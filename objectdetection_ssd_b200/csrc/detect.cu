// Detection post-processing: softmax + score threshold, per-class greedy NMS, global top-k.
// Reference: inference(), Losses.py:11-98 (decode Util.py:86-91, corner form Util.py:93-96, IoU Util.py:252-301).
//
// What the reference computes per image: for every foreground class a full greedy NMS over the candidates with
// prob >= min_score (descending prob), the kept lists concatenated class-major, and - if more than top_k boxes
// survive - the top_k of them by descending prob (Losses.py:77-81).  Whether a candidate is kept depends only on the
// HIGHER-scored candidates of its own class.  So the 20 per-class sweeps can be run as ONE sweep over the image's
// candidates in descending (prob, then lower class, then lower prior) order, suppression tested within a class only:
// every keep/suppress decision is the one the per-class sweep takes, kept boxes come out in exactly the order of the
// final global top-k (T7: equal prob -> earlier class-major position = lower class, then earlier rank = lower prior),
// and the sweep may stop as soon as top_k + 1 boxes are kept - the other ~20 x top_k kept boxes the per-class
// formulation produces can never reach the output.  If the list runs out with <= top_k boxes kept the output is
// the class-major concatenation (Losses.py:71-73), produced by a stable partition of the kept list by class.
//
// Two routes with identical outputs.  The SHORT-LIST route (large calls; detect_stream_kernel + detect_sweep_kernel,
// described at SAMPLE_STRIDE below) lists only the candidates above a sampled score floor and falls back, per image and
// inside the sweep kernel, to the full list when that was not enough.  The EXHAUSTIVE route (small calls, a
// max_candidates cap below P, or SSDHEAD_DETECT_SHORTLIST=0) lists every candidate:
//   detect_score_kernel  grid (row tiles, B), 256 rows per CTA: the tile's conf rows arrive in shared memory with one
//                        1-D TMA bulk copy (plain loads when unaligned), one thread per prior does the softmax and
//                        appends a 64-bit key (prob bits << 32 | ~(class << 24 | prior)) to the image's candidate list
//                        for every class with prob >= min_score (one atomic per warp), and counts the keys into a
//                        coarse log-probability histogram of the image (256 bins, 32 per octave).  HBM bound.
//                        Boxes are NOT decoded here: only the few hundred candidates the sweep touches need one.
//   detect_nms_kernel    one CTA per image: the coarse histogram cuts the list into SLICES of descending score
//                        (about 1.5 x top_k keys first, doubling); a slice is filtered into shared memory, sorted
//                        exactly by an adaptive counting sort on the full 64-bit key (2048 linear bins between the
//                        slice's min and max key, in-bin ranking, crowded bins re-binned), its boxes decoded, and
//                        swept in blocks of 64: each candidate against the kept boxes OF ITS CLASS, then a 64x64
//                        same-class suppression bit mask resolved by one warp with shuffles.  The IoU test needs
//                        no division unless the ratio is within 2^-20 of the threshold, where the reference's exact
//                        `inter/union >= thr` is evaluated (bit-exact keep lists).  The CTA writes the detections.
#include <algorithm>
#include "common.cuh"

namespace ssdhead {

#ifdef SSDHEAD_PHASE_TIMES      // developer build: SM clock at the phase boundaries of the first image's sweep CTA
__device__ long long g_phase[16];
#define PHASE(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_phase[i] = clock64(); } while (0)
// stream kernel, per CTA: [0] items, [1] consumer warp 0: clocks waiting for item data, [2] clocks working on rows,
// [3] producer: clocks waiting for a free stage, [4] clocks of its bookkeeping, [5] [6] global timer at start / end,
// [7] clocks of the sampling prologue
__device__ long long g_stream[2048][8];
__device__ __forceinline__ long long gtimer() { long long v; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(v)); return v; }
#define STREAM_STAT(stmt) do { stmt; } while (0)
#else
#define STREAM_STAT(stmt) do { } while (0)
#define PHASE(i) do { } while (0)
#endif

constexpr int SC_T = 256;          // score kernel: threads = rows per tile
#ifndef SSDHEAD_NMS_THREADS
#define SSDHEAD_NMS_THREADS 512
#endif
constexpr int NT = SSDHEAD_NMS_THREADS;   // nms kernel threads
constexpr int NPART = NT / 64;     // threads per candidate in a block of 64
constexpr int CBINS = 256;         // coarse log-probability rank bins of an image (0 = [1, ..), 32 per octave)
constexpr int FBINS = 2048;        // bins of the in-slice counting sort
constexpr int SL = 2048;           // slice keys sorted in shared memory; larger slices use the global scratch
constexpr int CROWD = 64;          // bins with more keys are re-binned instead of ranked quadratically
constexpr int MAXSEG = 512;        // crowded bins remembered per level
static_assert(SC_T == CBINS, "one thread per coarse bin in the score kernel");
static_assert(FBINS % NT == 0 && CBINS <= NT, "scan ownership");

struct DetectWs {
    unsigned long long* cand;      // [B][capI] candidate keys of an image: one chunk per score tile, each chunk ordered
                                   //           by coarse rank bin (highest probabilities first)
    unsigned long long* scr_a;     // [B][capI] slice buffers for slices that do not fit shared memory
    unsigned long long* scr_b;     // [B][capI]
    unsigned short* dir;           // [B][T][CBINS] per chunk: keys in the coarse rank bins BEFORE each bin (exclusive prefix sums; rewritten by every call)
    unsigned int* dir_base;        // [B][T][2] start of the chunk in the image's list, keys in the chunk
    unsigned int* cand_cnt;        // [B]       zero on entry, zero on exit
    unsigned int* overflow;        // [B]       zero on entry, zero on exit
    // short-list route (score floor from a sample of the rows)
    unsigned long long* floor;     // [B]       1 << 32 | bits of the image's score floor (>= min_score) once it is known; zero on entry, zero on exit
    unsigned int* flag_cnt;        // [1]       images whose short list did not decide the output (reset by the next call's sampling kernel)
    unsigned int* work;            // [2]       next score item, CTAs that left the stream kernel; zero on entry, zero on exit
};

static inline int detect_cap_image(int P, int C, int n) { return (C - 1) * (n > 0 ? std::min(n, P) : P); }
static inline int detect_tiles(int P) { return (P + SC_T - 1) / SC_T; }

static size_t detect_ws_layout(int B, int P, int C, int n, DetectWs* w, void* base)
{
    const size_t capI = (size_t)detect_cap_image(P, C, n);
    const size_t T = (size_t)detect_tiles(P) + SSDHEAD_MAX_LEVELS;   // per-level calls: at most one partial tile more per level
    size_t off = 0;
    char* b = (char*)base;
    auto take = [&](size_t bytes) { size_t o = off; off += round_up(bytes, 256); return b ? (void*)(b + o) : nullptr; };
    void* p0 = take((size_t)B * capI * 8);
    void* p1 = take((size_t)B * capI * 8);
    void* p2 = take((size_t)B * capI * 8);
    void* p3 = take((size_t)B * T * CBINS * 2);
    void* p4 = take((size_t)B * T * 8);
    void* p5 = take((size_t)B * 4);
    void* p6 = take((size_t)B * 4);
    void* p7 = take((size_t)B * 8);
    void* p9 = take(16);
    void* p10 = take(16);
    if (w) { w->floor = (unsigned long long*)p7; w->flag_cnt = (unsigned int*)p9; w->work = (unsigned int*)p10; }
    if (w) { w->cand = (unsigned long long*)p0; w->scr_a = (unsigned long long*)p1; w->scr_b = (unsigned long long*)p2;
             w->dir = (unsigned short*)p3; w->dir_base = (unsigned int*)p4;
             w->cand_cnt = (unsigned int*)p5; w->overflow = (unsigned int*)p6; }
    return off;
}

size_t detect_workspace_bytes(int B, int P, int C, int n)
{
    if (B <= 0 || P <= 0 || C < 2) return 0;
    return detect_ws_layout(B, P, C, n, nullptr, nullptr);
}

// key = score word << 32 | ~(class << 24 | prior): descending key order = descending prob, then lower class, then
// lower prior (T5, T7).  The score word is the probability's bits (score_word below).
__device__ __forceinline__ unsigned long long make_key(unsigned word, int cls, int prior) {
    return ((unsigned long long)word << 32) | (unsigned long long)(0xffffffffu - (((unsigned)cls << 24) | (unsigned)prior));
}
__device__ __forceinline__ int key_cls(unsigned long long key) { return (int)((0xffffffffu - (unsigned)(key & 0xffffffffull)) >> 24); }
__device__ __forceinline__ unsigned key_prior(unsigned long long key) { return (0xffffffffu - (unsigned)(key & 0xffffffffull)) & 0xffffffu; }
// coarse rank bin of a probability: 0 holds [1, ..), bin r the probabilities 2^(-r/32) steps below; the last bin
// holds everything smaller.  Monotone (non-increasing) in the probability.
__device__ __forceinline__ int coarse_rank(unsigned pbits) {
    const int d = (int)(0x3f800000u >> 18) - (int)(pbits >> 18);
    return min(CBINS - 1, max(0, d));
}
// The score word of a key (its upper 32 bits).  A softmax probability is >= +0, so its bits already order it.  The scores
// given to ssdhead_detect_from_scores can be anything: -0.0 must tie with +0.0 and a negative score rank below both (as in
// the reference's descending sort), so there the word is the order-preserving map of common.cuh (-0 -> +0, non-negative
// scores -> bits | 2^31, negative ones -> ~bits).  SCORE_TOP is what the word of 0x3f800000 (1.0) becomes.
template <bool FROM_SCORES> __device__ __forceinline__ unsigned score_word(float p) {
    return FROM_SCORES ? float_order_key(p) : __float_as_uint(p);
}
template <bool FROM_SCORES> __device__ __forceinline__ float word_score(unsigned w) {
    return __uint_as_float(!FROM_SCORES ? w : (w & 0x80000000u) ? (w ^ 0x80000000u) : ~w);
}
template <bool FROM_SCORES> constexpr unsigned SCORE_TOP = FROM_SCORES ? 0x80000000u : 0u;
// coarse rank bin of a score word; negative given scores fall into the last bin
template <bool FROM_SCORES> __device__ __forceinline__ int coarse_rank_w(unsigned w) {
    return !FROM_SCORES ? coarse_rank(w) : (w & 0x80000000u) ? coarse_rank(w ^ 0x80000000u) : CBINS - 1;
}

// Head outputs given per pyramid level (ssdhead_detect_levels; see ssdhead.h): level l holds cnt[l] priors per image,
// priors start[l] .. start[l+1]-1 of the global order; an image's score tiles tile0[l] .. tile0[l+1]-1 belong to level l.
constexpr int MAX_LEVELS = SSDHEAD_MAX_LEVELS;
struct DetLevels {
    int n;
    int cnt[MAX_LEVELS];
    int start[MAX_LEVELS + 1];
    int tile0[MAX_LEVELS + 1];
    int item0[MAX_LEVELS + 1];     // the same for the 480-row items of a sweep CTA that lists its image again
    const float* conf[MAX_LEVELS];
    const float* loc[MAX_LEVELS];
};

// ------------------------------------------------------------------------------------------------
// Where the conf rows of score tile `tile` of image b sit: first prior of the tile (global order), rows, source pointer.
template <int C, bool LEVELS>
__device__ __forceinline__ void
score_tile_rows(const float* __restrict__ conf, int P, int b, int tile, const DetLevels* __restrict__ dl,
                int& r0, int& nrows, const float*& src)
{
    r0 = tile * SC_T;
    nrows = min(SC_T, P - r0);
    src = conf + ((size_t)b * P + r0) * C;
    if (LEVELS) {
        int l = 0;
#pragma unroll
        for (int q = 1; q < MAX_LEVELS; ++q) if (q < dl->n && tile >= dl->tile0[q]) l = q;
        const int off = (tile - dl->tile0[l]) * SC_T;
        nrows = min(SC_T, dl->cnt[l] - off);
        r0 = dl->start[l] + off;
        src = dl->conf[l] + ((size_t)b * dl->cnt[l] + off) * C;
    }
}

// The same for the short-list route's items of ROWS rows (256: the score tiles; 480: a sweep CTA listing its image again).
template <int C, bool LEVELS, int ROWS>
__device__ __forceinline__ void
item_rows(const float* __restrict__ conf, int P, int b, int j, const DetLevels* __restrict__ dl, int& r0, int& nrows, const float*& src)
{
    r0 = j * ROWS;
    nrows = min(ROWS, P - r0);
    src = conf + ((size_t)b * P + r0) * C;
    if (LEVELS) {
        const int* first = ROWS == SC_T ? dl->tile0 : dl->item0;
        int l = 0;
#pragma unroll
        for (int q = 1; q < MAX_LEVELS; ++q) if (q < dl->n && j >= first[q]) l = q;
        const int off = (j - first[l]) * ROWS;
        nrows = min(ROWS, dl->cnt[l] - off);
        r0 = dl->start[l] + off;
        src = dl->conf[l] + ((size_t)b * dl->cnt[l] + off) * C;
    }
}
// first prior (global order) of item j, rows given at run time
template <bool LEVELS>
__device__ __forceinline__ int item_first_row(const DetLevels* __restrict__ dl, int rows, int j)
{
    if (!LEVELS) return j * rows;
    const int* first = rows == SC_T ? dl->tile0 : dl->item0;
    int l = 0;
#pragma unroll
    for (int q = 1; q < MAX_LEVELS; ++q) if (q < dl->n && j >= first[q]) l = q;
    return dl->start[l] + (j - first[l]) * rows;
}

// One score tile of image b in the EXHAUSTIVE route (every candidate >= min_score is listed).  s_bar is initialised by
// the caller (count 1); `parity` is the phase this call waits for; T = score tiles per image.
template <int C, bool FROM_SCORES, bool LEVELS>
__device__ __forceinline__ void
detect_score_body(const int b, const int tile, const int T, uint64_t* s_bar_p, const uint32_t parity,
                  const float* __restrict__ conf, int P, float min_score, int capI,
                  unsigned long long* __restrict__ cand, unsigned int* __restrict__ cand_cnt,
                  unsigned short* __restrict__ dir, unsigned int* __restrict__ dir_base,
                  unsigned int* __restrict__ overflow, const DetLevels* __restrict__ dl)
{
    constexpr int NF = C - 1;
    constexpr int NW = SC_T / 32;
    static_assert(NF <= 32, "class mask is one 32-bit word");
    __shared__ __align__(128) float s_conf[SC_T * C];
    __shared__ unsigned int s_ch[CBINS];            // keys per coarse rank bin, then their exclusive prefix sums
    __shared__ unsigned int s_fill[CBINS];
    __shared__ unsigned short s_stq[SC_T * NF];     // per warp: (lane << 5 | class) of its candidates, compact
    __shared__ unsigned int s_wtot[NW];
    __shared__ unsigned int s_wsum[NW];
    __shared__ unsigned int s_base;
    uint64_t& s_bar = *s_bar_p;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    int r0, nrows;
    const float* src;
    score_tile_rows<C, LEVELS>(conf, P, b, tile, dl, r0, nrows, src);
    const uint32_t bytes = (uint32_t)nrows * C * 4u;
    const bool bulk = ((reinterpret_cast<uintptr_t>(src) | (uintptr_t)bytes) & 15u) == 0;

    s_ch[t] = 0u;
    s_fill[t] = 0u;
    __syncthreads();
    if (bulk) {
        if (t == 0) { mbar_expect_tx(&s_bar, bytes); bulk_g2s(s_conf, src, bytes, &s_bar); }
        mbar_wait(&s_bar, parity);
    } else if (((reinterpret_cast<uintptr_t>(src) | (uintptr_t)bytes) & 7u) == 0) {
        // 8-byte aligned rows (e.g. an odd image of a level with an odd half-count of priors): float2 loads
        const float2* src2 = reinterpret_cast<const float2*>(src);
        float2* dst2 = reinterpret_cast<float2*>(s_conf);
        for (int i = t; i < (nrows * C) / 2; i += SC_T) dst2[i] = __ldg(src2 + i);
        __syncthreads();
    } else {
        for (int i = t; i < nrows * C; i += SC_T) s_conf[i] = __ldg(src + i);
        __syncthreads();
    }

    // thread per prior: class probabilities, written back over the row's logits; bit q of cmask <=> prob[q] >= min_score
    float* x = s_conf + t * C;
    unsigned cmask = 0u;
    if (t < nrows) {
        float p[NF];
        if (FROM_SCORES) {
#pragma unroll
            for (int q = 0; q < NF; ++q) p[q] = x[q];
        } else {
            // softmax: exp(x - max) * (1 / sum)  (Losses.py:25)
            float e[C];
#pragma unroll
            for (int q = 0; q < C; ++q) e[q] = x[q];
            float m = e[0];
#pragma unroll
            for (int q = 1; q < C; ++q) m = fmaxf(m, e[q]);
            float s = 0.0f;
#pragma unroll
            for (int q = 0; q < C; ++q) { e[q] = fast_exp_ftz(__fsub_rn(e[q], m)); s = __fadd_rn(s, e[q]); }   // rel. error ~2e-7
            const float inv = __fdiv_rn(1.0f, s);
#pragma unroll
            for (int q = 0; q < NF; ++q) { p[q] = __fmul_rn(e[q], inv); x[q] = p[q]; }
        }
#pragma unroll
        for (int q = 0; q < NF; ++q) cmask |= (p[q] >= min_score ? 1u : 0u) << q;                              // Losses.py:32
    }
    // Rows with a weak background logit pass in many classes at once (heavy tail), so per-thread emission would run
    // at the pace of the warp's busiest lane.  Each lane only lists its candidates as (lane, class) descriptors,
    // compacted across the warp; the warp then handles 32 candidates at a time.
    const unsigned ncand = (unsigned)__popc(cmask);
    unsigned incl = ncand;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += o;
    }
    const unsigned wtotal = __shfl_sync(FULL, incl, 31);
    if (lane == 0) s_wtot[warp] = wtotal;
    unsigned short* st_q = s_stq + warp * (32 * NF);
    {
        unsigned o = incl - ncand;
        unsigned mm = cmask;
        while (mm) {
            const int q = __ffs(mm) - 1;
            mm &= mm - 1u;
            st_q[o++] = (unsigned short)((lane << 5) | q);
        }
    }
    __syncthreads();
    // the CTA's keys form one chunk of the image's list: reserve it (the atomic's latency hides behind the histogram)
    unsigned total = 0u, chunk = 0u;
    if (t == 0) {
#pragma unroll
        for (int w = 0; w < NW; ++w) total += s_wtot[w];
        if (total) chunk = atomicAdd(&cand_cnt[b], total);
    }
    const float* wrow = s_conf + warp * (32 * C);
#pragma unroll 1                         // ~3 trips: an unrolled body only adds a preamble
    for (unsigned j = lane; j < wtotal; j += 32) {
        const unsigned lq = st_q[j];
        const float pj = wrow[(lq >> 5) * C + (lq & 31u)];
        atomicAdd(&s_ch[coarse_rank_w<FROM_SCORES>(score_word<FROM_SCORES>(pj))], 1u);
    }
    __syncthreads();
    // exclusive prefix sums over the 256 rank bins: the chunk is written ordered by bin, highest probabilities first,
    // and its per-bin counts go to the image's directory - the sweep kernel then reads only the keys of a score slice
    const unsigned h = s_ch[t];
    unsigned hin = h;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(FULL, hin, d);
        if (lane >= d) hin += o;
    }
    if (lane == 31) s_wsum[warp] = hin;
    if (t == 0) {
        const bool fits = chunk + total <= (unsigned)capI;
        s_base = fits ? chunk : 0xffffffffu;
        dir_base[((size_t)b * T + tile) * 2] = fits ? chunk : 0u;
        dir_base[((size_t)b * T + tile) * 2 + 1] = fits ? total : 0u;
        if (!fits) atomicOr(&overflow[b], 1u);                   // the whole chunk is dropped; out_cnt[b] becomes -1
    }
    __syncthreads();
    unsigned wb = 0u;
#pragma unroll
    for (int w = 0; w < NW; ++w) if (w < warp) wb += s_wsum[w];
    s_ch[t] = wb + hin - h;
    const unsigned base = s_base;
    // the directory row of this chunk: keys before each rank bin (a chunk holds at most 20 x 256 keys: 16 bits).  Prefix sums
    // instead of counts: the sweep kernel gets a slice's position in the chunk with two loads, and the image's coarse
    // prefix sums are the column sums of the rows - no scan on its side
    dir[((size_t)b * T + tile) * CBINS + t] = base != 0xffffffffu ? (unsigned short)(wb + hin - h) : (unsigned short)0;
    __syncthreads();
    if (base != 0xffffffffu) {
        unsigned long long* seg = cand + (size_t)b * capI + base;
#pragma unroll 1
        for (unsigned j = lane; j < wtotal; j += 32) {
            const unsigned lq = st_q[j];
            const float pj = wrow[(lq >> 5) * C + (lq & 31u)];
            const unsigned w = score_word<FROM_SCORES>(pj);
            const int rb = coarse_rank_w<FROM_SCORES>(w);
            seg[s_ch[rb] + atomicAdd(&s_fill[rb], 1u)] = make_key(w, (int)(lq & 31u), r0 + warp * 32 + (int)(lq >> 5));
        }
    }
}

template <int C, bool FROM_SCORES, bool LEVELS>
__device__ __forceinline__ void
detect_score_grid(const float* __restrict__ conf, int P, float min_score, int capI,
                  unsigned long long* __restrict__ cand, unsigned int* __restrict__ cand_cnt,
                  unsigned short* __restrict__ dir, unsigned int* __restrict__ dir_base,
                  unsigned int* __restrict__ overflow, const DetLevels* __restrict__ dl, unsigned int* __restrict__ flag_cnt)
{
    __shared__ __align__(8) uint64_t s_bar;
    if (threadIdx.x == 0) { mbar_init(&s_bar, 1); mbar_fence_init(); }
    pdl_trigger();                       // the sweep kernel may become resident; it waits for this grid to finish
    pdl_wait();                          // the previous call's sweep may still be reading the lists we overwrite
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *flag_cnt = 0u;   // ssdhead_detect_fallbacks: none on this route
    detect_score_body<C, FROM_SCORES, LEVELS>(blockIdx.y, blockIdx.x, gridDim.x, &s_bar, 0u, conf, P, min_score, capI,
                                              cand, cand_cnt, dir, dir_base, overflow, dl);
}

template <int C, bool FROM_SCORES>
__global__ void __launch_bounds__(SC_T)
detect_score_kernel(const float* __restrict__ conf, int P, float min_score, int capI,
                    unsigned long long* __restrict__ cand, unsigned int* __restrict__ cand_cnt,
                    unsigned short* __restrict__ dir, unsigned int* __restrict__ dir_base,
                    unsigned int* __restrict__ overflow, unsigned int* __restrict__ flag_cnt)
{
    detect_score_grid<C, FROM_SCORES, false>(conf, P, min_score, capI, cand, cand_cnt, dir, dir_base, overflow, nullptr, flag_cnt);
}

template <int C>
__global__ void __launch_bounds__(SC_T)
detect_score_levels_kernel(int P, float min_score, int capI,
                           unsigned long long* __restrict__ cand, unsigned int* __restrict__ cand_cnt,
                           unsigned short* __restrict__ dir, unsigned int* __restrict__ dir_base,
                           unsigned int* __restrict__ overflow, unsigned int* __restrict__ flag_cnt, const __grid_constant__ DetLevels dl)
{
    detect_score_grid<C, false, true>(nullptr, P, min_score, capI, cand, cand_cnt, dir, dir_base, overflow, &dl, flag_cnt);
}

// ------------------------------------------------------------------------------------------------
// Short-list route.  At min_score = 0.01 an image has tens of thousands of candidates, and the sweep stops after a few
// hundred of them: listing all of them is what made the score kernel issue-bound.
//   detect_stream_kernel  persistent, warp-specialised, 8 consumer warps + a producer lane.  Prologue: the consumer warps of
//                         CTA c look at every SAMPLE_STRIDE-th row of the images c, c + grid, ... and pick each image's score
//                         FLOOR (an edge of the coarse rank bins, >= min_score) above which about SAMPLE_STRIDE x
//                         SAMPLE_TARGET candidates are expected - while the producer's first copies are in flight.  Main
//                         loop: the producer draws 256-row ITEMS from a global counter and moves them into a two-stage ring
//                         with bulk copies (full/empty mbarriers); a consumer warp works on its own 32 rows without any
//                         CTA-wide barrier - thread-per-row softmax (the exhaustive route's arithmetic), class mask against
//                         the image's floor, one shared-memory atomic per lane that holds a candidate for its place in the
//                         item's key segment, keys straight to global memory.  No dense passes, no directory.
//   detect_sweep_kernel   one CTA per image: the sweep of the exhaustive route on the short list.  A candidate's fate
//                         depends only on higher-scored candidates, so if the sweep keeps top_k + 1 boxes inside the short
//                         list - or the floor never rose above min_score - the output is the exhaustive route's, bit for
//                         bit.  Otherwise the CTA lists the image AGAIN itself with the floor at min_score (the same
//                         producer/consumer loop over its own items, 15 consumer warps) and sweeps the full list: the
//                         output never depends on the floor, and nothing runs behind the kernel.
// An item's keys go to a fixed segment of the image's list - 20 keys per row, at 20 x (first row) - so nothing can overflow.
constexpr int SAMPLE_STRIDE = 35;     // coprime with the 4 / 6 priors per cell: every aspect ratio is sampled; SSD300: one row per thread
constexpr int SAMPLE_TARGET = 46;     // sampled candidates above the floor: ~1600 listed keys per image
#ifndef SSDHEAD_STREAM_CTAS
#define SSDHEAD_STREAM_CTAS 4         // resident CTAs per SM the stream kernel is built for
#endif
#ifndef SSDHEAD_STREAM_STAGES
#define SSDHEAD_STREAM_STAGES 2       // stages of its item ring (measured at batch 256: 2 x 4 CTAs 66.8 us, 3 x 3 67.9, 4 x 2 76.7, 2 x 5 82.2)
#endif
constexpr int SST = SSDHEAD_STREAM_STAGES;
constexpr int SCW = 8;                // consumer warps of the stream kernel: items of 256 rows (the score tiles of the exhaustive route)
constexpr int RCW = NT / 32 - 1;      // consumer warps when a sweep CTA lists its image again: items of 480 rows
static_assert(SCW * 32 == SC_T, "the stream kernel's items are the exhaustive route's score tiles");

// row -> foreground probabilities p[0..NF), exactly the exhaustive route's arithmetic; returns the row's best one
template <int C, bool FROM_SCORES>
__device__ __forceinline__ float row_probs(const float* __restrict__ x, float (&e)[C], float& m, float& inv)
{
    constexpr int NF = C - 1;
#pragma unroll
    for (int q = 0; q < C; ++q) e[q] = x[q];
    inv = 1.0f;
    m = 0.0f;
    if (!FROM_SCORES) {
        m = e[0];
#pragma unroll
        for (int q = 1; q < C; ++q) m = fmaxf(m, e[q]);
        float s = 0.0f;
#pragma unroll
        for (int q = 0; q < C; ++q) { e[q] = fast_exp_ftz(__fsub_rn(e[q], m)); s = __fadd_rn(s, e[q]); }
        inv = __fdiv_rn(1.0f, s);
    }
    float best = e[0];
#pragma unroll
    for (int q = 1; q < NF; ++q) best = fmaxf(best, e[q]);
    return FROM_SCORES ? best : __fmul_rn(best, inv);          // rounding is monotone: max(e) * inv == max(e * inv)
}
// probability of class q of a row recomputed from the row (same operations => same bits as row_probs)
template <bool FROM_SCORES>
__device__ __forceinline__ float prob_again(const float* __restrict__ x, int q, float m, float inv)
{
    return FROM_SCORES ? x[q] : __fmul_rn(fast_exp_ftz(__fsub_rn(x[q], m)), inv);
}

// barrier of the first 256 threads of a CTA (the stream kernel's consumer warps), or of a whole 256-thread CTA
template <bool NAMED> __device__ __forceinline__ void sync256() {
    if (NAMED) asm volatile("bar.sync 1, 256;" ::: "memory"); else __syncthreads();
}

// Score floor of image b from every SAMPLE_STRIDE-th row, by 256 threads (t = 0 .. 255); valid in thread 0.
template <int C, bool FROM_SCORES, bool LEVELS, bool NAMED>
__device__ __forceinline__ float
sample_floor(const int b, const float* __restrict__ conf, int P, float min_score, const DetLevels* __restrict__ dl)
{
    constexpr int NF = C - 1;
    __shared__ unsigned int s_h[CBINS];
    __shared__ unsigned int s_ws[SC_T / 32];
    __shared__ int s_r;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    s_h[t] = 0u;
    if (t == 0) s_r = CBINS;
    sync256<NAMED>();
    for (int r = t * SAMPLE_STRIDE; r < P; r += SC_T * SAMPLE_STRIDE) {
        const float* x = conf + ((size_t)b * P + r) * C;
        if (LEVELS) {
            int l = 0;
#pragma unroll
            for (int q = 1; q < MAX_LEVELS; ++q) if (q < dl->n && r >= dl->start[q]) l = q;
            x = dl->conf[l] + ((size_t)b * dl->cnt[l] + (r - dl->start[l])) * C;
        }
        float e[C], m, inv;
        const float best = row_probs<C, FROM_SCORES>(x, e, m, inv);
        if (best >= min_score) {
#pragma unroll
            for (int q = 0; q < NF; ++q) {
                const float p = FROM_SCORES ? e[q] : __fmul_rn(e[q], inv);
                if (p >= min_score) atomicAdd(&s_h[coarse_rank_w<FROM_SCORES>(score_word<FROM_SCORES>(p))], 1u);
            }
        }
    }
    sync256<NAMED>();
    // the first rank bin (from the top) at which the sampled candidates reach the target: its lower edge is the floor
    const unsigned h = s_h[t];
    unsigned incl = h;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_ws[warp] = incl;
    sync256<NAMED>();
#pragma unroll
    for (int w = 0; w < SC_T / 32; ++w) if (w < warp) incl += s_ws[w];
    if (incl >= (unsigned)SAMPLE_TARGET && incl - h < (unsigned)SAMPLE_TARGET) s_r = t;
    sync256<NAMED>();
    float F = min_score;                 // too few candidates in the sample: list everything (the exhaustive semantics)
    const int r = s_r;
    if (r < CBINS - 1) {
        const float edge = __uint_as_float(((0x3f800000u >> 18) - (unsigned)r) << 18);
        if (edge > min_score) F = edge;
    }
    sync256<NAMED>();                    // s_r / s_h are reused by the next image
    return F;
}

// ------------------------------------------------------------------------------------------------
// `a` suppresses `b`  <=>  inter / union >= thr, evaluated exactly as the reference does (Util.py:262-265,
// 294-301, Losses.py:51) but without the division when the answer is not within 2^-20 of the threshold.
__device__ __forceinline__ bool iou_ge(const float4 a, const float aa, const float4 b, const float ab,
                                       const float thr, const float thr_lo, const float thr_hi)
{
    const float dx = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.0f);
    const float dy = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.0f);
    const float inter = __fmul_rn(dx, dy);
    const float uni = __fsub_rn(__fadd_rn(aa, ab), inter);
    if (uni > 0.0f && thr > 0.0f) {
        if (inter < __fmul_rn(uni, thr_lo)) return false;
        if (inter > __fmul_rn(uni, thr_hi)) return true;
    }
    return __fdiv_rn(inter, uni) >= thr;
}

// The same predicate with a cheap filter in front.  In real arithmetic inter/union >= thr <=> inter >= T (aa + ab) with
// T = thr / (1 + thr); the fp32 evaluation of either side is off by less than 2^-21 relative (no cancellation: inter <=
// union), so outside a 2^-18 band around T (aa + ab) the answer is certain and inside it the reference's own expression
// decides.  t_lo/t_hi = T (1 -+ 2^-18), or -inf/+inf when thr is not inside (0, 1) (always the exact path); NaNs fail
// both comparisons and reach the exact path too.
struct IouThr { float thr, thr_lo, thr_hi, t_lo, t_hi; };
__device__ __forceinline__ IouThr make_iou_thr(float thr) {
    IouThr r;
    r.thr = thr;
    r.thr_lo = __fmul_rn(thr, 1.0f - 9.5367431640625e-07f);   // thr * (1 - 2^-20)
    r.thr_hi = __fmul_rn(thr, 1.0f + 9.5367431640625e-07f);
    const bool ok = thr > 0.0f && thr < 1.0f;
    const float T = __fdiv_rn(thr, __fadd_rn(1.0f, thr));
    r.t_lo = ok ? __fmul_rn(T, 1.0f - 3.814697265625e-06f) : __int_as_float(0xff800000);
    r.t_hi = ok ? __fmul_rn(T, 1.0f + 3.814697265625e-06f) : __int_as_float(0x7f800000);
    return r;
}
__device__ __forceinline__ bool iou_ge_fast(const float4 a, const float aa, const float4 b, const float ab, const IouThr& q)
{
    const float dx = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.0f);
    const float dy = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.0f);
    const float inter = __fmul_rn(dx, dy);
    const float sum = __fadd_rn(aa, ab);
    bool res = inter > __fmul_rn(sum, q.t_hi);
    if (!res && !(inter < __fmul_rn(sum, q.t_lo)))            // rare: inside the band (or NaN)
        res = __fdiv_rn(inter, __fsub_rn(sum, inter)) >= q.thr;
    return res;
}

struct NmsBlock {                  // one block of up to 64 sorted candidates
    float4 cbox[64];
    unsigned long long ckey[64];
    unsigned long long mask[64];
    float carea[64];
    int ccls[64];
    unsigned int supp[2];
    unsigned long long alive;
};

struct SortShared {
    unsigned long long kmin, kmax;
    int2 seg[2][MAXSEG];
    int nseg[2];
    unsigned int wsum[NT / 32];
};

struct Kept {                      // kept boxes in sweep order + per-class index lists
    float4* box;
    unsigned long long* key;
    float* area;
    unsigned short* idx;           // [NF][cap]
    int* cnt;                      // [NF]
    int cap;
};

// exclusive prefix sum of one value per thread over the CTA (two barriers; s_wsum is reusable afterwards)
__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned int* s_wsum, unsigned& total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    unsigned wbase = 0u;
    total = 0u;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) { const unsigned x = s_wsum[w]; if (w < warp) wbase += x; total += x; }
    __syncthreads();
    return wbase + incl - v;
}

// exclusive prefix sums of s_cnt[0..FBINS) into s_S[0..FBINS], counters reset to zero (thread t owns FBINS/NT bins)
__device__ __forceinline__ void scan_bins(unsigned int* s_cnt, unsigned int* s_S, unsigned int* s_wsum)
{
    constexpr int per = FBINS / NT;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    unsigned v[per], mine = 0u;
#pragma unroll
    for (int q = 0; q < per; ++q) { v[q] = s_cnt[t * per + q]; mine += v[q]; s_cnt[t * per + q] = 0u; }
    unsigned incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned o = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    unsigned wbase = 0u;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) if (w < warp) wbase += s_wsum[w];
    unsigned run = wbase + incl - mine;
#pragma unroll
    for (int q = 0; q < per; ++q) { s_S[t * per + q] = run; run += v[q]; }
    if (t == NT - 1) s_S[FBINS] = run;
    __syncthreads();
}

// Linear map of a key range onto FBINS bins, bin 0 = largest keys (keys outside the range are clamped: still monotone).
struct BinMap {
    unsigned long long kmax;
    int shift;
    __device__ __forceinline__ BinMap(unsigned long long kmin_, unsigned long long kmax_) : kmax(kmax_) {
        const unsigned long long range = kmax_ - kmin_;
        shift = range ? max(0, 64 - __clzll((long long)range) - 11) : 0;                      // (range >> shift) < FBINS
    }
    __device__ __forceinline__ int operator()(unsigned long long k) const {
        return k >= kmax ? 0 : (int)min((kmax - k) >> shift, (unsigned long long)(FBINS - 1));
    }
};

// Sorts X[0,n) in descending key order (keys are distinct); Y is scratch of the same size.  X/Y may be shared or
// global memory.  Adaptive counting sort: FBINS linear bins between the segment's min and max key, keys scattered
// bin-grouped into Y, ranked inside their bin back into X; a bin with more than CROWD keys becomes a segment of the
// next level (its own min/max spread its keys again), so ties in the probability cost one more level, not n^2.
// `pre`: the caller already knows bounds [kmin0, kmax0] of the keys and has counted them into s_cnt with
// BinMap(kmin0, kmax0) (the slice filter does this on the fly), so the first level starts at the prefix sums.
// place(pos, key) is called once per key when its final position is known.
template <typename Place>
__device__ void sort_desc(unsigned long long* X, unsigned long long* Y, int n,
                          unsigned int* s_S, unsigned int* s_cnt, SortShared& ss,
                          bool pre, unsigned long long kmin0, unsigned long long kmax0, Place place)
{
    const int t = threadIdx.x;
    if (t == 0) { ss.seg[0][0] = make_int2(0, n); ss.nseg[0] = 1; ss.nseg[1] = 0; }
    __syncthreads();
    for (int level = 0; level < 8; ++level) {
        const int cur = level & 1;
        const int ns = min(ss.nseg[cur], MAXSEG);
        if (ns == 0) break;
        for (int si = 0; si < ns; ++si) {
            const int a = ss.seg[cur][si].x, m = ss.seg[cur][si].y - a;
            unsigned long long kmin = kmin0, kmax = kmax0;
            const bool counted = pre && level == 0;
            if (!counted) {
                if (t == 0) { ss.kmin = ~0ull; ss.kmax = 0ull; }
                for (int i = t; i < FBINS; i += NT) s_cnt[i] = 0u;
                __syncthreads();
                unsigned long long lo = ~0ull, hi = 0ull;
                for (int i = t; i < m; i += NT) { const unsigned long long k = X[a + i]; lo = min(lo, k); hi = max(hi, k); }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    lo = min(lo, __shfl_xor_sync(FULL, lo, d));
                    hi = max(hi, __shfl_xor_sync(FULL, hi, d));
                }
                if ((t & 31) == 0 && lo <= hi) { atomicMin(&ss.kmin, lo); atomicMax(&ss.kmax, hi); }
                __syncthreads();
                kmin = ss.kmin; kmax = ss.kmax;
                if (kmax == kmin) {                              // one key (or equal keys): nothing to order
                    for (int i = t; i < m; i += NT) place(a + i, X[a + i]);
                    __syncthreads();
                    continue;
                }
            }
            const BinMap bin_of(kmin, kmax);
            if (!counted) {
                for (int i = t; i < m; i += NT) atomicAdd(&s_cnt[bin_of(X[a + i])], 1u);
                __syncthreads();
            }
            scan_bins(s_cnt, s_S, ss.wsum);
            for (int i = t; i < m; i += NT) {
                const unsigned long long k = X[a + i];
                const int f = bin_of(k);
                Y[a + s_S[f] + atomicAdd(&s_cnt[f], 1u)] = k;
            }
            __syncthreads();
            // crowded bins become segments of the next level (marked in s_cnt); without room they are ranked in place
            for (int f = t; f < FBINS; f += NT) {
                const int lo = (int)s_S[f], c = (int)s_S[f + 1] - lo;
                unsigned mark = 0u;
                if (c > CROWD) {
                    const int at = atomicAdd(&ss.nseg[cur ^ 1], 1);
                    if (at < MAXSEG) { ss.seg[cur ^ 1][at] = make_int2(a + lo, a + lo + c); mark = 1u; }
                }
                s_cnt[f] = mark;
            }
            __syncthreads();
            for (int i = t; i < m; i += NT) {
                const unsigned long long k = Y[a + i];
                const int f = bin_of(k);
                if (s_cnt[f]) { X[a + i] = k; continue; }     // re-binned at the next level
                const int lo = (int)s_S[f], hi = (int)s_S[f + 1];
                int r = 0;
                for (int j = lo; j < hi; ++j) r += (Y[a + j] > k) ? 1 : 0;
                X[a + lo + r] = k;
                place(a + lo + r, k);
            }
            __syncthreads();
        }
        if (t == 0) ss.nseg[cur] = 0;
        __syncthreads();
    }
}

// One block of up to 64 sorted candidates (Losses.py:44-55): against the kept boxes of their class, then among
// themselves.  Returns the new kept count; kept boxes are appended in sweep order.
template <typename BoxOf>
__device__ __forceinline__ int nms_block(NmsBlock& s, const unsigned long long* keys, int base, int m, BoxOf box_of,
                                         const Kept kp, int K, float iou_thr, float thr_lo, float thr_hi)
{
    const int t = threadIdx.x;
    if (t < 64) {
        float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
        unsigned long long key = 0ull;
        int cls = -1;
        if (t < m) {
            key = keys[base + t];
            box = box_of(base + t, key);
            cls = key_cls(key);
        }
        s.cbox[t] = box;
        s.carea[t] = box_area(box);
        s.ckey[t] = key;
        s.ccls[t] = cls;
        s.mask[t] = 0ull;
    }
    if (t < 2) s.supp[t] = 0u;
    __syncthreads();
    unsigned long long bits = 0ull;
    {
        const int cnd = t & 63, part = t >> 6;
        if (cnd < m) {
            const float4 cb = s.cbox[cnd];
            const float ca = s.carea[cnd];
            const int c = s.ccls[cnd];
            // (a) against the boxes of class c kept so far, the list split NPART ways
            const int kc = kp.cnt[c];
            const unsigned short* il = kp.idx + (size_t)c * kp.cap;
            for (int k = part; k < kc; k += NPART) {
                const int id = il[k];
                if (iou_ge(kp.box[id], kp.area[id], cb, ca, iou_thr, thr_lo, thr_hi)) {
                    atomicOr(&s.supp[cnd >> 5], 1u << (cnd & 31));
                    break;
                }
            }
            // (b) inside the block: row cnd tests the later same-class columns of its part
            constexpr int CW = 64 / NPART;
#pragma unroll
            for (int q = 0; q < CW; ++q) {
                const int col = part * CW + q;
                if (col > cnd && col < m && s.ccls[col] == c &&
                    iou_ge(cb, ca, s.cbox[col], s.carea[col], iou_thr, thr_lo, thr_hi))
                    bits |= 1ull << col;
            }
            if (bits) atomicOr(&s.mask[cnd], bits);
        }
    }
    const unsigned long long valid = m == 64 ? ~0ull : ((1ull << m) - 1ull);
    unsigned long long alive;
    if (__syncthreads_or(bits != 0ull)) {
        if (t < 32) {
            // (c) serial resolve: a box that is still alive suppresses the later boxes it overlaps.  The 64 mask rows
            // are pulled into registers first (two per lane); the dependent chain is ALU + shuffles.
            const unsigned long long m_lo = s.mask[t], m_hi = s.mask[t + 32];
            unsigned long long al = valid & ~((unsigned long long)s.supp[0] | ((unsigned long long)s.supp[1] << 32));
            unsigned nz_lo = __ballot_sync(FULL, m_lo != 0ull), nz_hi = __ballot_sync(FULL, m_hi != 0ull);
            while (nz_lo) {                                   // only rows that overlap somebody, in sweep order
                const int i = __ffs(nz_lo) - 1;
                nz_lo &= nz_lo - 1u;
                const unsigned long long mk = __shfl_sync(FULL, m_lo, i);
                if ((al >> i) & 1ull) al &= ~mk;
            }
            while (nz_hi) {
                const int i = __ffs(nz_hi) - 1;
                nz_hi &= nz_hi - 1u;
                const unsigned long long mk = __shfl_sync(FULL, m_hi, i);
                if ((al >> (i + 32)) & 1ull) al &= ~mk;
            }
            if (t == 0) s.alive = al;
        }
        __syncthreads();
        alive = s.alive;
    } else {
        // no overlapping same-class pair inside the block (the common case): nothing to resolve
        alive = valid & ~((unsigned long long)s.supp[0] | ((unsigned long long)s.supp[1] << 32));
    }
    if (t < m && ((alive >> t) & 1ull)) {
        const int pos = K + __popcll(alive & ((1ull << t) - 1ull));
        if (pos < kp.cap) {
            kp.box[pos] = s.cbox[t]; kp.area[pos] = s.carea[t]; kp.key[pos] = s.ckey[t];
            const int c = s.ccls[t];
            kp.idx[(size_t)c * kp.cap + atomicAdd(&kp.cnt[c], 1)] = (unsigned short)pos;
        }
    }
    __syncthreads();
    return K + __popcll(alive);
}

__device__ __forceinline__ int compact_kept(const unsigned long long* X, const float4* s_box, const unsigned char* s_keep, int cnt,
                                            unsigned int* s_wsum, const Kept kp, int K);

// Sweep of one sorted slice held in shared memory (keys X[0,cnt), boxes s_box[0,cnt), cnt <= SL).  Suppression only
// acts inside a class, so the greedy NMS of a class (Losses.py:44-55) runs inside ONE warp, all classes side by side and
// without a block-wide barrier: (1) a stable partition of the slice positions by class (match_any inside chunks of 32 +
// per-class prefix sums over the chunks), (2) per class, 32 candidates at a time in lanes: tested against the boxes of
// the class kept earlier (previous slices, previous rounds), then all pairs of the round through register shuffles
// (lane i's box is broadcast, one ballot = row i of the overlap matrix), resolved in score order - only boxes that
// are still alive and overlap somebody are walked, (3) the kept flags are compacted in slice (= global score) order
// onto the kept list.  `scratch` is at least 16 KB of shared memory that is free during the sweep.  Returns the new
// kept count.
__device__ __noinline__ int sweep_slice_by_class(const unsigned long long* X, const float4* s_box, int cnt, int NF, unsigned char* scratch,
                                    unsigned int* s_wsum, const Kept kp, int K, const IouThr q)
{
    constexpr int NW = NT / 32;
    constexpr int NFP = 32;                                    // row stride of the per-chunk class counts
    unsigned short* s_order = reinterpret_cast<unsigned short*>(scratch);              // [SL] positions, grouped by class
    unsigned char* s_keep = scratch + SL * 2;                                          // [SL]
    unsigned short* s_cc = reinterpret_cast<unsigned short*>(scratch + SL * 3);        // [SL/32][NFP]
    int* s_cstart = reinterpret_cast<int*>(scratch + SL * 3 + (SL / 32) * NFP * 2);    // [NFP + 1]
    static_assert(SL * 3 + (SL / 32) * NFP * 2 + (NFP + 1) * 4 <= SL * 8, "sweep scratch layout");
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int nchunk = (cnt + 31) >> 5;
    PHASE(8);

    for (int i = t; i < nchunk * NFP; i += NT) s_cc[i] = 0;
    for (int i = t; i < cnt; i += NT) s_keep[i] = 0;
    __syncthreads();
    for (int ch = warp; ch < nchunk; ch += NW) {
        const int i = ch * 32 + lane;
        const int c = i < cnt ? key_cls(X[i]) : NFP - 1;       // padding lanes form their own group
        const unsigned peers = __match_any_sync(FULL, c);
        if (lane == __ffs(peers) - 1) s_cc[ch * NFP + c] = (unsigned short)__popc(peers);
    }
    __syncthreads();
    if (t < NFP) {
        int run = 0;
        for (int ch = 0; ch < nchunk; ++ch) { const int v = s_cc[ch * NFP + t]; s_cc[ch * NFP + t] = (unsigned short)run; run += v; }
        // class starts: exclusive prefix over the classes (one warp)
        int incl = t < NF ? run : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += o;
        }
        s_cstart[t + 1] = incl;
        if (t == 0) s_cstart[0] = 0;
    }
    __syncthreads();
    for (int ch = warp; ch < nchunk; ch += NW) {
        const int i = ch * 32 + lane;
        const int c = i < cnt ? key_cls(X[i]) : NFP - 1;
        const unsigned peers = __match_any_sync(FULL, c);
        if (i < cnt) s_order[s_cstart[c] + s_cc[ch * NFP + c] + __popc(peers & lt)] = (unsigned short)i;
    }
    __syncthreads();
    PHASE(9);

    for (int c = warp; c < NF; c += NW) {
        const int n_c = s_cstart[c + 1] - s_cstart[c];
        unsigned short* L = s_order + s_cstart[c];
        const int kc0 = kp.cnt[c];
        const unsigned short* il = kp.idx + (size_t)c * kp.cap;
        int m_c = 0;                                           // kept in this slice so far: their positions are L[0, m_c)
        for (int r0 = 0; r0 < n_c; r0 += 32) {
            const int j = r0 + lane;
            const bool v = j < n_c;
            const int pos = v ? (int)L[j] : 0;
            const float4 bx = v ? s_box[pos] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float ar = box_area(bx);
            bool sup = false;
            for (int k = 0; k < kc0; ++k) {
                const int id = il[k];
                sup = sup || iou_ge_fast(kp.box[id], kp.area[id], bx, ar, q);
            }
            for (int k = 0; k < m_c; ++k) {
                const float4 b2 = s_box[L[k]];
                sup = sup || iou_ge_fast(b2, box_area(b2), bx, ar, q);
            }
            // all pairs of the round: the box of lane i is broadcast with shuffles, every later lane tests itself against
            // it, and one ballot is the row of the 32 x 32 overlap matrix that lane i keeps (the later lanes its box
            // overlaps) - no shared-memory traffic and no dependent loads inside the loop; then only rows that overlap
            // somebody are walked in score order
            const int nr = min(32, n_c - r0);
            unsigned row = 0u;
#pragma unroll 4
            for (int i = 0; i < nr - 1; ++i) {
                const float4 bi = make_float4(__shfl_sync(FULL, bx.x, i), __shfl_sync(FULL, bx.y, i),
                                              __shfl_sync(FULL, bx.z, i), __shfl_sync(FULL, bx.w, i));
                const float ai = __shfl_sync(FULL, ar, i);
                const bool ov = lane > i && v && iou_ge_fast(bi, ai, bx, ar, q);
                const unsigned m = __ballot_sync(FULL, ov);
                if (lane == i) row = m;
            }
            unsigned alive = __ballot_sync(FULL, v && !sup);
            unsigned todo = __ballot_sync(FULL, row != 0u);
            while (todo) {
                const int i = __ffs(todo) - 1;
                todo &= todo - 1u;
                const unsigned r = __shfl_sync(FULL, row, i);
                if ((alive >> i) & 1u) alive &= ~r;
            }
            __syncwarp();
            if ((alive >> lane) & 1u) { L[m_c + __popc(alive & lt)] = (unsigned short)pos; s_keep[pos] = 1; }
            m_c += __popc(alive);
            __syncwarp();
        }
    }
    __syncthreads();
    PHASE(10);

    const int Kn = compact_kept(X, s_box, s_keep, cnt, s_wsum, kp, K);
    PHASE(11);
    return Kn;
}

// kept flags of a swept slice -> the kept list (boxes, areas, keys in slice = global score order, per-class index lists).
// Returns the new kept count (entries past the list's capacity are counted, not stored: the caller stops at top_k + 1).
__device__ __forceinline__ int compact_kept(const unsigned long long* X, const float4* s_box, const unsigned char* s_keep, int cnt,
                                            unsigned int* s_wsum, const Kept kp, int K)
{
    const int t = threadIdx.x;
    const int per = (cnt + NT - 1) / NT;
    const int lo = min(cnt, t * per), hi = min(cnt, lo + per);
    unsigned local = 0u;
    for (int i = lo; i < hi; ++i) local += s_keep[i];
    unsigned total;
    int g = K + (int)block_excl_scan(local, s_wsum, total);
    for (int i = lo; i < hi; ++i) {
        if (!s_keep[i]) continue;
        if (g < kp.cap) {
            const unsigned long long key = X[i];
            const float4 bx = s_box[i];
            kp.box[g] = bx; kp.area[g] = box_area(bx); kp.key[g] = key;
            const int c = key_cls(key);
            kp.idx[(size_t)c * kp.cap + atomicAdd(&kp.cnt[c], 1)] = (unsigned short)g;
        }
        ++g;
    }
    __syncthreads();
    return K + (int)total;
}

static size_t nms_smem_bytes(int NF, int top_k, int T)
{
    const size_t kcap = (size_t)top_k + 65;
    size_t off = 0;
    off += kcap * 16;                  // kept boxes
    off += (size_t)SL * 16;            // decoded boxes of the sorted slice
    off += (size_t)SL * 8 * 2;         // slice buffers
    off += kcap * 8;                   // kept keys
    off += (size_t)(FBINS + 1 + 3) * 4;// prefix sums (padded to 16 bytes)
    off += (size_t)FBINS * 4;          // counters
    off += kcap * 4;                   // kept areas
    off += 32 * 4;                     // per-class kept counts
    off += (size_t)T * 5 * 4;          // per-chunk base, key count; start, length, offset of the current slice
    off += (size_t)NF * kcap * 2;      // per-class index lists
    return (off + 15) & ~(size_t)15;
}

// FLOOR: the short-list route (the image's keys sit in one fixed segment per score item + a coarse histogram) instead
// of the exhaustive route's chunks and directory; fl.* are used by it alone.
struct FloorArgs {
    unsigned long long* floor;     // [B] valid flag << 32 | floor bits: one word, so a reader needs no second load and no fence
    unsigned int* icnt;            // [B][items per image] keys listed by each item
    unsigned int* work;            // [2]
    unsigned int* flag_cnt;        // [1] images listed twice (statistic)
    float min_score;
};
// how an image's rows were cut into items when its short list was written
struct ItemLayout {
    int rows;                      // rows per item
    int n;                         // items per image
    bool raised;                   // the list holds only candidates above a floor > min_score
};

// Returns false when the image was not decided (FLOOR only; nothing has been written then).
template <bool FROM_SCORES, bool LEVELS, bool FLOOR>
__device__ __forceinline__ bool
detect_nms_body(const int b, const FloorArgs fl, const ItemLayout il,
                  const DetLevels* __restrict__ dl, const float4* __restrict__ loc_or_boxes, const float4* __restrict__ pri_cxcywh,
                  unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a,
                  unsigned long long* __restrict__ scr_b, const unsigned short* __restrict__ dir,
                  const unsigned int* __restrict__ dir_base, unsigned int* __restrict__ cand_cnt,
                  unsigned int* __restrict__ overflow,
                  const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                  float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                  int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int kcap = top_k + 65;
    unsigned char* sp = smem_raw;
    float4* s_kbox = reinterpret_cast<float4*>(sp);                          sp += (size_t)kcap * 16;
    float4* s_box = reinterpret_cast<float4*>(sp);                           sp += (size_t)SL * 16;
    unsigned long long* s_buf_a = reinterpret_cast<unsigned long long*>(sp); sp += (size_t)SL * 8;
    unsigned long long* s_buf_b = reinterpret_cast<unsigned long long*>(sp); sp += (size_t)SL * 8;
    unsigned long long* s_kkey = reinterpret_cast<unsigned long long*>(sp);  sp += (size_t)kcap * 8;
    unsigned int* s_S = reinterpret_cast<unsigned int*>(sp);                 sp += (size_t)(FBINS + 4) * 4;
    unsigned int* s_cnt = reinterpret_cast<unsigned int*>(sp);               sp += (size_t)FBINS * 4;
    float* s_karea = reinterpret_cast<float*>(sp);                           sp += (size_t)kcap * 4;
    int* s_kcnt = reinterpret_cast<int*>(sp);                                sp += 32 * 4;
    unsigned int* s_cbase = reinterpret_cast<unsigned int*>(sp);             sp += (size_t)T * 4;
    unsigned int* s_cstart = reinterpret_cast<unsigned int*>(sp);            sp += (size_t)T * 4;
    unsigned int* s_clen = reinterpret_cast<unsigned int*>(sp);              sp += (size_t)T * 4;
    unsigned int* s_coff = reinterpret_cast<unsigned int*>(sp);              sp += (size_t)T * 4;
    unsigned int* s_ctot = reinterpret_cast<unsigned int*>(sp);              sp += (size_t)T * 4;
    unsigned short* s_kidx = reinterpret_cast<unsigned short*>(sp);
    // the image's directory (T x 256 counts) is kept in the box buffer, which is idle while a slice is gathered
    bool dir_cached = (size_t)T * CBINS * 2 <= (size_t)SL * 16;       // until the first slice's boxes overwrite it
    unsigned short* s_dir = reinterpret_cast<unsigned short*>(s_box);
    __shared__ NmsBlock s;
    __shared__ SortShared ss;
    __shared__ unsigned int s_CS[CBINS + 1];
    __shared__ unsigned int s_col[CBINS];
    __shared__ int s_rc1;
    __shared__ unsigned int s_gcnt;

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t < CBINS) s_col[t] = 0u;
    if (t < 32) s_kcnt[t] = 0;
    if (t == 0) s_CS[CBINS] = 0u;
    __syncthreads();
    PHASE(0);
    const unsigned long long* seg = cand + (size_t)b * capI;
    const unsigned short* gdir = dir + (size_t)b * T * CBINS;
    const size_t bP = (size_t)b * P;
    float4* ob = out_boxes + (size_t)b * top_k;
    float* op = out_prob + (size_t)b * top_k;
    int* oc = out_cls + (size_t)b * top_k;
    int* oi = out_prior ? out_prior + (size_t)b * top_k : nullptr;

    int fl_n = 0;                                            // keys in the image's short list
    bool fl_parked = false;                                  // ... and they sit in s_buf_b (until the first sort uses it as scratch)
    if (FLOOR) {
        // the items' key counts: where every item's segment starts in the list and in the flat numbering of the image's keys
        const unsigned n_j = t < il.n ? (unsigned)ld_cg_s32(reinterpret_cast<const int*>(fl.icnt) + (size_t)b * T + t) : 0u;
        unsigned ntot;
        const unsigned off_j = block_excl_scan(n_j, ss.wsum, ntot);
        if (t < il.n) { s_coff[t] = off_j; s_cbase[t] = (unsigned)item_first_row<LEVELS>(dl, il.rows, t) * (unsigned)NF; }
        fl_n = (int)ntot;
        fl_parked = fl_n <= SL;
        __syncthreads();
        // one pass over the keys: the image's coarse histogram (s_col was zeroed above) -> prefix sums
        for (int f0 = 0; f0 < fl_n; f0 += 4 * NT) {
            unsigned long long kk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int f = f0 + u * NT + t;
                kk[u] = 0ull;
                if (f < fl_n) {
                    int lo = 0, hi = il.n - 1;
                    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s_coff[mid] <= (unsigned)f) lo = mid; else hi = mid - 1; }
                    kk[u] = ld_cg_u64(seg + s_cbase[lo] + ((unsigned)f - s_coff[lo]));
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (f0 + u * NT + t < fl_n) {
                    atomicAdd(&s_col[coarse_rank_w<FROM_SCORES>((unsigned)(kk[u] >> 32))], 1u);
                    if (fl_parked) s_buf_b[f0 + u * NT + t] = kk[u];     // the first slice is picked out of shared memory
                }
        }
        __syncthreads();
        unsigned total;
        const unsigned ex = block_excl_scan(t < CBINS ? s_col[t] : 0u, ss.wsum, total);
        if (t < CBINS) s_CS[t] = ex;
        if (t == 0) s_CS[CBINS] = total;
        __syncthreads();
    } else
    // column sums of the directory rows (per-chunk prefix sums) = the image's coarse prefix sums: CS[r] = number of keys in
    // rank bins < r (bin 0 = highest probabilities); CS[CBINS] = all keys of the image
    {
        constexpr int G = NT / CBINS;                        // thread groups sharing the chunks of a column
        const int col = t % CBINS, g = t / CBINS;
        unsigned sum = 0u;
#pragma unroll 4
        for (int c = g; c < T; c += G) {
            const unsigned short v = ld_cg_u16(gdir + (size_t)c * CBINS + col);
            if (dir_cached) s_dir[c * CBINS + col] = v;
            sum += v;
        }
        if (g < G && sum) atomicAdd(&s_col[col], sum);
        for (int c = t; c < T; c += NT) {
            const unsigned long long w2 = ld_cg_u64(reinterpret_cast<const unsigned long long*>(dir_base) + (size_t)b * T + c);
            const unsigned tot_c = (unsigned)(w2 >> 32);
            s_cbase[c] = (unsigned)w2;
            s_ctot[c] = tot_c;
            if (tot_c) atomicAdd(&s_CS[CBINS], tot_c);
        }
        __syncthreads();
        if (t < CBINS) s_CS[t] = s_col[t];
        __syncthreads();
    }

    PHASE(1);
    const float thr_lo = __fmul_rn(iou_thr, 1.0f - 9.5367431640625e-07f);   // thr * (1 - 2^-20)
    const float thr_hi = __fmul_rn(iou_thr, 1.0f + 9.5367431640625e-07f);
    const Kept kp = {s_kbox, s_kkey, s_karea, s_kidx, s_kcnt, kcap};
    auto load_box = [&](unsigned long long key) {
        const unsigned prior = key_prior(key);
        float4 v;
        if (LEVELS) {
            int l = 0;
#pragma unroll
            for (int q = 1; q < MAX_LEVELS; ++q) if (q < dl->n && (int)prior >= dl->start[q]) l = q;
            v = reinterpret_cast<const float4*>(dl->loc[l])[(size_t)b * dl->cnt[l] + (prior - (unsigned)dl->start[l])];
        } else {
            v = loc_or_boxes[bP + prior];
        }
        if (!FROM_SCORES) v = decode_box(v, pri_cxcywh[prior]);             // Losses.py:23
        return cxcywh_to_xyxy(v);                                           // Losses.py:41,71
    };

    int K = 0;
    int rc0 = 0;                                    // rank bins < rc0 are done
    int target = max(top_k + top_k / 2 + 1, 96);
    while (K <= top_k && rc0 < CBINS && s_CS[CBINS] - s_CS[rc0] > 0u) {
        // slice = rank bins [rc0, rc1): the fewest bins holding at least `target` keys, or all that is left
        if (t == 0) s_rc1 = CBINS;
        __syncthreads();
        if (t < CBINS) {
            const int rc = t + 1;
            if (rc > rc0 && s_CS[rc] - s_CS[rc0] >= (unsigned)target && s_CS[rc - 1] - s_CS[rc0] < (unsigned)target) s_rc1 = rc;
        }
        __syncthreads();
        const int rc1 = s_rc1;
        const int cnt = (int)(s_CS[rc1] - s_CS[rc0]);
        const bool in_smem = cnt <= SL;
        unsigned long long* X = in_smem ? s_buf_a : scr_a + (size_t)b * capI;
        unsigned long long* Y = in_smem ? s_buf_b : scr_b + (size_t)b * capI;
        // key bounds of the slice from its coarse bins (the open-ended last bin has none: the sort measures them)
        const bool pre = rc1 < CBINS;
        const unsigned top18 = 0x3f800000u >> 18;
        constexpr unsigned long long top = SCORE_TOP<FROM_SCORES>;
        const unsigned long long kmax0 = rc0 == 0 ? ((0x3f800000ull + top) << 32 | 0xffffffffull)
                                                  : (((unsigned long long)((top18 - rc0 + 1) << 18) + top) << 32) - 1ull;
        const unsigned long long kmin0 = pre ? ((unsigned long long)((top18 - (rc1 - 1)) << 18) + top) << 32 : 0ull;
        const BinMap bin0(kmin0, kmax0);
        if (pre) for (int i = t; i < FBINS; i += NT) s_cnt[i] = 0u;
        if (FLOOR) {
            // the short list is unordered: one pass over its keys picks the slice's (the sort below orders them)
            if (t == 0) s_gcnt = 0u;
            __syncthreads();
            if (fl_parked) {
                for (int f = t; f < fl_n; f += NT) {
                    const unsigned long long k = s_buf_b[f];
                    const int r = coarse_rank_w<FROM_SCORES>((unsigned)(k >> 32));
                    if (r >= rc0 && r < rc1) {
                        X[atomicAdd(&s_gcnt, 1u)] = k;
                        if (pre) atomicAdd(&s_cnt[bin0(k)], 1u);
                    }
                }
                fl_parked = false;
            } else
            // flat key f sits in the item whose range of the flat numbering holds f (binary search over the items' offsets);
            // four keys per thread are requested before any is looked at
            for (int f0 = 0; f0 < fl_n; f0 += 4 * NT) {
                unsigned long long kk[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int f = f0 + u * NT + t;
                    kk[u] = 0ull;
                    if (f < fl_n) {
                        int lo = 0, hi = il.n - 1;
                        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s_coff[mid] <= (unsigned)f) lo = mid; else hi = mid - 1; }
                        kk[u] = ld_cg_u64(seg + s_cbase[lo] + ((unsigned)f - s_coff[lo]));
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (f0 + u * NT + t >= fl_n) continue;
                    const int r = coarse_rank_w<FROM_SCORES>((unsigned)(kk[u] >> 32));
                    if (r >= rc0 && r < rc1) {
                        X[atomicAdd(&s_gcnt, 1u)] = kk[u];
                        if (pre) atomicAdd(&s_cnt[bin0(kk[u])], 1u);
                    }
                }
            }
            __syncthreads();
        } else {
        // where the slice sits in every chunk: chunks are ordered by rank bin, so it is one contiguous piece per chunk -
        // from the chunk's prefix sums, two loads
        for (int c = t; c < T; c += NT) {
            const unsigned p0 = dir_cached ? s_dir[c * CBINS + rc0] : ld_cg_u16(gdir + (size_t)c * CBINS + rc0);
            const unsigned p1 = rc1 >= CBINS ? s_ctot[c]
                                             : (dir_cached ? (unsigned)s_dir[c * CBINS + rc1] : (unsigned)ld_cg_u16(gdir + (size_t)c * CBINS + rc1));
            s_cstart[c] = p0;
            s_clen[c] = p1 - p0;
        }
        __syncthreads();
        for (int c0 = 0; c0 < T; c0 += NT) {                    // T <= NT: one round
            unsigned total;
            const int c = c0 + t;
            const unsigned ex = block_excl_scan(c < T ? s_clen[c] : 0u, ss.wsum, total);
            if (c < T) s_coff[c] = ex;
        }
        __syncthreads();
        for (int c = warp; c < T; c += NT / 32) {
            const unsigned long long* src = seg + s_cbase[c] + s_cstart[c];
            const int len = (int)s_clen[c], off = (int)s_coff[c];
            for (int i = lane; i < len; i += 32) {
                const unsigned long long k = ld_cg_u64(src + i);
                X[off + i] = k;
                if (pre) atomicAdd(&s_cnt[bin0(k)], 1u);
            }
        }
        __syncthreads();
        }
        PHASE(2);
        if (in_smem) {
            // boxes are decoded as soon as a key's final position is known
            sort_desc(X, Y, cnt, s_S, s_cnt, ss, pre, kmin0, kmax0, [&](int pos, unsigned long long key) { s_box[pos] = load_box(key); });
            PHASE(3);
            PHASE(4);
            K = sweep_slice_by_class(X, s_box, cnt, NF, reinterpret_cast<unsigned char*>(Y), ss.wsum, kp, K, make_iou_thr(iou_thr));
        } else {
            sort_desc(X, Y, cnt, s_S, s_cnt, ss, pre, kmin0, kmax0, [](int, unsigned long long) {});
            for (int base = 0; base < cnt && K <= top_k; base += 64)
                K = nms_block(s, X, base, min(64, cnt - base), [&](int, unsigned long long key) { return load_box(key); },
                              kp, K, iou_thr, thr_lo, thr_hi);
        }
        rc0 = rc1;
        dir_cached = false;
        if (target < (1 << 28)) target *= 2;
        PHASE(5);
    }

    if (FLOOR && K <= top_k && il.raised) return false;     // the short list ran out before top_k + 1 boxes were kept and
                                                             // candidates below the floor exist: not decided here
    float sx = 1.0f, sy = 1.0f;
    if (img_wh) { sx = img_wh[2 * b]; sy = img_wh[2 * b + 1]; }
    auto emit = [&](int slot, int i) {
        const unsigned long long key = s_kkey[i];
        const float4 v = s_kbox[i];
        ob[slot] = img_wh ? make_float4(__fmul_rn(v.x, sx), __fmul_rn(v.y, sy), __fmul_rn(v.z, sx), __fmul_rn(v.w, sy)) : v;   // Losses.py:89
        op[slot] = word_score<FROM_SCORES>((unsigned)(key >> 32));
        oc[slot] = key_cls(key);
        if (oi) oi[slot] = (int)key_prior(key);
    };
    int nout;
    if (K > top_k) {
        // more than top_k survive: the top_k by descending prob, ties -> earlier class-major position (Losses.py:77-81, T7)
        // - the first top_k boxes of the sweep
        nout = top_k;
        for (int i = t; i < top_k; i += NT) emit(i, i);
    } else {
        // class-major, each class in descending score order (Losses.py:71-73): stable partition of the sweep order
        nout = K;
        for (int i = t; i < K; i += NT) {
            const int c = key_cls(s_kkey[i]);
            int pos = 0;
            for (int q = 0; q < c; ++q) pos += s_kcnt[q];
            for (int j = 0; j < i; ++j) pos += (key_cls(s_kkey[j]) == c) ? 1 : 0;
            emit(pos, i);
        }
    }
    if (t == 0) {
        if (FLOOR) {
            out_cnt[b] = nout;
        } else {
            out_cnt[b] = ld_cg_s32(reinterpret_cast<const int*>(overflow) + b) ? -1 : nout;     // -1: the candidate list exceeded the caller's cap
            overflow[b] = 0u;
            cand_cnt[b] = 0u;
        }
    }
    PHASE(6);
    return true;
}

// The same sweep, as two kernels' entry: the exhaustive route's (lists and directory from detect_score_kernel) ...
template <bool FROM_SCORES>
__global__ void __launch_bounds__(NT, 2)
detect_nms_kernel(const float4* __restrict__ loc_or_boxes, const float4* __restrict__ pri_cxcywh,
                  unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a,
                  unsigned long long* __restrict__ scr_b, const unsigned short* __restrict__ dir,
                  const unsigned int* __restrict__ dir_base, unsigned int* __restrict__ cand_cnt,
                  unsigned int* __restrict__ overflow,
                  const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                  float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                  int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    pdl_wait();                                              // the score kernel's lists and directory are complete
    detect_nms_body<FROM_SCORES, false, false>(blockIdx.x, FloorArgs{}, ItemLayout{}, nullptr, loc_or_boxes, pri_cxcywh, cand, scr_a, scr_b, dir, dir_base,
                                               cand_cnt, overflow, img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt);
}

__global__ void __launch_bounds__(NT, 2)
detect_nms_levels_kernel(const __grid_constant__ DetLevels dl, const float4* __restrict__ pri_cxcywh,
                         unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a,
                         unsigned long long* __restrict__ scr_b, const unsigned short* __restrict__ dir,
                         const unsigned int* __restrict__ dir_base, unsigned int* __restrict__ cand_cnt,
                         unsigned int* __restrict__ overflow,
                         const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                         float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                         int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    pdl_wait();
    detect_nms_body<false, true, false>(blockIdx.x, FloorArgs{}, ItemLayout{}, &dl, nullptr, pri_cxcywh, cand, scr_a, scr_b, dir, dir_base,
                                        cand_cnt, overflow, img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt);
}

// ... and the short-list route's.  Scoring loop shared by detect_stream_kernel (items of all images from a global counter,
// NCW = 8 consumer warps) and by a sweep CTA that lists its image again (its own items, NCW = 15): warp NCW's lane 0 is
// the producer, warps 0 .. NCW-1 consume.  `ring`: 2 x NCW x 32 rows of shared memory.  Items w in [w_begin, w_end) drawn
// from *counter (global) or counted privately (counter == nullptr); item w = image w / ipi, item w % ipi of that image.
// SAMPLE (stream kernel only): before their first item the consumer warps compute the floors of the images
// blockIdx.x, blockIdx.x + gridDim.x, ... and publish them (floor[b], then ready[b] with release) - while the producer's
// first copies are already in flight; a producer that needs the floor of an image waits for its flag.  Every CTA of the
// grid is resident - the grid is sized with the occupancy query and launched cooperatively, so this holds even when
// kernels of other streams occupy part of the GPU - and no CTA waits before its own images are published, so the flags
// always arrive.
struct ItemDesc {                  // what the producer tells the consumers about the item in a stage
    int item;                      // -1: no more items
    int b, r0, nrows, bulk;
    float F;
    const float* src;
};

// one consumer warp's 32 rows of an item: class mask against the floor, the warp's place in the item's segment (one
// shared-memory atomic), keys to global memory.  `x`: the lane's row (shared or global memory - two instantiations, so
// the compiler knows the address space)
template <int C, bool FROM_SCORES, typename Ptr>
__device__ __forceinline__ void
score_rows(Ptr x, const bool valid, const float F, const int prior, unsigned int* s_icnt_st, unsigned long long* __restrict__ seg0)
{
    constexpr int NF = C - 1;
    unsigned cmask = 0u;
    float m = 0.0f, inv = 1.0f;
    if (valid) {
        float e[C];
        row_probs<C, FROM_SCORES>(x, e, m, inv);
#pragma unroll
        for (int q = 0; q < NF; ++q) cmask |= ((FROM_SCORES ? e[q] : __fmul_rn(e[q], inv)) >= F ? 1u : 0u) << q;
    }
    if (cmask) {                                             // about one lane in five: its keys' place in the item's segment
        unsigned long long* seg = seg0 + atomicAdd(s_icnt_st, (unsigned)__popc(cmask));
        do {
            const int q = __ffs(cmask) - 1;
            cmask &= cmask - 1u;
            *seg++ = make_key(score_word<FROM_SCORES>(prob_again<FROM_SCORES>(x, q, m, inv)), q, prior);
        } while (cmask);
    }
}

template <int C, bool FROM_SCORES, bool LEVELS, int NCW, int NST, bool SAMPLE>
__device__ __forceinline__ void
score_items(unsigned char* ring, unsigned int* counter, const int w_begin, const int w_end, const int ipi, const int B,
            unsigned long long* __restrict__ floor, const float f_const,
            const float* __restrict__ conf, const int P, const DetLevels* __restrict__ dl,
            unsigned long long* __restrict__ cand, const int capI, unsigned int* __restrict__ icnt, const int icnt_stride)
{
    constexpr int NF = C - 1;
    constexpr int ROWS = NCW * 32;
    constexpr uint32_t STAGE_BYTES = ROWS * C * 4;
    __shared__ __align__(8) uint64_t s_full[NST];
    __shared__ __align__(8) uint64_t s_empty[NST];
    __shared__ ItemDesc s_desc[NST];
    __shared__ unsigned int s_icnt[NST];                     // keys the stage's item has listed so far
    __shared__ int s_it[NST];                                // item whose key count is still to be published, per stage
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) {
#pragma unroll
        for (int q = 0; q < NST; ++q) { mbar_init(&s_full[q], 1); mbar_init(&s_empty[q], NCW); s_icnt[q] = 0u; s_it[q] = -1; }
        mbar_fence_init();
    }
    __syncthreads();
    int st = 0;
    uint32_t ph = 0u;
    if (warp == NCW) {
        if (lane == 0) {
            // Nothing the producer needs per item may cost it a round trip to L2 - it serves the whole CTA: the index of
            // the item after the next (w2) and the floor word of the next item (fw1) are requested one item ahead.
            if (SAMPLE) pdl_wait();                          // (no-op for the ordinary launch the stream kernel gets by default)
            unsigned w1 = counter ? atomicAdd(counter, 1u) : (unsigned)w_begin;
            unsigned w2 = counter ? atomicAdd(counter, 1u) : w1 + 1u;
            unsigned long long fw1 = 0ull;
            if (SAMPLE && (int)w1 < w_end) fw1 = ld_relaxed_gpu_u64(floor + (int)w1 / ipi);
#ifdef SSDHEAD_PHASE_TIMES
            long long pw = 0, pb = 0, pc0, pc1;
            if (SAMPLE && blockIdx.x < 2048) g_stream[blockIdx.x][5] = gtimer();
#endif
            for (;;) {
                STREAM_STAT(pc0 = clock64());
                mbar_wait(&s_empty[st], ph ^ 1u);            // the stage is free: the item that was in it is complete
                STREAM_STAT(pc1 = clock64(); pw += pc1 - pc0);
                const int fin = s_it[st];
                if (fin >= 0) icnt[(size_t)(fin / ipi) * icnt_stride + fin % ipi] = s_icnt[st];
                s_it[st] = -1;
                s_icnt[st] = 0u;
                const int d = (int)w1 < w_end ? (int)w1 : -1;
                s_desc[st].item = d;
                if (d < 0) { mbar_arrive(&s_full[st]); break; }
                const int b = d / ipi;
                int r0, nrows; const float* src;
                item_rows<C, LEVELS, ROWS>(conf, P, b, d - b * ipi, dl, r0, nrows, src);
                const uint32_t bytes = (uint32_t)nrows * C * 4u;
                const bool bulk = ((reinterpret_cast<uintptr_t>(src) | (uintptr_t)bytes) & 15u) == 0;
                // the copy first (its bytes are counted on the barrier whenever they land; the phase cannot complete before
                // this thread's own arrival below), then everything else the consumers need to know
                if (bulk) bulk_g2s(ring + (size_t)st * STAGE_BYTES, src, bytes, &s_full[st]);
                s_it[st] = d;
                float F = f_const;
                if (SAMPLE) {
                    int spins = 0;
                    while ((fw1 >> 32) == 0ull) {            // the image's floor is still being sampled (first items of a call only)
                        if (++spins > (1 << 22)) __trap();   // seconds: fail loudly, do not hang
                        fw1 = ld_relaxed_gpu_u64(floor + b);
                    }
                    F = __uint_as_float((unsigned)fw1);
                }
                s_desc[st].b = b; s_desc[st].r0 = r0; s_desc[st].nrows = nrows; s_desc[st].bulk = bulk ? 1 : 0;
                s_desc[st].F = F; s_desc[st].src = src;
                if (bulk) mbar_expect_tx(&s_full[st], bytes); else mbar_arrive(&s_full[st]);   // not 16-byte aligned: the consumers read global memory
                w1 = w2;
                if (SAMPLE && (int)w1 < w_end) fw1 = ld_relaxed_gpu_u64(floor + (int)w1 / ipi);
                w2 = counter ? atomicAdd(counter, 1u) : w2 + 1u;
                if (++st == NST) { st = 0; ph ^= 1u; }
                STREAM_STAT(pb += clock64() - pc1);
            }
#ifdef SSDHEAD_PHASE_TIMES
            if (SAMPLE && blockIdx.x < 2048) { g_stream[blockIdx.x][3] = pw; g_stream[blockIdx.x][4] = pb; }
#endif
        }
        __syncwarp();
    } else if (warp < NCW) {
        if (SAMPLE) {
            pdl_wait();                                      // (the stream kernel is the first kernel of a call)
#ifdef SSDHEAD_PHASE_TIMES
            const long long sc0 = clock64();
#endif
            for (int b = blockIdx.x; b < B; b += gridDim.x) {
                const float F = sample_floor<C, FROM_SCORES, LEVELS, true>(b, conf, P, f_const, dl);
                if (t == 0) st_relaxed_gpu_u64(floor + b, (1ull << 32) | (unsigned long long)__float_as_uint(F));   // one word: flag and value
            }
#ifdef SSDHEAD_PHASE_TIMES
            if (t == 0 && blockIdx.x < 2048) g_stream[blockIdx.x][7] = clock64() - sc0;
#endif
        }
#ifdef SSDHEAD_PHASE_TIMES
        long long cw = 0, cr = 0, cn = 0, cc0, cc1;
#endif
        for (;;) {
            STREAM_STAT(cc0 = clock64());
            mbar_wait(&s_full[st], ph);
            STREAM_STAT(cc1 = clock64(); cw += cc1 - cc0);
            const int d = s_desc[st].item;
            if (d < 0) break;
            const int b = s_desc[st].b, r0 = s_desc[st].r0;
            const int row = warp * 32 + lane;
            const bool valid = row < s_desc[st].nrows;
            unsigned long long* seg0 = cand + (size_t)b * capI + (size_t)r0 * NF;
            if (s_desc[st].bulk) {
                extern __shared__ __align__(16) unsigned char smem_ring[];      // == ring: the address space is known here
                score_rows<C, FROM_SCORES>(reinterpret_cast<const float*>(smem_ring + (size_t)st * STAGE_BYTES) + row * C, valid,
                                           s_desc[st].F, r0 + row, &s_icnt[st], seg0);
            } else {
                score_rows<C, FROM_SCORES>(s_desc[st].src + (size_t)row * C, valid, s_desc[st].F, r0 + row, &s_icnt[st], seg0);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&s_empty[st]);        // release: the warp's keys and its count are ordered before the producer's read
            if (++st == NST) { st = 0; ph ^= 1u; }
            STREAM_STAT(cr += clock64() - cc1; ++cn);
        }
#ifdef SSDHEAD_PHASE_TIMES
        if (SAMPLE && t == 0 && blockIdx.x < 2048) { long long* g = g_stream[blockIdx.x]; g[0] = cn; g[1] = cw; g[2] = cr; g[6] = gtimer(); }
#endif
    }
    __syncthreads();                                         // every consumer warp has left: all items are complete
    if (t == NCW * 32) {
#pragma unroll
        for (int q = 0; q < NST; ++q)
            if (s_it[q] >= 0) icnt[(size_t)(s_it[q] / ipi) * icnt_stride + s_it[q] % ipi] = s_icnt[q];
    }
    __syncthreads();
}

template <int C, bool FROM_SCORES, bool LEVELS>
__device__ __forceinline__ void
detect_stream_body(const FloorArgs fl, const float* __restrict__ conf, const int B, const int P, const int ipi,
                   const DetLevels* __restrict__ dl, unsigned long long* __restrict__ cand, const int capI, const int icnt_stride)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_trigger();                       // the sweep kernel may become resident; it waits for this grid to finish
    // An ordinary launch: everything in front of this call is complete, so the producer requests conf at once while the
    // consumer warps sample the floors.
    if (blockIdx.x == 0 && threadIdx.x == 0) fl.flag_cnt[0] = 0u;
    score_items<C, FROM_SCORES, LEVELS, SCW, SST, true>(smem_raw, fl.work, 0, B * ipi, ipi, B, fl.floor, fl.min_score,
                                                   conf, P, dl, cand, capI, fl.icnt, icnt_stride);
    // the last CTA to leave resets the work counters (every other CTA has drawn its last index by then)
    if (threadIdx.x == 0) {
        const unsigned e = atomicAdd(&fl.work[1], 1u);
        if (e == gridDim.x - 1) { fl.work[0] = 0u; fl.work[1] = 0u; }
    }
}

template <int C, bool FROM_SCORES>
__global__ void __launch_bounds__((SCW + 1) * 32, SSDHEAD_STREAM_CTAS)
detect_stream_kernel(const FloorArgs fl, const float* __restrict__ conf, const int B, const int P, const int ipi,
                     unsigned long long* __restrict__ cand, const int capI, const int icnt_stride)
{
    detect_stream_body<C, FROM_SCORES, false>(fl, conf, B, P, ipi, nullptr, cand, capI, icnt_stride);
}
template <int C>
__global__ void __launch_bounds__((SCW + 1) * 32, SSDHEAD_STREAM_CTAS)
detect_stream_levels_kernel(const FloorArgs fl, const int B, const int P, const int ipi, const __grid_constant__ DetLevels dl,
                            unsigned long long* __restrict__ cand, const int capI, const int icnt_stride)
{
    detect_stream_body<C, false, true>(fl, nullptr, B, P, ipi, &dl, cand, capI, icnt_stride);
}

template <int C, bool FROM_SCORES, bool LEVELS>
__device__ __forceinline__ void
detect_sweep_body(const FloorArgs fl, const float* __restrict__ conf, const int ipi_a, const int ipi_b,
                  const DetLevels* __restrict__ dl, const float4* __restrict__ loc_or_boxes, const float4* __restrict__ pri_cxcywh,
                  unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a, unsigned long long* __restrict__ scr_b,
                  const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                  float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                  int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x;
    pdl_trigger();
    pdl_wait();                                              // the stream kernel's short lists are complete
    const ItemLayout la = {SC_T, ipi_a, __uint_as_float((unsigned)ld_cg_u64(fl.floor + b)) > fl.min_score};
    __syncthreads();
    if (threadIdx.x == 0) fl.floor[b] = 0ull;
    if (detect_nms_body<FROM_SCORES, LEVELS, true>(b, fl, la, dl, loc_or_boxes, pri_cxcywh, cand, scr_a, scr_b, nullptr, nullptr, nullptr, nullptr,
                                                   img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt))
        return;
    // Not decided: the short list ran out with at most top_k boxes kept and candidates below the floor exist.  List the
    // image again with the floor at min_score - every candidate, as the exhaustive route does - and sweep that list.
    if (threadIdx.x == 0) atomicAdd(fl.flag_cnt, 1u);
    fence_proxy_async_smem();                                // the sweep wrote the ring's bytes with ordinary stores
    __syncthreads();
    score_items<C, FROM_SCORES, LEVELS, RCW, 2, false>(smem_raw, nullptr, b * ipi_b, (b + 1) * ipi_b, ipi_b, 0, nullptr, fl.min_score,
                                                    conf, P, dl, cand, capI, fl.icnt, T);
    const ItemLayout lb = {RCW * 32, ipi_b, false};
    detect_nms_body<FROM_SCORES, LEVELS, true>(b, fl, lb, dl, loc_or_boxes, pri_cxcywh, cand, scr_a, scr_b, nullptr, nullptr, nullptr, nullptr,
                                               img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt);
}

template <int C, bool FROM_SCORES>
__global__ void __launch_bounds__(NT, 2)
detect_sweep_kernel(const FloorArgs fl, const float* __restrict__ conf, const int ipi_a, const int ipi_b,
                    const float4* __restrict__ loc_or_boxes, const float4* __restrict__ pri_cxcywh,
                    unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a, unsigned long long* __restrict__ scr_b,
                    const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                    float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                    int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    detect_sweep_body<C, FROM_SCORES, false>(fl, conf, ipi_a, ipi_b, nullptr, loc_or_boxes, pri_cxcywh, cand, scr_a, scr_b,
                                             img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt);
}
template <int C>
__global__ void __launch_bounds__(NT, 2)
detect_sweep_levels_kernel(const FloorArgs fl, const int ipi_a, const int ipi_b, const __grid_constant__ DetLevels dl,
                           const float4* __restrict__ pri_cxcywh,
                           unsigned long long* __restrict__ cand, unsigned long long* __restrict__ scr_a, unsigned long long* __restrict__ scr_b,
                           const float* __restrict__ img_wh, int P, int NF, int T, int capI, int top_k, float iou_thr,
                           float4* __restrict__ out_boxes, float* __restrict__ out_prob, int* __restrict__ out_cls,
                           int* __restrict__ out_prior, int* __restrict__ out_cnt)
{
    detect_sweep_body<C, false, true>(fl, nullptr, ipi_a, ipi_b, &dl, nullptr, pri_cxcywh, cand, scr_a, scr_b,
                                      img_wh, P, NF, T, capI, top_k, iou_thr, out_boxes, out_prob, out_cls, out_prior, out_cnt);
}

// Which route serves a call.  SSDHEAD_DETECT_SHORTLIST=0 forces the exhaustive route, =1 the short-list route (the two give
// identical outputs; read per call so that tests can compare them in one process).  Unset: the short-list route from
// ~900 k rows per call (batch 104 of SSD300) - measured on B200, batch 256 / 128 / 64 / 32 / 8 / 1: short list 65.9 /
// 49.8 / 43.1 / 38.7 / 34.1 / 26.7 us, exhaustive 85.0 / 52.9 / 36.8 / 29.3 / 22.5 / 21.4 us (small batches pay the
// sampling prologue and the sweep's extra pass over the keys without having the rows to amortise them).
static bool shortlist_enabled(int B, int P)
{
    const char* e = getenv("SSDHEAD_DETECT_SHORTLIST");
    if (e) return atoi(e) != 0;
    return (long long)B * P >= 900000;
}


template <bool FROM_SCORES>
static int run_detect(const float* loc, const float* conf, const float* pri_cxcywh, int B, int P, int C,
                      float min_score, float iou_thr, int top_k, const float* img_wh,
                      float* out_boxes, float* out_prob, int32_t* out_cls, int32_t* out_prior, int32_t* out_cnt,
                      void* ws, size_t ws_bytes, int n_cap, cudaStream_t st, const DetLevels* dl = nullptr)
{
    if (B < 0 || P <= 0 || top_k <= 0 || n_cap < 0) return SSDHEAD_E_BADARG;
    if ((!dl && (!loc || !conf)) || (!FROM_SCORES && !pri_cxcywh) || !out_boxes || !out_prob || !out_cls || !out_cnt || !ws) return SSDHEAD_E_BADARG;
    if (C != 21) return SSDHEAD_E_UNSUPPORTED;
    if (B == 0) return 0;
    if (B > 65535 || P >= (1 << 24) || top_k > 60000) return SSDHEAD_E_UNSUPPORTED;
    if ((!dl && !aligned16(loc)) || (!FROM_SCORES && !aligned16(pri_cxcywh)) || !aligned16(out_boxes) || !aligned16(ws)) return SSDHEAD_E_ALIGN;
    const int NF = C - 1;
    const int T = dl ? dl->tile0[dl->n] : detect_tiles(P);
    if (T > NT) return SSDHEAD_E_UNSUPPORTED;                                 // P <= 131072
    const size_t smem_nms = nms_smem_bytes(NF, top_k, T);
    if (smem_nms > 200 * 1024) return SSDHEAD_E_UNSUPPORTED;                 // 20 classes: top_k <= 1729 at SSD300 (T = 35),
                                                                              // <= 1589 at T = 512
    DetectWs w;
    const size_t need = detect_ws_layout(B, P, C, n_cap, &w, ws);
    if (ws_bytes < need) return SSDHEAD_E_WORKSPACE;
    const int capI = detect_cap_image(P, C, n_cap);
    // the short-list route gives every row its 20 key slots in the image's list (a max_candidates below P rules it out)
    const bool fast = shortlist_enabled(B, P) && capI == NF * P && (long long)B * T < (1ll << 30);

    if (fast) {
        const int ipi_a = T;                                                  // 256-row items = the score tiles
        const int ipi_b = dl ? dl->item0[dl->n] : (P + RCW * 32 - 1) / (RCW * 32);
        const FloorArgs fl = {w.floor, w.dir_base, w.work, w.flag_cnt, min_score};
        const size_t smem_stream = (size_t)SST * SCW * 32 * C * 4;
        const size_t smem_sweep = std::max(smem_nms, (size_t)2 * RCW * 32 * C * 4);
        int per_sm = 0;
        // stream kernel (a cooperative launch without early start: everything in front of this call is complete when it
        // starts, which lets its producers request conf at once, and its CTAs wait on each other's floors, so all of them
        // must be resident even when other streams' kernels hold SMs): floors + short lists; sweep kernel
        if (dl) {
            auto ks = detect_stream_levels_kernel<21>;
            auto kw = detect_sweep_levels_kernel<21>;
            SSD_CHECK_CUDA(smem_limit_once(ks));
            SSD_CHECK_CUDA(smem_limit_once(kw));
            SSD_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ks, (SCW + 1) * 32, smem_stream));
            if (per_sm < 1) return SSDHEAD_E_UNSUPPORTED;
            const int grid = (int)std::min<long long>((long long)B * ipi_a, (long long)per_sm * device_sm_count());
            SSD_CHECK_CUDA(launch_coop(ks, dim3(grid), dim3((SCW + 1) * 32), smem_stream, st, fl, B, P, ipi_a, *dl, w.cand, capI, T));
            SSD_CHECK_CUDA(launch_pdl(kw, dim3(B), dim3(NT), smem_sweep, st, fl, ipi_a, ipi_b, *dl, (const float4*)pri_cxcywh,
                                      w.cand, w.scr_a, w.scr_b, img_wh, P, NF, T, capI, top_k, iou_thr,
                                      (float4*)out_boxes, out_prob, out_cls, out_prior, out_cnt));
        } else {
            auto ks = detect_stream_kernel<21, FROM_SCORES>;
            auto kw = detect_sweep_kernel<21, FROM_SCORES>;
            SSD_CHECK_CUDA(smem_limit_once(ks));
            SSD_CHECK_CUDA(smem_limit_once(kw));
            SSD_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ks, (SCW + 1) * 32, smem_stream));
            if (per_sm < 1) return SSDHEAD_E_UNSUPPORTED;
            const int grid = (int)std::min<long long>((long long)B * ipi_a, (long long)per_sm * device_sm_count());
            SSD_CHECK_CUDA(launch_coop(ks, dim3(grid), dim3((SCW + 1) * 32), smem_stream, st, fl, conf, B, P, ipi_a, w.cand, capI, T));
            SSD_CHECK_CUDA(launch_pdl(kw, dim3(B), dim3(NT), smem_sweep, st, fl, conf, ipi_a, ipi_b, (const float4*)loc, (const float4*)pri_cxcywh,
                                      w.cand, w.scr_a, w.scr_b, img_wh, P, NF, T, capI, top_k, iou_thr,
                                      (float4*)out_boxes, out_prob, out_cls, out_prior, out_cnt));
        }
        count_launch(2);
        return 0;
    }

    // the exhaustive route
    const dim3 g1(T, B);
    if (dl) {
        SSD_CHECK_CUDA(smem_limit_once(detect_nms_levels_kernel));
        SSD_CHECK_CUDA(launch_pdl(detect_score_levels_kernel<21>, g1, dim3(SC_T), 0, st,
                                  P, min_score, capI, w.cand, w.cand_cnt, w.dir, w.dir_base, w.overflow, w.flag_cnt, *dl));
        SSD_CHECK_CUDA(launch_pdl(detect_nms_levels_kernel, dim3(B), dim3(NT), smem_nms, st,
                                  *dl, (const float4*)pri_cxcywh, w.cand, w.scr_a, w.scr_b, (const unsigned short*)w.dir,
                                  (const unsigned int*)w.dir_base, w.cand_cnt, w.overflow, img_wh, P, NF, T, capI, top_k, iou_thr,
                                  (float4*)out_boxes, out_prob, out_cls, out_prior, out_cnt));
    } else {
        SSD_CHECK_CUDA(smem_limit_once(detect_nms_kernel<FROM_SCORES>));
        SSD_CHECK_CUDA(launch_pdl(detect_score_kernel<21, FROM_SCORES>, g1, dim3(SC_T), 0, st,
                                  conf, P, min_score, capI, w.cand, w.cand_cnt, w.dir, w.dir_base, w.overflow, w.flag_cnt));
        SSD_CHECK_CUDA(launch_pdl(detect_nms_kernel<FROM_SCORES>, dim3(B), dim3(NT), smem_nms, st,
                                  (const float4*)loc, (const float4*)pri_cxcywh, w.cand, w.scr_a, w.scr_b, (const unsigned short*)w.dir,
                                  (const unsigned int*)w.dir_base, w.cand_cnt, w.overflow, img_wh, P, NF, T, capI, top_k, iou_thr,
                                  (float4*)out_boxes, out_prob, out_cls, out_prior, out_cnt));
    }
    count_launch(2);
    return 0;
}

}  // namespace ssdhead

using namespace ssdhead;

extern "C" {

int ssdhead_detect(const float* loc, const float* conf, const float* pri_cxcywh, int B, int P, int C,
                   float min_score, float iou_thr, int top_k, const float* img_wh, int max_candidates,
                   float* out_boxes, float* out_prob, int32_t* out_cls, int32_t* out_prior, int32_t* out_cnt,
                   void* ws, size_t ws_bytes, void* stream)
{
    return run_detect<false>(loc, conf, pri_cxcywh, B, P, C, min_score, iou_thr, top_k, img_wh,
                             out_boxes, out_prob, out_cls, out_prior, out_cnt, ws, ws_bytes, max_candidates, (cudaStream_t)stream);
}

int ssdhead_detect_from_scores(const float* boxes_cxcywh, const float* probs, int B, int P, int C,
                               float min_score, float iou_thr, int top_k, const float* img_wh, int max_candidates,
                               float* out_boxes, float* out_prob, int32_t* out_cls, int32_t* out_prior, int32_t* out_cnt,
                               void* ws, size_t ws_bytes, void* stream)
{
    return run_detect<true>(boxes_cxcywh, probs, nullptr, B, P, C, min_score, iou_thr, top_k, img_wh,
                            out_boxes, out_prob, out_cls, out_prior, out_cnt, ws, ws_bytes, max_candidates, (cudaStream_t)stream);
}

int ssdhead_detect_levels(const ssdhead_levels* levels, const float* pri_cxcywh,
                          int B, int P, int C, float min_score, float iou_thr, int top_k,
                          const float* img_wh, int max_candidates,
                          float* out_boxes, float* out_prob, int32_t* out_cls, int32_t* out_prior, int32_t* out_cnt,
                          void* ws, size_t ws_bytes, void* stream)
{
    if (!levels || levels->num_levels < 1 || levels->num_levels > MAX_LEVELS) return SSDHEAD_E_BADARG;
    DetLevels dl = {};
    dl.n = levels->num_levels;
    int sum = 0, t0 = 0, i0 = 0;
    for (int l = 0; l < dl.n; ++l) {
        const int n = levels->count[l];
        if (n <= 0 || !levels->conf[l] || !levels->loc[l]) return SSDHEAD_E_BADARG;
        if (!aligned16(levels->loc[l])) return SSDHEAD_E_ALIGN;             // float4 rows; conf rows may sit anywhere
        dl.cnt[l] = n; dl.start[l] = sum; dl.tile0[l] = t0; dl.item0[l] = i0;
        dl.conf[l] = levels->conf[l]; dl.loc[l] = levels->loc[l];
        sum += n;
        t0 += (n + SC_T - 1) / SC_T;
        i0 += (n + RCW * 32 - 1) / (RCW * 32);
    }
    for (int l = dl.n; l <= MAX_LEVELS; ++l) { dl.start[l] = sum; dl.tile0[l] = t0; dl.item0[l] = i0; }
    if (sum != P) return SSDHEAD_E_BADARG;
    return run_detect<false>(nullptr, nullptr, pri_cxcywh, B, P, C, min_score, iou_thr, top_k, img_wh,
                             out_boxes, out_prob, out_cls, out_prior, out_cnt, ws, ws_bytes, max_candidates,
                             (cudaStream_t)stream, &dl);
}

int ssdhead_detect_fallbacks(const void* ws, size_t ws_bytes, int B, int P, int C, int max_candidates, int32_t* host_count, void* stream)
{
    if (!ws || !host_count || B <= 0 || P <= 0 || C < 2 || max_candidates < 0) return SSDHEAD_E_BADARG;
    DetectWs w;
    if (ws_bytes < detect_ws_layout(B, P, C, max_candidates, &w, const_cast<void*>(ws))) return SSDHEAD_E_WORKSPACE;
    SSD_CHECK_CUDA(cudaMemcpyAsync(host_count, w.flag_cnt, sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    SSD_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

#ifdef SSDHEAD_PHASE_TIMES
int ssdhead_debug_phases(long long* out16) { return (int)cudaMemcpyFromSymbol(out16, g_phase, sizeof(long long) * 16); }
int ssdhead_debug_stream(long long* out, int n_ctas) { return (int)cudaMemcpyFromSymbol(out, g_stream, sizeof(long long) * 8 * (size_t)n_ctas); }
#endif

}  // extern "C"
