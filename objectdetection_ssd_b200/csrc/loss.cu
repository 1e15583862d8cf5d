// Multibox loss: cross entropy + L1 + hard-negative mining, forward and gradients.
// Reference: ssd / ssd1_, Losses.py:119-199.
//
// The gradient of this loss is SPARSE: only positives and mined negatives (about 4*npos of the
// 8732 rows of an image) have a non-zero conf gradient, and only positives touch loc at all.
// The path is therefore split into one streaming kernel and one small per-image kernel:
//
//   ce_stream_kernel   persistent CTAs, one producer warp + 8 consumer warps.  The producer moves
//                      256-row tiles of conf (21 504 B) into a 2-stage shared-memory ring with 1-D
//                      TMA bulk copies (mbarrier full/empty pipeline) and, from a zeroed tile in
//                      shared memory, bulk-stores the zero background of grad_conf / grad_loc.
//                      Consumers do thread-per-row log-softmax out of shared memory (row stride 21
//                      words: bank-conflict free) and write one CE value per prior, scored against
//                      the BACKGROUND class (~99 % of the rows; positives are re-scored by
//                      mine_kernel).  With MATCH = true the same thread also computes the natural
//                      match of its prior (best gt, T1) and feeds the per-gt arg-max over priors (T2):
//                      the kernel is HBM-bound, the match rides in its spare issue slots.  conf is
//                      read exactly once; the tile grid is flat over B*P rows so every bulk copy is
//                      16-byte aligned whatever P is.
//   mine_kernel        one CTA per image: (FIN) forced-match override of the image from the arg-max
//                      keys (T3); CE row + class bytes -> keys in shared memory; exact selection of
//                      the k = 3*npos largest background CE (linear-bin histogram + direct ranking of
//                      the boundary bin; radix select 11/11/10 bits when ties crowd it), ties to the
//                      lower prior index (T4; positives rank with value 0, Losses.py:190); then
//                      thread-per-row over the ~4*npos selected rows only: re-read that conf row, write
//                      (softmax - onehot)/N into grad_conf, and for positives the L1 term and sign/(4N)
//                      into grad_loc.  N is the batch-global positive count: with FIN the CTAs of the
//                      (cooperative) grid exchange it through a counter, and - for a batch sharded over
//                      several GPUs - with their peers through stores into NVLink peer memory, as they
//                      do the two loss sums.  Loss partials are reduced in fp64 in a fixed order by the
//                      last CTA -> run-to-run deterministic.
//   match_finalize_kernel   the forced-match override as a separate small kernel (the NCCL route of a
//                      sharded batch, or when the batch does not fit a co-resident grid).
//   *_levels_kernel    the same two kernel bodies reading the head outputs per pyramid level in place (a level
//                      table in the constant bank instead of the concatenated [B,P,*] tensors; SURVEY 8(f) #3).
//   For batches with many gts per image the streaming kernel also records the best gt of every prior (2 B/row) so the
//   mining kernel does not walk the image's gts for every positive row.
//
// HBM traffic per image: conf in once (733 KB) + CE out/in (2 x 35 KB, L2-resident between the two
// kernels) + dense gradients out once (873 KB) + ~4*npos sparse rows: the algorithmic minimum.
#include <algorithm>
#include <tuple>
#include <type_traits>
#include "common.cuh"

namespace ssdhead {

#ifdef SSDHEAD_PHASE_TIMES      // developer build: SM clock at the phase boundaries of the first image's mining CTA
__device__ long long g_phase_loss[16];
#define LPHASE(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_phase_loss[i] = clock64(); } while (0)
__device__ long long g_cta[1024][12];    // per mining CTA: clocks from its wait to [0] selection done, [1] gradient rows done, [2] end; [3] = nsel;
                                          // [4] batch total known; row-loop trips 0/1: [5],[6] warp 0 done, [7],[8] last warp done, [9],[10] warp 0's conf part done
__device__ unsigned long long g_gt[8];    // global-timer marks: [0] last streaming CTA done, [1]/[2] first/last mining CTA past its wait, [3] last mining CTA done
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long v; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(v)); return v; }
#define GMARK_MAX(i) do { if (threadIdx.x == 0) atomicMax(&g_gt[i], gtimer()); } while (0)
#define GMARK_MIN(i) do { if (threadIdx.x == 0) atomicMin(&g_gt[i], gtimer()); } while (0)
#else
#define LPHASE(i) do { } while (0)
#define GMARK_MAX(i) do { } while (0)
#define GMARK_MIN(i) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------
// per-row cross entropy, -(x_c - max - log(sum exp(x - max))): the order ATen's log_softmax uses
// ------------------------------------------------------------------------------------------------
// FAST = true (streaming kernel only): exp through one ex2.approx.ftz per element (d <= 0; relative error
// <= (2 + 1.16|d|) ulp, i.e. an absolute error of ~2e-7 on log(sum)); the gradient and positive-row paths use expf.
template <int C, bool FAST = false>
__device__ __forceinline__ float row_cross_entropy(const float* __restrict__ row, int c)
{
    float x[C];
#pragma unroll
    for (int q = 0; q < C; ++q) x[q] = row[q];
    float m = x[0];
#pragma unroll
    for (int q = 1; q < C; ++q) m = fmaxf(m, x[q]);
    float s = 0.0f, xc = 0.0f;
#pragma unroll
    for (int q = 0; q < C; ++q) {
        const float d = __fsub_rn(x[q], m);
        s = __fadd_rn(s, FAST ? fast_exp_ftz(d) : expf(d));
        if (q == c) xc = d;
    }
    const float ce = __fsub_rn(logf(s), xc);
    return __fadd_rn(ce, 0.0f);                  // -0.0 -> +0.0 so the bit pattern orders like the value
}

// ------------------------------------------------------------------------------------------------
// Natural match fused into the streaming kernel (Losses.py:150-157): the consumer thread that scores prior p of
// image b also finds the best gt of that prior (T1) and takes part in the per-gt arg-max over priors (T2, merged with
// 64-bit atomicMax exactly as match_kernel does).  The streaming kernel is HBM-bound with issue slots to spare, so
// the ~G*15 extra instructions per row ride along for free and the separate match kernel leaves the critical path.
// Called by all 32 lanes of a warp together (`valid` masks rows past the end).
// ------------------------------------------------------------------------------------------------
struct FusedMatch {
    const float4* gt_xyxy;
    const float* gt_cls;
    const int* gt_off;
    const float4* pri_xyxy;
    int P, bg_class;
    float pos_iou;
    uint8_t* cls_u8;
    unsigned long long* best_key;
    int* npos_acc;
    unsigned short* obj_u16;     // nullable: natural best gt (local index) of every prior, for batches with many gts per image
    const float* seed_lb;        // batches with many gts per image (else nullptr): a lower bound of every gt's best IoU
    int sumG;                    // capacity of the gt arrays (match_seed_kernel's grid); a warp skips the gts that can neither make one of its priors positive
};                               // nor be best matched by one of them

// Everything the match of one row needs from global memory, fetched ONE TILE AHEAD so the two dependent L2 round trips
// (gt offsets -> gt boxes) and the prior box are in flight while the previous tile is being scored.
struct FusedPre {
    float4 pb;          // prior box of this row
    float4 gbox;        // lane l: gt l of the first image this warp touches (first 32 gts)
    float gcls;         //         and its class
    int b, p;           // image / prior of this row (-1 / 0 past the end)
    int b_first, b_last, off0, G;
};

__device__ __forceinline__ FusedPre fused_prefetch_bp(const FusedMatch& m, int b, int p, bool valid)
{
    FusedPre r;
    const int lane = threadIdx.x & 31;
    r.b = valid ? b : -1;
    r.p = valid ? p : 0;
    r.b_first = (int)__reduce_min_sync(FULL, valid ? (unsigned)r.b : 0x7fffffffu);
    r.b_last = __reduce_max_sync(FULL, r.b);
    r.pb = m.pri_xyxy[r.p];                                  // unconditional (p = 0 past the end): issued at once
    r.off0 = 0; r.G = 0;
    r.gbox = make_float4(0.f, 0.f, 0.f, 0.f);
    r.gcls = 0.0f;
    if (r.b_last >= 0) {
        r.off0 = m.gt_off[r.b_first];
        r.G = m.gt_off[r.b_first + 1] - r.off0;
        if (lane < min(r.G, 32)) { r.gbox = m.gt_xyxy[r.off0 + lane]; r.gcls = m.gt_cls[r.off0 + lane]; }
    }
    return r;
}

__device__ __forceinline__ FusedPre fused_prefetch(const FusedMatch& m, unsigned row, bool valid)
{
    const int b = (int)(row / (unsigned)m.P);
    return fused_prefetch_bp(m, b, (int)(row - (unsigned)b * (unsigned)m.P), valid);
}

template <bool MULTI = false>       // MULTI: a warp may span three or more images (per-level layout only)
__device__ __forceinline__ void fused_match_rows(const FusedMatch& m, unsigned row, bool valid, const FusedPre& pre)
{
    const int lane = threadIdx.x & 31;
    if (pre.b_last < 0) return;                              // no valid row in this warp
    const int b = pre.b, p = pre.p;
    const float4 pb = pre.pb;
    const float pa = box_area(pb);
    if (MULTI && pre.b_last - pre.b_first >= 2) {
        // The warp's 32 rows belong to three or more images (only the per-level layout does this, in the levels with a
        // handful of priors per image): walking the images one after the other would leave most lanes idle for a long
        // chain.  Each lane matches its own row against its own image's gts instead; the per-gt arg-max goes straight
        // to the 64-bit atomicMax (same key: highest IoU, then lowest prior - T2), the per-prior best stays strict-> (T1).
        if (valid) {
            const int off0 = m.gt_off[b], G = m.gt_off[b + 1] - off0;
            float bst = 0.0f;
            int obj_b = 0;
            float cls_b = G > 0 ? m.gt_cls[off0] : (float)m.bg_class;
            for (int g = 0; g < G; ++g) {
                const float4 gb = m.gt_xyxy[off0 + g];
                const float dx = __fsub_rn(fminf(gb.z, pb.z), fmaxf(gb.x, pb.x));
                const float dy = __fsub_rn(fminf(gb.w, pb.w), fmaxf(gb.y, pb.y));
                float v = 0.0f;
                if (dx > 0.0f && dy > 0.0f) {
                    const float inter = __fmul_rn(dx, dy);
                    v = __fdiv_rn(inter, __fsub_rn(__fadd_rn(box_area(gb), pa), inter));
                    if (v > bst) { bst = v; cls_b = m.gt_cls[off0 + g]; obj_b = g; }
                }
                if (v != 0.0f || p == 0)                    // an all-zero IoU row resolves to prior 0 (T2)
                    atomicMax(&m.best_key[off0 + g],
                              ((unsigned long long)(__float_as_uint(v) | 0x80000000u) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)p));
            }
            const bool hit = (G > 0) && !(bst < m.pos_iou);                           // T6
            const int c = hit ? (int)cls_b : m.bg_class;
            m.cls_u8[row] = (uint8_t)c;
            if (m.obj_u16) m.obj_u16[row] = (unsigned short)obj_b;
            if (c != m.bg_class) atomicAdd(&m.npos_acc[b], 1);
        }
        return;
    }
    float best = 0.0f;                 // IoU >= 0 and ties keep the first gt: (0, gt 0) equals max() over the column
    int g_mine = 0, obj_mine = 0;
    float cls_mine = (float)m.bg_class;
    // bounding box of the warp's 32 consecutive priors: a gt that misses it has IoU 0 with all of them, so the whole
    // pair test, the reduction and the atomic are skipped for that gt (about 3 of 4 gts for the dense 38x38 level)
    float wx1 = pb.x, wy1 = pb.y, wx2 = pb.z, wy2 = pb.w;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        wx1 = fminf(wx1, __shfl_xor_sync(FULL, wx1, d));
        wy1 = fminf(wy1, __shfl_xor_sync(FULL, wy1, d));
        wx2 = fmaxf(wx2, __shfl_xor_sync(FULL, wx2, d));
        wy2 = fmaxf(wy2, __shfl_xor_sync(FULL, wy2, d));
    }
    // Many gts per image (m.cull): IoU(prior, gt) <= min(area) / max(area), so with [amin, amax] the areas of the warp's
    // priors no pair of the warp with gt g can exceed ub(g) = 1 if area_g lies inside, area_g / amin below, amax / area_g
    // above.  A gt whose ub is below BOTH pos_iou (it cannot make a prior of the warp positive - the only use of the
    // per-prior maximum) and the gt's seed (match_seed_kernel: the IoU of a real prior, so strictly smaller values cannot
    // win the arg-max; ties keep the rule of the atomicMax) is skipped; the margin covers the rounding of the fp32 IoU.
    // The seeds are read-only during this kernel: cached loads next to the gt boxes, no extra round trip to L2.
    float amin = 0.0f, amax = 0.0f;
    if (m.seed_lb) {
        amin = valid ? pa : __int_as_float(0x7f800000);
        amax = valid ? pa : 0.0f;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            amin = fminf(amin, __shfl_xor_sync(FULL, amin, d));
            amax = fmaxf(amax, __shfl_xor_sync(FULL, amax, d));
        }
    }
    for (int bb = pre.b_first; bb <= pre.b_last; ++bb) {     // one image per warp except where a warp straddles two
        const bool first = (bb == pre.b_first);
        const int off0 = first ? pre.off0 : m.gt_off[bb];
        const int G = first ? pre.G : m.gt_off[bb + 1] - off0;
        const bool act = (b == bb);
        if (act) g_mine = G;
        const bool owns_p0 = __any_sync(FULL, act && p == 0);   // the arg-max of an all-zero IoU row is prior 0 (T2)
        for (int g0 = 0; g0 < G; g0 += 32) {
            // lane l holds gt g0+l (box + class): one coalesced round trip per 32 gts instead of one per gt;
            // the loop below broadcasts them with shuffles
            const int gc = min(32, G - g0);
            float4 mybox = pre.gbox;
            float mycls = pre.gcls;
            if (!(first && g0 == 0)) {
                mybox = make_float4(0.f, 0.f, 0.f, 0.f);
                mycls = 0.0f;
                if (lane < gc) { mybox = m.gt_xyxy[off0 + g0 + lane]; mycls = m.gt_cls[off0 + g0 + lane]; }
            }
            const float myarea = box_area(mybox);
            int chunk_best = -1;
            bool useful = true;
            if (m.seed_lb && lane < gc) {
                const float lb = __ldg(m.seed_lb + off0 + g0 + lane);                           // 0: no overlap in the sample
                const float ub = myarea < amin ? __fdiv_rn(myarea, amin) : (myarea > amax ? __fdiv_rn(amax, myarea) : 1.0f);
                useful = !(__fmul_rn(ub, 1.00002f) < fminf(m.pos_iou, lb));
            }
            // lanes whose gt can touch the warp's priors (the warp owning prior 0 must visit every gt: an all-zero
            // IoU row resolves to prior 0)
            unsigned todo = __ballot_sync(FULL, lane < gc && (owns_p0 || (useful && mybox.z > wx1 && mybox.x < wx2 && mybox.w > wy1 && mybox.y < wy2)));
            while (todo) {
                const int g = __ffs(todo) - 1;
                todo &= todo - 1;
                const float gx = __shfl_sync(FULL, mybox.x, g), gy = __shfl_sync(FULL, mybox.y, g);
                const float gz = __shfl_sync(FULL, mybox.z, g), gw = __shfl_sync(FULL, mybox.w, g);
                const float ga = __shfl_sync(FULL, myarea, g);
                float v = 0.0f;
                if (act) {
                    const float dx = __fsub_rn(fminf(gz, pb.z), fmaxf(gx, pb.x));
                    const float dy = __fsub_rn(fminf(gw, pb.w), fmaxf(gy, pb.y));
                    if (dx > 0.0f && dy > 0.0f) {            // disjoint boxes have IoU == +0 exactly
                        const float inter = __fmul_rn(dx, dy);
                        v = __fdiv_rn(inter, __fsub_rn(__fadd_rn(ga, pa), inter));
                        if (v > best) { best = v; chunk_best = g; }                   // T1: strict > keeps the first gt
                    }
                }
                const uint32_t mx = __reduce_max_sync(FULL, __float_as_uint(v));      // IoU >= 0: bits order like values
                if (mx != 0u || owns_p0) {
                    const unsigned ball = __ballot_sync(FULL, act && __float_as_uint(v) == mx);
                    const int wp = __shfl_sync(FULL, p, __ffs(ball) - 1);             // T2: lowest lane = lowest prior
                    if (lane == 0)
                        atomicMax(&m.best_key[off0 + g0 + g],
                                  ((unsigned long long)(mx | 0x80000000u) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)wp));
                }
            }
            // class of the best gt so far: gt 0 by default (first chunk), else the arg-max found in this chunk
            const float c_first = __shfl_sync(FULL, mycls, 0);
            const float c_best = __shfl_sync(FULL, mycls, chunk_best < 0 ? 0 : chunk_best);
            if (act) {
                if (chunk_best >= 0) { cls_mine = c_best; obj_mine = g0 + chunk_best; }
                else if (g0 == 0) cls_mine = c_first;
            }
        }
    }
    if (valid) {
        const bool hit = (g_mine > 0) && !(best < m.pos_iou);                     // T6
        const int c = hit ? (int)cls_mine : m.bg_class;
        m.cls_u8[row] = (uint8_t)c;                                               // natural class; forced matches patched later
        if (m.obj_u16) m.obj_u16[row] = (unsigned short)obj_mine;
        if (c != m.bg_class) atomicAdd(&m.npos_acc[b], 1);
    }
}

// Batches with many gts per image: a lower bound of every gt's best IoU - its best IoU over every SEED_STRIDE-th prior.
// One warp per gt.  The fused match then skips, per warp, the gts whose IoU with its priors cannot reach that bound.
// The sampled priors are staged in shared memory once per CTA (every warp of the grid walks all of them); a warp then
// takes gts in turn.  The packed gt arrays may be longer than the batch (`sumG` is their capacity): the warps stop at
// gt_off[B], read here, so a captured graph replays with whatever count the offsets hold.
constexpr int SEED_STRIDE = 16;                              // (stress shape: stride 8 / 16 / 32 leaves 8.0 / 8.6 / 10.3 of 23.2 gts per warp to visit)
constexpr int SEED_CAP = 65536;                              // gts of a batch the cull has seeds for (a fixed tail of the loss workspace:
                                                             // written before it is read, so it needs no cleaning)
constexpr int SEED_MAX = 8192;                               // sampled priors held in shared memory (128 KB)
__global__ void __launch_bounds__(256)
match_seed_kernel(const float4* __restrict__ gt_xyxy, const int* __restrict__ gt_off, int B, const float4* __restrict__ pri_xyxy,
                  int nsamp, int stride, float* __restrict__ seed_lb)
{
    extern __shared__ __align__(16) float4 s_pri[];
    const int t = threadIdx.x, lane = t & 31;
    const int n = gt_off[B];
    for (int i = t; i < nsamp; i += 256) s_pri[i] = pri_xyxy[(size_t)i * stride];
    __syncthreads();
    for (int g = blockIdx.x * 8 + (t >> 5); g < n; g += gridDim.x * 8) {
        const float4 gb = gt_xyxy[g];
        const float ga = box_area(gb);
        float best = 0.0f;
#pragma unroll 4
        for (int i = lane; i < nsamp; i += 32) {
            const float4 pb = s_pri[i];
            const float dx = __fsub_rn(fminf(gb.z, pb.z), fmaxf(gb.x, pb.x));
            const float dy = __fsub_rn(fminf(gb.w, pb.w), fmaxf(gb.y, pb.y));
            if (dx > 0.0f && dy > 0.0f) {                    // the fused match's own expression: the same bits
                const float inter = __fmul_rn(dx, dy);
                best = fmaxf(best, __fdiv_rn(inter, __fsub_rn(__fadd_rn(ga, box_area(pb)), inter)));
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) best = fmaxf(best, __shfl_xor_sync(FULL, best, d));
        if (lane == 0) seed_lb[g] = best;
    }
}

// After the streaming kernel: forced-match override (Losses.py:164-167) + positive counts.  One small CTA per image.
__global__ void __launch_bounds__(64)
match_finalize_kernel(const float* __restrict__ gt_cls, const int* __restrict__ gt_off, int B, int P, int bg_class,
                      int* __restrict__ best_prior, int* __restrict__ npos, uint8_t* __restrict__ cls_u8,
                      unsigned long long* __restrict__ best_key, int* __restrict__ npos_acc, unsigned int* __restrict__ image_counter)
{
    constexpr int CAP = 128;                                 // gts handled out of shared memory
    __shared__ int s_bp[CAP];
    __shared__ int s_extra;
    const int b = blockIdx.x, t = threadIdx.x;
    const int off0 = gt_off[b];
    const int G = gt_off[b + 1] - off0;
    pdl_trigger();                                           // let the mining kernel become resident behind us
    pdl_wait();                                              // everything below reads what the streaming kernel wrote
    const int acc0 = ld_cg_s32(&npos_acc[b]);                // independent of the gts: issue early
    if (t == 0) s_extra = 0;
    // one round of loads: best prior + class of every gt of the image
    int my_p[CAP / 64], my_c[CAP / 64];
#pragma unroll
    for (int q = 0; q < CAP / 64; ++q) {
        const int g = t + 64 * q;
        my_p[q] = -1; my_c[q] = bg_class;
        if (g < G) {
            my_p[q] = (int)(0xffffffffu - (uint32_t)(ld_cg_u64(&best_key[off0 + g]) & 0xffffffffull));
            my_c[q] = (int)gt_cls[off0 + g];
        }
    }
#pragma unroll
    for (int q = 0; q < CAP / 64; ++q) {
        const int g = t + 64 * q;
        if (g < G) { s_bp[g] = my_p[q]; best_prior[off0 + g] = my_p[q]; best_key[off0 + g] = 0ull; }
    }
    for (int g = CAP + t; g < G; g += 64) {                  // images with more than CAP gts: through global memory
        best_prior[off0 + g] = (int)(0xffffffffu - (uint32_t)(ld_cg_u64(&best_key[off0 + g]) & 0xffffffffull));
        best_key[off0 + g] = 0ull;
    }
    __syncthreads();
    int extra = 0;
    for (int g = t; g < G; g += 64) {
        const int p = g < CAP ? s_bp[g] : best_prior[off0 + g];
        bool winner = true;                                  // T3: the highest gt index keeps the prior
        for (int g2 = g + 1; g2 < G; ++g2) winner = winner && ((g2 < CAP ? s_bp[g2] : best_prior[off0 + g2]) != p);
        if (winner) {
            const int c_new = (g < CAP) ? my_c[g / 64] : (int)gt_cls[off0 + g];
            const int c_nat = (int)cls_u8[(size_t)b * P + p];
            extra += (c_new != bg_class ? 1 : 0) - (c_nat != bg_class ? 1 : 0);
            cls_u8[(size_t)b * P + p] = (uint8_t)c_new;
        }
    }
    if (extra) atomicAdd(&s_extra, extra);
    __syncthreads();
    if (t == 0) {
        npos[b] = acc0 + s_extra;
        npos_acc[b] = 0;
        __threadfence();
        const unsigned done = atomicAdd(image_counter, 1u);
        if (done == gridDim.x - 1) {                         // last image: batch total, fixed order
            __threadfence();
            int tot = 0;
            for (int i = 0; i < B; ++i) tot += ld_relaxed_gpu_s32(&npos[i]);   // other CTAs of this grid wrote them: coherent loads
            npos[B] = tot;
            *image_counter = 0u;
        }
    }
}

constexpr int CE_ROWS = 256;                      // rows per tile = consumer threads
// Ring depth, resident CTAs per SM and zero-tile size of the streaming kernel (compile-time: tools/variants.py builds and
// times alternatives).  Measured on B200 at B=256 / 128 (step, us): 4 stages + a whole zeroed tile (round 1) 106.6 / 66.4;
// 3 stages 104.4 / 64.4; 2 stages + a 64-row zero tile 103.6 / 62.8 (two CTAs x two 21.5 KB tiles in flight per SM
// still cover HBM's latency-bandwidth product, and the smaller shared-memory footprint - 97 KB instead of 215 KB per SM -
// leaves the L1 to the match's loads); three CTAs per SM (72-register cap) 111.1.  Staging the tile's prior boxes through
// the ring as well changed nothing at any depth.
#ifndef SSDHEAD_CE_STAGES
#define SSDHEAD_CE_STAGES 2
#endif
#ifndef SSDHEAD_CE_CTAS
#define SSDHEAD_CE_CTAS 2
#endif
#ifndef SSDHEAD_CE_ZERO_ROWS
#define SSDHEAD_CE_ZERO_ROWS 64
#endif
constexpr int CE_STAGES = SSDHEAD_CE_STAGES;      // stages of the conf ring
constexpr int CE_CTAS = SSDHEAD_CE_CTAS;          // resident CTAs per SM the kernel is built for
constexpr int CE_ZERO_ROWS = SSDHEAD_CE_ZERO_ROWS;// rows of the zeroed tile the gradient background is bulk-stored from
static_assert(CE_ZERO_ROWS * 21 * 4 >= 256 * 16 && (CE_ZERO_ROWS * 21 * 4) % 16 == 0, "the zero tile must cover one tile of loc rows");
constexpr int CE_THREADS = CE_ROWS + 32;          // + one producer warp

// Head outputs given PER PYRAMID LEVEL (SURVEY.md 8(f) #3): the reference permutes every conv output to NHWC and
// concatenates the six levels into [B,8732,4] / [B,8732,21] (Model.py:212-235) - a full extra HBM round trip.  An
// NHWC conv output already IS the row layout [B, n_l, 21] of its level, so the kernels can read the level tensors in
// place: level l holds n_l = cnt[l] priors per image, its rows are flat [B * n_l], priors start[l] .. start[l+1]-1 of the
// global order.  The streaming kernel walks one virtual tile space: tile0[l] .. tile0[l+1]-1 are the full 256-row tiles
// of level l (tiles straddle images inside a level exactly as they do in the concatenated layout).
constexpr int MAX_LEVELS = SSDHEAD_MAX_LEVELS;
struct LevelTab {
    int n;
    int cnt[MAX_LEVELS];
    int start[MAX_LEVELS + 1];
    int tile0[MAX_LEVELS + 1];
    int rows[MAX_LEVELS];        // B * cnt[l]; the last tile of a level may be partial (then rows % 4 == 0: 16-byte sizes)
    int perm_stride, perm_inc;   // the k-th tile a CTA visits is virtual tile (k * stride) mod total: levels interleave, so the
                                 // match-heavy tiles of the coarse levels hide under the memory time of the fine ones
    const float* conf[MAX_LEVELS];
    const float* loc[MAX_LEVELS];
    float* gconf[MAX_LEVELS];
    float* gloc[MAX_LEVELS];
};
__device__ __forceinline__ int level_of_tile(const LevelTab& lv, int vt) {
    int l = 0;
#pragma unroll
    for (int q = 1; q < MAX_LEVELS; ++q) if (q < lv.n && vt >= lv.tile0[q]) l = q;
    return l;
}
__device__ __forceinline__ int level_of_prior(const LevelTab& lv, int j) {
    int l = 0;
#pragma unroll
    for (int q = 1; q < MAX_LEVELS; ++q) if (q < lv.n && j >= lv.start[q]) l = q;
    return l;
}

template <int C, bool ZERO_FILL, bool MATCH, bool LEVELS>
__device__ __forceinline__ void
ce_stream_body(const float* __restrict__ conf, float* __restrict__ ce_out,
               float* __restrict__ grad_conf, float* __restrict__ grad_loc, long long total_rows, int use_tma,
               const FusedMatch& fm, const LevelTab* __restrict__ lvp)
{
    constexpr uint32_t TILE_BYTES = CE_ROWS * C * 4;
    constexpr uint32_t ZERO_BYTES = CE_ZERO_ROWS * C * 4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t s_full[CE_STAGES];
    __shared__ __align__(8) uint64_t s_empty[CE_STAGES];
    float* zero_tile = reinterpret_cast<float*>(smem_raw + (size_t)CE_STAGES * TILE_BYTES);

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long long full_tiles = LEVELS ? lvp->tile0[lvp->n] : (use_tma ? total_rows / CE_ROWS : 0);
    const int P = fm.P;

    if (t == 0) {
#pragma unroll
        for (int s = 0; s < CE_STAGES; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], CE_ROWS / 32); }
        mbar_fence_init();
    }
    if (ZERO_FILL) {
        for (int i = t; i < (int)(ZERO_BYTES / 16); i += CE_THREADS)
            reinterpret_cast<float4*>(zero_tile)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        fence_proxy_async_smem();
    }
    pdl_trigger();                                           // the finaliser may become resident now (it waits for us)
    pdl_wait();                                              // the previous step may still be reading the buffers we overwrite
    __syncthreads();

    if (warp == CE_ROWS / 32) {
        // ---------------- producer warp: one elected lane drives the TMA engine ----------------
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            int vt = LEVELS ? (int)(((long long)blockIdx.x * lvp->perm_stride) % full_tiles) : 0;
            for (long long k = blockIdx.x; k < full_tiles; k += gridDim.x) {
                const long long tile = LEVELS ? (long long)vt : k;
                if (LEVELS) { vt += lvp->perm_inc; if (vt >= (int)full_tiles) vt -= (int)full_tiles; }
                mbar_wait(&s_empty[s], ph ^ 1u);
                const float* src = conf + (size_t)tile * CE_ROWS * C;
                float* gc = grad_conf + (size_t)tile * CE_ROWS * C;
                float* gl = grad_loc + (size_t)tile * CE_ROWS * 4;
                uint32_t nr = CE_ROWS;
                if (LEVELS) {
                    const int l = level_of_tile(*lvp, (int)tile);
                    const size_t r0 = (size_t)((int)tile - lvp->tile0[l]) * CE_ROWS;
                    nr = (uint32_t)min((long long)CE_ROWS, (long long)lvp->rows[l] - (long long)r0);
                    src = lvp->conf[l] + r0 * C;
                    if (ZERO_FILL) { gc = lvp->gconf[l] + r0 * C; gl = lvp->gloc[l] + r0 * 4; }
                }
                mbar_expect_tx(&s_full[s], nr * C * 4);
                bulk_g2s(smem_raw + (size_t)s * TILE_BYTES, src, nr * C * 4, &s_full[s]);
                if (ZERO_FILL) {
                    for (uint32_t o = 0; o < nr * C * 4; o += ZERO_BYTES)       // the conf rows' background in zero-tile sized pieces
                        bulk_s2g(reinterpret_cast<unsigned char*>(gc) + o, zero_tile, min(ZERO_BYTES, nr * C * 4 - o));
                    bulk_s2g(gl, zero_tile, nr * 16);
                    bulk_commit();
                }
                if (++s == CE_STAGES) { s = 0; ph ^= 1u; }
            }
            if (ZERO_FILL) bulk_wait_read_all();
        }
    } else {
        // ---------------- consumer warps: thread per row ----------------
        int s = 0;
        uint32_t ph = 0;
        // global row (b * P + prior) of this thread's row in virtual tile `tile`
        FusedPre pre, nxt;
        if (!LEVELS) {
            if (MATCH && (long long)blockIdx.x < full_tiles) pre = fused_prefetch(fm, (unsigned)(blockIdx.x * CE_ROWS + t), true);
            for (long long tile = blockIdx.x; tile < full_tiles; tile += gridDim.x) {
                const long long row = tile * CE_ROWS + t;
                if (MATCH) {
                    // issue the next tile's match inputs now; score this tile's match (independent of the conf tile)
                    if (tile + gridDim.x < full_tiles) nxt = fused_prefetch(fm, (unsigned)((tile + gridDim.x) * CE_ROWS + t), true);
                    fused_match_rows(fm, (unsigned)row, true, pre);
                    pre = nxt;
                }
                mbar_wait(&s_full[s], ph);
                const float ce = row_cross_entropy<C, true>(reinterpret_cast<const float*>(smem_raw + (size_t)s * TILE_BYTES) + t * C, C - 1);
                __syncwarp();
                if (lane == 0) mbar_arrive(&s_empty[s]);
                ce_out[row] = ce;
                if (++s == CE_STAGES) { s = 0; ph ^= 1u; }
            }
        } else {
            // image / prior of this thread's row in virtual tile `tile` (b = -1 past the end of a partial last tile)
            auto locate = [&](int tile, int& b, int& p) {
                const int l = level_of_tile(*lvp, tile);
                const unsigned lr = (unsigned)(tile - lvp->tile0[l]) * CE_ROWS + (unsigned)t, n = (unsigned)lvp->cnt[l];
                if (lr >= (unsigned)lvp->rows[l]) { b = -1; p = 0; return; }
                const unsigned bb = lr / n;
                b = (int)bb;
                p = lvp->start[l] + (int)(lr - bb * n);
            };
            int cb = -1, cp = 0, nb = -1, np = 0;
            const int T = (int)full_tiles;
            int vt = T > 0 ? (int)(((long long)blockIdx.x * lvp->perm_stride) % T) : 0;       // same walk as the producer
            if ((long long)blockIdx.x < full_tiles) { locate(vt, cb, cp); pre = fused_prefetch_bp(fm, cb, cp, cb >= 0); }
            for (long long k = blockIdx.x; k < full_tiles; k += gridDim.x) {
                const bool valid = cb >= 0;
                const long long row = (long long)cb * P + cp;
                vt += lvp->perm_inc;
                if (vt >= T) vt -= T;
                if (k + gridDim.x < full_tiles) { locate(vt, nb, np); nxt = fused_prefetch_bp(fm, nb, np, nb >= 0); }
                fused_match_rows<true>(fm, (unsigned)row, valid, pre);
                pre = nxt;
                mbar_wait(&s_full[s], ph);
                float ce = 0.0f;
                if (valid) ce = row_cross_entropy<C, true>(reinterpret_cast<const float*>(smem_raw + (size_t)s * TILE_BYTES) + t * C, C - 1);
                __syncwarp();
                if (lane == 0) mbar_arrive(&s_empty[s]);
                if (valid) ce_out[row] = ce;
                cb = nb; cp = np;
                if (++s == CE_STAGES) { s = 0; ph ^= 1u; }
            }
        }
        // rows past the last full tile (or every row when the pointers are not 16-byte aligned): plain loads
        if (!LEVELS) {
            const long long rest0 = full_tiles * CE_ROWS;
            for (long long row0 = rest0 + (long long)blockIdx.x * CE_ROWS; row0 < total_rows; row0 += (long long)gridDim.x * CE_ROWS) {
                const long long row = row0 + t;                  // the loop bound is CTA-uniform: warps stay converged
                const bool valid = row < total_rows;
                if (MATCH) fused_match_rows(fm, (unsigned)row, valid, fused_prefetch(fm, (unsigned)row, valid));
                if (valid) {
                    ce_out[row] = row_cross_entropy<C, true>(conf + (size_t)row * C, C - 1);
                    if (ZERO_FILL) {
#pragma unroll
                        for (int q = 0; q < C; ++q) grad_conf[(size_t)row * C + q] = 0.0f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) grad_loc[(size_t)row * 4 + q] = 0.0f;
                    }
                }
            }
        } else {
            // per level: the rows after its last full tile (fewer than 256 when B * n_l is not a multiple of 256)
            for (int l = 0; l < lvp->n; ++l) {
                const unsigned n = (unsigned)lvp->cnt[l];
                const long long rows_l = total_rows / P * n;     // B * n_l
                const long long rest0 = (long long)(lvp->tile0[l + 1] - lvp->tile0[l]) * CE_ROWS;
                // each level's tail starts on a different CTA (otherwise CTA 0 would walk all of them one after the other)
                const unsigned first = (blockIdx.x + gridDim.x - ((unsigned)l * (gridDim.x / MAX_LEVELS + 1)) % gridDim.x) % gridDim.x;
                for (long long r0 = rest0 + (long long)first * CE_ROWS; r0 < rows_l; r0 += (long long)gridDim.x * CE_ROWS) {
                    const long long lr = r0 + t;
                    const bool valid = lr < rows_l;
                    const unsigned b = valid ? (unsigned)(lr / n) : 0u;
                    const long long row = valid ? (long long)b * P + lvp->start[l] + (int)(lr - (long long)b * n) : total_rows;
                    if (MATCH) fused_match_rows<true>(fm, (unsigned)row, valid, fused_prefetch(fm, (unsigned)row, valid));
                    if (valid) {
                        ce_out[row] = row_cross_entropy<C, true>(lvp->conf[l] + (size_t)lr * C, C - 1);
                        if (ZERO_FILL) {
#pragma unroll
                            for (int q = 0; q < C; ++q) lvp->gconf[l][(size_t)lr * C + q] = 0.0f;
#pragma unroll
                            for (int q = 0; q < 4; ++q) lvp->gloc[l][(size_t)lr * 4 + q] = 0.0f;
                        }
                    }
                }
            }
        }
    }
    __syncthreads();
    GMARK_MAX(0);
}

template <int C, bool ZERO_FILL, bool MATCH>
__global__ void __launch_bounds__(CE_THREADS, CE_CTAS)
ce_stream_kernel(const float* __restrict__ conf, float* __restrict__ ce_out,
                 float* __restrict__ grad_conf, float* __restrict__ grad_loc, long long total_rows, int use_tma,
                 const FusedMatch fm)
{
    ce_stream_body<C, ZERO_FILL, MATCH, false>(conf, ce_out, grad_conf, grad_loc, total_rows, use_tma, fm, nullptr);
}

// the same kernel reading / zero-filling per-level tensors in place (no concatenated [B,P,*] tensors exist)
template <int C, bool ZERO_FILL>
__global__ void __launch_bounds__(CE_THREADS, CE_CTAS)
ce_stream_levels_kernel(float* __restrict__ ce_out, long long total_rows, const FusedMatch fm, const __grid_constant__ LevelTab lv)
{
    ce_stream_body<C, ZERO_FILL, true, true>(nullptr, ce_out, nullptr, nullptr, total_rows, 1, fm, &lv);
}

// ------------------------------------------------------------------------------------------------
// mine_kernel
// ------------------------------------------------------------------------------------------------
constexpr int MN_T = 512;
constexpr int MN_W = MN_T / 32;
constexpr int MN_BINS = 2048;

struct MineParams {
    const float* loc;
    const float* conf;
    const float* ce;             // CE of every row against the BACKGROUND class (ce_stream_kernel)
    float* ce_w;                 // host-side convenience: the same buffer, writable (level entry point)
    float* ce_tap;               // nullable: receives the true CE of positive rows (debug tap)
    const uint8_t* cls_u8;
    const float4* gt_xyxy;
    const float* gt_cls;
    const int* gt_off;
    const float4* pri_xyxy;
    const float4* pri_cxcywh;
    const int* best_prior;
    const int* npos;
    const int* npos_norm;
    int B, P, neg_ratio, bg_class;
    float pos_iou;
    double* sums;
    float* losses;
    float* grad_loc;
    float* grad_conf;
    uint32_t* mined_mask;
    double* partials;            // [B][2]
    unsigned int* done_counter;  // self-resetting
    // fused forced-match finaliser (FIN = true; cooperative launch, all CTAs co-resident):
    unsigned short* obj_u16;     // nullable: best gt per prior from the streaming kernel (forced ones patched by FIN)
    uint8_t* cls_rw;             // class bytes, patched in place
    int* best_prior_w;           // [sumG] out
    int* npos_w;                 // [B+1] out
    unsigned long long* best_key;   // match workspace: per-gt arg-max keys (left zeroed)
    int* npos_acc;                  //                  natural positives per image (left zeroed)
    unsigned long long* arrive_total;  // workspace word: CTAs that published (high half) | batch positive count (low), left zeroed
    // cross-GPU exchange of the positive count and the loss sums over NVLink peer memory (xchg.R > 1):
    // every rank owns an exchange buffer of XCHG_WORDS 64-bit words that its PEERS write into (and it spins on).
    Xchg xchg;
    // sparse gradient return (SPARSE = true; ssdhead_mine_sparse): the rows that carry a gradient, packed per image
    // instead of scattered into dense [B,P,*] tensors.  Slot s of image b: sp_idx[b*cap+s] = prior, sp_conf[(b*cap+s)*C..]
    // its conf-gradient row; the first sp_cnt[2b+1] slots are the positives and also own sp_loc[(b*cap+s)*4..].
    float* sp_conf;
    float* sp_loc;
    int* sp_idx;
    int* sp_cnt;                    // [B][2]: rows of the image (may exceed cap: then only cap were stored), positives
    int sp_cap;
    // resident gradient tensors (ssdhead_multibox_step_resident): grad_conf / grad_loc are all-zero except for the rows
    // the PREVIOUS step wrote, which are listed here; this step retracts them, writes its own rows and lists those
    unsigned char* res_base;        // per image one record of res_stride bytes (independent of B): int32 rows, int32 positives,
    size_t res_stride;              // then uint16 [P] the rows of the image that carry a gradient, positives first (nullable)
};


// exclusive prefix sum over the MN_T threads of the CTA; *total receives the block sum
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* s_warp /*[MN_W+1]*/, uint32_t* total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(FULL, inc, d);
        if (lane >= d) inc += o;
    }
    __syncthreads();                              // protect s_warp against the previous use
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t base = 0u, tot = 0u;
#pragma unroll
    for (int w = 0; w < MN_W; ++w) { const uint32_t c = s_warp[w]; if (w < warp) base += c; tot += c; }
    *total = tot;
    return base + inc - v;
}

constexpr int MN_GC = 64;        // gt boxes staged in shared memory
constexpr int MN_CAND = 512;     // boundary-bin candidates ranked directly (one per thread)

template <int C, bool GRADS, bool FIN, bool LEVELS, bool SPARSE = false>
__device__ __forceinline__ void mine_body(const MineParams& p, const LevelTab* __restrict__ lvp)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t* s_key = reinterpret_cast<uint32_t*>(smem_raw);            // [P]  CE bit pattern, 0 for positives; bit 31 = selected
    uint32_t* s_hist = s_key + p.P;                                      // [MN_BINS]
    uint16_t* s_list = reinterpret_cast<uint16_t*>(s_hist + MN_BINS);    // [P]  rows that carry a gradient (P < 65536)
    uint8_t* s_cls = reinterpret_cast<uint8_t*>(s_list + ((p.P + 7) & ~7)); // [P]  class bytes (16-byte aligned)
    __shared__ uint32_t s_warp[MN_W + 1];
    __shared__ uint32_t s_sel[3];
    __shared__ uint32_t s_nsel, s_ncand, s_max;
    // positives are listed from the END of s_list downwards, mined rows from its start upwards (together at most P
    // entries): the box part of the positive rows runs as its own pass (step 4a)
    __shared__ uint32_t s_npl;
    __shared__ uint32_t s_ckey[MN_CAND], s_cidx[MN_CAND];
    __shared__ float4 s_gbox[MN_GC];
    __shared__ float s_garea[MN_GC];
    __shared__ int s_gbp[MN_GC];
    __shared__ double s_redd[2][MN_W];

    const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int P = p.P;
    const size_t row0 = (size_t)b * P;
    const int off0 = p.gt_off[b];
    const int G = p.gt_off[b + 1] - off0;
    double acc_l1 = 0.0, acc_ce = 0.0;
    // row j of this image in the head tensors: the concatenated [B,P,*] tensors, or the tensor of j's pyramid level
    auto conf_row = [&](int j) -> const float* {
        if (!LEVELS) return p.conf + (row0 + j) * C;
        const int l = level_of_prior(*lvp, j);
        return lvp->conf[l] + ((size_t)b * lvp->cnt[l] + (size_t)(j - lvp->start[l])) * C;
    };
    auto gconf_row = [&](int j) -> float* {
        if (!LEVELS) return p.grad_conf + (row0 + j) * C;
        const int l = level_of_prior(*lvp, j);
        return lvp->gconf[l] + ((size_t)b * lvp->cnt[l] + (size_t)(j - lvp->start[l])) * C;
    };
    auto loc_row = [&](int j) -> const float4* {
        if (!LEVELS) return reinterpret_cast<const float4*>(p.loc) + row0 + j;
        const int l = level_of_prior(*lvp, j);
        return reinterpret_cast<const float4*>(lvp->loc[l]) + (size_t)b * lvp->cnt[l] + (size_t)(j - lvp->start[l]);
    };
    auto gloc_row = [&](int j) -> float4* {
        if (!LEVELS) return reinterpret_cast<float4*>(p.grad_loc) + row0 + j;
        const int l = level_of_prior(*lvp, j);
        return reinterpret_cast<float4*>(lvp->gloc[l]) + (size_t)b * lvp->cnt[l] + (size_t)(j - lvp->start[l]);
    };

    // ---- 1. keys: CE bits for negatives, 0 for positives (Losses.py:188-190); class bytes; gts ----
    if (t == 0) { s_nsel = 0u; s_ncand = 0u; s_max = 0u; s_npl = 0u; }
    if (t < min(G, MN_GC)) {
        const float4 bx = p.gt_xyxy[off0 + t];               // inputs of the step: may be read before the wait
        s_gbox[t] = bx;
        s_garea[t] = box_area(bx);
    }
    pdl_trigger();
    pdl_wait();                                              // CE, class bytes, best priors, positive counts are ready
    __syncthreads();                                         // s_max / s_nsel / gt staging above are visible
    int* res_cnt = nullptr;
    unsigned short* res_rows = nullptr;
    if (GRADS && !SPARSE && p.res_base) {
        // resident gradient tensors: zero the rows the previous step left in this image (everything else is zero
        // already), so no dense zero background is written at all.  The new rows are written after several barriers.
        res_cnt = reinterpret_cast<int*>(p.res_base + (size_t)b * p.res_stride);
        res_rows = reinterpret_cast<unsigned short*>(p.res_base + (size_t)b * p.res_stride + 8);
        const int n_prev = res_cnt[0], npl_prev = res_cnt[1];
        for (int i = t; i < n_prev; i += MN_T) {
            const int j = (int)res_rows[i];
            float* g = gconf_row(j);
#pragma unroll
            for (int q = 0; q < C; ++q) g[q] = 0.0f;
            if (i < npl_prev) *gloc_row(j) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    LPHASE(0);
    GMARK_MIN(1); GMARK_MAX(2);
#ifdef SSDHEAD_PHASE_TIMES
    const long long cta_t0 = clock64();
#endif
    // The forced-match inputs are requested first, then the keys are built from the NATURAL classes while those loads
    // are in flight; the override below patches the few forced priors in shared memory (and in the global class map).
    int acc0 = 0;
    unsigned long long bk0 = 0ull;
    if (FIN) {
        acc0 = ld_cg_s32(&p.npos_acc[b]);
        if (t < G) bk0 = ld_cg_u64(&p.best_key[off0 + t]);
    }
    uint32_t kmax = 0u;
    const bool vec_ok = ((P & 3) == 0) && (((row0 * 4) & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.ce) & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.cls_u8) & 3) == 0);
    if (vec_ok) {
        const float4* ce4 = reinterpret_cast<const float4*>(p.ce + row0);
        const uchar4* cl4 = reinterpret_cast<const uchar4*>(p.cls_u8 + row0);
        const int nvec = P >> 2;
        // 16-byte CE loads + 4-byte class loads; KU of each are issued per thread before the first is used
        // (SSD300: 2183 vectors / 512 threads -> the whole image in one round of loads)
        constexpr int KU = 5;
        for (int v0 = t; v0 < nvec; v0 += KU * MN_T) {
            float4 e5[KU];
            uchar4 c5[KU];
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int v = v0 + u * MN_T;
                if (v < nvec) { e5[u] = ce4[v]; c5[u] = cl4[v]; }
            }
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int v = v0 + u * MN_T;
                if (v >= nvec) break;
                const float4 e = e5[u];
                const uchar4 c = c5[u];
                const float ev[4] = {e.x, e.y, e.z, e.w};
                const uint8_t cv[4] = {c.x, c.y, c.z, c.w};
                uint32_t kv[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const bool pos = (int)cv[q] != p.bg_class;
                    kv[q] = pos ? 0u : (__float_as_uint(ev[q]) & 0x7fffffffu);
                    kmax = max(kmax, kv[q]);
                }
                reinterpret_cast<uint4*>(s_key)[v] = make_uint4(kv[0], kv[1], kv[2], kv[3]);
                reinterpret_cast<uchar4*>(s_cls)[v] = c;
            }
        }
    } else {
        for (int j = t; j < P; j += MN_T) {
            const float ce = p.ce[row0 + j];
            const uint8_t c = p.cls_u8[row0 + j];
            const bool pos = (int)c != p.bg_class;
            const uint32_t key = pos ? 0u : (__float_as_uint(ce) & 0x7fffffffu);
            s_key[j] = key;
            s_cls[j] = c;
            kmax = max(kmax, key);
        }
    }
    kmax = __reduce_max_sync(FULL, kmax);
    if (lane == 0) atomicMax(&s_max, kmax);
    LPHASE(1);
    int npos_b;
    if (FIN) {
        // ---- 0. forced-match override of THIS image (Losses.py:164-167), fused here so that no separate finaliser
        // kernel sits between the streaming kernel and this one.  The batch-global positive count, which only the
        // gradient scale needs, is exchanged through a counter the CTAs of this (cooperative) grid wait on later.
        __shared__ int s_fin_extra, s_fin_npos;
        if (t == 0) s_fin_extra = 0;
        for (int g = t; g < G; g += MN_T) {
            const unsigned long long bkv = g == t ? bk0 : ld_cg_u64(&p.best_key[off0 + g]);
            const int bp = (int)(0xffffffffu - (uint32_t)(bkv & 0xffffffffull));
            p.best_key[off0 + g] = 0ull;                     // leave the workspace zeroed
            p.best_prior_w[off0 + g] = bp;
            if (g < MN_GC) s_gbp[g] = bp;
        }
        __syncthreads();
        int extra = 0;
        for (int g = t; g < G; g += MN_T) {
            const int bp = g < MN_GC ? s_gbp[g] : p.best_prior_w[off0 + g];
            bool winner = true;                              // T3: the highest gt index keeps the prior
            for (int g2 = g + 1; g2 < G; ++g2) winner = winner && ((g2 < MN_GC ? s_gbp[g2] : p.best_prior_w[off0 + g2]) != bp);
            if (winner) {
                const int c_new = (int)p.gt_cls[off0 + g];
                const int c_nat = (int)s_cls[bp];            // the natural class, staged a moment ago
                extra += (c_new != p.bg_class ? 1 : 0) - (c_nat != p.bg_class ? 1 : 0);
                p.cls_rw[row0 + bp] = (uint8_t)c_new;
                s_cls[bp] = (uint8_t)c_new;                  // a prior has one winner: no two threads patch the same entry
                const uint32_t key = c_new != p.bg_class ? 0u : (__float_as_uint(p.ce[row0 + bp]) & 0x7fffffffu);
                s_key[bp] = key;
                // a gt labelled with the background class turns a positive into a negative: its key rises from 0 to
                // its CE, which the histogram range (s_max) must cover - a NaN / inf key sends the image to the radix path
                if (c_new == p.bg_class) atomicMax(&s_max, key);
                if (p.obj_u16) p.obj_u16[row0 + bp] = (unsigned short)g;
            }
        }
        if (extra) atomicAdd(&s_fin_extra, extra);
        __syncthreads();
        if (t == 0) {
            const int nb = acc0 + s_fin_extra;
            s_fin_npos = nb;
            p.npos_w[b] = nb;
            p.npos_acc[b] = 0;
            // one 64-bit atomic carries both the arrival (high word) and the image's positives (low word): whoever sees
            // gridDim.x arrivals sees the complete batch count in the same word - no fence between two atomics
            const unsigned long long before = atomicAdd(p.arrive_total, (1ull << 32) | (unsigned long long)(unsigned)nb);
            if (p.xchg.R > 1 && (unsigned)(before >> 32) == gridDim.x - 1u)
                xchg_publish_count(p.xchg, (unsigned)before + (unsigned)nb);    // last image of this GPU: the count is complete
        }
        __syncthreads();
        npos_b = s_fin_npos;
    } else {
        if (t < min(G, MN_GC)) s_gbp[t] = p.best_prior[off0 + t];
        __syncthreads();
        npos_b = p.npos[b];
    }
    const int* bprior = FIN ? p.best_prior_w : p.best_prior;
    __syncthreads();
    kmax = s_max;                                            // covers every key: the override folded in the keys it raised;
    LPHASE(2);                                               // a key it lowered to 0 (made positive) only widens the bins

    // ---- 2. the k largest keys, ties to the lower prior index (T4): mark them with bit 31 ----
    const long long kk = (long long)p.neg_ratio * (long long)npos_b;
    const uint32_t k = (uint32_t)min((long long)P, max(0ll, kk));
    bool listed = false;                         // the row list was already built by the fast path
    if (k >= (uint32_t)P) {
        for (int j = t; j < P; j += MN_T) s_key[j] |= 0x80000000u;
    } else if (k > 0u) {
        bool done = false;
        const float vmax = __uint_as_float(kmax);
        if (kmax > 0u && kmax < 0x7f800000u) {
            // fast path: one histogram over 2048 LINEAR bins of [0, max] (monotone in the key), then the few
            // keys of the boundary bin are ranked against each other directly.
            const float scale = __fdiv_rn(2047.0f, vmax);
            for (int i = t; i < MN_BINS; i += MN_T) s_hist[i] = 0u;
            __syncthreads();
            for (int j = t; j < P; j += MN_T)
                atomicAdd(&s_hist[(int)__fmul_rn(__uint_as_float(s_key[j]), scale)], 1u);
            __syncthreads();
            constexpr int per = MN_BINS / MN_T;
            uint32_t c4[per], mine = 0u;
#pragma unroll
            for (int q = 0; q < per; ++q) { c4[q] = s_hist[MN_BINS - 1 - (t * per + q)]; mine += c4[q]; }
            uint32_t tot;
            uint32_t above = block_exclusive_scan(mine, s_warp, &tot);
            if (above < k && above + mine >= k) {
#pragma unroll
                for (int q = 0; q < per; ++q) {
                    if (above + c4[q] >= k) { s_sel[0] = (uint32_t)(MN_BINS - 1 - (t * per + q)); s_sel[1] = above; s_sel[2] = c4[q]; break; }
                    above += c4[q];
                }
            }
            __syncthreads();
            const int bq = (int)s_sel[0];
            const uint32_t need = k - s_sel[1], cnt = s_sel[2];
            if (cnt <= (uint32_t)MN_CAND) {
                done = true;
                listed = true;
                // one pass: rows above the boundary bin are mined, rows in it become candidates, positives are listed
                for (int j = t; j < P; j += MN_T) {
                    const uint32_t key = s_key[j];
                    const bool pos = (int)s_cls[j] != p.bg_class;
                    const int bin = (int)__fmul_rn(__uint_as_float(key), scale);
                    if (pos) {
                        s_list[P - 1 - (int)atomicAdd(&s_npl, 1u)] = (uint16_t)j;
                    } else if (bin > bq) {
                        acc_ce += (double)__uint_as_float(key);
                        if (p.mined_mask) atomicOr(&p.mined_mask[(size_t)b * ((P + 31) / 32) + (j >> 5)], 1u << (j & 31));
                        if (GRADS) s_list[atomicAdd(&s_nsel, 1u)] = (uint16_t)j;
                    } else if (bin == bq) {
                        const uint32_t s = atomicAdd(&s_ncand, 1u);
                        s_ckey[s] = key;
                        s_cidx[s] = (uint32_t)j;
                    }
                }
                __syncthreads();
                // positives in the boundary bin (key 0, only when bq == 0) were listed above, not made candidates;
                // they still occupy ranks: `need` counts them, so rank them through the candidate count of bin 0
                const uint32_t ncand = s_ncand;
                if ((uint32_t)t < ncand) {
                    const uint32_t mk = s_ckey[t], mi = s_cidx[t];
                    uint32_t rank = 0u;
                    for (uint32_t q = 0; q < ncand; ++q) {
                        const uint32_t ok = s_ckey[q], oi = s_cidx[q];
                        rank += (ok > mk || (ok == mk && oi < mi)) ? 1u : 0u;
                    }
                    if (bq == 0) {
                        // positives (value 0) tie with zero-CE negatives: ties go to the lower prior index
                        if (mk == 0u) for (int j = 0; j < (int)mi; ++j) rank += ((int)s_cls[j] != p.bg_class) ? 1u : 0u;
                    }
                    if (rank < need) {
                        acc_ce += (double)__uint_as_float(mk);
                        if (p.mined_mask) atomicOr(&p.mined_mask[(size_t)b * ((P + 31) / 32) + (mi >> 5)], 1u << (mi & 31));
                        if (GRADS) s_list[atomicAdd(&s_nsel, 1u)] = (uint16_t)mi;
                    }
                }
            }
        }
        if (!done) {
            // general path (many equal keys, or non-finite CE): exact radix select, digits of 11 / 11 / 10 bits
            uint32_t prefix = 0u, mask = 0u, need = k;
#pragma unroll 1
            for (int pass = 0; pass < 3; ++pass) {
                const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
                const int bins = pass == 2 ? 1024 : 2048;
                __syncthreads();
                for (int i = t; i < bins; i += MN_T) s_hist[i] = 0u;
                __syncthreads();
                for (int j = t; j < P; j += MN_T) {
                    const uint32_t key = s_key[j];
                    if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & (uint32_t)(bins - 1)], 1u);
                }
                __syncthreads();
                const int per = bins / MN_T;          // 4 or 2
                uint32_t c4[4] = {0u, 0u, 0u, 0u}, mine = 0u;
#pragma unroll
                for (int q = 0; q < 4; ++q) if (q < per) { c4[q] = s_hist[bins - 1 - (t * per + q)]; mine += c4[q]; }
                uint32_t tot;
                uint32_t above = block_exclusive_scan(mine, s_warp, &tot);
                if (above < need && above + mine >= need) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) if (q < per) {
                        if (above + c4[q] >= need) { s_sel[0] = (uint32_t)(bins - 1 - (t * per + q)); s_sel[1] = above; s_sel[2] = c4[q]; break; }
                        above += c4[q];
                    }
                }
                __syncthreads();
                prefix |= s_sel[0] << shift;
                mask |= (uint32_t)(bins - 1) << shift;
                need -= s_sel[1];
            }
            const uint32_t T = prefix;               // take every key > T and the first `need` keys == T in prior order
            int per = (P + MN_T - 1) / MN_T;
            per |= 1;                                // odd stride: fewer shared-memory bank conflicts
            const int j0 = min(P, t * per), j1 = min(P, j0 + per);
            uint32_t ties = 0u;
            for (int j = j0; j < j1; ++j) ties += (s_key[j] == T) ? 1u : 0u;
            uint32_t tot_ties;
            uint32_t rank = block_exclusive_scan(ties, s_warp, &tot_ties);
            for (int j = j0; j < j1; ++j) {
                const uint32_t key = s_key[j];
                if (key > T) s_key[j] = key | 0x80000000u;
                else if (key == T) { if (rank < need) s_key[j] = key | 0x80000000u; ++rank; }
            }
        }
    }
    __syncthreads();

    // ---- 3. mined CE sum, list of rows that carry a gradient ----
    if (!listed) {
        for (int j = t; j < P; j += MN_T) {
            const uint32_t key = s_key[j];
            const bool pos = (int)s_cls[j] != p.bg_class;
            const bool mined = (key >> 31) && !pos;
            if (mined) {
                acc_ce += (double)__uint_as_float(key & 0x7fffffffu);
                if (p.mined_mask) atomicOr(&p.mined_mask[(size_t)b * ((P + 31) / 32) + (j >> 5)], 1u << (j & 31));
            }
            if (pos) s_list[P - 1 - (int)atomicAdd(&s_npl, 1u)] = (uint16_t)j;
            else if (GRADS && mined) s_list[atomicAdd(&s_nsel, 1u)] = (uint16_t)j;
        }
    }
    __syncthreads();

    // ---- 4. the selected rows only: conf gradient, and for positives the L1 term + loc gradient ----
    LPHASE(3);
    const uint32_t npl = s_npl;                  // positives, listed from the end
    const uint32_t nsel = s_nsel + npl;
    if (SPARSE && t == 0) { p.sp_cnt[2 * b] = (int)nsel; p.sp_cnt[2 * b + 1] = (int)npl; }
    if (GRADS && !SPARSE && res_rows && t == 0) { res_cnt[0] = (int)nsel; res_cnt[1] = (int)npl; }
#ifdef SSDHEAD_PHASE_TIMES
    if (t == 0 && b < 1024) { g_cta[b][0] = clock64() - cta_t0; g_cta[b][3] = nsel; }
#endif
    int npos_total;
    if (FIN) {
        // every CTA of the grid is co-resident (cooperative launch) and published its count long ago (step 0); a bounded
        // wait that expires is reported (trap on one GPU, err_flag for a peer that never arrived), never papered over
        __shared__ int s_total;
        if (t == 0) {
            if (p.xchg.R > 1) {
                s_total = xchg_gather_count(p.xchg);     // sharded batch: the counts of all ranks, written by their last CTAs
            } else {
                // The launch is cooperative, so every CTA of the grid is resident and has published its count microseconds
                // ago.  The spin is still bounded (~2 s) so that a broken launch contract cannot hang the GPU - but it
                // never continues with a partial count: it traps, and the host sees a launch failure.
                unsigned spins = 0;
                unsigned long long w;
                while ((unsigned)((w = ld_relaxed_gpu_u64(p.arrive_total)) >> 32) < gridDim.x && ++spins < (1u << 25)) __nanosleep(64);
                if ((unsigned)(w >> 32) < gridDim.x) __trap();
                s_total = (int)(unsigned)w;
            }
        }
        __syncthreads();
        npos_total = s_total;
    } else {
        npos_total = *p.npos_norm;
    }
    LPHASE(4);
#ifdef SSDHEAD_PHASE_TIMES
    if (t == 0 && b < 1024) { g_cta[b][4] = clock64() - cta_t0; for (int q = 5; q < 11; ++q) g_cta[b][q] = 0; }
#endif
    const float nrm = (float)npos_total;
    const float gs_conf = __fdiv_rn(1.0f, nrm);
    const float gs_loc = __fdiv_rn(1.0f, __fmul_rn(4.0f, nrm));
    // The rows are scattered over the image, 84 bytes each: a thread-per-row access touches 32 rows per instruction
    // (32 sectors for 128 useful bytes).  With gradients the warp therefore moves its 32 rows through shared memory:
    // flat, coalesced loads of the 32 x 21 logits, thread-per-row arithmetic in place, flat coalesced stores - about
    // seven times fewer L2 transactions on the latency chain every CTA of the step waits for.  The staging area is the
    // key + histogram region, dead since the selection.
    // ---- 4a. the box part of the positive rows (target encoding, L1 term, loc gradient): its own pass, one thread per
    // positive, handed out from the LAST thread downwards.  The conf trip below is a serial chain of about a thousand
    // instructions per warp and its rows are packed into the first warps, so in most images the last warps are free to
    // do this meanwhile, and neither loop carries the other's registers (measured: 112.0 -> 105.6 us per step at B=256,
    // 36.9 -> 34.3 at B=32, no spills left in the gradient kernel; same bits).
    auto box_pass = [&]() {      // (kept as a lambda: this is the form whose code generation was measured and tested)
        for (uint32_t i = (uint32_t)(MN_T - 1 - t); i < npl; i += MN_T) {
            const int j = (int)s_list[P - 1 - (int)i];
            const float4 pb = p.pri_xyxy[j];
            const float4 pc = p.pri_cxcywh[j];
            const float4 l = *loc_row(j);
            const float pa = box_area(pb);
            int obj = -1, ng = 0;
            float nb = 0.0f;
            if (FIN && p.obj_u16) obj = (int)p.obj_u16[row0 + j];   // recorded by the match: no walk over the image's gts
            else for (int g = 0; g < G; ++g) {
                float4 gb; float ga; int bp;
                if (g < MN_GC) { gb = s_gbox[g]; ga = s_garea[g]; bp = s_gbp[g]; }
                else { gb = p.gt_xyxy[off0 + g]; ga = box_area(gb); bp = bprior[off0 + g]; }
                if (bp == j) obj = g;
                const float v = iou_sparse(gb, ga, pb, pa);
                if (v > nb) { nb = v; ng = g; }
            }
            if (obj < 0) obj = ng;
            const float4 gbox = obj < MN_GC ? s_gbox[obj] : p.gt_xyxy[off0 + obj];
            const float4 tgt = encode_box(xyxy_to_cxcywh(gbox), pc);
            const float dx = __fsub_rn(l.x, tgt.x), dy = __fsub_rn(l.y, tgt.y);
            const float dz = __fsub_rn(l.z, tgt.z), dw = __fsub_rn(l.w, tgt.w);
            acc_l1 += (double)fabsf(dx) + (double)fabsf(dy) + (double)fabsf(dz) + (double)fabsf(dw);
            if (GRADS) {
                float4 gl;
                gl.x = dx > 0.f ? gs_loc : (dx < 0.f ? -gs_loc : 0.f);
                gl.y = dy > 0.f ? gs_loc : (dy < 0.f ? -gs_loc : 0.f);
                gl.z = dz > 0.f ? gs_loc : (dz < 0.f ? -gs_loc : 0.f);
                gl.w = dw > 0.f ? gs_loc : (dw < 0.f ? -gs_loc : 0.f);
                if (SPARSE) { if (i < (uint32_t)p.sp_cap) reinterpret_cast<float4*>(p.sp_loc)[(size_t)b * p.sp_cap + i] = gl; }
                else *gloc_row(j) = gl;
            }
        }
    };
    box_pass();
    const bool staged = GRADS && (size_t)P * 4 + (size_t)MN_BINS * 4 >= (size_t)MN_W * 32 * C * 4;
    float* wstage = reinterpret_cast<float*>(smem_raw) + warp * (32 * C);
    for (uint32_t base = 0; base < nsel; base += MN_T) {
        const uint32_t idx = base + t;
        const bool valid = idx < nsel;
        const uint32_t wbase = base + (uint32_t)warp * 32u;
        const int nrw = wbase < nsel ? (int)min(32u, nsel - wbase) : 0;
        const int j = valid ? (int)(idx < npl ? s_list[P - 1 - (int)idx] : s_list[idx - npl]) : 0;   // positives first
        const float* my_crow = LEVELS ? conf_row(j) : nullptr;      // per-level tensors: locate the row once, pass pointers
        float* my_grow = (LEVELS && GRADS) ? gconf_row(j) : nullptr;
        if (SPARSE && valid && idx < (uint32_t)p.sp_cap) p.sp_idx[(size_t)b * p.sp_cap + idx] = j;
        if (GRADS && !SPARSE && res_rows && valid) res_rows[idx] = (unsigned short)j;
        if (staged) {
            // element e = lane + 32 i of the warp's 32 x C block belongs to row e / C, whose index lane e / C holds;
            // all loads are issued before the first shared-memory store (which the compiler must assume may alias)
            float v[C];
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const int e = lane + 32 * i, r = e / C, q = e - r * C;
                const float* rp;
                if (LEVELS) rp = reinterpret_cast<const float*>(__shfl_sync(FULL, (unsigned long long)my_crow, r));
                else rp = conf_row(__shfl_sync(FULL, j, r));
                v[i] = r < nrw ? __ldg(rp + q) : 0.0f;
            }
#pragma unroll
            for (int i = 0; i < C; ++i) wstage[lane + 32 * i] = v[i];
            __syncwarp();
        }
        const int c = valid ? (int)s_cls[j] : p.bg_class;
        const bool pos = c != p.bg_class;
        float x[C];
        if (valid && (GRADS || pos)) {
            if (staged) {
#pragma unroll
                for (int q = 0; q < C; ++q) x[q] = wstage[lane * C + q];
            } else {
                const float* row = LEVELS ? my_crow : conf_row(j);
#pragma unroll
                for (int q = 0; q < C; ++q) x[q] = __ldg(row + q);
            }
        }
        if (!GRADS && pos) {
            // the streaming kernel scored every row against the background class; a positive row gets its
            // true-class CE here, from the row it re-reads anyway (same code -> same bits as a direct evaluation)
            const float ce = row_cross_entropy<C>(x, c);
            acc_ce += (double)ce;
            if (p.ce_tap) p.ce_tap[row0 + j] = ce;
        }
        if (GRADS && valid) {
            float m = x[0];
#pragma unroll
            for (int q = 1; q < C; ++q) m = fmaxf(m, x[q]);
            float s = 0.0f, xc = 0.0f;
#pragma unroll
            for (int q = 0; q < C; ++q) {
                const float d = __fsub_rn(x[q], m);
                if (q == c) xc = d;
                x[q] = expf(d);
                s = __fadd_rn(s, x[q]);
            }
            if (pos) {
                // max, exponentials and their sum (same order) are exactly row_cross_entropy's: the true-class CE of a
                // positive row falls out of the softmax its gradient needs anyway
                const float ce = __fadd_rn(__fsub_rn(logf(s), xc), 0.0f);
                acc_ce += (double)ce;
                if (p.ce_tap) p.ce_tap[row0 + j] = ce;
            }
            const float inv = __fdiv_rn(1.0f, s);
            if (staged) {
#pragma unroll
                for (int q = 0; q < C; ++q)
                    wstage[lane * C + q] = __fmul_rn(__fsub_rn(__fmul_rn(x[q], inv), q == c ? 1.0f : 0.0f), gs_conf);
            } else {
                float* grow = SPARSE ? p.sp_conf + ((size_t)b * p.sp_cap + idx) * C : (LEVELS ? my_grow : gconf_row(j));
                if (!SPARSE || idx < (uint32_t)p.sp_cap) {
#pragma unroll
                    for (int q = 0; q < C; ++q)
                        grow[q] = __fmul_rn(__fsub_rn(__fmul_rn(x[q], inv), q == c ? 1.0f : 0.0f), gs_conf);
                }
            }
        }
        if (staged) {
            __syncwarp();
            float v[C];
#pragma unroll
            for (int i = 0; i < C; ++i) v[i] = wstage[lane + 32 * i];
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const int e = lane + 32 * i, r = e / C, q = e - r * C;
                float* rp;
                if (SPARSE) {
                    // the warp's 32 slots are contiguous in the packed output: one flat, fully coalesced block
                    rp = p.sp_conf + ((size_t)b * p.sp_cap + (wbase + (uint32_t)r)) * C;
                    if (r < nrw && wbase + (uint32_t)r < (uint32_t)p.sp_cap) rp[q] = v[i];
                    continue;
                }
                if (LEVELS) rp = reinterpret_cast<float*>(__shfl_sync(FULL, (unsigned long long)my_grow, r));
                else rp = gconf_row(__shfl_sync(FULL, j, r));
                if (r < nrw) rp[q] = v[i];
            }
            __syncwarp();
        }
#ifdef SSDHEAD_PHASE_TIMES
        if (lane == 0 && warp == 0 && b < 1024 && base < 2 * MN_T) g_cta[b][9 + base / MN_T] = clock64() - cta_t0;
#endif
#ifdef SSDHEAD_PHASE_TIMES
        __syncwarp();
        if (lane == 0 && (warp == 0 || warp == MN_W - 1) && b < 1024 && base < 2 * MN_T)
            g_cta[b][5 + (warp ? 2 : 0) + base / MN_T] = clock64() - cta_t0;
#endif
    }

#ifdef SSDHEAD_PHASE_TIMES
    if (t == 0 && b < 1024) g_cta[b][1] = clock64() - cta_t0;
#endif
    LPHASE(5);
    // ---- 5. loss sums: per-image partial -> the last CTA reduces all partials in a fixed order ----
    acc_l1 = warp_sum(acc_l1);
    acc_ce = warp_sum(acc_ce);
    if (lane == 0) { s_redd[0][warp] = acc_l1; s_redd[1][warp] = acc_ce; }
    __syncthreads();
    // The publisher is the LAST thread of the CTA: its fence only has to drain its own stores, and unlike thread 0 it
    // normally wrote no gradient row (rows go to threads 0..nsel-1).  The CTA that draws the last ticket adds the
    // partials in a fixed order (run-to-run deterministic).  (A fence-free variant - sign bit of the non-negative sums as
    // a "valid" mark, one fixed CTA polling - was measured 1-2 us SLOWER per step, and taught a hardware lesson: its
    // polls must be relaxed gpu-scope loads; an ld.cg poll spun forever on a stale copy of the line in the SM's near L2
    // partition while the plain store from the other die sat in the far one.)
    __shared__ int s_is_last;
    if (t == MN_T - 1) {
        double a = 0.0, c = 0.0;
        for (int w = 0; w < MN_W; ++w) { a += s_redd[0][w]; c += s_redd[1][w]; }
        p.partials[2 * b] = a;
        p.partials[2 * b + 1] = c;
        __threadfence();
        const unsigned done = atomicAdd(p.done_counter, 1u);
        s_is_last = (done == gridDim.x - 1u) ? 1 : 0;
    }
    __syncthreads();
    LPHASE(6);
    if (s_is_last) {
        __threadfence();
        double a = 0.0, c = 0.0;
        for (int s = t; s < (int)gridDim.x; s += MN_T) {     // written by the other CTAs of this grid: coherent loads
            a += __longlong_as_double((long long)ld_relaxed_gpu_u64(reinterpret_cast<const unsigned long long*>(p.partials) + 2 * (size_t)s));
            c += __longlong_as_double((long long)ld_relaxed_gpu_u64(reinterpret_cast<const unsigned long long*>(p.partials) + 2 * (size_t)s + 1));
        }
        a = warp_sum(a);
        c = warp_sum(c);
        __syncthreads();
        if (lane == 0) { s_redd[0][warp] = a; s_redd[1][warp] = c; }
        __syncthreads();
        if (t == 0) {
            a = 0.0; c = 0.0;
            for (int w = 0; w < MN_W; ++w) { a += s_redd[0][w]; c += s_redd[1][w]; }
            if (FIN && p.xchg.R > 1) xchg_allreduce_sums(p.xchg, a, c);
            p.sums[0] = a;
            p.sums[1] = c;
            losses_from_sums(p.losses, a, c, npos_total);
            *p.done_counter = 0u;
            if (FIN) {                   // every CTA has read the total (it did so before it reported done)
                p.npos_w[p.B] = (p.xchg.R > 1) ? (int)(unsigned)ld_cg_u64(p.arrive_total) : npos_total;    // this rank's own count
                *p.arrive_total = 0ull;
            }
        }
    }
    GMARK_MAX(3);
#ifdef SSDHEAD_PHASE_TIMES
    if (t == 0 && b < 1024) g_cta[b][2] = clock64() - cta_t0;
#endif
}


template <int C, bool GRADS, bool FIN>
__global__ void __launch_bounds__(MN_T, 2)    // two CTAs per SM: B = 256 images stay co-resident (cooperative launch)
mine_kernel(const MineParams p)
{
    mine_body<C, GRADS, FIN, false>(p, nullptr);
}

// the mining kernel with the gradient rows returned PACKED (ssdhead_mine_sparse): no dense [B,P,*] gradient tensor exists
template <int C>
__global__ void __launch_bounds__(MN_T, 2)
mine_sparse_kernel(const MineParams p)
{
    mine_body<C, true, false, false, true>(p, nullptr);
}

// the same kernel on per-level head tensors (ssdhead_multibox_step_levels)
template <int C, bool GRADS, bool FIN>
__global__ void __launch_bounds__(MN_T, 2)
mine_levels_kernel(const MineParams p, const __grid_constant__ LevelTab lv)
{
    mine_body<C, GRADS, FIN, true>(p, &lv);
}


__global__ void finish_loss_kernel(const double* __restrict__ sums, const int* __restrict__ npos_norm, float* __restrict__ losses)
{
    losses_from_sums(losses, sums[0], sums[1], *npos_norm);
}

__global__ void __launch_bounds__(256)
scale_grads_kernel(float4* __restrict__ gl, size_t n4_loc, float* __restrict__ gl_tail, int tail_loc,
                   float4* __restrict__ gc, size_t n4_conf, float* __restrict__ gc_tail, int tail_conf,
                   const float* __restrict__ gout)
{
    const float a = gout[0], c = gout[1];
    if (a == 1.0f && c == 1.0f) return;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a != 1.0f) {
        for (size_t i = tid; i < n4_loc; i += stride) { float4 v = gl[i]; v.x *= a; v.y *= a; v.z *= a; v.w *= a; gl[i] = v; }
        if (tid < (size_t)tail_loc) gl_tail[tid] *= a;
    }
    if (c != 1.0f) {
        for (size_t i = tid; i < n4_conf; i += stride) { float4 v = gc[i]; v.x *= c; v.y *= c; v.z *= c; v.w *= c; gc[i] = v; }
        if (tid < (size_t)tail_conf) gc_tail[tid] *= c;
    }
}

static size_t mine_smem_bytes(int P) { return (size_t)P * 4 + MN_BINS * 4 + (size_t)((P + 7) & ~7) * 2 + round_up((size_t)P, 16); }

// Loss workspace (16-byte aligned): done counter [0,16) | partials double[2B] | CE float[B*P] (when the caller passes no
// ce buffer) | best-gt map u16[B*P] of the steps | seeds float[SEED_CAP] of the fused match's cull.  The counter and the
// partials are kept zero between calls.
struct LossWs {
    unsigned int* done_counter;
    double* partials;
    float* ce;
    unsigned short* obj;
    float* seed;
};
static LossWs loss_ws(void* ws, int B, int P)
{
    uintptr_t w = (uintptr_t)ws;
    LossWs l;
    l.done_counter = (unsigned int*)w;            w += 16;
    l.partials = (double*)w;                      w += round_up((size_t)B * 2 * sizeof(double), 16);
    l.ce = (float*)w;                             w += round_up((size_t)B * P * sizeof(float), 16);
    l.obj = (unsigned short*)w;                   w += round_up((size_t)B * P * sizeof(unsigned short), 16);
    l.seed = (float*)w;
    return l;
}
size_t loss_workspace_bytes(int B, int P, int C)
{
    if (mine_smem_bytes(P) > 220 * 1024 || P >= 65536) return 0;   // P <= ~31 000 priors
    return (uintptr_t)loss_ws(nullptr, B, P).seed + (size_t)SEED_CAP * sizeof(float);
}
// Bytes from the start of a loss workspace that hold the done counter and the partials of any batch of up to maxB
// images, plus 256 bytes that no field needs (they reach into the CE rows, which every call rewrites).
size_t loss_ws_header_bytes(int maxB) { return (uintptr_t)loss_ws(nullptr, maxB, 0).ce + 256; }

// rows workspace of the resident-gradient step: one record per image, the same for every batch size - int32 rows,
// int32 positives, uint16 [P] row indices (P < 65536)
static size_t resident_row_stride(int P) { return round_up(8 + (size_t)P * sizeof(unsigned short), 16); }
size_t resident_rows_bytes(int B, int P)
{
    if (B <= 0 || P <= 0 || P >= 65536) return 0;
    return (size_t)B * resident_row_stride(P);
}

static int num_sms() { return device_sm_count(); }

// The streaming CE kernel over [B*P] rows (lv == nullptr) or over the per-level tensors of lv
template <int C, bool GRADS, bool MATCH>
static int launch_ce_stream(const float* conf, float* ce, float* grad_conf, float* grad_loc, long long rows,
                            const FusedMatch& fm, const LevelTab* lv, cudaStream_t st)
{
    constexpr size_t tile = (size_t)CE_ROWS * C * 4;
    const size_t smem_ce = tile * CE_STAGES + (GRADS ? (size_t)CE_ZERO_ROWS * C * 4 : 0);
    const long long tiles = (rows + CE_ROWS - 1) / CE_ROWS + (lv ? lv->n : 0);
    const int grid_ce = (int)std::min<long long>(tiles, (long long)CE_CTAS * num_sms());
    if (MATCH && fm.seed_lb) {
        const int stride = std::max(SEED_STRIDE, (fm.P + SEED_MAX - 1) / SEED_MAX);
        const int nsamp = (fm.P + stride - 1) / stride;
        const size_t smem_seed = (size_t)nsamp * 16;
        SSD_CHECK_CUDA(smem_limit_once(match_seed_kernel));
        const int grid_seed = std::min((fm.sumG + 7) / 8, 2 * num_sms());      // sized by the capacity
        const int B = (int)(rows / fm.P);                                       // rows = B * P in every caller
        match_seed_kernel<<<grid_seed, 256, smem_seed, st>>>(fm.gt_xyxy, fm.gt_off, B, fm.pri_xyxy, nsamp, stride,
                                                             const_cast<float*>(fm.seed_lb));
        SSD_LAUNCH_CHECK();
        count_launch();
    }
    if (MATCH && lv) {
        auto kce = ce_stream_levels_kernel<C, GRADS>;
        SSD_CHECK_CUDA(smem_limit_once(kce));
        // stride ~ 0.618 T, coprime with T: consecutive visits land in different levels in proportion to their sizes
        LevelTab lt = *lv;
        const long long T = lt.tile0[lt.n];
        auto gcd = [](long long a, long long b) { while (b) { const long long c = a % b; a = b; b = c; } return a; };
        long long S = std::max<long long>(1, (long long)(0.6180339887 * (double)T));
        while (S > 1 && gcd(S, T) != 1) --S;
        lt.perm_stride = (int)S;
        lt.perm_inc = T > 0 ? (int)(((long long)grid_ce * S) % T) : 0;
        SSD_CHECK_CUDA(launch_pdl(kce, dim3(grid_ce), dim3(CE_THREADS), smem_ce, st, ce, rows, fm, lt));
    } else {
        auto kce = ce_stream_kernel<C, GRADS, MATCH>;
        SSD_CHECK_CUDA(smem_limit_once(kce));
        const int use_tma = (aligned16(conf) && (!GRADS || (aligned16(grad_conf) && aligned16(grad_loc)))) ? 1 : 0;
        SSD_CHECK_CUDA(launch_pdl(kce, dim3(grid_ce), dim3(CE_THREADS), smem_ce, st, conf, ce, grad_conf, grad_loc, rows, use_tma, fm));
    }
    count_launch();
    return 0;
}

// Whether `st` is capturing into a graph (a failed query counts as capturing: the caller then takes the launch that
// cannot be refused).
static bool stream_capturing(cudaStream_t st)
{
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) {
        (void)cudaGetLastError();
        return true;
    }
    return cs != cudaStreamCaptureStatusNone;
}

// Whether a grid of B CTAs of the mining kernel kmn can be co-resident (*fits); the kernel's dynamic shared memory limit
// is raised first (once per device), as its launch needs and the occupancy query reads it.
template <typename... KArgs>
static int mine_fits_coresident(void (*kmn)(KArgs...), int B, int P, bool* fits)
{
    const size_t smem_mn = mine_smem_bytes(P);
    SSD_CHECK_CUDA(smem_limit_once(kmn));
    int per_sm = 0;
    SSD_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kmn, MN_T, smem_mn));
    *fits = (long long)per_sm * num_sms() >= B;
    return 0;
}

// A mining kernel on one CTA per image.  FIN: the forced-match finaliser is fused in, so every CTA must be co-resident
// (they exchange the batch positive count through a counter) - a cooperative launch, which returns 1 (not an error)
// when the grid does not fit.
template <bool FIN, typename... KArgs, typename... Args>
static int launch_mine(void (*kmn)(KArgs...), int B, int P, cudaStream_t st, Args... args)
{
    const size_t smem_mn = mine_smem_bytes(P);
    if (!FIN) {
        SSD_CHECK_CUDA(smem_limit_once(kmn));
        SSD_CHECK_CUDA(launch_pdl(kmn, dim3(B), dim3(MN_T), smem_mn, st, args...));
        count_launch();
        return 0;
    }
    bool fits = false;
    const int rc = mine_fits_coresident(kmn, B, P, &fits);
    if (rc || !fits) return rc ? rc : 1;
    // cooperative (co-residency guaranteed) AND programmatic stream serialization (the grid may become resident while
    // the streaming kernel drains; it waits in pdl_wait()).  Runtimes that refuse the combination get the plain
    // cooperative launch.  The combination is first tried on an eager launch: a refused launch inside a stream capture
    // would invalidate the capture, so a capture takes it only once an eager launch has shown it is accepted.  What was
    // learnt is kept per device (threads may launch on several at once).
    static std::atomic<int> pdl_state[MAX_DEVICES];          // 0: not tried yet, 1: accepted, -1: refused
    int dev = 0;
    SSD_CHECK_CUDA(cudaGetDevice(&dev));
    std::atomic<int> untracked{0};
    std::atomic<int>& with_pdl = dev < MAX_DEVICES ? pdl_state[dev] : untracked;
    const int known = with_pdl.load(std::memory_order_relaxed);
    const bool capturing = known >= 0 && stream_capturing(st);
    if (known == 1 || (known == 0 && !capturing)) {
        const cudaError_t e = launch_pdl<true>(kmn, dim3(B), dim3(MN_T), smem_mn, st, args...);
        if (e == cudaSuccess) { with_pdl.store(1, std::memory_order_relaxed); count_launch(); return 0; }
        if (capturing) return (int)e;
        (void)cudaGetLastError();
        with_pdl.store(-1, std::memory_order_relaxed);
    }
    static_assert(std::is_same<std::tuple<std::decay_t<Args>...>, std::tuple<std::decay_t<KArgs>...>>::value,
                  "the cooperative launch passes the arguments by address: they must have the kernel's parameter types");
    void* ptrs[] = {(void*)&args...};
    SSD_CHECK_CUDA(cudaLaunchCooperativeKernel((const void*)kmn, dim3(B), dim3(MN_T), ptrs, smem_mn, st));
    count_launch();
    return 0;
}

// The walk over an image's gts in the mining kernel costs G x ~25 instructions per positive row, on the latency chain
// of the step's last kernel; the streaming kernel can record the best gt of every prior instead (2 bytes per row, +1 %
// of its traffic) and the walk disappears.  Measured at 1-10 gts per image: 112.4 -> 111.5 us per step at B=256 with the
// map, 671 -> 565 us at 100 gts per image - so the steps use the map whenever a gt index fits its 16 bits.
// The seeded cull of the fused match pays from a few dozen gts per image (the stress shape has 100); the ordinary
// batches (<= 10 gts per image) keep the plain loop.  SSDHEAD_MATCH_CULL_MIN overrides the average gt count it starts at.
static bool match_cull_enabled(int B, int sumG)
{
    const char* e = getenv("SSDHEAD_MATCH_CULL_MIN");          // read per call: a test compares the two paths in one process
    const int min_avg = e ? atoi(e) : 24;
    return B > 0 && sumG >= (long long)min_avg * B && sumG <= SEED_CAP;
}

static int check_xchg(const Xchg& x, bool seq_required)
{
    if (x.R < 1 || x.R > XCHG_MAX_R || x.rank < 0 || x.rank >= x.R || (seq_required && x.seq == 0u)) return SSDHEAD_E_BADARG;
    if (x.R > 1 && (!x.peers || !x.local || !x.err_flag)) return SSDHEAD_E_BADARG;
    return 0;
}

// What the mining kernel reads beyond the match; `flat`: the head tensors loc and conf (the per-level steps take a table).
// Their alignment is checked by the caller, where a batch of B = 0 has always been checked for it or not.
static int check_mine(const StepArgs& a, bool flat)
{
    if ((flat && (!a.loc || !a.conf)) || !a.pri_cxcywh || !a.sums || !a.losses || a.neg_ratio < 0) return SSDHEAD_E_BADARG;
    return 0;
}

// What every loss entry point needs: the sizes, the class count, the gradient pair and the loss workspace.  A batch of
// B = 0 passes before the alignment and workspace checks: it has nothing to do.
static int check_loss(int B, int P, int C, const float* grad_loc, const float* grad_conf, const void* ws, size_t ws_bytes)
{
    if (B < 0 || P <= 0 || !ws || (grad_loc == nullptr) != (grad_conf == nullptr)) return SSDHEAD_E_BADARG;
    if (C != 21) return SSDHEAD_E_UNSUPPORTED;          // VOC head of the reference (Losses.py:184 hard-codes 21)
    if (B == 0) return 0;
    if ((grad_loc && !aligned16(grad_loc)) || !aligned16(ws)) return SSDHEAD_E_ALIGN;
    const size_t need = loss_workspace_bytes(B, P, C);
    if (need == 0) return SSDHEAD_E_UNSUPPORTED;
    return ws_bytes < need ? SSDHEAD_E_WORKSPACE : 0;
}

// ... and what the fused match needs (every step)
static int check_match(const StepArgs& a)
{
    if (a.sumG < 0 || !a.gt_off || !a.pri_xyxy || !a.cls_u8 || !a.npos || !a.ws_match) return SSDHEAD_E_BADARG;
    if (a.sumG > 0 && (!a.gt_xyxy || !a.gt_cls || !a.best_prior)) return SSDHEAD_E_BADARG;
    const int rc = check_loss(a.B, a.P, a.C, a.grad_loc, a.grad_conf, a.ws_loss, a.ws_loss_bytes);
    if (rc || a.B == 0) return rc;
    if ((long long)a.B * a.P >= (1ll << 31)) return SSDHEAD_E_UNSUPPORTED;
    if (!aligned16(a.ws_match) || !aligned16(a.pri_xyxy) || (a.sumG > 0 && !aligned16(a.gt_xyxy))) return SSDHEAD_E_ALIGN;
    return a.ws_match_bytes < match_ws_bytes(a.B, a.sumG) ? SSDHEAD_E_WORKSPACE : 0;
}

static int check_resident(const StepArgs& a)
{
    if (!a.ws_rows || !a.grad_loc || !a.grad_conf || a.B < 0 || a.P <= 0 || a.P >= 65536) return SSDHEAD_E_BADARG;
    if (!aligned16(a.ws_rows) || !aligned16(a.grad_loc)) return SSDHEAD_E_ALIGN;
    if (a.ws_rows_bytes < resident_rows_bytes(a.B, a.P)) return SSDHEAD_E_WORKSPACE;
    return 0;
}

// The level table as the kernels index it: the levels partition the P priors, all or none of them carry gradients.
// With B = 0 only the table's size is checked: an empty batch may pass levels without tensors.
static int check_levels(const ssdhead_levels* levels, int B, int P, LevelTab* lv)
{
    if (!levels || levels->num_levels < 1 || levels->num_levels > MAX_LEVELS) return SSDHEAD_E_BADARG;
    if (B == 0) return 0;
    lv->n = levels->num_levels;
    int sum = 0, with_grads = 0;
    int t0 = 0;
    for (int l = 0; l < lv->n; ++l) {
        const int n = levels->count[l];
        if (n <= 0 || !levels->conf[l] || !levels->loc[l]) return SSDHEAD_E_BADARG;
        if (!aligned16(levels->loc[l])) return SSDHEAD_E_ALIGN;                        // float4 rows
        const bool g = levels->grad_conf[l] != nullptr;
        if (g != (levels->grad_loc[l] != nullptr)) return SSDHEAD_E_BADARG;
        if (g && !aligned16(levels->grad_loc[l])) return SSDHEAD_E_ALIGN;
        // conf / grad_conf rows are 84 bytes: a level whose pointers are not 16-byte aligned (e.g. a view into a larger
        // tensor) cannot ride the TMA pipeline and goes through the plain-load path entirely
        const bool tma_ok = aligned16(levels->conf[l]) && (!g || aligned16(levels->grad_conf[l]));
        with_grads += g ? 1 : 0;
        lv->cnt[l] = n; lv->start[l] = sum; lv->tile0[l] = t0;
        lv->conf[l] = levels->conf[l]; lv->loc[l] = levels->loc[l]; lv->gconf[l] = levels->grad_conf[l]; lv->gloc[l] = levels->grad_loc[l];
        sum += n;
        const long long rows_l = (long long)B * n;
        lv->rows[l] = (int)rows_l;
        // the partial last tile of a level rides the TMA pipeline too when its byte counts are multiples of 16
        if (tma_ok) t0 += (int)(rows_l / CE_ROWS) + ((rows_l % CE_ROWS) != 0 && (rows_l % 4) == 0 ? 1 : 0);
    }
    for (int l = lv->n; l <= MAX_LEVELS; ++l) { lv->start[l] = sum; lv->tile0[l] = t0; }
    if (sum != P) return SSDHEAD_E_BADARG;
    if (with_grads != 0 && with_grads != lv->n) return SSDHEAD_E_BADARG;
    return 0;
}

// The natural match that rides in the streaming kernel
static FusedMatch bind_match(const StepArgs& a, const MatchWs& mw, unsigned short* obj_u16, const float* seed_lb)
{
    FusedMatch fm = {};
    fm.gt_xyxy = (const float4*)a.gt_xyxy; fm.gt_cls = a.gt_cls; fm.gt_off = a.gt_off; fm.pri_xyxy = (const float4*)a.pri_xyxy;
    fm.P = a.P; fm.bg_class = a.C - 1; fm.pos_iou = a.pos_iou; fm.cls_u8 = a.cls_u8; fm.best_key = mw.best_key; fm.npos_acc = mw.npos_acc;
    fm.obj_u16 = obj_u16; fm.sumG = a.sumG; fm.seed_lb = seed_lb;
    return fm;
}

// The mining kernel's parameters; `mw` (the steps): the forced-match finaliser fused in, writing the match outputs
static MineParams bind_mine(const StepArgs& a, const LossWs& lw, const int32_t* npos_norm, const MatchWs* mw)
{
    MineParams prm = {};
    prm.loc = a.loc; prm.conf = a.conf; prm.cls_u8 = a.cls_u8;
    prm.gt_xyxy = (const float4*)a.gt_xyxy; prm.gt_cls = a.gt_cls; prm.gt_off = a.gt_off;
    prm.pri_xyxy = (const float4*)a.pri_xyxy; prm.pri_cxcywh = (const float4*)a.pri_cxcywh;
    prm.best_prior = a.best_prior; prm.npos = a.npos; prm.npos_norm = npos_norm;
    prm.B = a.B; prm.P = a.P; prm.neg_ratio = a.neg_ratio; prm.bg_class = a.C - 1; prm.pos_iou = a.pos_iou;
    prm.sums = a.sums; prm.losses = a.losses; prm.grad_loc = a.grad_loc; prm.grad_conf = a.grad_conf;
    prm.mined_mask = a.mined_mask;
    prm.done_counter = lw.done_counter;
    prm.partials = lw.partials;
    prm.ce = a.ce ? a.ce : lw.ce;
    prm.ce_tap = a.ce;
    if (mw) {
        prm.cls_rw = a.cls_u8; prm.best_prior_w = a.best_prior; prm.npos_w = a.npos;
        prm.best_key = mw->best_key; prm.npos_acc = mw->npos_acc; prm.arrive_total = mw->arrive_total;
    }
    return prm;
}

// The forced-match finaliser on its own: one CTA per image after the streaming kernel's natural match
static int launch_finalize(const StepArgs& a, const MatchWs& mw, cudaStream_t st)
{
    match_finalize_kernel<<<a.B, 64, 0, st>>>(a.gt_cls, a.gt_off, a.B, a.P, a.C - 1, a.best_prior, a.npos, a.cls_u8,
                                              mw.best_key, mw.npos_acc, mw.image_counter);
    SSD_LAUNCH_CHECK();
    count_launch();
    return 0;
}

// The mining kernel of a step, with the finaliser fused in; a batch that does not fit co-resident (B > 2 CTAs x SMs)
// gets the finaliser and the ordinary mining kernel instead, except a sharded one: its peer exchange needs the
// co-resident grid.
template <bool GRADS>
static int launch_mine_step(const StepArgs& a, const MineParams& prm, const LevelTab* lv, const MatchWs& mw, cudaStream_t st)
{
    int rc = lv ? launch_mine<true>(mine_levels_kernel<21, GRADS, true>, a.B, a.P, st, prm, *lv)
                : launch_mine<true>(mine_kernel<21, GRADS, true>, a.B, a.P, st, prm);
    if (rc != 1) return rc;
    if (prm.xchg.R > 1) return SSDHEAD_E_UNSUPPORTED;
    rc = launch_finalize(a, mw, st);
    if (rc) return rc;
    return lv ? launch_mine<false>(mine_levels_kernel<21, GRADS, false>, a.B, a.P, st, prm, *lv)
              : launch_mine<false>(mine_kernel<21, GRADS, false>, a.B, a.P, st, prm);
}

// The whole training-head step of one GPU in two kernels, on checked arguments with B > 0: the streaming CE kernel
// with the fused natural match over [B*P] rows (lv == nullptr) or the per-level tensors of lv, then the mining kernel
// with the forced-match finaliser fused in.  ws_rows: resident gradient tensors - the streaming kernel writes no zero
// background (it runs forward-only), the mining kernel retracts the previous step's rows and writes this step's.
static int step_impl(const StepArgs& a, const LevelTab* lv, const Xchg& x, void* ws_rows)
{
    cudaStream_t st = (cudaStream_t)a.stream;
    const LossWs lw = loss_ws(a.ws_loss, a.B, a.P);
    const MatchWs mw = match_ws(a.ws_match, a.B, a.sumG);
    unsigned short* obj = a.sumG <= 65535 ? lw.obj : nullptr;
    const FusedMatch fm = bind_match(a, mw, obj, !lv && match_cull_enabled(a.B, a.sumG) ? lw.seed : nullptr);
    MineParams prm = bind_mine(a, lw, a.npos + a.B, &mw);
    prm.obj_u16 = obj;
    prm.xchg = x;
    if (ws_rows) {
        prm.res_base = (unsigned char*)ws_rows;
        prm.res_stride = resident_row_stride(a.P);
    }
    if (lv) prm.ce_w = lw.ce;
    const bool grads = lv ? lv->gconf[0] != nullptr : a.grad_loc != nullptr;
    if (x.R > 1) {
        // a sharded batch has no three-kernel fallback (its peer exchange needs the co-resident grid): one that does not
        // fit is refused here, before the streaming kernel adds into the match workspace or writes any gradient
        bool fits = false;
        const int frc = lv ? (grads ? mine_fits_coresident(mine_levels_kernel<21, true, true>, a.B, a.P, &fits)
                                    : mine_fits_coresident(mine_levels_kernel<21, false, true>, a.B, a.P, &fits))
                           : (grads ? mine_fits_coresident(mine_kernel<21, true, true>, a.B, a.P, &fits)
                                    : mine_fits_coresident(mine_kernel<21, false, true>, a.B, a.P, &fits));
        if (frc) return frc;
        if (!fits) return SSDHEAD_E_UNSUPPORTED;
    }
    const bool ce_grads = grads && !ws_rows;
    const long long rows = (long long)a.B * a.P;
    float* ce = a.ce ? a.ce : lw.ce;
    int rc = ce_grads ? launch_ce_stream<21, true, true>(a.conf, ce, a.grad_conf, a.grad_loc, rows, fm, lv, st)
                      : launch_ce_stream<21, false, true>(a.conf, ce, nullptr, nullptr, rows, fm, lv, st);
    if (rc) return rc;
    if (a.mined_mask) SSD_CHECK_CUDA(cudaMemsetAsync(a.mined_mask, 0, (size_t)a.B * ((a.P + 31) / 32) * sizeof(uint32_t), st));
    return grads ? launch_mine_step<true>(a, prm, lv, mw, st) : launch_mine_step<false>(a, prm, lv, mw, st);
}

static int step_flat(const StepArgs& a, const Xchg& x, void* ws_rows)
{
    int rc = check_mine(a, true);
    if (!rc && (!aligned16(a.loc) || !aligned16(a.pri_cxcywh))) rc = SSDHEAD_E_ALIGN;
    if (!rc) rc = check_match(a);
    if (rc || a.B == 0) return rc;
    return step_impl(a, nullptr, x, ws_rows);
}

static int step_levels(const StepArgs& a, const Xchg& x)
{
    LevelTab lv = {};
    int rc = check_mine(a, false);
    if (!rc) rc = check_match(a);
    if (!rc) rc = check_levels(a.levels, a.B, a.P, &lv);
    if (rc || a.B == 0) return rc;
    if (!aligned16(a.pri_cxcywh)) return SSDHEAD_E_ALIGN;
    return step_impl(a, &lv, x, nullptr);
}

// A sharded step needs a sequence number; the resident step takes R = 1 with any as one GPU.
int run_step(StepKind kind, const StepArgs& a, const Xchg* x)
{
    const bool resident = kind == StepKind::resident;
    int rc = resident ? check_resident(a) : 0;
    if (!rc && x) rc = check_xchg(*x, !resident || x->R > 1);
    if (rc) return rc;
    const Xchg none = {};
    const Xchg& xr = x ? *x : none;
    return kind == StepKind::levels ? step_levels(a, xr) : step_flat(a, xr, resident ? a.ws_rows : nullptr);
}

}  // namespace ssdhead

using namespace ssdhead;

extern "C" {

int ssdhead_ce_stream(const float* conf, int B, int P, int C, float* ce, float* grad_loc, float* grad_conf,
                      void* ws, size_t ws_bytes, void* stream)
{
    if (!conf) return SSDHEAD_E_BADARG;
    const int rc = check_loss(B, P, C, grad_loc, grad_conf, ws, ws_bytes);
    if (rc || B == 0) return rc;
    float* ce_buf = ce ? ce : loss_ws(ws, B, P).ce;
    const long long rows = (long long)B * P;
    FusedMatch none = {};
    return grad_loc ? launch_ce_stream<21, true, false>(conf, ce_buf, grad_conf, grad_loc, rows, none, nullptr, (cudaStream_t)stream)
                    : launch_ce_stream<21, false, false>(conf, ce_buf, nullptr, nullptr, rows, none, nullptr, (cudaStream_t)stream);
}

// ssdhead_ce_stream with the natural match fused in, followed by the per-image forced-match finaliser: produces
// everything ssdhead_match produces for the loss (cls_u8, best_prior, npos) without a separate pass over the priors.
// It records no best-gt map: ssdhead_mine walks the gts.
int ssdhead_ce_match_stream(const float* conf, const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                            const float* pri_xyxy, int B, int P, int C, int sumG, float pos_iou,
                            float* ce, float* grad_loc, float* grad_conf,
                            uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                            void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes,
                            int run_finalizer, void* stream)
{
    const StepArgs a = {.conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off, .pri_xyxy = pri_xyxy,
                        .B = B, .P = P, .C = C, .sumG = sumG, .pos_iou = pos_iou, .grad_loc = grad_loc,
                        .grad_conf = grad_conf, .cls_u8 = cls_u8, .best_prior = best_prior, .npos = npos, .ce = ce,
                        .ws_loss = ws_loss, .ws_loss_bytes = ws_loss_bytes, .ws_match = ws_match,
                        .ws_match_bytes = ws_match_bytes, .stream = stream};
    if (!conf) return SSDHEAD_E_BADARG;
    int rc = check_match(a);
    if (rc || B == 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const LossWs lw = loss_ws(ws_loss, B, P);
    const MatchWs mw = match_ws(ws_match, B, sumG);
    const FusedMatch fm = bind_match(a, mw, nullptr, match_cull_enabled(B, sumG) ? lw.seed : nullptr);
    float* ce_buf = ce ? ce : lw.ce;
    const long long rows = (long long)B * P;
    rc = grad_loc ? launch_ce_stream<21, true, true>(conf, ce_buf, grad_conf, grad_loc, rows, fm, nullptr, st)
                  : launch_ce_stream<21, false, true>(conf, ce_buf, nullptr, nullptr, rows, fm, nullptr, st);
    if (rc || !run_finalizer) return rc;
    return launch_finalize(a, mw, st);
}

// The whole training-head step of ONE GPU in two kernels: the streaming CE kernel with the fused natural match,
// then the mining kernel with the forced-match finaliser fused in (cooperative launch).  When the batch does not fit
// co-resident (B > 2 CTAs x SMs) the finaliser and the ordinary mining kernel run separately (three kernels).
int ssdhead_multibox_step(const float* loc, const float* conf,
                          const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                          const float* pri_xyxy, const float* pri_cxcywh,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums, float* losses, float* grad_loc, float* grad_conf,
                          uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                          uint32_t* mined_mask, float* ce,
                          void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes, void* stream)
{
    return run_step(StepKind::flat,
                    {.loc = loc, .conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off,
                     .pri_xyxy = pri_xyxy, .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C, .sumG = sumG,
                     .neg_ratio = neg_ratio, .pos_iou = pos_iou, .sums = sums, .losses = losses,
                     .grad_loc = grad_loc, .grad_conf = grad_conf, .cls_u8 = cls_u8, .best_prior = best_prior,
                     .npos = npos, .mined_mask = mined_mask, .ce = ce, .ws_loss = ws_loss,
                     .ws_loss_bytes = ws_loss_bytes, .ws_match = ws_match, .ws_match_bytes = ws_match_bytes,
                     .stream = stream},
                    nullptr);
}

// The same two kernels for a batch sharded by image over R GPUs: the mining kernel exchanges the positive count (before
// it scales any gradient) and the two loss sums with its peers by storing into their exchange buffers over NVLink -
// no NCCL call, no extra kernel.  `peers_dev` is a device table of R peer-mapped exchange buffers (XCHG words each,
// zero-filled once), `seq` a step counter starting at 1 that every rank advances in lock step.
int ssdhead_multibox_step_sharded(const float* loc, const float* conf,
                          const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                          const float* pri_xyxy, const float* pri_cxcywh,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums, float* losses, float* grad_loc, float* grad_conf,
                          uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                          void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes,
                          int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev, int32_t* err_flag_dev,
                          void* stream)
{
    const Xchg x = {R, rank, seq, (unsigned long long* const*)peers_dev, (unsigned long long*)xchg_local_dev, err_flag_dev};
    return run_step(StepKind::flat,
                    {.loc = loc, .conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off,
                     .pri_xyxy = pri_xyxy, .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C, .sumG = sumG,
                     .neg_ratio = neg_ratio, .pos_iou = pos_iou, .sums = sums, .losses = losses,
                     .grad_loc = grad_loc, .grad_conf = grad_conf, .cls_u8 = cls_u8, .best_prior = best_prior,
                     .npos = npos, .ws_loss = ws_loss, .ws_loss_bytes = ws_loss_bytes, .ws_match = ws_match,
                     .ws_match_bytes = ws_match_bytes, .stream = stream},
                    &x);
}

// ssdhead_multibox_step with RESIDENT gradient tensors: grad_loc / grad_conf are all-zero when first handed over (together
// with a zero-filled rows workspace) and are then only ever written by this call.  The gradient of this loss is
// sparse (about 4 * Npos of the P rows of an image), so instead of writing 873 KB of zero background per image per step
// the step retracts the ~200 rows the previous step wrote and writes its own - the tensors hold exactly the dense
// gradient of this step afterwards (Losses.py:177-197 + autograd), bit-identical to ssdhead_multibox_step's.
// With R > 1 the batch is sharded as in ssdhead_multibox_step_sharded.
int ssdhead_multibox_step_resident(const float* loc, const float* conf,
                          const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                          const float* pri_xyxy, const float* pri_cxcywh,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums, float* losses, float* grad_loc, float* grad_conf,
                          uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                          void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes,
                          void* ws_rows, size_t ws_rows_bytes,
                          int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev, int32_t* err_flag_dev,
                          void* stream)
{
    const Xchg x = {R, rank, seq, (unsigned long long* const*)peers_dev, (unsigned long long*)xchg_local_dev, err_flag_dev};
    return run_step(StepKind::resident,
                    {.loc = loc, .conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off,
                     .pri_xyxy = pri_xyxy, .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C, .sumG = sumG,
                     .neg_ratio = neg_ratio, .pos_iou = pos_iou, .sums = sums, .losses = losses,
                     .grad_loc = grad_loc, .grad_conf = grad_conf, .cls_u8 = cls_u8, .best_prior = best_prior,
                     .npos = npos, .ws_loss = ws_loss, .ws_loss_bytes = ws_loss_bytes, .ws_match = ws_match,
                     .ws_match_bytes = ws_match_bytes, .ws_rows = ws_rows, .ws_rows_bytes = ws_rows_bytes,
                     .stream = stream},
                    &x);
}

// ssdhead_multibox_step on per-level head tensors (SURVEY.md 8(f) #3, Model.py:212-235 without the permute/cat copies)
int ssdhead_multibox_step_levels(const ssdhead_levels* levels,
                                 const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                                 const float* pri_xyxy, const float* pri_cxcywh,
                                 int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                                 double* sums, float* losses,
                                 uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                                 void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes, void* stream)
{
    return run_step(StepKind::levels,
                    {.levels = levels, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off, .pri_xyxy = pri_xyxy,
                     .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C, .sumG = sumG, .neg_ratio = neg_ratio,
                     .pos_iou = pos_iou, .sums = sums, .losses = losses, .cls_u8 = cls_u8,
                     .best_prior = best_prior, .npos = npos, .ws_loss = ws_loss, .ws_loss_bytes = ws_loss_bytes,
                     .ws_match = ws_match, .ws_match_bytes = ws_match_bytes, .stream = stream},
                    nullptr);
}

// the per-level step of a batch sharded by image over R GPUs (peer-memory exchange inside the mining kernel, as in
// ssdhead_multibox_step_sharded)
int ssdhead_multibox_step_levels_sharded(const ssdhead_levels* levels,
                                 const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                                 const float* pri_xyxy, const float* pri_cxcywh,
                                 int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                                 double* sums, float* losses,
                                 uint8_t* cls_u8, int32_t* best_prior, int32_t* npos,
                                 void* ws_loss, size_t ws_loss_bytes, void* ws_match, size_t ws_match_bytes,
                                 int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev, int32_t* err_flag_dev,
                                 void* stream)
{
    const Xchg x = {R, rank, seq, (unsigned long long* const*)peers_dev, (unsigned long long*)xchg_local_dev, err_flag_dev};
    return run_step(StepKind::levels,
                    {.levels = levels, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off, .pri_xyxy = pri_xyxy,
                     .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C, .sumG = sumG, .neg_ratio = neg_ratio,
                     .pos_iou = pos_iou, .sums = sums, .losses = losses, .cls_u8 = cls_u8,
                     .best_prior = best_prior, .npos = npos, .ws_loss = ws_loss, .ws_loss_bytes = ws_loss_bytes,
                     .ws_match = ws_match, .ws_match_bytes = ws_match_bytes, .stream = stream},
                    &x);
}

size_t ssdhead_xchg_bytes(void) { return (size_t)XCHG_WORDS * 8; }

// The mining kernel alone, on the match of an earlier call; sp_cnt != nullptr: the gradient returns as packed rows
static int mine_impl(const StepArgs& a, const int32_t* npos_norm,
                     int sp_cap, int32_t* sp_cnt, int32_t* sp_idx, float* sp_conf, float* sp_loc)
{
    if (!a.gt_off || !a.pri_xyxy || !a.npos || !npos_norm || !a.cls_u8) return SSDHEAD_E_BADARG;
    const bool sparse = sp_cnt != nullptr;
    if (sparse && (sp_cap <= 0 || !sp_idx || !sp_conf || !sp_loc || a.grad_loc)) return SSDHEAD_E_BADARG;
    int rc = check_mine(a, true);
    if (!rc) rc = check_loss(a.B, a.P, a.C, a.grad_loc, a.grad_conf, a.ws_loss, a.ws_loss_bytes);
    if (rc || a.B == 0) return rc;
    if (!aligned16(a.loc) || !aligned16(a.pri_xyxy) || !aligned16(a.pri_cxcywh) || (a.gt_xyxy && !aligned16(a.gt_xyxy)) ||
        (sparse && !aligned16(sp_loc)))
        return SSDHEAD_E_ALIGN;
    cudaStream_t st = (cudaStream_t)a.stream;
    MineParams prm = bind_mine(a, loss_ws(a.ws_loss, a.B, a.P), npos_norm, nullptr);
    prm.sp_cap = sp_cap; prm.sp_cnt = sp_cnt; prm.sp_idx = sp_idx; prm.sp_conf = sp_conf; prm.sp_loc = sp_loc;
    if (a.mined_mask) SSD_CHECK_CUDA(cudaMemsetAsync(a.mined_mask, 0, (size_t)a.B * ((a.P + 31) / 32) * sizeof(uint32_t), st));
    if (sparse) return launch_mine<false>(mine_sparse_kernel<21>, a.B, a.P, st, prm);
    return a.grad_loc ? launch_mine<false>(mine_kernel<21, true, false>, a.B, a.P, st, prm)
                      : launch_mine<false>(mine_kernel<21, false, false>, a.B, a.P, st, prm);
}

// (the match outputs in StepArgs are writable for the steps that produce them; the mining kernel only reads them)
int ssdhead_mine(const float* loc, const float* conf,
                 const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                 const float* pri_xyxy, const float* pri_cxcywh,
                 const int32_t* best_prior, const int32_t* npos, const int32_t* npos_norm, const uint8_t* cls_u8,
                 int B, int P, int C, int neg_ratio, float pos_iou,
                 double* sums, float* losses, float* grad_loc, float* grad_conf,
                 uint32_t* mined_mask, float* ce,
                 void* ws, size_t ws_bytes, void* stream)
{
    const StepArgs a = {.loc = loc, .conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off,
                        .pri_xyxy = pri_xyxy, .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C,
                        .neg_ratio = neg_ratio, .pos_iou = pos_iou, .sums = sums, .losses = losses,
                        .grad_loc = grad_loc, .grad_conf = grad_conf, .cls_u8 = const_cast<uint8_t*>(cls_u8),
                        .best_prior = const_cast<int32_t*>(best_prior), .npos = const_cast<int32_t*>(npos),
                        .mined_mask = mined_mask, .ce = ce, .ws_loss = ws, .ws_loss_bytes = ws_bytes,
                        .stream = stream};
    return mine_impl(a, npos_norm, 0, nullptr, nullptr, nullptr, nullptr);
}

int ssdhead_mine_sparse(const float* loc, const float* conf,
                 const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                 const float* pri_xyxy, const float* pri_cxcywh,
                 const int32_t* best_prior, const int32_t* npos, const int32_t* npos_norm, const uint8_t* cls_u8,
                 int B, int P, int C, int neg_ratio, float pos_iou,
                 double* sums, float* losses,
                 int row_cap, int32_t* row_cnt, int32_t* row_idx, float* grad_conf_rows, float* grad_loc_rows,
                 void* ws, size_t ws_bytes, void* stream)
{
    if (!row_cnt) return SSDHEAD_E_BADARG;
    const StepArgs a = {.loc = loc, .conf = conf, .gt_xyxy = gt_xyxy, .gt_cls = gt_cls, .gt_off = gt_off,
                        .pri_xyxy = pri_xyxy, .pri_cxcywh = pri_cxcywh, .B = B, .P = P, .C = C,
                        .neg_ratio = neg_ratio, .pos_iou = pos_iou, .sums = sums, .losses = losses,
                        .cls_u8 = const_cast<uint8_t*>(cls_u8), .best_prior = const_cast<int32_t*>(best_prior),
                        .npos = const_cast<int32_t*>(npos), .ws_loss = ws, .ws_loss_bytes = ws_bytes,
                        .stream = stream};
    return mine_impl(a, npos_norm, row_cap, row_cnt, row_idx, grad_conf_rows, grad_loc_rows);
}

int ssdhead_multibox_loss(const float* loc, const float* conf,
                          const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                          const float* pri_xyxy, const float* pri_cxcywh,
                          const int32_t* best_prior, const int32_t* npos, const int32_t* npos_norm, const uint8_t* cls_u8,
                          int B, int P, int C, int neg_ratio, float pos_iou,
                          double* sums, float* losses, float* grad_loc, float* grad_conf,
                          uint32_t* mined_mask, float* ce,
                          void* ws, size_t ws_bytes, void* stream)
{
    const int rc = ssdhead_ce_stream(conf, B, P, C, ce, grad_loc, grad_conf, ws, ws_bytes, stream);
    if (rc != 0) return rc;
    return ssdhead_mine(loc, conf, gt_xyxy, gt_cls, gt_off, pri_xyxy, pri_cxcywh, best_prior, npos, npos_norm, cls_u8,
                        B, P, C, neg_ratio, pos_iou, sums, losses, grad_loc, grad_conf, mined_mask, ce, ws, ws_bytes, stream);
}

int ssdhead_finish_loss(const double* sums, const int32_t* npos_norm, float* losses, void* stream)
{
    if (!sums || !npos_norm || !losses) return SSDHEAD_E_BADARG;
    finish_loss_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sums, npos_norm, losses);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

int ssdhead_scale_grads(float* grad_loc, size_t n_loc, float* grad_conf, size_t n_conf, const float* gout, void* stream)
{
    if (!grad_loc || !grad_conf || !gout) return SSDHEAD_E_BADARG;
    if (!aligned16(grad_loc) || !aligned16(grad_conf)) return SSDHEAD_E_ALIGN;
    const size_t n4l = n_loc / 4, n4c = n_conf / 4;
    scale_grads_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(
        (float4*)grad_loc, n4l, grad_loc + n4l * 4, (int)(n_loc - n4l * 4),
        (float4*)grad_conf, n4c, grad_conf + n4c * 4, (int)(n_conf - n4c * 4), gout);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

#ifdef SSDHEAD_PHASE_TIMES
int ssdhead_debug_phases_loss(long long* out16) { return (int)cudaMemcpyFromSymbol(out16, ssdhead::g_phase_loss, sizeof(long long) * 16); }
int ssdhead_debug_cta(long long* out, int n) { return (int)cudaMemcpyFromSymbol(out, ssdhead::g_cta, sizeof(long long) * 12 * n); }
int ssdhead_debug_gmarks(unsigned long long* out8, int reset) {
    int rc = (int)cudaMemcpyFromSymbol(out8, ssdhead::g_gt, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0ull, ~0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull}; rc |= (int)cudaMemcpyToSymbol(ssdhead::g_gt, z, sizeof(z)); }
    return rc;
}
#endif

}  // extern "C"
