// Matching of ground-truth boxes against the prior set, dense IoU, and the box-format /
// offset elementwise ops.  Reference: Losses.py:150-171, Util.py:57-63, 86-102, 252-265,
// 288-301, 333-352.
//
// match_kernel: grid (tiles, B), 256 threads, each thread owns 4 CONSECUTIVE priors (64 B of the
// L2-resident prior table).  The gt boxes of the image are staged in shared memory; each thread keeps
// the best gt of its priors (T1: first maximal gt) and, per gt, its own best prior (lowest index on
// ties); one redux.max + ballot per gt then gives the warp's best prior (T2), merged across warps and
// tiles with 64-bit atomicMax on (iou_key << 32 | ~prior).  Pairs that do not intersect skip the IEEE
// division (0/union == +0 exactly).  The last tile of an image to finish applies the forced-match
// override (T3: highest gt index wins) and publishes best_prior / npos[b]; the last image to finish
// publishes the batch total npos[B].  The workspace is left zeroed (self-cleaning): no memsets.
// HBM traffic is negligible (gt + priors in, one class byte per prior out); the kernel exists so the
// loss kernels know the class of every prior and the batch-global positive count.
#include <algorithm>
#include "common.cuh"

namespace ssdhead {

constexpr int MT = 256;          // threads per CTA
constexpr int MPPT = 4;          // consecutive priors per thread
constexpr int MTILE = MT * MPPT; // priors per CTA
constexpr int MGC = 64;          // gt boxes staged per chunk

__global__ void __launch_bounds__(MT, 5)
match_kernel(const float4* __restrict__ gt_xyxy, const float* __restrict__ gt_cls, const int* __restrict__ gt_off,
             const float4* __restrict__ pri_xyxy, int B, int P, int bg_class, float pos_iou,
             int* __restrict__ best_prior, int* __restrict__ npos, uint8_t* __restrict__ cls_u8,
             int* __restrict__ obj_idx, int* __restrict__ cls_out,
             unsigned long long* __restrict__ best_key, unsigned int* __restrict__ tile_counter,
             int* __restrict__ npos_acc, unsigned int* __restrict__ image_counter)
{
    __shared__ float4 s_box[MGC];
    __shared__ float s_area[MGC];
    __shared__ unsigned long long s_key[MGC];
    __shared__ int s_red[MT / 32];
    __shared__ int s_last;

    const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int off0 = gt_off[b];
    const int G = gt_off[b + 1] - off0;
    const int ntiles = (P + MTILE - 1) / MTILE;
    const bool one_chunk = G <= MGC;                 // the usual case: gts staged once, per-gt keys merged over the CTA's tiles
    int cnt = 0;

    if (one_chunk) {
        if (t < G) {
            const float4 bx = gt_xyxy[off0 + t];
            s_box[t] = bx;
            s_area[t] = box_area(bx);
            s_key[t] = 0ull;
        }
        __syncthreads();
    }

    // a CTA walks several tiles of its image so that the fixed latencies (gt fetch, fences, counters) are paid once
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int p0 = tile * MTILE + t * MPPT;      // first prior of this thread
        float4 pb[MPPT];
        float pa[MPPT], best[MPPT];
        int bestg[MPPT];
#pragma unroll
        for (int i = 0; i < MPPT; ++i) {
            pb[i] = (p0 + i < P) ? pri_xyxy[p0 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
            pa[i] = box_area(pb[i]);
            best[i] = 0.0f;        // IoU >= 0 and ties keep the first gt: starting at (0, gt 0) equals max() over the column
            bestg[i] = 0;
        }
        const bool first_warp = (tile == 0 && warp == 0);   // owns prior 0: the argmax of an all-zero IoU row (T2)
        // bounding box of the warp's 128 priors: a gt that misses it has IoU 0 with all of them (warp-uniform skip)
        float wx1 = fminf(fminf(pb[0].x, pb[1].x), fminf(pb[2].x, pb[3].x));
        float wy1 = fminf(fminf(pb[0].y, pb[1].y), fminf(pb[2].y, pb[3].y));
        float wx2 = fmaxf(fmaxf(pb[0].z, pb[1].z), fmaxf(pb[2].z, pb[3].z));
        float wy2 = fmaxf(fmaxf(pb[0].w, pb[1].w), fmaxf(pb[2].w, pb[3].w));
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            wx1 = fminf(wx1, __shfl_xor_sync(FULL, wx1, d));
            wy1 = fminf(wy1, __shfl_xor_sync(FULL, wy1, d));
            wx2 = fmaxf(wx2, __shfl_xor_sync(FULL, wx2, d));
            wy2 = fmaxf(wy2, __shfl_xor_sync(FULL, wy2, d));
        }

        for (int g0 = 0; g0 < G; g0 += MGC) {
            const int gc = min(MGC, G - g0);
            if (!one_chunk) {
                __syncthreads();
                if (t < gc) {
                    const float4 bx = gt_xyxy[off0 + g0 + t];
                    s_box[t] = bx;
                    s_area[t] = box_area(bx);
                    s_key[t] = 0ull;
                }
                __syncthreads();
            }
            for (int g = 0; g < gc; ++g) {
                const float4 gb = s_box[g];
                const float ga = s_area[g];
                float tv = 0.0f;       // this thread's best IoU for gt g (IoU >= 0), lowest prior on ties
                int ti = 0;
                const bool near = (gb.z > wx1) && (gb.x < wx2) && (gb.w > wy1) && (gb.y < wy2);
                if (!near && !first_warp) continue;
                if (near) {
#pragma unroll
                    for (int i = 0; i < MPPT; ++i) {
                        // disjoint boxes (the common case) have IoU == +0 exactly: no multiply, no IEEE division
                        const float dx = __fsub_rn(fminf(gb.z, pb[i].z), fmaxf(gb.x, pb[i].x));
                        const float dy = __fsub_rn(fminf(gb.w, pb[i].w), fmaxf(gb.y, pb[i].y));
                        if (dx > 0.0f && dy > 0.0f) {
                            const float inter = __fmul_rn(dx, dy);
                            const float v = __fdiv_rn(inter, __fsub_rn(__fadd_rn(ga, pa[i]), inter));
                            if (v > best[i]) { best[i] = v; bestg[i] = g0 + g; }  // T1: strict > keeps the first gt
                            if (v > tv) { tv = v; ti = i; }                       // strict > keeps the lower prior
                        }
                    }
                }
                const uint32_t m = __reduce_max_sync(FULL, __float_as_uint(tv));  // IoU >= 0: bits order like values
                if (m != 0u || first_warp) {                                      // some IoU > 0, or the warp owning prior 0
                    const unsigned ball = __ballot_sync(FULL, __float_as_uint(tv) == m);
                    const int src = __ffs(ball) - 1;                              // T2: lowest lane = lowest prior
                    const int wi = __shfl_sync(FULL, ti, src);
                    if (lane == 0) {
                        const uint32_t wprior = (uint32_t)(tile * MTILE + (warp * 32 + src) * MPPT + wi);
                        atomicMax(&s_key[g], ((unsigned long long)(m | 0x80000000u) << 32) | (unsigned long long)(0xffffffffu - wprior));
                    }
                }
            }
            if (!one_chunk) {
                __syncthreads();
                if (t < gc && s_key[t] != 0ull) atomicMax(&best_key[off0 + g0 + t], s_key[t]);
            }
        }

        // natural (pre-override) match of this tile: one class byte per prior
        uint32_t packed = 0u;
#pragma unroll
        for (int i = 0; i < MPPT; ++i) {
            const int p = p0 + i;
            const bool hit = (G > 0) && !(best[i] < pos_iou);                   // T6: matched <=> not (iou < thr)
            const int c = (hit && p < P) ? (int)gt_cls[off0 + bestg[i]] : bg_class;
            packed |= (uint32_t)(c & 0xff) << (8 * i);
            if (p < P) {
                cnt += (c != bg_class) ? 1 : 0;                                 // positive <=> class != bg (Losses.py:179)
                if (obj_idx) obj_idx[(size_t)b * P + p] = off0 + bestg[i];
                if (cls_out) cls_out[(size_t)b * P + p] = c;
            }
        }
        uint8_t* dst = cls_u8 + (size_t)b * P + p0;
        if (p0 + MPPT <= P && ((reinterpret_cast<uintptr_t>(dst) & 3u) == 0)) {
            *reinterpret_cast<uint32_t*>(dst) = packed;
        } else {
#pragma unroll
            for (int i = 0; i < MPPT; ++i) if (p0 + i < P) dst[i] = (uint8_t)(packed >> (8 * i));
        }
    }
    if (one_chunk) {
        __syncthreads();
        if (t < G && s_key[t] != 0ull) atomicMax(&best_key[off0 + t], s_key[t]);
    }

    cnt = warp_sum(cnt);
    if (lane == 0) s_red[warp] = cnt;
    __syncthreads();
    if (t == 0) {
        int c = 0;
        for (int w = 0; w < MT / 32; ++w) c += s_red[w];
        if (c) atomicAdd(&npos_acc[b], c);
        __threadfence();
        const unsigned done = atomicAdd(&tile_counter[b], 1u);
        s_last = (done == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();

    // ---- last tile of image b: forced-match override (Losses.py:164-167) ----
    int extra = 0;
    if (one_chunk) {
        // all gts of the image are still staged in s_box / s_area: one round of loads, then shared memory only
        uint32_t* s_bp = reinterpret_cast<uint32_t*>(s_key);                    // reuse: best prior per gt
        uint32_t p = 0u;
        if (t < G) {
            p = 0xffffffffu - (uint32_t)(ld_relaxed_gpu_u64(&best_key[off0 + t]) & 0xffffffffull);
            best_key[off0 + t] = 0ull;                                          // leave the workspace zeroed
            best_prior[off0 + t] = (int)p;
        }
        __syncthreads();
        if (t < G) s_bp[t] = p;
        __syncthreads();
        if (t < G) {
            bool winner = true;                                                 // T3: the highest gt index keeps the prior
            for (int g2 = t + 1; g2 < G; ++g2) winner = winner && (s_bp[g2] != p);
            if (winner) {
                const float4 pbx = pri_xyxy[p];
                const float pax = box_area(pbx);
                float nb = 0.0f;
                int ng = 0;
                for (int g2 = 0; g2 < G; ++g2) {
                    const float v = iou_sparse(s_box[g2], s_area[g2], pbx, pax);
                    if (v > nb) { nb = v; ng = g2; }
                }
                const int c_nat = !(nb < pos_iou) ? (int)gt_cls[off0 + ng] : bg_class;   // what the tile pass counted
                const int c_new = (int)gt_cls[off0 + t];
                extra = (c_new != bg_class ? 1 : 0) - (c_nat != bg_class ? 1 : 0);
                cls_u8[(size_t)b * P + p] = (uint8_t)c_new;
                if (obj_idx) obj_idx[(size_t)b * P + p] = off0 + t;
                if (cls_out) cls_out[(size_t)b * P + p] = c_new;
            }
        }
    } else {
        for (int g = t; g < G; g += MT) {
            const uint32_t p = 0xffffffffu - (uint32_t)(ld_relaxed_gpu_u64(&best_key[off0 + g]) & 0xffffffffull);
            best_prior[off0 + g] = (int)p;
            bool winner = true;
            for (int g2 = g + 1; g2 < G; ++g2) {
                const uint32_t p2 = 0xffffffffu - (uint32_t)(ld_relaxed_gpu_u64(&best_key[off0 + g2]) & 0xffffffffull);
                if (p2 == p) { winner = false; break; }
            }
            if (!winner) continue;
            const float4 pbx = pri_xyxy[p];
            const float pax = box_area(pbx);
            float nb = 0.0f;
            int ng = 0;
            for (int g2 = 0; g2 < G; ++g2) {
                const float4 gb = gt_xyxy[off0 + g2];
                const float v = iou_sparse(gb, box_area(gb), pbx, pax);
                if (v > nb) { nb = v; ng = g2; }
            }
            const int c_nat = !(nb < pos_iou) ? (int)gt_cls[off0 + ng] : bg_class;
            const int c_new = (int)gt_cls[off0 + g];
            extra += (c_new != bg_class ? 1 : 0) - (c_nat != bg_class ? 1 : 0);
            cls_u8[(size_t)b * P + p] = (uint8_t)c_new;
            if (obj_idx) obj_idx[(size_t)b * P + p] = off0 + g;
            if (cls_out) cls_out[(size_t)b * P + p] = c_new;
        }
        __syncthreads();                                                        // every best_key read above is done
        for (int g = t; g < G; g += MT) best_key[off0 + g] = 0ull;              // leave the workspace zeroed
    }
    extra = warp_sum(extra);
    __syncthreads();
    if (lane == 0) s_red[warp] = extra;
    __syncthreads();
    if (t == 0) {
        int e = 0;
        for (int w = 0; w < MT / 32; ++w) e += s_red[w];
        npos[b] = ld_relaxed_gpu_s32(&npos_acc[b]) + e;
        npos_acc[b] = 0;
        tile_counter[b] = 0u;
        __threadfence();
        const unsigned done = atomicAdd(image_counter, 1u);
        if (done == gridDim.y - 1) {                                            // last image: batch total, fixed order
            __threadfence();
            int tot = 0;
            for (int i = 0; i < B; ++i) tot += ld_relaxed_gpu_s32(&npos[i]);
            npos[B] = tot;
            *image_counter = 0u;
        }
    }
}

// ------------------------------------------------------------------------------- dense IoU
template <bool INTERSECTION_ONLY>
__global__ void __launch_bounds__(256)
iou_matrix_kernel(const float4* __restrict__ a, int n1, const float4* __restrict__ bxs, int n2, float* __restrict__ out)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = blockIdx.y * 8;
    if (j >= n2) return;
    const float4 pb = bxs[j];
    const float pa = box_area(pb);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int i = i0 + r;
        if (i >= n1) break;
        const float4 gb = a[i];
        if (INTERSECTION_ONLY) {                                  // find_intersection, Util.py:252-265
            const float dx = fmaxf(__fsub_rn(fminf(gb.z, pb.z), fmaxf(gb.x, pb.x)), 0.0f);
            const float dy = fmaxf(__fsub_rn(fminf(gb.w, pb.w), fmaxf(gb.y, pb.y)), 0.0f);
            out[(size_t)i * n2 + j] = __fmul_rn(dx, dy);
        } else {
            out[(size_t)i * n2 + j] = iou_xyxy(gb, box_area(gb), pb, pa);
        }
    }
}

// ------------------------------------------------------------------------------- match from a given IoU matrix
// map_prior_to_bb (Util.py:333-352): the legacy single-image entry takes the [G,P] jaccard matrix itself.
__global__ void __launch_bounds__(256)
match_iou_cols_kernel(const float* __restrict__ jacc, int G, int P, float* __restrict__ overlap, long long* __restrict__ obj)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    float best = jacc[p];
    int bg = 0;
    for (int g = 1; g < G; ++g) {
        const float v = jacc[(size_t)g * P + p];
        if (v > best) { best = v; bg = g; }                       // T1: first maximal gt
    }
    overlap[p] = best;
    obj[p] = bg;
}

__global__ void __launch_bounds__(256)
match_iou_rows_kernel(const float* __restrict__ jacc, int G, int P, int* __restrict__ best_prior)
{
    __shared__ unsigned long long s_best;
    const int g = blockIdx.x, t = threadIdx.x;
    if (t == 0) s_best = 0ull;
    __syncthreads();
    unsigned long long mine = 0ull;
    for (int p = t; p < P; p += blockDim.x) {
        const unsigned long long k = ((unsigned long long)float_order_key(jacc[(size_t)g * P + p]) << 32) |
                                     (unsigned long long)(0xffffffffu - (unsigned)p);
        mine = max(mine, k);                                      // T2: lowest prior index on ties
    }
    atomicMax(&s_best, mine);
    __syncthreads();
    if (t == 0) best_prior[g] = (int)(0xffffffffu - (unsigned)(s_best & 0xffffffffull));
}

__global__ void match_iou_finish_kernel(const float* __restrict__ classes, const int* __restrict__ best_prior, int G, int P,
                                        float thr, float bg_class, float* __restrict__ overlap, long long* __restrict__ obj,
                                        float* __restrict__ cls_out)
{
    // forced override, sequential over gts so the last write wins (T3), then classes and the threshold
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int g = 0; g < G; ++g) { obj[best_prior[g]] = g; overlap[best_prior[g]] = 1.0f; }
    }
    __threadfence();
    __syncthreads();
    if (blockIdx.x != 0) return;
    for (int p = threadIdx.x; p < P; p += blockDim.x)
        cls_out[p] = (overlap[p] < thr) ? bg_class : classes[obj[p]];
}

// ------------------------------------------------------------------------------- elementwise box ops
template <int OP>
__global__ void __launch_bounds__(256)
box_op_kernel(const float4* __restrict__ in, const float4* __restrict__ pri, float4* __restrict__ out, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 v = in[i];
    float4 r;
    if (OP == 0) r = cxcywh_to_xyxy(v);
    else if (OP == 1) r = xyxy_to_cxcywh(v);
    else if (OP == 2) r = encode_box(v, pri[i]);
    else r = decode_box(v, pri[i]);
    out[i] = r;
}

template <int OP>
static int launch_box_op(const float* in, const float* pri, float* out, int n, void* stream)
{
    if (n < 0 || (n > 0 && (!in || !out || (OP >= 2 && !pri)))) return SSDHEAD_E_BADARG;
    if (n == 0) return 0;
    if (!aligned16(in) || !aligned16(out) || (OP >= 2 && !aligned16(pri))) return SSDHEAD_E_ALIGN;
    box_op_kernel<OP><<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        (const float4*)in, (const float4*)pri, (float4*)out, n);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

}  // namespace ssdhead

using namespace ssdhead;

extern "C" {

int ssdhead_cxcywh_to_xyxy(const float* in, float* out, int n, void* stream) { return launch_box_op<0>(in, nullptr, out, n, stream); }
int ssdhead_xyxy_to_cxcywh(const float* in, float* out, int n, void* stream) { return launch_box_op<1>(in, nullptr, out, n, stream); }
int ssdhead_encode(const float* c, const float* p, float* out, int n, void* stream) { return launch_box_op<2>(c, p, out, n, stream); }
int ssdhead_decode(const float* g, const float* p, float* out, int n, void* stream) { return launch_box_op<3>(g, p, out, n, stream); }

int ssdhead_iou_matrix(const float* a, int n1, const float* b, int n2, float* out, void* stream)
{
    if (n1 < 0 || n2 < 0) return SSDHEAD_E_BADARG;
    if (n1 == 0 || n2 == 0) return 0;
    if (!a || !b || !out) return SSDHEAD_E_BADARG;
    if (!aligned16(a) || !aligned16(b)) return SSDHEAD_E_ALIGN;
    dim3 grid((n2 + 255) / 256, (n1 + 7) / 8);
    if (grid.y > 65535) return SSDHEAD_E_UNSUPPORTED;
    iou_matrix_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)a, n1, (const float4*)b, n2, out);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

int ssdhead_intersection_matrix(const float* a, int n1, const float* b, int n2, float* out, void* stream)
{
    if (n1 < 0 || n2 < 0) return SSDHEAD_E_BADARG;
    if (n1 == 0 || n2 == 0) return 0;
    if (!a || !b || !out) return SSDHEAD_E_BADARG;
    if (!aligned16(a) || !aligned16(b)) return SSDHEAD_E_ALIGN;
    dim3 grid((n2 + 255) / 256, (n1 + 7) / 8);
    if (grid.y > 65535) return SSDHEAD_E_UNSUPPORTED;
    iou_matrix_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)a, n1, (const float4*)b, n2, out);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

int ssdhead_match_from_iou(const float* jacc, const float* classes, int G, int P, float thr, int bg_class,
                           float* cls_out, long long* obj_out, float* overlap_ws, int32_t* best_prior_ws, void* stream)
{
    if (G <= 0 || P <= 0 || !jacc || !classes || !cls_out || !obj_out || !overlap_ws || !best_prior_ws) return SSDHEAD_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    match_iou_cols_kernel<<<(P + 255) / 256, 256, 0, st>>>(jacc, G, P, overlap_ws, obj_out);
    match_iou_rows_kernel<<<G, 256, 0, st>>>(jacc, G, P, best_prior_ws);
    match_iou_finish_kernel<<<1, 256, 0, st>>>(classes, best_prior_ws, G, P, thr, (float)bg_class, overlap_ws, obj_out, cls_out);
    count_launch(3);
    SSD_LAUNCH_CHECK();
    return 0;
}

int ssdhead_match(const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off, const float* pri_xyxy,
                  int B, int P, int C, int sumG, float pos_iou,
                  int32_t* best_prior, int32_t* npos, uint8_t* cls_u8, int32_t* obj_idx, int32_t* cls,
                  void* ws, size_t ws_bytes, void* stream)
{
    if (B < 0 || P <= 0 || C < 2 || C > 256 || sumG < 0) return SSDHEAD_E_BADARG;
    if (B == 0) return 0;
    if (!gt_off || !pri_xyxy || !npos || !cls_u8 || !ws) return SSDHEAD_E_BADARG;
    if (sumG > 0 && (!gt_xyxy || !gt_cls || !best_prior)) return SSDHEAD_E_BADARG;
    if (B > 65535) return SSDHEAD_E_UNSUPPORTED;
    if (!aligned16(pri_xyxy) || (sumG > 0 && !aligned16(gt_xyxy)) || !aligned16(ws)) return SSDHEAD_E_ALIGN;
    if (ws_bytes < match_ws_bytes(B, sumG)) return SSDHEAD_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const MatchWs mw = match_ws(ws, B, sumG);
    // enough CTAs per image to fill the machine about once (5 CTAs/SM), never more than the image has tiles
    const int ntiles = (P + MTILE - 1) / MTILE;
    const int per_image = std::max(1, std::min(ntiles, (5 * 148) / B));
    dim3 grid(per_image, B);
    match_kernel<<<grid, MT, 0, st>>>((const float4*)gt_xyxy, gt_cls, gt_off, (const float4*)pri_xyxy, B, P, C - 1, pos_iou,
                                      best_prior, npos, cls_u8, obj_idx, cls, mw.best_key, mw.tile_counter, mw.npos_acc, mw.image_counter);
    count_launch();
    SSD_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
