// Shared device helpers for libssdhead (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include "../../include/ssdhead.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libssdhead is written for sm_100a (B200) only"
#endif

namespace ssdhead {

extern unsigned long long g_launch_count;   // host-side counter of kernel launches (api.cu)
inline void count_launch(int n = 1) { g_launch_count += (unsigned long long)n; }

#define SSD_CHECK_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return (int)_e; } while (0)
#define SSD_LAUNCH_CHECK() do { cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) return (int)_e; } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr unsigned FULL = 0xffffffffu;

// ---------------------------------------------------------------------------------------------
// Box arithmetic.  Only IEEE + - * / min max, in the reference's operation order
// (Util.py:262-265, 294-301), written with _rn intrinsics so nothing is contracted into an FMA:
// the IoU is then bit-identical to the torch-CPU value and every index derived from it is exact.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float box_area(const float4 b) {
    return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}

__device__ __forceinline__ float iou_xyxy(const float4 a, const float area_a, const float4 b, const float area_b) {
    const float lx = fmaxf(a.x, b.x), ly = fmaxf(a.y, b.y);
    const float hx = fminf(a.z, b.z), hy = fminf(a.w, b.w);
    const float dx = fmaxf(__fsub_rn(hx, lx), 0.0f);
    const float dy = fmaxf(__fsub_rn(hy, ly), 0.0f);
    const float inter = __fmul_rn(dx, dy);
    const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
    return __fdiv_rn(inter, uni);
}

// IoU with the division skipped for disjoint boxes: inter == +0 -> 0/union == +0 for any union > 0
// (priors have positive area, so union > 0 whenever the gt area is not negative).
__device__ __forceinline__ float iou_sparse(const float4 a, const float area_a, const float4 b, const float area_b) {
    const float lx = fmaxf(a.x, b.x), ly = fmaxf(a.y, b.y);
    const float hx = fminf(a.z, b.z), hy = fminf(a.w, b.w);
    const float dx = fmaxf(__fsub_rn(hx, lx), 0.0f);
    const float dy = fmaxf(__fsub_rn(hy, ly), 0.0f);
    const float inter = __fmul_rn(dx, dy);
    if (inter == 0.0f && area_a >= 0.0f) return 0.0f;
    return __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
}

// Util.py:93-96
__device__ __forceinline__ float4 cxcywh_to_xyxy(const float4 b) {
    const float hw = __fdiv_rn(b.z, 2.0f), hh = __fdiv_rn(b.w, 2.0f);
    return make_float4(__fsub_rn(b.x, hw), __fsub_rn(b.y, hh), __fadd_rn(b.x, hw), __fadd_rn(b.y, hh));
}
// Util.py:57-63
__device__ __forceinline__ float4 xyxy_to_cxcywh(const float4 b) {
    return make_float4(__fdiv_rn(__fadd_rn(b.z, b.x), 2.0f), __fdiv_rn(__fadd_rn(b.w, b.y), 2.0f),
                       __fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}
// Util.py:98-102: (c - pc) / (pwh / 10), log(wh / pwh) * 5
__device__ __forceinline__ float4 encode_box(const float4 c, const float4 p) {
    return make_float4(__fdiv_rn(__fsub_rn(c.x, p.x), __fdiv_rn(p.z, 10.0f)),
                       __fdiv_rn(__fsub_rn(c.y, p.y), __fdiv_rn(p.w, 10.0f)),
                       __fmul_rn(logf(__fdiv_rn(c.z, p.z)), 5.0f),
                       __fmul_rn(logf(__fdiv_rn(c.w, p.w)), 5.0f));
}
// Util.py:86-91: g * pwh / 10 + pc, exp(g / 5) * pwh
__device__ __forceinline__ float4 decode_box(const float4 g, const float4 p) {
    return make_float4(__fadd_rn(__fdiv_rn(__fmul_rn(g.x, p.z), 10.0f), p.x),
                       __fadd_rn(__fdiv_rn(__fmul_rn(g.y, p.w), 10.0f), p.y),
                       __fmul_rn(expf(__fdiv_rn(g.z, 5.0f)), p.z),
                       __fmul_rn(expf(__fdiv_rn(g.w, 5.0f)), p.w));
}

// exp(d) through one ex2.approx.ftz (no denormal pre-scaling: results below 2^-126 flush to zero, which no caller can
// tell from a denormal).  Same value as __expf(d) everywhere else; relative error <= (2 + 1.16|d|) ulp.
__device__ __forceinline__ float fast_exp_ftz(float d) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fmul_rn(d, 1.4426950408889634f)));
    return r;
}

// Order-preserving map float -> uint32 (total order of the reals; -0 and +0 collapse).
__device__ __forceinline__ uint32_t float_order_key(float f) {
    f = __fadd_rn(f, 0.0f);                      // -0.0 -> +0.0
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + 1-D bulk async copies (TMA engine, SASS UBLKCP) + proxy fences.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy, completion signalled on an mbarrier (bytes % 16 == 0, 16B-aligned both sides)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global bulk copy (bulk_group completion)
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// order generic-proxy shared-memory writes before async-proxy (TMA) reads
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ uint64_t ld_cg_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// Polling load: ld.cg may keep hitting a stale copy of the line in the SM's near L2 partition when the data was written
// with a plain store from the other die (observed on B200: a poll that never saw the store); a relaxed gpu-scope load is
// coherent at the point the writer's store becomes visible.
__device__ __forceinline__ uint64_t ld_relaxed_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_relaxed_gpu_s32(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned short ld_cg_u16(const unsigned short* p) {
    unsigned short v;
    asm volatile("ld.global.cg.u16 %0, [%1];" : "=h"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ld_cg_v4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_cg_s32(const int* p) {
    int v;
    asm volatile("ld.global.cg.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Programmatic dependent launch (PDL): a kernel launched with launch_pdl() may become resident while its predecessor
// in the stream is still running; it must call pdl_wait() before touching anything the predecessor produces (or
// anything the predecessor still reads, before overwriting it).  pdl_trigger() lets the NEXT kernel start early.
// Both are no-ops for a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// COOP: also a cooperative launch (every CTA co-resident).
template <bool COOP = false, typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeCooperative;
    attr[1].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = COOP ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Workspace of the match (ssdhead_match, and the match fused into the loss steps), zero on entry and on exit:
// best_key u64[sumG] | tile_counter u32[B] | npos_acc i32[B] | image_counter u32, and in the same 16-byte tail the
// u64 arrive_total of the mining kernel's fused finaliser.
struct MatchWs {
    unsigned long long* best_key;
    unsigned int* tile_counter;
    int* npos_acc;
    unsigned int* image_counter;
    unsigned long long* arrive_total;
};
static inline MatchWs match_ws(void* ws, int B, int sumG)
{
    uintptr_t w = (uintptr_t)ws;
    MatchWs m;
    m.best_key = (unsigned long long*)w;          w += round_up((size_t)sumG * 8, 16);
    m.tile_counter = (unsigned int*)w;            w += round_up((size_t)B * 4, 16);
    m.npos_acc = (int*)w;                         w += round_up((size_t)B * 4, 16);
    m.image_counter = (unsigned int*)w;
    m.arrive_total = (unsigned long long*)(w + 8);
    return m;
}
static inline size_t match_ws_bytes(int B, int sumG) { return (uintptr_t)match_ws(nullptr, B, sumG).image_counter + 16; }

// system-scope accesses for the cross-GPU exchange over NVLink peer memory (sharded batches)
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// Cross-GPU exchange buffer of a sharded batch: every rank owns XCHG_WORDS 64-bit words that its PEERS write into over
// NVLink (and it polls locally).  Slots are double-buffered by the parity of the step sequence number.
constexpr int XCHG_MAX_R = 16;
constexpr int XCHG_WORDS = 2 * 4 * XCHG_MAX_R;     // parity x {npos, sum_l1, sum_ce, sums_flag} x rank
__host__ __device__ __forceinline__ int xchg_slot(unsigned seq, int what, int rank) { return ((int)(seq & 1u) * 4 + what) * XCHG_MAX_R + rank; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

}  // namespace ssdhead
