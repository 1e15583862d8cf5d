// Context front end: owns streams, events, device buffers and workspaces so that one C call runs a
// whole step - either on device-resident tensors (fork/join of the match beside the CE stream kernel)
// or on HOST buffers, with the copies pipelined against the kernels in image chunks.
// Reference call sites: ssd() train_function.py:82 (loss), inference() Losses.py:11-98 (detect).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#ifdef __linux__
#include <sched.h>
#endif
#include "common.cuh"

using namespace ssdhead;

namespace ssdhead {
size_t loss_ws_header_bytes(int maxB);     // loss.cu

// Util.py:93-96 on the host for the one-off prior table (same fp32 operations as the device helper)
static void priors_xyxy_host(const float* cxcywh, float* xyxy, int P)
{
    for (int i = 0; i < P; ++i) {
        const float cx = cxcywh[4 * i], cy = cxcywh[4 * i + 1];
        const volatile float hw = cxcywh[4 * i + 2] / 2.0f, hh = cxcywh[4 * i + 3] / 2.0f;
        xyxy[4 * i] = cx - hw; xyxy[4 * i + 1] = cy - hh; xyxy[4 * i + 2] = cx + hw; xyxy[4 * i + 3] = cy + hh;
    }
}
__global__ void sum_chunks_kernel(const double* __restrict__ chunk_sums, int nchunks, const int* __restrict__ npos_norm,
                                  double* __restrict__ sums, float* __restrict__ losses)
{
    double a = 0.0, c = 0.0;
    for (int i = 0; i < nchunks; ++i) { a += chunk_sums[2 * i]; c += chunk_sums[2 * i + 1]; }
    sums[0] = a; sums[1] = c;
    const double N = (double)(*npos_norm);
    losses[0] = (float)(a / (4.0 * N));
    losses[1] = (float)(c / N);
}

// Sharded batches through the host-buffer entry points: the same exchange buffers the fused mining kernel uses
// (common.cuh), driven by two single-thread kernels.  xchg_npos_kernel: this rank's positive count goes to every rank,
// the global count comes back - before any chunk is mined (it scales the gradients, Losses.py:182,197).
struct XchgArgs {
    int R, rank;
    unsigned int seq;
    unsigned long long* const* peers;
    unsigned long long* local;
    int* err_flag;
};
__global__ void xchg_npos_kernel(const int* __restrict__ npos_local, int* __restrict__ npos_global, const XchgArgs x)
{
    const unsigned long long word = ((unsigned long long)x.seq << 32) | (unsigned)(*npos_local);
    for (int q = 0; q < x.R; ++q) st_relaxed_sys_u64(x.peers[q] + xchg_slot(x.seq, 0, x.rank), word);   // self-validating word
    unsigned spins = 0;
    int tot = 0;
    for (int q = 0; q < x.R; ++q) {
        unsigned long long w;
        while ((unsigned)((w = ld_acquire_sys_u64(x.local + xchg_slot(x.seq, 0, q))) >> 32) != x.seq && ++spins < (1u << 27)) __nanosleep(64);
        tot += (int)(unsigned)w;
    }
    if (spins >= (1u << 27)) *x.err_flag = 1;
    *npos_global = tot;
}
// The chunk sums of this rank -> global sums (added in rank order on every rank: identical bits everywhere) -> losses.
__global__ void sum_chunks_xchg_kernel(const double* __restrict__ chunk_sums, int nchunks, const int* __restrict__ npos_norm,
                                       double* __restrict__ sums, float* __restrict__ losses, const XchgArgs x)
{
    double a = 0.0, c = 0.0;
    for (int i = 0; i < nchunks; ++i) { a += chunk_sums[2 * i]; c += chunk_sums[2 * i + 1]; }
    for (int q = 0; q < x.R; ++q) {
        st_relaxed_sys_u64(x.peers[q] + xchg_slot(x.seq, 1, x.rank), (unsigned long long)__double_as_longlong(a));
        st_relaxed_sys_u64(x.peers[q] + xchg_slot(x.seq, 2, x.rank), (unsigned long long)__double_as_longlong(c));
    }
    __threadfence_system();                      // values before flags
    for (int q = 0; q < x.R; ++q) st_relaxed_sys_u64(x.peers[q] + xchg_slot(x.seq, 3, x.rank), (unsigned long long)x.seq);
    unsigned spins = 0;
    a = 0.0; c = 0.0;
    for (int q = 0; q < x.R; ++q) {
        while ((unsigned)ld_acquire_sys_u64(x.local + xchg_slot(x.seq, 3, q)) != x.seq && ++spins < (1u << 27)) __nanosleep(64);
        a += __longlong_as_double((long long)ld_relaxed_sys_u64(x.local + xchg_slot(x.seq, 1, q)));
        c += __longlong_as_double((long long)ld_relaxed_sys_u64(x.local + xchg_slot(x.seq, 2, q)));
    }
    if (spins >= (1u << 27)) *x.err_flag = 1;
    sums[0] = a; sums[1] = c;
    const double N = (double)(*npos_norm);
    losses[0] = (float)(a / (4.0 * N));
    losses[1] = (float)(c / N);
}
}  // namespace ssdhead

// A few host threads that live as long as the context: they zero the caller's DENSE gradient buffers while the inputs
// of a host-buffer loss call stream in (spawning threads per call would cost ~0.1 ms of every call).  All waiting is
// on condition variables: a rank that waits burns no core (eight ranks share the host's cores).
struct ZeroPool {
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv, cv_done;
    std::function<void(int)> job;          // job(thread index); valid while a generation is running
    unsigned generation = 0;
    int finished = 0;
    int chunk_done[16] = {};               // threads that finished chunk k of the current generation
    bool stop = false;

    int size() const { return (int)threads.size(); }
    void start(int n) {
        for (int ti = 0; ti < n; ++ti)
            threads.emplace_back([this, ti]() {
                unsigned seen = 0;
                for (;;) {
                    std::function<void(int)> j;
                    {
                        std::unique_lock<std::mutex> lk(m);
                        cv.wait(lk, [&] { return stop || generation != seen; });
                        if (stop) return;
                        seen = generation;
                        j = job;
                    }
                    j(ti);
                    { std::lock_guard<std::mutex> lk(m); ++finished; }
                    cv_done.notify_all();
                }
            });
    }
    void run(std::function<void(int)> j) {                 // returns at once; wait() blocks until every thread is done
        {
            std::lock_guard<std::mutex> lk(m);
            finished = 0;
            for (int& c : chunk_done) c = 0;
            job = std::move(j);
            ++generation;
        }
        cv.notify_all();
    }
    void mark_chunk(int k) {                                // called by a worker when its part of chunk k is zero
        { std::lock_guard<std::mutex> lk(m); ++chunk_done[k]; }
        cv_done.notify_all();
    }
    void wait_chunk(int k) {
        std::unique_lock<std::mutex> lk(m);
        cv_done.wait(lk, [&] { return chunk_done[k] >= size(); });
    }
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        cv_done.wait(lk, [&] { return finished >= size(); });
    }
    void shutdown() {
        { std::lock_guard<std::mutex> lk(m); stop = true; }
        cv.notify_all();
        for (auto& t : threads) if (t.joinable()) t.join();
        threads.clear();
    }
};

// Zeroing threads of one context: the host's cores are shared by all ranks of the box (one process per GPU), so the
// pool takes its share of what this process may run on - (affinity-mask cores / LOCAL_WORLD_SIZE) / 2, between 1 and 8
// (memset throughput saturates near 8 threads beside the DMA traffic).  SSDHEAD_ZERO_THREADS overrides.
static int zero_pool_threads()
{
    if (const char* e = getenv("SSDHEAD_ZERO_THREADS")) return std::max(1, std::min(64, atoi(e)));
    unsigned cores = std::thread::hardware_concurrency();
#ifdef __linux__
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) cores = (unsigned)CPU_COUNT(&set);
#endif
    int ranks = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, atoi(e));
    return (int)std::min(8u, std::max(1u, cores / (unsigned)ranks / 2u));
}

struct ssdhead_ctx {
    ZeroPool pool;
    int device, maxB, P, C, max_sumG, top_k, last_detect_B, last_loss_B;
    // cross-GPU exchange (sharded batches)
    int xchg_R, xchg_rank;
    unsigned int xchg_seq;
    void* xchg_local;
    void** xchg_peers_dev;
    void* xchg_opened[16];
    int* err_flag;
    cudaStream_t s_main, s_aux, s_h2d, s_d2h;
    cudaEvent_t ev_fork, ev_join, ev_gt, ev_done;
    std::vector<cudaEvent_t> ev_in, ev_out;            // per chunk
    // prior tables
    float *pri_cxcywh, *pri_xyxy;
    // gt + match outputs
    float *gt_xyxy, *gt_cls;
    int32_t *gt_off, *best_prior, *npos;
    uint8_t* cls_u8;
    // head tensors (host-buffer path)
    float *loc, *conf, *grad_loc, *grad_conf;
    double *sums, *chunk_sums;
    float *losses;
    // workspaces
    void *ws_match, *ws_loss, *ws_detect;
    // resident gradient tensors (ssdhead_ctx_multibox_loss_dev_resident): rows workspace + the tensors it describes
    void* ws_rows;
    size_t ws_rows_bytes;
    float *res_grad_loc, *res_grad_conf;
    int res_B;                              // images of the two tensors that were zero-filled at the hand-over
    size_t ws_match_bytes, ws_loss_bytes, ws_loss_total, ws_detect_bytes;
    // detect outputs (host-buffer path)
    float *det_boxes, *det_prob;
    int32_t *det_cls, *det_prior, *det_cnt;
    // pinned scratch for small results
    float* h_losses;
    // host-buffer path of a sharded batch: global positive count (device int)
    int32_t* npos_global;
    // sparse gradient return into pageable host buffers: device staging (grown on demand)
    int32_t *sp_cnt, *sp_idx;
    float *sp_conf, *sp_loc;
    size_t sp_rows;                                     // capacity of the staging in rows (B * row_cap)
};

// Device-visible alias of a page-locked host buffer (UVA maps cudaHostAlloc / cudaHostRegister memory), or null for
// pageable / unaligned memory.  Kernels that touch only a few rows of a tensor read it in place instead of copying it.
static const float* mapped_host_alias(const float* host)
{
    cudaPointerAttributes attr;
    float* mapped = nullptr;
    if (cudaPointerGetAttributes(&attr, host) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
        cudaHostGetDevicePointer((void**)&mapped, (void*)host, 0) == cudaSuccess && mapped && aligned16(mapped))
        return mapped;
    (void)cudaGetLastError();
    return nullptr;
}

// The loss workspace keeps its counters and per-image partial sums zeroed between steps, but their extent depends on
// the batch size (include/ssdhead.h: "re-zero a buffer before reusing it with another shape"): re-zero the headers of
// all chunk workspaces when B changes.
static int ctx_loss_ws_for(ssdhead_ctx* c, int B, cudaStream_t st)
{
    if (c->last_loss_B == B) return 0;
    const size_t head = loss_ws_header_bytes(c->maxB);
    for (size_t off = 0; off + head <= c->ws_loss_total; off += c->ws_loss_bytes)
        SSD_CHECK_CUDA(cudaMemsetAsync((char*)c->ws_loss + off, 0, std::min(head, c->ws_loss_bytes), st));
    c->last_loss_B = B;
    return 0;
}

#define CTX_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { rc = (int)_e; goto fail; } } while (0)

static const int kMaxChunks = 16;

extern "C" {

// gt collate on the host (Dataset.py:24-36, train_function.py:62-63, Losses.py:129-130): see ssdhead.h
int ssdhead_pack_gt(const float* const* boxes, const float* const* classes, const uint8_t* const* difficult,
                    const int32_t* counts, int B, int keep_difficult, const float* img_wh,
                    float* out_xyxy, float* out_cls, int32_t* out_off, int capacity)
{
    if (B < 0 || capacity < 0 || !out_off || (B > 0 && (!boxes || !classes || !counts))) return SSDHEAD_E_BADARG;
    int n = 0;
    out_off[0] = 0;
    for (int i = 0; i < B; ++i) {
        if (counts[i] < 0 || (counts[i] > 0 && (!boxes[i] || !classes[i]))) return SSDHEAD_E_BADARG;
        const uint8_t* dif = (difficult && !keep_difficult) ? difficult[i] : nullptr;
        const int before = n;
        for (int g = 0; g < counts[i]; ++g) {
            if (dif && dif[g]) continue;                                        // Dataset.py:28-30
            if (n >= capacity || !out_xyxy || !out_cls) return SSDHEAD_E_WORKSPACE;
            const float* bx = boxes[i] + 4 * (size_t)g;
            float* o = out_xyxy + 4 * (size_t)n;
            if (img_wh) {                                                       // Dataset.py:35-36: bboxes / [w, h, w, h]
                const float w = img_wh[2 * i], h = img_wh[2 * i + 1];
                o[0] = bx[0] / w; o[1] = bx[1] / h; o[2] = bx[2] / w; o[3] = bx[3] / h;
            } else {
                o[0] = bx[0]; o[1] = bx[1]; o[2] = bx[2]; o[3] = bx[3];
            }
            out_cls[n] = classes[i][g];
            ++n;
        }
        if (n == before) return SSDHEAD_E_STATE;                                // an image without objects (Losses.py:153)
        out_off[i + 1] = n;
    }
    return n;
}

void* ssdhead_host_alloc(size_t bytes)
{
    void* p = nullptr;
    return cudaHostAlloc(&p, bytes, cudaHostAllocDefault) == cudaSuccess ? p : nullptr;
}
void ssdhead_host_free(void* p) { if (p) cudaFreeHost(p); }

void ssdhead_ctx_destroy(ssdhead_ctx* c)
{
    if (!c) return;
    c->pool.shutdown();
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    void* bufs[] = {c->pri_cxcywh, c->pri_xyxy, c->gt_xyxy, c->gt_cls, c->gt_off, c->best_prior, c->npos, c->cls_u8,
                    c->loc, c->conf, c->grad_loc, c->grad_conf, c->sums, c->chunk_sums, c->losses,
                    c->ws_match, c->ws_loss, c->ws_detect, c->det_boxes, c->det_prob, c->det_cls, c->det_prior, c->det_cnt};
    for (void* b : bufs) if (b) cudaFree(b);
    if (c->h_losses) cudaFreeHost(c->h_losses);
    for (int q = 0; q < 16; ++q) if (c->xchg_opened[q]) cudaIpcCloseMemHandle(c->xchg_opened[q]);
    if (c->xchg_local) cudaFree(c->xchg_local);
    if (c->xchg_peers_dev) cudaFree(c->xchg_peers_dev);
    if (c->err_flag) cudaFree(c->err_flag);
    if (c->ws_rows) cudaFree(c->ws_rows);
    void* more[] = {c->npos_global, c->sp_cnt, c->sp_idx, c->sp_conf, c->sp_loc};
    for (void* b : more) if (b) cudaFree(b);
    cudaStream_t st[] = {c->s_main, c->s_aux, c->s_h2d, c->s_d2h};
    for (cudaStream_t s : st) if (s) cudaStreamDestroy(s);
    cudaEvent_t ev[] = {c->ev_fork, c->ev_join, c->ev_gt, c->ev_done};
    for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->ev_in) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->ev_out) if (e) cudaEventDestroy(e);
    delete c;
}

int ssdhead_ctx_create(ssdhead_ctx** out, int device, int maxB, int P, int C, int max_sumG, int top_k,
                       const float* pri_cxcywh_host)
{
    if (!out || maxB <= 0 || P <= 0 || C < 2 || max_sumG < 0 || top_k <= 0 || !pri_cxcywh_host) return SSDHEAD_E_BADARG;
    int rc = 0;
    ssdhead_ctx* c = new ssdhead_ctx();
    c->device = device; c->maxB = maxB; c->P = P; c->C = C; c->max_sumG = std::max(max_sumG, 1); c->top_k = top_k;
    {
        const size_t nrow = (size_t)maxB * P;
        std::vector<float> xy((size_t)P * 4);
        priors_xyxy_host(pri_cxcywh_host, xy.data(), P);
        CTX_CUDA(cudaSetDevice(device));
        CTX_CUDA(cudaStreamCreateWithFlags(&c->s_main, cudaStreamNonBlocking));
        CTX_CUDA(cudaStreamCreateWithFlags(&c->s_aux, cudaStreamNonBlocking));
        CTX_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
        CTX_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
        CTX_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CTX_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        CTX_CUDA(cudaEventCreateWithFlags(&c->ev_gt, cudaEventDisableTiming));
        CTX_CUDA(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
        c->ev_in.assign(kMaxChunks, nullptr);
        c->ev_out.assign(kMaxChunks, nullptr);
        for (int i = 0; i < kMaxChunks; ++i) {
            CTX_CUDA(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
            CTX_CUDA(cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming));
        }
        CTX_CUDA(cudaMalloc(&c->pri_cxcywh, (size_t)P * 16));
        CTX_CUDA(cudaMalloc(&c->pri_xyxy, (size_t)P * 16));
        CTX_CUDA(cudaMemcpy(c->pri_cxcywh, pri_cxcywh_host, (size_t)P * 16, cudaMemcpyHostToDevice));
        CTX_CUDA(cudaMemcpy(c->pri_xyxy, xy.data(), (size_t)P * 16, cudaMemcpyHostToDevice));
        CTX_CUDA(cudaMalloc(&c->gt_xyxy, (size_t)c->max_sumG * 16));
        CTX_CUDA(cudaMalloc(&c->gt_cls, (size_t)c->max_sumG * 4));
        CTX_CUDA(cudaMalloc(&c->gt_off, (size_t)(maxB + 1) * 4));
        CTX_CUDA(cudaMalloc(&c->best_prior, (size_t)c->max_sumG * 4));
        CTX_CUDA(cudaMalloc(&c->npos, (size_t)(maxB + 1) * 4));
        CTX_CUDA(cudaMalloc(&c->cls_u8, round_up(nrow, 16)));
        CTX_CUDA(cudaMalloc(&c->loc, nrow * 16));
        CTX_CUDA(cudaMalloc(&c->conf, nrow * C * 4));
        CTX_CUDA(cudaMalloc(&c->grad_loc, nrow * 16));
        CTX_CUDA(cudaMalloc(&c->grad_conf, nrow * C * 4));
        CTX_CUDA(cudaMalloc(&c->sums, 2 * sizeof(double)));
        CTX_CUDA(cudaMalloc(&c->chunk_sums, 2 * kMaxChunks * sizeof(double)));
        CTX_CUDA(cudaMalloc(&c->losses, 2 * sizeof(float)));
        c->ws_match_bytes = ssdhead_workspace_bytes(SSDHEAD_WS_MATCH, maxB, P, C, c->max_sumG);
        c->ws_loss_bytes = ssdhead_workspace_bytes(SSDHEAD_WS_LOSS, maxB, P, C, 0);
        c->ws_detect_bytes = ssdhead_workspace_bytes(SSDHEAD_WS_DETECT, maxB, P, C, 0);
        CTX_CUDA(cudaMalloc(&c->ws_match, c->ws_match_bytes));
        CTX_CUDA(cudaMemset(c->ws_match, 0, c->ws_match_bytes));
        if (c->ws_loss_bytes) {
            // one workspace per chunk slot so chunk i+1 can stream while chunk i is being mined
            c->ws_loss_total = c->ws_loss_bytes * kMaxChunks;
            CTX_CUDA(cudaMalloc(&c->ws_loss, c->ws_loss_bytes * kMaxChunks));
            CTX_CUDA(cudaMemset(c->ws_loss, 0, c->ws_loss_bytes * kMaxChunks));
        }
        if (c->ws_detect_bytes) {
            CTX_CUDA(cudaMalloc(&c->ws_detect, c->ws_detect_bytes));
            CTX_CUDA(cudaMemset(c->ws_detect, 0, c->ws_detect_bytes));
        }
        CTX_CUDA(cudaMalloc(&c->det_boxes, (size_t)maxB * top_k * 16));
        CTX_CUDA(cudaMalloc(&c->det_prob, (size_t)maxB * top_k * 4));
        CTX_CUDA(cudaMalloc(&c->det_cls, (size_t)maxB * top_k * 4));
        CTX_CUDA(cudaMalloc(&c->det_prior, (size_t)maxB * top_k * 4));
        CTX_CUDA(cudaMalloc(&c->det_cnt, (size_t)maxB * 4));
        CTX_CUDA(cudaHostAlloc(&c->h_losses, 64, cudaHostAllocDefault));
        CTX_CUDA(cudaMalloc(&c->xchg_local, ssdhead_xchg_bytes()));
        CTX_CUDA(cudaMemset(c->xchg_local, 0, ssdhead_xchg_bytes()));
        CTX_CUDA(cudaMalloc(&c->xchg_peers_dev, 16 * sizeof(void*)));
        CTX_CUDA(cudaMalloc(&c->err_flag, sizeof(int)));
        CTX_CUDA(cudaMemset(c->err_flag, 0, sizeof(int)));
        CTX_CUDA(cudaMalloc(&c->npos_global, sizeof(int32_t)));
        c->xchg_R = 1;
    }
    *out = c;
    return 0;
fail:
    ssdhead_ctx_destroy(c);
    return rc;
}

// Sharded batches: the step in two halves around the all-reduce of the positive count (SURVEY.md 8(e)).
// begin: the CE streaming kernel with the fused natural match + the forced-match finaliser; on return
// *npos_total_dev points to this rank's int32 positive count (device memory owned by the context).
int ssdhead_ctx_multibox_loss_begin(ssdhead_ctx* c, const float* conf,
                                    const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off, int B, int sumG,
                                    float pos_iou, float* grad_loc, float* grad_conf, int32_t** npos_total_dev, void* stream)
{
    if (!c) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB || sumG < 0 || sumG > c->max_sumG) return SSDHEAD_E_STATE;
    cudaStream_t st = (cudaStream_t)stream;
    { const int zr = ctx_loss_ws_for(c, B, st); if (zr) return zr; }
    // the natural match rides inside the CE streaming kernel; a small finaliser applies the forced-match override
    const int rc = ssdhead_ce_match_stream(conf, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, B, c->P, c->C, sumG, pos_iou,
                                           nullptr, grad_loc, grad_conf, c->cls_u8, c->best_prior, c->npos,
                                           c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes, 1, st);
    if (rc) return rc;
    if (npos_total_dev) *npos_total_dev = c->npos + B;
    return 0;
}

// end: the mining kernel, normalised by *npos_norm_dev (null = this rank's own count).
int ssdhead_ctx_multibox_loss_end(ssdhead_ctx* c, const float* loc, const float* conf,
                                  const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off, int B,
                                  int neg_ratio, float pos_iou, const int32_t* npos_norm_dev,
                                  double* sums, float* losses, float* grad_loc, float* grad_conf, void* stream)
{
    if (!c) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB) return SSDHEAD_E_STATE;
    return ssdhead_mine(loc, conf, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, c->best_prior, c->npos,
                        npos_norm_dev ? npos_norm_dev : c->npos + B,
                        c->cls_u8, B, c->P, c->C, neg_ratio, pos_iou, sums, losses, grad_loc, grad_conf, nullptr, nullptr,
                        c->ws_loss, c->ws_loss_bytes, (cudaStream_t)stream);
}

// One training-head step on DEVICE tensors: ssdhead_multibox_step, or the sharded step - two kernels on `stream`.
int ssdhead_ctx_multibox_loss_dev(ssdhead_ctx* c, const float* loc, const float* conf,
                                  const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off, int B, int sumG,
                                  int neg_ratio, float pos_iou,
                                  double* sums, float* losses, float* grad_loc, float* grad_conf, void* stream)
{
    if (!c) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB || sumG < 0 || sumG > c->max_sumG) return SSDHEAD_E_STATE;
    { const int zr = ctx_loss_ws_for(c, B, (cudaStream_t)stream); if (zr) return zr; }
    if (c->xchg_R > 1)
        return ssdhead_multibox_step_sharded(loc, conf, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, B, c->P, c->C, sumG,
                                             neg_ratio, pos_iou, sums, losses, grad_loc, grad_conf, c->cls_u8, c->best_prior, c->npos,
                                             c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes,
                                             c->xchg_R, c->xchg_rank, ++c->xchg_seq, c->xchg_peers_dev, c->xchg_local, c->err_flag, stream);
    return ssdhead_multibox_step(loc, conf, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, B, c->P, c->C, sumG,
                                 neg_ratio, pos_iou, sums, losses, grad_loc, grad_conf, c->cls_u8, c->best_prior, c->npos,
                                 nullptr, nullptr, c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes, stream);
}

int ssdhead_ctx_multibox_loss_dev_resident(ssdhead_ctx* c, const float* loc, const float* conf,
                                  const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off, int B, int sumG,
                                  int neg_ratio, float pos_iou,
                                  double* sums, float* losses, float* grad_loc, float* grad_conf, int fresh, void* stream)
{
    if (!c || !grad_loc || !grad_conf) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB || sumG < 0 || sumG > c->max_sumG) return SSDHEAD_E_STATE;
    cudaStream_t st = (cudaStream_t)stream;
    if (!c->ws_rows) {
        SSD_CHECK_CUDA(cudaSetDevice(c->device));
        c->ws_rows_bytes = ssdhead_workspace_bytes(SSDHEAD_WS_ROWS, c->maxB, c->P, c->C, 0);
        if (c->ws_rows_bytes == 0) return SSDHEAD_E_UNSUPPORTED;
        SSD_CHECK_CUDA(cudaMalloc(&c->ws_rows, c->ws_rows_bytes));
        fresh = 1;
    }
    if (fresh) {
        SSD_CHECK_CUDA(cudaMemsetAsync(c->ws_rows, 0, c->ws_rows_bytes, st));
        SSD_CHECK_CUDA(cudaMemsetAsync(grad_loc, 0, (size_t)B * c->P * 4 * sizeof(float), st));
        SSD_CHECK_CUDA(cudaMemsetAsync(grad_conf, 0, (size_t)B * c->P * c->C * sizeof(float), st));
        c->res_grad_loc = grad_loc; c->res_grad_conf = grad_conf; c->res_B = B;
    } else if (grad_loc != c->res_grad_loc || grad_conf != c->res_grad_conf || B > c->res_B) {
        return SSDHEAD_E_STATE;                          // not the tensors the rows workspace describes, or images beyond the clean part
    }
    { const int zr = ctx_loss_ws_for(c, B, st); if (zr) return zr; }
    const bool sharded = c->xchg_R > 1;
    return ssdhead_multibox_step_resident(loc, conf, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, B, c->P, c->C, sumG,
                                          neg_ratio, pos_iou, sums, losses, grad_loc, grad_conf, c->cls_u8, c->best_prior, c->npos,
                                          c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes, c->ws_rows, c->ws_rows_bytes,
                                          sharded ? c->xchg_R : 1, sharded ? c->xchg_rank : 0, sharded ? ++c->xchg_seq : 0u,
                                          sharded ? c->xchg_peers_dev : nullptr, sharded ? c->xchg_local : nullptr,
                                          sharded ? c->err_flag : nullptr, stream);
}

int ssdhead_ctx_multibox_loss_levels_dev(ssdhead_ctx* c, const ssdhead_levels* levels,
                                         const float* gt_xyxy, const float* gt_cls, const int32_t* gt_off,
                                         int B, int sumG, int neg_ratio, float pos_iou,
                                         double* sums, float* losses, void* stream)
{
    if (!c || !levels) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB || sumG < 0 || sumG > c->max_sumG) return SSDHEAD_E_STATE;
    { const int zr = ctx_loss_ws_for(c, B, (cudaStream_t)stream); if (zr) return zr; }
    if (c->xchg_R > 1)
        return ssdhead_multibox_step_levels_sharded(levels, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, B, c->P, c->C, sumG,
                                                    neg_ratio, pos_iou, sums, losses, c->cls_u8, c->best_prior, c->npos,
                                                    c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes,
                                                    c->xchg_R, c->xchg_rank, ++c->xchg_seq, c->xchg_peers_dev, c->xchg_local, c->err_flag, stream);
    return ssdhead_multibox_step_levels(levels, gt_xyxy, gt_cls, gt_off, c->pri_xyxy, c->pri_cxcywh, B, c->P, c->C, sumG,
                                        neg_ratio, pos_iou, sums, losses, c->cls_u8, c->best_prior, c->npos,
                                        c->ws_loss, c->ws_loss_bytes, c->ws_match, c->ws_match_bytes, stream);
}

int ssdhead_ctx_xchg_export(ssdhead_ctx* c, void* handle64_out)
{
    if (!c || !handle64_out) return SSDHEAD_E_BADARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    SSD_CHECK_CUDA(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    SSD_CHECK_CUDA(cudaIpcGetMemHandle(&h, c->xchg_local));
    std::memcpy(handle64_out, &h, 64);
    return 0;
}

int ssdhead_ctx_xchg_import(ssdhead_ctx* c, const void* handles, int R, int rank)
{
    if (!c || !handles || R < 1 || R > 16 || rank < 0 || rank >= R) return SSDHEAD_E_BADARG;
    SSD_CHECK_CUDA(cudaSetDevice(c->device));
    void* table[16] = {};
    for (int q = 0; q < R; ++q) {
        if (q == rank) { table[q] = c->xchg_local; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, (const char*)handles + 64 * q, 64);
        SSD_CHECK_CUDA(cudaIpcOpenMemHandle(&table[q], h, cudaIpcMemLazyEnablePeerAccess));
        c->xchg_opened[q] = table[q];
    }
    SSD_CHECK_CUDA(cudaMemcpy(c->xchg_peers_dev, table, sizeof(table), cudaMemcpyHostToDevice));
    c->xchg_R = R; c->xchg_rank = rank; c->xchg_seq = 0;
    return 0;
}

int ssdhead_ctx_xchg_error(ssdhead_ctx* c)
{
    if (!c) return SSDHEAD_E_BADARG;
    int e = 0;
    if (cudaMemcpy(&e, c->err_flag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    return e;
}

// ssd() on HOST buffers (pass page-locked memory, e.g. ssdhead_host_alloc, for asynchronous copies).
// gt goes first and the match starts at once; conf/loc travel in image chunks, each chunk is streamed
// (CE) and mined as soon as it lands while the next one is in flight.  Gradients come back either DENSE (the caller's
// [B,P,*] host tensors) or SPARSE (packed rows, ssdhead_ctx_multibox_loss_host_sparse).  After ssdhead_ctx_xchg_import
// the batch is one shard of a batch spread over R GPUs: the positive count and the loss sums cross GPUs through the
// exchange buffers (two single-thread kernels, NVLink peer stores), so losses and gradients carry the GLOBAL
// normalisation of Losses.py:182,197; all ranks must call in lock step.  Blocks until the results are in host memory.
static int loss_host_impl(ssdhead_ctx* c, const float* loc_h, const float* conf_h,
                          const float* gt_xyxy_h, const float* gt_cls_h, const int32_t* gt_off_h,
                          int B, int neg_ratio, float pos_iou, float* losses_h,
                          float* grad_loc_h, float* grad_conf_h,
                          int row_cap, int32_t* row_cnt_h, int32_t* row_idx_h, float* gconf_rows_h, float* gloc_rows_h)
{
    if (!c || !loc_h || !conf_h || !gt_off_h || !losses_h) return SSDHEAD_E_BADARG;
    if ((grad_loc_h == nullptr) != (grad_conf_h == nullptr)) return SSDHEAD_E_BADARG;
    const bool rows = row_cnt_h != nullptr;                   // sparse gradient return
    if (rows && (row_cap <= 0 || !row_idx_h || !gconf_rows_h || !gloc_rows_h || grad_loc_h)) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB) return SSDHEAD_E_STATE;
    const int sumG = gt_off_h[B];
    if (sumG < 0 || sumG > c->max_sumG || (sumG > 0 && (!gt_xyxy_h || !gt_cls_h))) return SSDHEAD_E_STATE;
    SSD_CHECK_CUDA(cudaSetDevice(c->device));
    const int P = c->P, C = c->C;
    const bool grads = grad_loc_h != nullptr;
    { const int zr = ctx_loss_ws_for(c, -B, c->s_main); if (zr) return zr; }   // (-B: the chunked layout of batch B)

    // gt -> device, match on the auxiliary stream
    if (sumG > 0) {
        SSD_CHECK_CUDA(cudaMemcpyAsync(c->gt_xyxy, gt_xyxy_h, (size_t)sumG * 16, cudaMemcpyHostToDevice, c->s_aux));
        SSD_CHECK_CUDA(cudaMemcpyAsync(c->gt_cls, gt_cls_h, (size_t)sumG * 4, cudaMemcpyHostToDevice, c->s_aux));
    }
    SSD_CHECK_CUDA(cudaMemcpyAsync(c->gt_off, gt_off_h, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, c->s_aux));
    int rc = ssdhead_match(c->gt_xyxy, c->gt_cls, c->gt_off, c->pri_xyxy, B, P, C, sumG, pos_iou,
                           c->best_prior, c->npos, c->cls_u8, nullptr, nullptr, c->ws_match, c->ws_match_bytes, c->s_aux);
    if (rc) return rc;
    const bool sharded = c->xchg_R > 1;
    XchgArgs xa = {};
    const int32_t* npos_norm = c->npos + B;
    if (sharded) {
        xa.R = c->xchg_R; xa.rank = c->xchg_rank; xa.seq = ++c->xchg_seq;
        xa.peers = (unsigned long long* const*)c->xchg_peers_dev; xa.local = (unsigned long long*)c->xchg_local; xa.err_flag = c->err_flag;
        xchg_npos_kernel<<<1, 1, 0, c->s_aux>>>(c->npos + B, c->npos_global, xa);
        count_launch();
        SSD_LAUNCH_CHECK();
        npos_norm = c->npos_global;
    }
    SSD_CHECK_CUDA(cudaEventRecord(c->ev_join, c->s_aux));

    const float* loc_alias = mapped_host_alias(loc_h);
    // >= 8 images per chunk, at most 8 chunks (measured on B200/PCIe5: 1 chunk 8.2 ms, 4: 5.8, 8: 5.6, 16: 6.3 at B=256)
    const int nchunks = std::min(8, std::max(1, B / 8));
    const int per = (B + nchunks - 1) / nchunks;
    int used = 0;

    // DENSE return.  The gradient is sparse (about 4 Npos of the B x P rows): when the caller's gradient buffers are
    // page-locked, the dense zero background never crosses PCIe.  Host threads zero the buffers chunk by chunk while the
    // inputs stream in, the streaming kernel runs without its zero-fill, and the mining kernel stores its few hundred
    // rows per image straight into the host buffers through their UVA aliases.  Same bits in the caller's buffers.
    float* gl_alias = grads ? const_cast<float*>(mapped_host_alias(grad_loc_h)) : nullptr;
    float* gc_alias = grads ? const_cast<float*>(mapped_host_alias(grad_conf_h)) : nullptr;
    const bool sparse = gl_alias && gc_alias;
    int T = 0;
    if (sparse) {
        if (c->pool.size() == 0) c->pool.start(zero_pool_threads());
        T = c->pool.size();
        ZeroPool* pool = &c->pool;
        c->pool.run([=](int ti) {
            for (int k = 0, b0 = 0; b0 < B; ++k, b0 += per) {
                const int nb = std::min(per, B - b0);
                const size_t r0 = (size_t)b0 * P, nr = (size_t)nb * P;
                auto zero_part = [&](float* base, size_t floats) {
                    const size_t part = ((floats + T - 1) / T + 15) & ~(size_t)15;     // T parts cover everything
                    const size_t lo = std::min(floats, part * ti), hi = std::min(floats, lo + part);
                    if (hi > lo) std::memset(base + lo, 0, (hi - lo) * sizeof(float));
                };
                zero_part(grad_conf_h + r0 * C, nr * C);
                zero_part(grad_loc_h + r0 * 4, nr * 4);
                pool->mark_chunk(k);
            }
        });
    }
    // ROW return: packed rows; page-locked output buffers are written in place by the mining kernel, pageable ones
    // through device staging copied back at the end.  No zero background exists on either side.
    int32_t* rc_dev = nullptr; int32_t* ri_dev = nullptr; float* rgc_dev = nullptr; float* rgl_dev = nullptr;
    bool rows_staged = false;
    if (rows) {
        rc_dev = (int32_t*)mapped_host_alias((const float*)row_cnt_h);
        ri_dev = (int32_t*)mapped_host_alias((const float*)row_idx_h);
        rgc_dev = const_cast<float*>(mapped_host_alias(gconf_rows_h));
        rgl_dev = const_cast<float*>(mapped_host_alias(gloc_rows_h));
        if (!rc_dev || !ri_dev || !rgc_dev || !rgl_dev) {
            const size_t need_rows = (size_t)B * row_cap;
            if (c->sp_rows < need_rows) {
                void* old[] = {c->sp_cnt, c->sp_idx, c->sp_conf, c->sp_loc};
                for (void* o : old) if (o) cudaFree(o);
                c->sp_cnt = nullptr; c->sp_idx = nullptr; c->sp_conf = nullptr; c->sp_loc = nullptr; c->sp_rows = 0;
                SSD_CHECK_CUDA(cudaMalloc(&c->sp_cnt, (size_t)c->maxB * 2 * 4));
                SSD_CHECK_CUDA(cudaMalloc(&c->sp_idx, need_rows * 4));
                SSD_CHECK_CUDA(cudaMalloc(&c->sp_conf, need_rows * C * 4));
                SSD_CHECK_CUDA(cudaMalloc(&c->sp_loc, need_rows * 16));
                c->sp_rows = need_rows;
            }
            rc_dev = c->sp_cnt; ri_dev = c->sp_idx; rgc_dev = c->sp_conf; rgl_dev = c->sp_loc;
            rows_staged = true;
        }
    }
    auto join_all = [&]() { if (sparse) c->pool.wait(); };     // the job references the caller's buffers: never return before it is done
#define CTX_HOST_CHECK(expr) do { const int _rc = (expr); if (_rc) { join_all(); return _rc; } } while (0)

    // all input copies first (they depend on nothing), then the kernels chunk by chunk
    for (int k = 0, b0 = 0; b0 < B; ++k, b0 += per) {
        const int nb = std::min(per, B - b0);
        const size_t r0 = (size_t)b0 * P, nr = (size_t)nb * P;
        CTX_HOST_CHECK((int)cudaMemcpyAsync(c->conf + r0 * C, conf_h + r0 * C, nr * C * 4, cudaMemcpyHostToDevice, c->s_h2d));
        // the mining kernel reads loc only for the positive rows (~50 per image): page-locked loc is read in place
        if (!loc_alias) CTX_HOST_CHECK((int)cudaMemcpyAsync(c->loc + r0 * 4, loc_h + r0 * 4, nr * 16, cudaMemcpyHostToDevice, c->s_h2d));
        CTX_HOST_CHECK((int)cudaEventRecord(c->ev_in[k], c->s_h2d));
    }
    for (int k = 0, b0 = 0; b0 < B; ++k, b0 += per) {
        const int nb = std::min(per, B - b0);
        const size_t r0 = (size_t)b0 * P, nr = (size_t)nb * P;
        CTX_HOST_CHECK((int)cudaStreamWaitEvent(c->s_main, c->ev_in[k], 0));
        void* ws = (char*)c->ws_loss + (size_t)k * c->ws_loss_bytes;
        float* gl = grads ? (sparse ? gl_alias + r0 * 4 : c->grad_loc + r0 * 4) : nullptr;
        float* gc = grads ? (sparse ? gc_alias + r0 * C : c->grad_conf + r0 * C) : nullptr;
        rc = ssdhead_ce_stream(c->conf + r0 * C, nb, P, C, nullptr, (sparse || rows) ? nullptr : gl, (sparse || rows) ? nullptr : gc, ws, c->ws_loss_bytes, c->s_main);
        CTX_HOST_CHECK(rc);
        if (k == 0) CTX_HOST_CHECK((int)cudaStreamWaitEvent(c->s_main, c->ev_join, 0));
        if (sparse) c->pool.wait_chunk(k);                       // chunk k's slices are zero (condition variable, no spinning)
        const float* loc_k = (loc_alias ? loc_alias : c->loc) + r0 * 4;
        if (rows)
            rc = ssdhead_mine_sparse(loc_k, c->conf + r0 * C, c->gt_xyxy, c->gt_cls, c->gt_off + b0, c->pri_xyxy, c->pri_cxcywh,
                                     c->best_prior, c->npos + b0, npos_norm, c->cls_u8 + r0, nb, P, C, neg_ratio, pos_iou,
                                     c->chunk_sums + 2 * k, c->losses, row_cap, rc_dev + 2 * (size_t)b0, ri_dev + (size_t)b0 * row_cap,
                                     rgc_dev + (size_t)b0 * row_cap * C, rgl_dev + (size_t)b0 * row_cap * 4,
                                     ws, c->ws_loss_bytes, c->s_main);
        else
            rc = ssdhead_mine(loc_k, c->conf + r0 * C, c->gt_xyxy, c->gt_cls, c->gt_off + b0, c->pri_xyxy, c->pri_cxcywh,
                              c->best_prior, c->npos + b0, npos_norm, c->cls_u8 + r0, nb, P, C, neg_ratio, pos_iou,
                              c->chunk_sums + 2 * k, c->losses, gl, gc, nullptr, nullptr, ws, c->ws_loss_bytes, c->s_main);
        CTX_HOST_CHECK(rc);
        if (grads && !sparse) {
            CTX_HOST_CHECK((int)cudaEventRecord(c->ev_out[k], c->s_main));
            CTX_HOST_CHECK((int)cudaStreamWaitEvent(c->s_d2h, c->ev_out[k], 0));
            CTX_HOST_CHECK((int)cudaMemcpyAsync(grad_conf_h + r0 * C, gc, nr * C * 4, cudaMemcpyDeviceToHost, c->s_d2h));
            CTX_HOST_CHECK((int)cudaMemcpyAsync(grad_loc_h + r0 * 4, gl, nr * 16, cudaMemcpyDeviceToHost, c->s_d2h));
        }
        used = k + 1;
    }
    join_all();
#undef CTX_HOST_CHECK
    if (sharded) sum_chunks_xchg_kernel<<<1, 1, 0, c->s_main>>>(c->chunk_sums, used, npos_norm, c->sums, c->losses, xa);
    else sum_chunks_kernel<<<1, 1, 0, c->s_main>>>(c->chunk_sums, used, npos_norm, c->sums, c->losses);
    count_launch();
    SSD_LAUNCH_CHECK();
    SSD_CHECK_CUDA(cudaMemcpyAsync(c->h_losses, c->losses, 2 * sizeof(float), cudaMemcpyDeviceToHost, c->s_main));
    if (rows_staged) {
        const size_t nrows = (size_t)B * row_cap;
        SSD_CHECK_CUDA(cudaMemcpyAsync(row_cnt_h, rc_dev, (size_t)B * 2 * 4, cudaMemcpyDeviceToHost, c->s_main));
        SSD_CHECK_CUDA(cudaMemcpyAsync(row_idx_h, ri_dev, nrows * 4, cudaMemcpyDeviceToHost, c->s_main));
        SSD_CHECK_CUDA(cudaMemcpyAsync(gconf_rows_h, rgc_dev, nrows * C * 4, cudaMemcpyDeviceToHost, c->s_main));
        SSD_CHECK_CUDA(cudaMemcpyAsync(gloc_rows_h, rgl_dev, nrows * 16, cudaMemcpyDeviceToHost, c->s_main));
    }
    SSD_CHECK_CUDA(cudaStreamSynchronize(c->s_main));
    if (grads && !sparse) SSD_CHECK_CUDA(cudaStreamSynchronize(c->s_d2h));
    losses_h[0] = c->h_losses[0];
    losses_h[1] = c->h_losses[1];
    return 0;
}

int ssdhead_ctx_multibox_loss_host(ssdhead_ctx* c, const float* loc_h, const float* conf_h,
                                   const float* gt_xyxy_h, const float* gt_cls_h, const int32_t* gt_off_h,
                                   int B, int neg_ratio, float pos_iou,
                                   float* losses_h, float* grad_loc_h, float* grad_conf_h)
{
    return loss_host_impl(c, loc_h, conf_h, gt_xyxy_h, gt_cls_h, gt_off_h, B, neg_ratio, pos_iou, losses_h,
                          grad_loc_h, grad_conf_h, 0, nullptr, nullptr, nullptr, nullptr);
}

int ssdhead_ctx_multibox_loss_host_sparse(ssdhead_ctx* c, const float* loc_h, const float* conf_h,
                                          const float* gt_xyxy_h, const float* gt_cls_h, const int32_t* gt_off_h,
                                          int B, int neg_ratio, float pos_iou, float* losses_h,
                                          int row_cap, int32_t* row_cnt_h, int32_t* row_idx_h,
                                          float* grad_conf_rows_h, float* grad_loc_rows_h)
{
    if (!row_cnt_h) return SSDHEAD_E_BADARG;
    return loss_host_impl(c, loc_h, conf_h, gt_xyxy_h, gt_cls_h, gt_off_h, B, neg_ratio, pos_iou, losses_h,
                          nullptr, nullptr, row_cap, row_cnt_h, row_idx_h, grad_conf_rows_h, grad_loc_rows_h);
}

// inference() over a batch on HOST buffers: copies in, ssdhead_detect, detections out.  Blocks.
int ssdhead_ctx_detect_host(ssdhead_ctx* c, const float* loc_h, const float* conf_h, int B,
                            float min_score, float iou_thr,
                            float* out_boxes_h, float* out_prob_h, int32_t* out_cls_h, int32_t* out_prior_h, int32_t* out_cnt_h)
{
    if (!c || !loc_h || !conf_h || !out_boxes_h || !out_prob_h || !out_cls_h || !out_cnt_h) return SSDHEAD_E_BADARG;
    if (B <= 0 || B > c->maxB || !c->ws_detect) return SSDHEAD_E_STATE;
    SSD_CHECK_CUDA(cudaSetDevice(c->device));
    const size_t nr = (size_t)B * c->P;
    if (c->last_detect_B != B) {
        // the detect workspace keeps its counters zeroed, but their position depends on B: re-zero on a shape change
        SSD_CHECK_CUDA(cudaMemsetAsync(c->ws_detect, 0, c->ws_detect_bytes, c->s_main));
        c->last_detect_B = B;
    }
    SSD_CHECK_CUDA(cudaMemcpyAsync(c->conf, conf_h, nr * c->C * 4, cudaMemcpyHostToDevice, c->s_main));
    // The sweep decodes only the few hundred boxes per image it actually visits, so the offsets need not cross PCIe in
    // full (16 % of the input bytes): page-locked host memory is mapped into the device's address space (UVA) and the
    // kernel reads those rows in place.  Pageable or unaligned buffers are copied as before.
    const float* loc_alias = mapped_host_alias(loc_h);
    const float* loc_dev = loc_alias ? loc_alias : c->loc;
    if (loc_dev == c->loc) SSD_CHECK_CUDA(cudaMemcpyAsync(c->loc, loc_h, nr * 16, cudaMemcpyHostToDevice, c->s_main));
    const int rc = ssdhead_detect(loc_dev, c->conf, c->pri_cxcywh, B, c->P, c->C, min_score, iou_thr, c->top_k, nullptr, 0,
                                  c->det_boxes, c->det_prob, c->det_cls, c->det_prior, c->det_cnt,
                                  c->ws_detect, c->ws_detect_bytes, c->s_main);
    if (rc) return rc;
    const size_t nk = (size_t)B * c->top_k;
    SSD_CHECK_CUDA(cudaMemcpyAsync(out_boxes_h, c->det_boxes, nk * 16, cudaMemcpyDeviceToHost, c->s_main));
    SSD_CHECK_CUDA(cudaMemcpyAsync(out_prob_h, c->det_prob, nk * 4, cudaMemcpyDeviceToHost, c->s_main));
    SSD_CHECK_CUDA(cudaMemcpyAsync(out_cls_h, c->det_cls, nk * 4, cudaMemcpyDeviceToHost, c->s_main));
    if (out_prior_h) SSD_CHECK_CUDA(cudaMemcpyAsync(out_prior_h, c->det_prior, nk * 4, cudaMemcpyDeviceToHost, c->s_main));
    SSD_CHECK_CUDA(cudaMemcpyAsync(out_cnt_h, c->det_cnt, (size_t)B * 4, cudaMemcpyDeviceToHost, c->s_main));
    SSD_CHECK_CUDA(cudaStreamSynchronize(c->s_main));
    return 0;
}

}  // extern "C"
