/*
 * ssdhead.h - C ABI of libssdhead.so: the SSD multibox head path on B200 (sm_100a).
 *
 * The reference (nitishsaDire/objectDetection_ssd) is pure Python and has no FFI; the
 * boundary it offers for this path is the call surface of Losses.py / Util.py.  Every
 * entry point below names the reference function (file:line under /root/reference) it
 * replaces; objectdetection_ssd_b200/{Losses,Util}.py bind them with ctypes under the
 * reference's own names (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes; no torch / C++ types; all tensors dense row-major fp32
 *     unless stated; "dev" pointers are CUDA device pointers, "host" pointers host memory.
 *   - return 0 = ok, <0 = SSDHEAD_E_* (bad argument / unsupported shape), >0 = cudaError_t.
 *   - device entry points are asynchronous on `stream` (a cudaStream_t passed as void*),
 *     allocate nothing, keep no global state and are re-entrant across streams when each
 *     call has its own workspace.  The caller owns every buffer.
 *   - workspaces: sized by ssdhead_workspace_bytes(); must be zero-filled before their first use with a given
 *     (B, P, C, n) - the kernels leave every counter zeroed again, so steady-state steps contain no memsets, but the
 *     position of the counters depends on the shape: re-zero a buffer before reusing it with another shape.
 *   - there is no CPU fallback anywhere in this library.
 *   - gt layout: boxes packed [sumG,4] fractional xyxy, classes [sumG] fp32 (Dataset.py:26),
 *     offsets int32 [B+1] (the cumsum of Losses.py:130).  Background class id = C-1
 *     (Losses.py:171).  Prior tables [P,4]: `pri_xyxy` and `pri_cxcywh` (Losses.py:6-7).
 *   - `sumG` is a CAPACITY: the number of gt rows the packed arrays, best_prior and the match workspace have room
 *     for.  It must be at least gt_off[B]; the rows past gt_off[B] are never read, and best_prior past gt_off[B] is
 *     never written.  Every kernel finds an image's gts through gt_off only, read on the device, so a caller with
 *     fixed buffers (a captured CUDA graph, or a context created with max_sumG) passes the capacity and lets the
 *     count change from call to call.  Results do not depend on the capacity; it selects routes that give the same
 *     bits (above 65 535 the steps do not record each prior's best gt, which costs time).
 *   - tie rules T1-T8 of SURVEY.md section 8.1 (repeated in DESIGN.md) are implemented exactly.
 */
#ifndef SSDHEAD_H_
#define SSDHEAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSDHEAD_ABI_VERSION 4   /* 2: sparse gradient return (ssdhead_mine_sparse, ssdhead_ctx_multibox_loss_host_sparse);
                                   3: resident gradient tensors (ssdhead_multibox_step_resident, ssdhead_ctx_multibox_loss_dev_resident);
                                   4: ssdhead_detect_fallbacks (short-list route of the detect kernels; larger detect workspace) */

#define SSDHEAD_E_BADARG      (-1)  /* null pointer / negative size */
#define SSDHEAD_E_UNSUPPORTED (-2)  /* shape outside what the kernels are built for */
#define SSDHEAD_E_WORKSPACE   (-3)  /* workspace too small */
#define SSDHEAD_E_ALIGN       (-4)  /* pointer not 16-byte aligned */
#define SSDHEAD_E_STATE       (-5)  /* host context misuse */

/* which workspace ssdhead_workspace_bytes() sizes */
#define SSDHEAD_WS_MATCH  0
#define SSDHEAD_WS_LOSS   1
#define SSDHEAD_WS_DETECT 2
#define SSDHEAD_WS_NMS    3
#define SSDHEAD_WS_ROWS   4   /* rows workspace of ssdhead_multibox_step_resident */

int         ssdhead_abi_version(void);
const char* ssdhead_error_string(int code);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
uint64_t    ssdhead_launch_count(void);

/* Bytes of device workspace an entry point needs.  `n` = total gt count (MATCH),
 * max candidates per (image,class) the caller wants to allow (DETECT/NMS; 0 = P: three key buffers of
 * B * (C-1) * P * 8 bytes - 4.2 MB per SSD300 image - plus a small directory). */
size_t ssdhead_workspace_bytes(int which, int B, int P, int C, int n);

/* ---- box format / offsets: Util.py:93-96, 57-63, 98-102, 86-91 ------------------- */
int ssdhead_cxcywh_to_xyxy(const float* in_dev, float* out_dev, int n, void* stream);   /* xywh_to_xyxy      */
int ssdhead_xyxy_to_cxcywh(const float* in_dev, float* out_dev, int n, void* stream);   /* xyxy_to_xywh      */
int ssdhead_encode(const float* cxcywh_dev, const float* pri_cxcywh_dev, float* out_dev, int n, void* stream); /* get_offsets_coords */
int ssdhead_decode(const float* gcxgcy_dev, const float* pri_cxcywh_dev, float* out_dev, int n, void* stream); /* gcxgcy_to_cxcy     */

/* ---- dense IoU: find_intersection + get_jaccard_tensor1, Util.py:252-265, 288-301 -- */
int ssdhead_iou_matrix(const float* a_xyxy_dev, int n1, const float* b_xyxy_dev, int n2,
                       float* out_dev /*[n1,n2]*/, void* stream);

/* find_intersection, Util.py:252-265: the [n1,n2] intersection areas only. */
int ssdhead_intersection_matrix(const float* a_xyxy_dev, int n1, const float* b_xyxy_dev, int n2,
                                float* out_dev /*[n1,n2]*/, void* stream);

/* map_prior_to_bb, Util.py:333-352: single-image match from a GIVEN jaccard matrix [G,P] and classes [G]
 * (fp32).  Outputs cls fp32 [P] (bg_class where overlap < thr), obj int64 [P] (local gt index after the
 * forced override, T1-T3).  overlap_ws fp32 [P] and best_prior_ws int32 [G] are scratch. */
int ssdhead_match_from_iou(const float* jacc_dev, const float* classes_dev, int G, int P, float thr, int bg_class,
                           float* cls_out_dev, long long* obj_out_dev, float* overlap_ws_dev, int32_t* best_prior_ws_dev,
                           void* stream);

/* ---- matching: Losses.py:150-171 (batched) / map_prior_to_bb Util.py:333-352 --------
 * Outputs: best_prior int32 [sumG] (argmax over priors per gt, T2);
 *          npos int32 [B+1]: positives per image, npos[B] = batch total;
 *          cls_u8 uint8 [B,P] class per prior after the forced override, C-1 = background
 *                 (what Losses.obj_forEach_prior___ holds; consumed by ssdhead_multibox_loss);
 *          obj_idx int32 [B,P] GLOBAL gt index after the forced override (nullable; debug tap);
 *          cls     int32 [B,P] the class map widened to int32 (nullable; debug tap).
 * The workspace must be zero-filled before its FIRST use; every call leaves it zeroed.      */
int ssdhead_match(const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                  const float* pri_xyxy_dev, int B, int P, int C, int sumG, float pos_iou,
                  int32_t* best_prior_dev, int32_t* npos_dev, uint8_t* cls_u8_dev,
                  int32_t* obj_idx_dev, int32_t* cls_dev,
                  void* ws_dev, size_t ws_bytes, void* stream);

/* ---- multibox loss fwd(+bwd): ssd / ssd1_, Losses.py:119-199 ------------------------
 * Two kernels, exposed separately so that the first can run CONCURRENTLY with ssdhead_match
 * (it does not depend on the match) and so that a sharded batch can all-reduce the positive
 * count between them:
 *
 * ssdhead_ce_stream  persistent streaming kernel: reads conf exactly once through a 4-stage
 *                    TMA/mbarrier shared-memory ring and writes, per prior, the cross entropy
 *                    against the BACKGROUND class (the class of ~99 % of the priors; positives
 *                    are re-scored by ssdhead_mine from the row it re-reads anyway).  When
 *                    grad_* are non-null it also bulk-stores the zero background of the dense
 *                    gradients.
 * ssdhead_mine       one CTA per image: selects the k = neg_ratio*npos largest background CE
 *                    exactly (descending CE, ties -> lower prior index, T4; positives rank with
 *                    value 0, Losses.py:190), sums the loss and writes the gradient rows of
 *                    positives and mined negatives only, for unit upstream gradients.
 * ssdhead_multibox_loss = both, back to back on one stream.
 *
 * `npos_dev`, `best_prior_dev`, `cls_u8_dev` are ssdhead_match's outputs; `npos_norm_dev`
 * points to the int32 positive count the losses/gradients are normalised by (npos_dev+B on
 * one GPU; the all-reduced total when the batch is sharded by image).
 * Outputs: sums double[2] = { sum |loc-enc| over positives, sum CE over positives+mined };
 *          losses float[2] = { sums[0]/(4N), sums[1]/N }  (loc_loss, conf_loss of ssd());
 *          grad_loc [B,P,4], grad_conf [B,P,C] dense (nullable as a pair; pass the same pair
 *                 to both calls);
 *          mined_mask uint32 [B, ceil(P/32)] bit p = mined negative (nullable; debug tap);
 *          ce [B,P] per-prior cross entropy (nullable: then it lives in the workspace; pass
 *                 the same pointer to both calls).
 * The workspace (same one for both calls) must be zero-filled before its FIRST use; every
 * call leaves its counter zeroed.  P <= ~31 000 (shared-memory bound of ssdhead_mine).      */
int ssdhead_ce_stream(const float* conf_dev, int B, int P, int C, float* ce_dev,
                      float* grad_loc_dev, float* grad_conf_dev,
                      void* ws_dev, size_t ws_bytes, void* stream);
/* ssdhead_ce_stream with the NATURAL MATCH FUSED IN (the hot path of ssd()): the consumer thread that scores prior
 * p of image b also finds the best gt of that prior and feeds the per-gt arg-max over priors; a small finaliser
 * kernel then applies the forced-match override.  Produces cls_u8 / best_prior / npos exactly as ssdhead_match does
 * (same IoU code, same tie rules), so no separate pass over the priors is needed.  `ws_match` is a
 * SSDHEAD_WS_MATCH workspace (zero-filled once; left zeroed).  B*P < 2^31.
 * run_finalizer: 1 = complete (streaming kernel + finaliser kernel).  0 = streaming kernel only: cls_u8 then holds
 * the NATURAL classes and the workspace the un-finalised arg-max keys - the state ssdhead_multibox_step's fused
 * mining kernel (or a profiler timing the dominant kernel alone, on a scratch workspace) continues from. */
int ssdhead_ce_match_stream(const float* conf_dev, const float* gt_xyxy_dev, const float* gt_cls_dev,
                            const int32_t* gt_off_dev, const float* pri_xyxy_dev,
                            int B, int P, int C, int sumG, float pos_iou,
                            float* ce_dev, float* grad_loc_dev, float* grad_conf_dev,
                            uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                            void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                            int run_finalizer, void* stream);
/* The whole training-head step of ONE GPU in two kernels: ssdhead_ce_match_stream's streaming kernel, then the
 * mining kernel with the forced-match finaliser fused in (cooperative launch: its CTAs exchange the batch positive
 * count through a counter they wait on, so all B CTAs must be co-resident).  Falls back by itself to the
 * three-kernel sequence (streaming, finaliser, mining) when B exceeds the co-resident capacity.  Outputs as
 * ssdhead_match (cls_u8, best_prior, npos) + ssdhead_mine (sums, losses, gradients, taps).  Not for sharded batches
 * (the all-reduce of the positive count has to sit between the kernels: use ce_match_stream + mine). */
int ssdhead_multibox_step(const float* loc_dev, const float* conf_dev,
                          const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                          const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                          uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                          uint32_t* mined_mask_dev, float* ce_dev,
                          void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                          void* stream);
/* ssdhead_multibox_step for a batch SHARDED BY IMAGE over R GPUs (one process per GPU): the same two kernels; the
 * mining kernel exchanges the positive count (before it scales any gradient) and the two loss sums with its peers by
 * storing into their exchange buffers over NVLink peer memory - no NCCL call and no extra kernel in the step.
 * `peers_dev`: device table of R pointers to the ranks' exchange buffers (ssdhead_xchg_bytes() each, zero-filled
 * once, mapped into this process with cudaIpcOpenMemHandle; entry `rank` is xchg_local_dev).  `seq` >= 1 is a step
 * counter every rank advances in lock step.  sums/losses come back GLOBAL, npos[B] is this rank's own count,
 * *err_flag_dev is set if a (10 s bounded) wait for a peer expired.  B must fit co-resident (else E_UNSUPPORTED:
 * use ssdhead_ce_match_stream + an all-reduce + ssdhead_mine). */
int ssdhead_multibox_step_sharded(const float* loc_dev, const float* conf_dev,
                          const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                          const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                          uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                          void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                          int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev,
                          int32_t* err_flag_dev, void* stream);
size_t ssdhead_xchg_bytes(void);
/* ssdhead_multibox_step with RESIDENT gradient tensors.  The gradient of this loss is sparse: only positives and mined
 * negatives (about 4 * Npos of the P rows of an image, Losses.py:177-197) carry one.  A caller that keeps the SAME
 * grad_loc / grad_conf tensors from step to step (a training loop does: they only feed the head's conv backward, which
 * reads them) hands them over once, zero-filled, together with a zero-filled SSDHEAD_WS_ROWS workspace; from then on
 * every call retracts the rows the previous call wrote and writes its own, so the tensors hold exactly this step's
 * dense gradient - bit-identical to ssdhead_multibox_step's - without 873 KB of zero background per image per step
 * ever being written (the streaming kernel runs forward-only: conf is read, nothing dense is stored).
 * Contract: between calls nobody else writes the two tensors or the rows workspace; after anything else touched them
 * (or the tensors were reallocated) zero-fill all three again.  A smaller batch may follow a larger one (the rows of
 * the images beyond B stay listed and are retracted when those images return).  R = 1: one GPU; R > 1: the batch is
 * sharded by image and the remaining arguments are those of ssdhead_multibox_step_sharded.  P < 65536. */
int ssdhead_multibox_step_resident(const float* loc_dev, const float* conf_dev,
                          const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                          const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                          int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                          double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                          uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                          void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                          void* ws_rows_dev, size_t ws_rows_bytes,
                          int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev,
                          int32_t* err_flag_dev, void* stream);
int ssdhead_mine(const float* loc_dev, const float* conf_dev,
                 const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                 const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                 const int32_t* best_prior_dev, const int32_t* npos_dev, const int32_t* npos_norm_dev,
                 const uint8_t* cls_u8_dev,
                 int B, int P, int C, int neg_ratio, float pos_iou,
                 double* sums_dev, float* losses_dev,
                 float* grad_loc_dev, float* grad_conf_dev,
                 uint32_t* mined_mask_dev, float* ce_dev,
                 void* ws_dev, size_t ws_bytes, void* stream);
/* ssdhead_mine with the gradients returned as PACKED ROWS instead of dense [B,P,*] tensors.  The gradient of this loss
 * is sparse - only positives and mined negatives (about 4 * Npos of the P rows of an image) carry one, Losses.py:177-197
 * - so a caller that scatters rows itself (or keeps its gradient buffers in host memory) needs no dense tensor at all.
 * Image b owns slots [b*row_cap, (b+1)*row_cap):  row_cnt[2b] = number of rows of the image (if it exceeds row_cap only
 * the first row_cap were stored - check it), row_cnt[2b+1] = how many of them are positives; slot s: row_idx = prior
 * index inside the image, grad_conf_rows [.,C] = (softmax - onehot)/N; the positives come first and also own
 * grad_loc_rows [.,4] = sign(loc - enc)/(4N).  The order of the rows inside an image is unspecified (the set is
 * deterministic).  Pair with ssdhead_ce_stream called WITHOUT gradient pointers (no zero background is needed). */
int ssdhead_mine_sparse(const float* loc_dev, const float* conf_dev,
                 const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                 const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                 const int32_t* best_prior_dev, const int32_t* npos_dev, const int32_t* npos_norm_dev,
                 const uint8_t* cls_u8_dev,
                 int B, int P, int C, int neg_ratio, float pos_iou,
                 double* sums_dev, float* losses_dev,
                 int row_cap, int32_t* row_cnt_dev /*[B,2]*/, int32_t* row_idx_dev /*[B,row_cap]*/,
                 float* grad_conf_rows_dev /*[B,row_cap,C]*/, float* grad_loc_rows_dev /*[B,row_cap,4]*/,
                 void* ws_dev, size_t ws_bytes, void* stream);
int ssdhead_multibox_loss(const float* loc_dev, const float* conf_dev,
                          const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                          const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                          const int32_t* best_prior_dev, const int32_t* npos_dev, const int32_t* npos_norm_dev,
                          const uint8_t* cls_u8_dev,
                          int B, int P, int C, int neg_ratio, float pos_iou,
                          double* sums_dev, float* losses_dev,
                          float* grad_loc_dev, float* grad_conf_dev,
                          uint32_t* mined_mask_dev, float* ce_dev,
                          void* ws_dev, size_t ws_bytes, void* stream);

/* losses[0..1] = { sums[0]/(4N), sums[1]/N } with N read from npos_norm_dev: used after the
 * loss sums of a sharded batch have been all-reduced. */
int ssdhead_finish_loss(const double* sums_dev, const int32_t* npos_norm_dev, float* losses_dev, void* stream);

/* grad_loc *= gout[0], grad_conf *= gout[1] (autograd upstream gradients of the two scalars,
 * read on the device; the kernel returns without touching memory when both are 1). */
int ssdhead_scale_grads(float* grad_loc_dev, size_t n_loc, float* grad_conf_dev, size_t n_conf,
                        const float* gout_dev /*[2]*/, void* stream);

/* ---- detection: inference(), Losses.py:11-98 ----------------------------------------
 * Per image: decode, softmax, per foreground class (0..C-2) keep prob >= min_score, sort by
 * descending prob (ties -> lower prior, T5), greedy NMS (suppress iou >= iou_thr), concatenate
 * class-major, and if more than top_k survive take the global top_k by descending prob
 * (ties -> earlier class-major position, T7).  Boxes are corner form, NOT clamped; fractional,
 * or multiplied by the image size when `img_wh_dev` [B,2] (w,h) is given (Losses.py:87-89).
 * `max_candidates` bounds the workspace: an image's candidate list holds (C-1) * max_candidates keys
 * (0 = P per class = every candidate, the reference's behaviour); if it overflows, out_cnt[b] = -1.
 * The per-class sweeps are run as ONE sweep per image in descending (prob, lower class, lower prior)
 * order with suppression tested inside a class only - the same keep/suppress decisions, the kept boxes
 * already in the order of the final global top-k - which stops once top_k + 1 boxes are kept: the
 * output is identical to the reference's full per-class sweeps (DESIGN.md 3.4).
 * Outputs: out_boxes [B,top_k,4], out_prob [B,top_k], out_cls int32 [B,top_k],
 *          out_prior int32 [B,top_k] (prior id of each detection; nullable), out_cnt int32 [B].
 * Kernels (short-list route, the default): a sampling kernel picks a score floor per image (>= min_score)
 * above which ~1600 candidates are expected; a persistent streaming kernel lists only the candidates above
 * it; the sweep kernel (per-image slice sort + class-parallel NMS + output) runs on that short list.  The
 * short list decides the output exactly when the sweep keeps top_k + 1 boxes inside it or the floor never
 * rose above min_score (a candidate's fate depends only on higher-scored candidates); for any other image
 * the sweep CTA lists the image again with the floor at min_score and sweeps the full list, so the output
 * never depends on the floor.  ssdhead_detect_fallbacks reports how many images of the last call needed
 * that.  The exhaustive route (two kernels: every candidate >= min_score listed, then the sweep) serves
 * calls with 0 < max_candidates < P, and every call when SSDHEAD_DETECT_SHORTLIST=0 is set in the
 * environment; only this route can report an overflowed cap (out_cnt[b] = -1).
 * P <= 131072, top_k <= ~1400.  Probabilities given to the _from_scores twin must be >= 0.
 * The workspace must be zero-filled before its FIRST use; every call leaves its counters zeroed. */
int ssdhead_detect(const float* loc_dev, const float* conf_dev, const float* pri_cxcywh_dev,
                   int B, int P, int C, float min_score, float iou_thr, int top_k,
                   const float* img_wh_dev, int max_candidates,
                   float* out_boxes_dev, float* out_prob_dev, int32_t* out_cls_dev, int32_t* out_prior_dev,
                   int32_t* out_cnt_dev, void* ws_dev, size_t ws_bytes, void* stream);

/* Stage-isolated twin of ssdhead_detect taking decoded boxes [B,P,4] (cxcywh) and class
 * probabilities [B,P,C] as given (the oracle's), so keep lists can be compared bit-exactly. */
int ssdhead_detect_from_scores(const float* boxes_cxcywh_dev, const float* probs_dev,
                               int B, int P, int C, float min_score, float iou_thr, int top_k,
                               const float* img_wh_dev, int max_candidates,
                               float* out_boxes_dev, float* out_prob_dev, int32_t* out_cls_dev, int32_t* out_prior_dev,
                               int32_t* out_cnt_dev, void* ws_dev, size_t ws_bytes, void* stream);

/* Number of images of the LAST ssdhead_detect* call on this workspace (same B, P, C, max_candidates) that the
 * short list did not decide and that were listed in full by their sweep CTA (0 .. B); blocks on `stream`.  A
 * caller that sees most images counted (heavy suppression: fewer than top_k survivors among the ~1600 best
 * candidates) may prefer SSDHEAD_DETECT_SHORTLIST=0.  No reference counterpart (a property of this implementation). */
int ssdhead_detect_fallbacks(const void* ws_dev, size_t ws_bytes, int B, int P, int C, int max_candidates,
                             int32_t* host_count, void* stream);

/* ---- evaluation: get_map(), Util.py:783-885 (VOC 11-point interpolated AP; consumer of the detect output) -------
 * Detections and ground truth are packed image-major with int32 offsets [num_images+1] (det_off, gt_off).  Per class:
 * detections ranked by descending score (ties -> lower detection index); walking that order, a detection is a true
 * positive iff its best-IoU gt of the same image and class (ties -> first gt) has IoU > iou_thr and is unclaimed
 * (Util.py:855-868); AP = mean over `recall_levels[11]` of the max precision at recall >= level; precision in fp64,
 * recall = cumTP * float32(1/#gt) as the reference's numpy/torch mix evaluates Util.py:872 (a class without detections
 * or without gt scores 0).  ap_out: double [num_fg]. */
size_t ssdhead_voc_ap_workspace_bytes(int N, int M, int num_fg);
int ssdhead_voc_ap(const float* det_boxes_xyxy_dev, const int32_t* det_cls_dev, const float* det_score_dev,
                   const int32_t* det_off_dev, int N,
                   const float* gt_boxes_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev, int M,
                   int num_images, int num_fg, float iou_thr, const double* recall_levels_dev /*[11]*/,
                   double* ap_out_dev, void* ws_dev, size_t ws_bytes, void* stream);

/* ---- head outputs per pyramid level (SURVEY.md 8(f) #3): Model.py:212-235 without the permute/cat round trip -----
 * The reference permutes each of its 12 conv outputs to NHWC, copies it (`.contiguous()`) and concatenates the six
 * levels into loc [B,8732,4] / conf [B,8732,21].  An NHWC (channels_last) conv output [B,H,W,A*21] already IS the row
 * layout [B, n_l, 21] of its level (n_l = H*W*A priors, cell-major then anchor - the prior order of Util.py:105-137),
 * so these entry points read the level tensors in place and write the gradients per level in the same layout:
 * no concatenated tensor exists in either direction.  count[l] priors per image in level l (sum = P), conf[l]
 * [B, count[l], C], loc[l] [B, count[l], 4], grads likewise (all or none); loc / grad_loc pointers 16-byte aligned, and
 * conf / grad_conf too for the fast (TMA) path - a level with unaligned conf pointers is read with plain loads. */
#define SSDHEAD_MAX_LEVELS 8
typedef struct ssdhead_levels {
    int32_t      num_levels;
    int32_t      count[SSDHEAD_MAX_LEVELS];
    const float* conf[SSDHEAD_MAX_LEVELS];
    const float* loc[SSDHEAD_MAX_LEVELS];
    float*       grad_conf[SSDHEAD_MAX_LEVELS];
    float*       grad_loc[SSDHEAD_MAX_LEVELS];
} ssdhead_levels;

/* ssdhead_multibox_step on per-level tensors: same two kernels, same outputs (the class map, best priors and counts
 * keep the global [B,P] prior indexing), results bit-identical to the concatenated call. */
int ssdhead_multibox_step_levels(const ssdhead_levels* levels,
                                 const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                 const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                                 int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                                 double* sums_dev, float* losses_dev,
                                 uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                                 void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                                 void* stream);
/* ... and of a batch sharded by image over R GPUs: ssdhead_multibox_step_sharded on per-level tensors. */
int ssdhead_multibox_step_levels_sharded(const ssdhead_levels* levels,
                                 const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                 const float* pri_xyxy_dev, const float* pri_cxcywh_dev,
                                 int B, int P, int C, int sumG, int neg_ratio, float pos_iou,
                                 double* sums_dev, float* losses_dev,
                                 uint8_t* cls_u8_dev, int32_t* best_prior_dev, int32_t* npos_dev,
                                 void* ws_loss_dev, size_t ws_loss_bytes, void* ws_match_dev, size_t ws_match_bytes,
                                 int R, int rank, unsigned int seq, void* const* peers_dev, void* xchg_local_dev,
                                 int32_t* err_flag_dev, void* stream);
/* ssdhead_detect on per-level tensors (grad pointers unused). */
int ssdhead_detect_levels(const ssdhead_levels* levels, const float* pri_cxcywh_dev,
                          int B, int P, int C, float min_score, float iou_thr, int top_k,
                          const float* img_wh_dev, int max_candidates,
                          float* out_boxes_dev, float* out_prob_dev, int32_t* out_cls_dev, int32_t* out_prior_dev,
                          int32_t* out_cnt_dev, void* ws_dev, size_t ws_bytes, void* stream);

/* ---- gt collate: Dataset.py:24-36 (difficult filter, standardisation) + train_function.py:62-63 (B small copies)
 * + Losses.py:129-130 (cat, cumsum) in one HOST pass ------------------------------------------------------------
 * B ragged host arrays -> the packed gt layout every entry point above takes: boxes [sumG,4], classes [sumG] fp32,
 * offsets int32 [B+1].  counts[i] boxes of image i are read from boxes[i] (xyxy, [counts[i],4]) and classes[i];
 * `difficult` (nullable, or null per image) drops boxes whose flag is non-zero unless keep_difficult != 0
 * (Dataset.py:28-30); `img_wh` (nullable, [B,2] = w,h) divides pixel boxes by (w,h,w,h) in fp32 (Dataset.py:35-36).
 * The outputs are host buffers with room for `capacity` boxes (page-locked memory from ssdhead_host_alloc makes the
 * single copy to the device asynchronous).  Returns sumG >= 0, SSDHEAD_E_WORKSPACE if `capacity` is too small, or
 * SSDHEAD_E_STATE if an image is left without a box (the reference fails on such a batch, Losses.py:153). */
int ssdhead_pack_gt(const float* const* boxes_host, const float* const* classes_host, const uint8_t* const* difficult_host,
                    const int32_t* counts, int B, int keep_difficult, const float* img_wh_host,
                    float* out_xyxy_host, float* out_cls_host, int32_t* out_off_host, int capacity);

/* ---- host-buffer front end (pinned staging + streams owned by the context) -----------
 * The same path for callers whose tensors live in host memory (what the reference's CPU
 * path sees).  Copies are pipelined against the kernels in image chunks. */
typedef struct ssdhead_ctx ssdhead_ctx;
int  ssdhead_ctx_create(ssdhead_ctx** out, int device, int maxB, int P, int C, int max_sumG, int top_k,
                        const float* pri_cxcywh_host);
void ssdhead_ctx_destroy(ssdhead_ctx* ctx);
/* page-locked host allocation helpers (so callers can hand in pinned buffers) */
void* ssdhead_host_alloc(size_t bytes);
void  ssdhead_host_free(void* p);

/* One training-head step on DEVICE tensors in a single call: ssdhead_multibox_step, or ssdhead_multibox_step_sharded
 * after ssdhead_ctx_xchg_import - two kernels on `stream`.  Asynchronous on `stream`;
 * sums double[2], losses float[2], grads nullable as a pair (all device pointers). */
int ssdhead_ctx_multibox_loss_dev(ssdhead_ctx* ctx, const float* loc_dev, const float* conf_dev,
                                  const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                  int B, int sumG, int neg_ratio, float pos_iou,
                                  double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                                  void* stream);
/* ssdhead_ctx_multibox_loss_dev with RESIDENT gradient tensors (ssdhead_multibox_step_resident; after ssdhead_ctx_xchg_import
 * the sharded step).  The context owns the rows workspace and remembers the two tensors.  fresh != 0: the context
 * zero-fills grad_loc [B,P,4] / grad_conf [B,P,C] and forgets the previous rows first (first call, new tensors, or
 * after anybody else wrote them); fresh == 0: the tensors must be the ones of the previous call and B at most the B
 * of the last fresh call - only that many images were zero-filled - (else SSDHEAD_E_STATE), and they must hold what
 * the previous call left in them. */
int ssdhead_ctx_multibox_loss_dev_resident(ssdhead_ctx* ctx, const float* loc_dev, const float* conf_dev,
                                  const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                  int B, int sumG, int neg_ratio, float pos_iou,
                                  double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                                  int fresh, void* stream);
/* ssdhead_ctx_multibox_loss_dev on per-level head tensors (ssdhead_levels, gradients inside the struct): one GPU, or
 * - after ssdhead_ctx_xchg_import - the sharded two-kernel step with global normalisation. */
int ssdhead_ctx_multibox_loss_levels_dev(ssdhead_ctx* ctx, const ssdhead_levels* levels,
                                         const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                         int B, int sumG, int neg_ratio, float pos_iou,
                                         double* sums_dev, float* losses_dev, void* stream);
/* The same step in two halves for a batch sharded by image over several GPUs: `begin` runs the match and
 * the CE streaming kernel and hands back a device pointer to this rank's int32 positive count; the
 * caller all-reduces it (NCCL, 4 bytes) and passes the total to `end` as npos_norm_dev (null = local
 * count), which mines and writes the gradients; the caller then all-reduces sums[2] and calls
 * ssdhead_finish_loss. */
int ssdhead_ctx_multibox_loss_begin(ssdhead_ctx* ctx, const float* conf_dev,
                                    const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                    int B, int sumG, float pos_iou, float* grad_loc_dev, float* grad_conf_dev,
                                    int32_t** npos_total_dev, void* stream);
int ssdhead_ctx_multibox_loss_end(ssdhead_ctx* ctx, const float* loc_dev, const float* conf_dev,
                                  const float* gt_xyxy_dev, const float* gt_cls_dev, const int32_t* gt_off_dev,
                                  int B, int neg_ratio, float pos_iou, const int32_t* npos_norm_dev,
                                  double* sums_dev, float* losses_dev, float* grad_loc_dev, float* grad_conf_dev,
                                  void* stream);
/* Sharded batches without NCCL: every rank exports the IPC handle of its exchange buffer (64 bytes), the handles are
 * gathered by the caller (e.g. torch.distributed.all_gather_object) and imported; from then on
 * ssdhead_ctx_multibox_loss_dev runs ssdhead_multibox_step_sharded and returns GLOBAL losses.  All ranks must call it
 * in lock step.  ssdhead_ctx_xchg_error returns 1 if a wait for a peer ever expired. */
int ssdhead_ctx_xchg_export(ssdhead_ctx* ctx, void* handle64_out);
int ssdhead_ctx_xchg_import(ssdhead_ctx* ctx, const void* handles /*[R][64]*/, int R, int rank);
int ssdhead_ctx_xchg_error(ssdhead_ctx* ctx);
/* ssd() with host buffers: losses_host[2] = (loc_loss, conf_loss); grads nullable as a pair.
 * Copies, kernels and copies back are pipelined in image chunks on the context's streams; pass
 * page-locked buffers (ssdhead_host_alloc) so the copies are asynchronous - a page-locked `loc` is not copied at
 * all (the kernels read the few rows they need in place), and page-locked gradient buffers are zeroed by host threads
 * and receive only their non-zero rows from the GPU.
 * Blocks until done. */
int ssdhead_ctx_multibox_loss_host(ssdhead_ctx* ctx, const float* loc_host, const float* conf_host,
                                   const float* gt_xyxy_host, const float* gt_cls_host, const int32_t* gt_off_host,
                                   int B, int neg_ratio, float pos_iou,
                                   float* losses_host, float* grad_loc_host, float* grad_conf_host);
/* ssd() with host buffers and the gradients returned as packed rows (layout: ssdhead_mine_sparse).  Nothing dense is
 * zeroed, copied or written on either side: page-locked output buffers receive their rows straight from the mining
 * kernel (about 100 bytes per row over PCIe); pageable ones go through device staging.  This is the cheap way to hand
 * the loss gradients to a host-side consumer: ~5 MB instead of 223 MB at batch 256.
 * After ssdhead_ctx_xchg_import BOTH host entry points treat the batch as one shard of a batch spread over R GPUs:
 * the positive count and the loss sums cross GPUs through the exchange buffers (NVLink peer stores from two
 * single-thread kernels), losses and gradients carry the global normalisation of Losses.py:182,197, and all ranks
 * must call in lock step. */
int ssdhead_ctx_multibox_loss_host_sparse(ssdhead_ctx* ctx, const float* loc_host, const float* conf_host,
                                          const float* gt_xyxy_host, const float* gt_cls_host, const int32_t* gt_off_host,
                                          int B, int neg_ratio, float pos_iou, float* losses_host,
                                          int row_cap, int32_t* row_cnt_host /*[B,2]*/, int32_t* row_idx_host /*[B,row_cap]*/,
                                          float* grad_conf_rows_host /*[B,row_cap,C]*/, float* grad_loc_rows_host /*[B,row_cap,4]*/);
/* inference() over a batch with host buffers; outputs as ssdhead_detect. */
int ssdhead_ctx_detect_host(ssdhead_ctx* ctx, const float* loc_host, const float* conf_host, int B,
                            float min_score, float iou_thr,
                            float* out_boxes_host, float* out_prob_host, int32_t* out_cls_host,
                            int32_t* out_prior_host, int32_t* out_cnt_host);

#ifdef __cplusplus
}
#endif
#endif /* SSDHEAD_H_ */
