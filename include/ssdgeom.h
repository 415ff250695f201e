/*
 * ssdgeom.h -- C ABI of libssdgeom.so: the B200-native (sm_100a) SSD box-geometry hot path.
 *
 * Drop-in boundary for the hot path of AcherStyx/SSD-Object-Detection.  The reference has no
 * FFI of its own (it is pure Python); each entry point below names the reference callable it
 * replaces (file:line relative to the reference root).  INTEGRATION.md shows the ctypes stub a
 * reference maintainer would add.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Unless a parameter says "host", every data pointer is a
 *    DEVICE pointer; inputs are const and never modified; outputs are fully overwritten.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All work is
 *    stream-ordered and asynchronous; nothing here synchronises unless documented.
 *  - The library never allocates device memory inside a compute entry point: the caller passes
 *    a workspace of at least ssdg_*_workspace_bytes() bytes (256-byte aligned).
 *  - Return value: 0 = OK; negative = argument error mirroring the reference's asserts
 *    (SSDG_ERR_*); positive = a cudaError_t (or SSDG_ERR_NCCL_BASE + ncclResult_t from
 *    ssdg_comm_*).  Nothing throws across the boundary.
 *  - Data-dependent errors that only the device can see (num_pos == 0, hard-negative k out of
 *    range) are reported through a status word in the result block, see each function.
 *  - There is no CPU fallback: without a CUDA device every compute entry point returns a
 *    cudaError_t.
 */
#ifndef SSDGEOM_H_
#define SSDGEOM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSDG_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define SSDG_API __attribute__((visibility("default")))
#else
#define SSDG_API
#endif

/* ---- status codes -------------------------------------------------------------------------- */
#define SSDG_OK 0
#define SSDG_ERR_ARG (-1)          /* null pointer / non-positive size / bad enum               */
#define SSDG_ERR_TOO_MANY_GT (-2)  /* n_targets > n_defaults           utils/bbox.py:50         */
#define SSDG_ERR_THRESH (-3)       /* thresh <= 0 (or NaN)             utils/bbox.py:51         */
#define SSDG_ERR_SHAPE (-4)        /* inconsistent shapes              models/ssd_model.py:347-351 */
#define SSDG_ERR_NO_POSITIVE (-5)  /* num_pos == 0 (reference: IndexError at models/ssd_model.py:369) */
#define SSDG_ERR_TOPK_RANGE (-6)   /* ratio*num_pos > B*A (reference: tf.math.top_k error, :368)     */
#define SSDG_ERR_WORKSPACE (-7)    /* workspace null, misaligned or too small                   */
#define SSDG_ERR_ALIGN (-8)        /* a pointer that must be 16-byte aligned is not             */
#define SSDG_ERR_LIMIT (-9)        /* size beyond an implementation limit (see function)        */
#define SSDG_ERR_POS_NEG_OVERLAP (-10) /* a positive prior was mined as negative  models/ssd_model.py:375 */
#define SSDG_ERR_NO_NCCL (-11)     /* ssdg_comm_*: libnccl.so.2 could not be loaded              */
#define SSDG_ERR_LABEL_RANGE (-12) /* a positive prior's class id is outside [0, C) (TensorFlow's
                                      sparse_softmax_cross_entropy_with_logits raises; :357)     */
#define SSDG_ERR_STALE_INDEX (-13) /* the prior index does not belong to these priors (content check) */
#define SSDG_ERR_NCCL_BASE 10000   /* ssdg_comm_*: SSDG_ERR_NCCL_BASE + ncclResult_t             */

/* element types for the box arrays whose dtype decides the matcher's rounding */
#define SSDG_F32 0
#define SSDG_F64 1
/* (ssdg_comm_allreduce_sum only) */
#define SSDG_I32 2
#define SSDG_I64 3

SSDG_API const char* ssdg_status_string(int status);
SSDG_API int ssdg_version(void);

/* ---- device / memory helpers (so host code needs no other CUDA binding) --------------------- */
SSDG_API int ssdg_device_count(int* count);
SSDG_API int ssdg_set_device(int device);
SSDG_API int ssdg_get_device(int* device);
SSDG_API int ssdg_device_alloc(void** dptr, size_t bytes);
SSDG_API int ssdg_device_free(void* dptr);
SSDG_API int ssdg_host_alloc(void** hptr, size_t bytes);           /* pinned */
SSDG_API int ssdg_host_free(void* hptr);
SSDG_API int ssdg_memcpy_h2d(void* dst, const void* src_host, size_t bytes, void* stream);
SSDG_API int ssdg_memcpy_d2h(void* dst_host, const void* src, size_t bytes, void* stream);
SSDG_API int ssdg_memset(void* dst, int value, size_t bytes, void* stream);
SSDG_API int ssdg_stream_create(void** stream);
SSDG_API int ssdg_stream_create_priority(void** stream, int high_priority); /* non-blocking; 0: lowest device priority, 1: highest, k >= 2: k-1 levels below the highest */
SSDG_API int ssdg_stream_destroy(void* stream);
SSDG_API int ssdg_stream_sync(void* stream);
SSDG_API int ssdg_event_create(void** event);
SSDG_API int ssdg_event_destroy(void* event);
SSDG_API int ssdg_event_record(void* event, void* stream);
SSDG_API int ssdg_stream_wait_event(void* stream, void* event);
SSDG_API int ssdg_event_elapsed_ms(void* start, void* stop, float* ms); /* synchronises on `stop` */

/* ---- per-kernel timing (for bench.py's roofline line) --------------------------------------------
 * When enabled, the dominant kernels (SSDG_PROF_MATCH: search + match_kernel, SSDG_PROF_CE: ce_kernel or
 * lossprep_kernel, SSDG_PROF_FILTER: filter_kernel, SSDG_PROF_NMS: nms_kernel, ...) are bracketed by CUDA
 * events on the stream they are launched on.  ssdg_profile_last_ms synchronises on the kernel's stop event
 * and returns the duration of its most recent launch on the CURRENT device.  A measurement aid: the switch is
 * process-wide and the events are per device, so enable it only from a driver that launches from one thread
 * per device (bench.py); it is off by default and compute entry points are otherwise free of global state. */
#define SSDG_PROF_MATCH 0
#define SSDG_PROF_CE 1
#define SSDG_PROF_FILTER 2
#define SSDG_PROF_NMS 3
#define SSDG_PROF_SEARCH 5      /* search_kernel (SSDG_PROF_MATCH covers search + per-image kernel) */
#define SSDG_PROF_LOSS_TAIL 6   /* select_kernel x2 + final_kernel */
#define SSDG_PROF_GRAD 7        /* grad_kernel */
SSDG_API int ssdg_profile_enable(int enable);
SSDG_API int ssdg_profile_last_ms(int which, float* ms);
/* Begin / end of the bracketed kernel relative to a caller-recorded event (ms): a timeline of one step. */
SSDG_API int ssdg_profile_span_ms(int32_t which, void* ref_event, float* begin_ms, float* end_ms);

/* ---- A1: anchors -------------------------------------------------------------------------------
 * Replaces SSDObjectDetectionModel._build_prior_box(size_list)      models/ssd_model.py:173-194
 * Level l (feat_h[l] x feat_w[l] cells, y outer / x inner) emits per cell, in this order:
 *   (s,s), (sqrt(s*s'),sqrt(s*s')), then for every ratio r of the level (s*sqrt r, s/sqrt r),
 *   (s/sqrt r, s*sqrt r), with s = s_k[l]/input_size, s' = s_k[l+1]/input_size; centres
 *   ((x+.5)/w, (y+.5)/h); float64, un-clipped -- bit-identical to the reference's host math.
 * All table pointers are HOST pointers.  ratio_offsets[l]..ratio_offsets[l+1] indexes `ratios`.
 */
SSDG_API int64_t ssdg_prior_count(const int32_t* feat_h, const int32_t* feat_w, const int32_t* ratio_offsets,
                         int32_t n_levels);
SSDG_API int ssdg_prior_boxes(const int32_t* feat_h, const int32_t* feat_w, const double* s_k /*[n_levels+1]*/,
                     const int32_t* ratio_offsets /*[n_levels+1]*/, const double* ratios,
                     int32_t n_levels, double input_size, double* out_priors /*dev [A,4]*/,
                     int64_t n_priors, void* stream);

/* ---- A3+A4+A5: target assignment -----------------------------------------------------------------
 * Replaces match_bbox(cls, bbox, default_box, thresh)               utils/bbox.py:44-91
 *      and apply_anchor_box(matched, default_box)                   utils/bbox.py:94-101
 *      as chained per image by get_train_set/batch_data_iter        models/ssd_model.py:211-224
 * for a whole batch: image i owns ground-truth rows gt_offsets[i]..gt_offsets[i+1] (CSR).
 *
 *   gt_boxes   [sum T,4] cxcywh, dtype gt_dtype (SSDG_F32 on the training path)
 *   gt_cls     [sum T]   float32 class ids (data_loaders/ssd/make_dataset.py:57); truncated to int32
 *   gt_offsets [B+1]     int32, device
 *   priors     [A,4]     cxcywh, dtype prior_dtype (SSDG_F64 on the training path), shared by the batch
 *   max_gt     upper bound on any image's T (sizes shared memory); images with T > max_gt or
 *              T > A raise bit 0 / bit 1 of the status word (ssdg_match_status)
 * Outputs (any may be NULL to skip it):
 *   out_cls   int32 [B,A]   labeled_cls      (0 where unmatched, as the reference)
 *   out_box   float [B,A,4] labeled_boxes    (matched ground-truth box, 0 where unmatched)
 *   out_loc   float [B,A,4] apply_anchor_box(labeled_boxes, priors) cast to float32
 *   out_mask  uint8 [B,A]   mask
 *   out_match int32 [B,A]   index (within the image) of the matched ground truth, -1 if none
 * Bit-exact contract: out_cls, out_box, out_mask, out_match equal the reference's; the IoU is
 * evaluated with the reference's exact operation order and dtype mix (no FMA contraction).
 * Limits: A < 2^21, max_gt <= 2048.
 */
SSDG_API size_t ssdg_match_workspace_bytes(int32_t batch, int32_t n_priors, int32_t max_gt);
/* Optional acceleration structure for a fixed prior set (the reference builds its priors once, in
 * __init__, models/ssd_model.py:60,164): a permutation that groups priors of identical shape into
 * spatially compact 32-prior tiles, plus per-tile statistics, so the matcher's tile-level IoU bound is
 * tight.  It changes no result.  ssdg_prior_index_build copies the priors to the host, sorts there and
 * SYNCHRONISES; call it once per prior set.  `index` is device memory of ssdg_prior_index_bytes bytes
 * (256-byte aligned) that must stay alive and unmodified while it is passed to ssdg_match_encode, on the device
 * it was built on.  The index remembers a content checksum of its priors: every ssdg_match_encode that is given
 * an index re-derives it on the device and raises status bit 3 (ssdg_match_status) when the priors were changed
 * afterwards (e.g. ssdg_priors_clip in place) or the index belongs to another array.  ssdg_prior_index_destroy
 * forgets the index (call it before freeing or reusing the memory). */
SSDG_API size_t ssdg_prior_index_bytes(int32_t n_priors);
SSDG_API int ssdg_prior_index_build(const void* priors, int32_t prior_dtype, int32_t n_priors, void* index,
                           size_t index_bytes, void* stream);
SSDG_API int ssdg_prior_index_destroy(void* index);
SSDG_API int ssdg_match_encode(const void* gt_boxes, int32_t gt_dtype, const float* gt_cls,
                      const int32_t* gt_offsets, const void* priors, int32_t prior_dtype,
                      const void* prior_index /* NULL or from ssdg_prior_index_build for these priors */,
                      int32_t batch, int32_t n_priors, int32_t max_gt, double thresh,
                      int32_t* out_cls, float* out_box, float* out_loc, uint8_t* out_mask,
                      int32_t* out_match, void* workspace, size_t workspace_bytes, void* stream);
/* Synchronous: copies the status word of the last ssdg_match_encode on `workspace` to *status
 * (bit 0: some T > max_gt, bit 1: some T > A -- those images were written as all-unmatched, where the reference
 * matches every box / asserts utils/bbox.py:50; bit 2: internal log overflow handled by rescan -- informational;
 * bit 3: the prior index does not belong to these priors -- results invalid).  The word is the second uint32 of
 * the workspace: an asynchronous caller copies workspace[4..8) itself (ssdgeom/pipeline.py does, with the results). */
SSDG_API int ssdg_match_status(const void* workspace, int32_t* status, void* stream);

/* Stand-alone encode / decode over [batch, A, 4] boxes against shared priors.
 * ssdg_encode replaces apply_anchor_box                             utils/bbox.py:94-101
 * ssdg_decode replaces the inline decode of visualize_dataset       models/ssd_model.py:466-467
 *   (xy = (t_xy*d_wh + d_xy)*scale, wh = exp(t_wh)*d_wh*scale; scale = 300 in the reference).
 * Arithmetic is float64 from exactly-converted inputs, rounded once to the output dtype. */
SSDG_API int ssdg_encode(const void* boxes, int32_t box_dtype, const void* priors, int32_t prior_dtype,
                int64_t batch, int32_t n_priors, void* out, int32_t out_dtype, void* stream);
SSDG_API int ssdg_decode(const float* loc, const void* priors, int32_t prior_dtype, int64_t batch,
                int32_t n_priors, double scale, float* out, void* stream);

/* Element-wise IoU of paired rows: replaces iou_n (utils/bbox.py:28-41; clamp 1e-10) when
 * clamp_eps != 0 and iou (utils/bbox.py:6-25; clamp 0.0) when clamp_eps == 0.  Each side is
 * evaluated in its own dtype and promoted as NumPy does; out dtype = SSDG_F64 if either side is. */
SSDG_API int ssdg_iou_pairs(const void* boxes_1, int32_t dtype_1, const void* boxes_2, int32_t dtype_2,
                   int64_t n, int32_t use_eps_clamp, void* out, void* stream);

/* ---- A6: multibox loss ------------------------------------------------------------------------------
 * Replaces SSDObjectDetectionModel._ssd_loss(y_true, y_pred)        models/ssd_model.py:341-396
 *   gt_cls int32 [B,A], gt_box float [B,A,4], gt_mask uint8 [B,A], pred_box float [B,A,4],
 *   pred_cls float [B,A,C] (16-byte aligned); background = class C-1 (:365); plain L1 (:384-386);
 *   hard negatives: every prior whose background CE >= the (neg_ratio*num_pos)-th largest over
 *   the WHOLE batch (:368-372, ties kept).
 * out_result: double[SSDG_LOSS_RESULT_LEN] on the device:
 *   [0] total  [1] "cls loss pos"  [2] "cls loss neg"  [3] "loc loss"
 *   [4] num_pos [5] num_neg [6] mining threshold (k-th largest background CE)
 *   [7] status: 0 OK, SSDG_ERR_NO_POSITIVE, SSDG_ERR_TOPK_RANGE, SSDG_ERR_POS_NEG_OVERLAP,
 *       SSDG_ERR_LABEL_RANGE (then [0..3] are NaN)
 *   [8] sum of positive CE [9] sum of mined-negative CE [10] sum of positive L1 (the separable
 *   sums a data-parallel caller all-reduces together with [4],[5]) [11] this shard's own positives
 *   [12] data-dependent errors seen by this shard (positives mined as negatives + class ids out of
 *        range): additive, so that every shard of a data-parallel run agrees on success
 * out_neg_mask (optional) uint8 [B,A]: the mined negative mask.
 * out_neg_ce   (optional) float [B,A]: per-prior background CE * (1-pos) (the mining input).
 * grad_box / grad_cls (optional, both or neither): d total / d pred_box, d total / d pred_cls --
 *   what tape.gradient back-propagates (models/ssd_model.py:248).
 */
#define SSDG_LOSS_RESULT_LEN 16
SSDG_API size_t ssdg_loss_workspace_bytes(int64_t batch, int32_t n_priors, int32_t n_classes);
SSDG_API int ssdg_multibox_loss(const int32_t* gt_cls, const float* gt_box, const uint8_t* gt_mask,
                       const float* pred_box, const float* pred_cls, int64_t batch,
                       int32_t n_priors, int32_t n_classes, int32_t neg_ratio, double* out_result,
                       uint8_t* out_neg_mask, float* out_neg_ce, float* grad_box, float* grad_cls,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Cross-shard (exact batch-global) mining: the same loss when the batch of models/ssd_model.py:341-396 is
 * split over several devices and the threshold of :368-372 must still be the k-th largest background CE
 * of the WHOLE batch (SURVEY.md section 8e, "exact-global option").  The loss runs in four stages; between
 * them the caller sums one exchange buffer over the shards (ncclAllReduce / torch.distributed, in place):
 *   stage 0  CE pass                 then sum  exchange 3 (int64 x1: positives) and exchange 0 (int32 x2048)
 *   stage 1  radix level 1           then sum  exchange 1 (int32 x2048)
 *   stage 2  radix level 2           then sum  exchange 2 (int32 x2048)
 *   stage 3  mask, sums, result      then sum  out_result[8..12] and [5]:  loss = ([8] + [10]) / sum[11] + [9] / sum[5],
 *                                              valid iff [7] == 0 and sum[12] == 0
 *   stage 4  gradient (optional; needs grad_box / grad_cls) -- AFTER the stage-3 exchange: it reads the summed
 *            num_neg [5] (and the global num_pos [4]), so the gradient of every shard is the slice of the
 *            single-device gradient of the whole batch
 * Every stage takes the arguments of ssdg_multibox_loss (same buffers each time) plus global_priors =
 * sum over shards of batch * n_priors, and optionally (both or neither, else NULL) the per-prior softmax statistics
 * of ssdg_detect_stage so that stage 0 skips its own pass over the logits (see ssdg_multibox_loss_fused).  After stage 3 out_result[4] is the global positive count, [11] the
 * shard's own, [6] the global threshold, and out_neg_mask equals the single-device mask of the whole batch.
 */
SSDG_API int ssdg_multibox_loss_stage(int32_t stage, int64_t global_priors, const float* row_ml,
                       const float* row_negbg, const int32_t* gt_cls,
                       const float* gt_box, const uint8_t* gt_mask, const float* pred_box,
                       const float* pred_cls, int64_t batch, int32_t n_priors, int32_t n_classes,
                       int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask, float* out_neg_ce,
                       float* grad_box, float* grad_cls, void* workspace, size_t workspace_bytes,
                       void* stream);
SSDG_API int ssdg_loss_exchange(void* workspace, int32_t which, void** out_ptr, int64_t* out_count);

/* The same loss when the post-processing branch has already streamed the same logits: ssdg_detect_stage(0, ...)
 * with out_row_ml / out_row_negbg leaves per prior (row max, log sum exp(x - max)) and the background CE; this
 * entry point then needs no second pass over pred_cls -- positives gather their one ground-truth logit.
 * row_ml float [B*A,2], row_negbg float [B*A]; everything else as ssdg_multibox_loss. */
SSDG_API int ssdg_multibox_loss_fused(const float* row_ml, const float* row_negbg, const int32_t* gt_cls,
                       const float* gt_box, const uint8_t* gt_mask, const float* pred_box,
                       const float* pred_cls, int64_t batch, int32_t n_priors, int32_t n_classes,
                       int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask, float* out_neg_ce,
                       float* grad_box, float* grad_cls, void* workspace, size_t workspace_bytes,
                       void* stream);

/* ---- data-parallel exchange (SURVEY.md section 8b / 8e) ---------------------------------------------------
 * The path shards by image (batch_data_iter is a per-image loop, models/ssd_model.py:211-215; NMS is per image
 * and class), so the only cross-device step is the loss's: with per-shard mining -- what the reference does per
 * slice under split_batch, models/ssd_model.py:235-256 -- the seven additive words out_result[4..10] are summed
 * once per step; with exact batch-global mining (:368-372) the exchange buffers of ssdg_multibox_loss_stage.
 * These entry points wrap NCCL (bound at run time from libnccl.so.2; SSDG_ERR_NO_NCCL if absent) so that a
 * TensorFlow or plain C host needs no other collective library:
 *   rank 0:  ssdg_comm_unique_id(id)  -> ship the SSDG_COMM_ID_BYTES bytes to every rank (any out-of-band channel)
 *   all:     ssdg_comm_init_rank(&comm, id, world, rank)      (collective; uses the current device)
 *   step:    ssdg_comm_allreduce_sum(comm, buf, count, dtype, stream)   in place, stream-ordered, asynchronous
 *   end:     ssdg_comm_destroy(comm)
 * ssdg_comm_allreduce_sum_multi sums n buffers as one NCCL group (one launch). */
#define SSDG_COMM_ID_BYTES 128
SSDG_API int ssdg_comm_available(int* nccl_version /* may be NULL */);
SSDG_API int ssdg_comm_unique_id(void* id_out /* host, SSDG_COMM_ID_BYTES */);
SSDG_API int ssdg_comm_init_rank(void** comm_out, const void* id /* host */, int32_t world, int32_t rank);
SSDG_API int ssdg_comm_world(void* comm, int32_t* world, int32_t* rank);
SSDG_API int ssdg_comm_allreduce_sum(void* comm, void* buf, int64_t count, int32_t dtype, void* stream);
SSDG_API int ssdg_comm_allreduce_sum_multi(void* comm, int32_t n, void* const* bufs, const int64_t* counts,
                                  const int32_t* dtypes, void* stream);
SSDG_API int ssdg_comm_destroy(void* comm);

/* ---- input glue (SURVEY.md section 8f, row 3) ----------------------------------------------------------
 * ssdg_gt_prepare replaces, for a whole batch of annotation rows at once,
 *   COCODataLoader.gen            data_loaders/coco/make_dataset.py:132   bbox[:, :2] += bbox[:, 2:] / 2
 *   SSDDataLoader._coco2ssd       data_loaders/ssd/make_dataset.py:43-44  box /= [w, h, w, h]
 * xywh [rows,4] pixel boxes (float64 as decoded from the annotation file, or float32), img_wh int32 [B,2]
 * (width, height of each image), gt_offsets int32 [B+1] (CSR rows per image) -> out_boxes float32
 * [rows,4] relative cxcywh: exactly the array the reference hands to match_bbox.
 * ssdg_image_normalize replaces batch_data_iter's (image - 0.5) * 2      models/ssd_model.py:214
 * on n float32 values (in and out may alias).
 */
SSDG_API int ssdg_gt_prepare(const void* xywh, int32_t dtype, const int32_t* img_wh, const int32_t* gt_offsets,
                    int64_t batch, int64_t rows, float* out_boxes, void* stream);
SSDG_API int ssdg_image_normalize(const float* in, float* out, int64_t n, void* stream);

/* ---- generalised anchor tables (SURVEY.md section 8f, row 4) --------------------------------------------
 * The reference's rule (models/ssd_model.py:173-194) neither clips priors nor uses variances; SSD variants do.
 * ssdg_priors_clip clamps every component of [A,4] cxcywh priors to [0,1] in place.  ssdg_loc_scale multiplies
 * encoded offsets [rows,4] by (sxy, sxy, swh, swh): 1/variance after ssdg_encode / ssdg_match_encode, variance
 * before ssdg_decode / ssdg_detect (in and out may alias).  Variance 1 and no clipping reproduce the reference. */
SSDG_API int ssdg_priors_clip(void* priors, int32_t dtype, int64_t n_priors, void* stream);
SSDG_API int ssdg_loc_scale(const float* in, float* out, int64_t rows, float scale_xy, float scale_wh, void* stream);

/* ---- A7+A8+A9: post-processing ------------------------------------------------------------------------
 * Replaces the head of SSDObjectDetectionModel.visualize            models/ssd_model.py:477-490
 *   (softmax, max foreground score, arg-max class, threshold mask) and the decode of
 *   visualize_dataset (:466-467, scale 1.0 here), and adds the per-class NMS the reference lacks
 *   (spec: oracle/ssd_oracle.py nms_per_class; PARITY UNPINNED, SURVEY.md section 8c):
 *   classes 0..C-2, candidates score > score_thresh, visit order (score desc, prior index asc),
 *   first top_k only, suppress when iou (utils/bbox.py:13-25, float32) > iou_thresh.
 * Outputs (any may be NULL except out_kept/out_count):
 *   out_kept   int32 [B,C-1,top_k] kept prior indices in visit order, -1 padded
 *   out_count  int32 [B,C-1]
 *   out_kept_score float [B,C-1,top_k] (0 padded)
 *   out_boxes  float [B,A,4] decoded cxcywh (relative units)
 *   out_probs  float [B,A,C] softmax (parity / debugging; large)
 *   head_*: score float [B,A], cls int32 [B,A], mask uint8 [B,A] at head_thresh (:481-488)
 * Limits: top_k <= 1024, batch * ceil(A/32) < 2^31.
 * Workspace: one candidate list per (image, class) with room for EVERY prior (no input can overflow it) --
 *   batch * (C-1) * ceil(A/32)*32 * 8 bytes (1.4 GB at SSD300 B=256, 23 GB at SSD512 B=1024; only the part that holds
 *   candidates, ~33 MB, is ever touched) -- plus the decoded boxes.  The size depends on the current device's SM count
 *   (the filter's launch geometry); query it on the device the call will run on.
 */
SSDG_API size_t ssdg_detect_workspace_bytes(int64_t batch, int32_t n_priors, int32_t n_classes, int32_t top_k);
SSDG_API int ssdg_detect(const float* pred_cls, const float* pred_box, const void* priors,
                int32_t prior_dtype, int64_t batch, int32_t n_priors, int32_t n_classes,
                float score_thresh, int32_t top_k, float iou_thresh, int32_t* out_kept,
                int32_t* out_count, float* out_kept_score, float* out_boxes, float* out_probs,
                float head_thresh, float* head_score, int32_t* head_cls, uint8_t* head_mask,
                void* workspace, size_t workspace_bytes, void* stream);
/* The same call in two stream-ordered stages sharing the workspace: stage 0 = softmax filter, decode and
 * the per-class candidate lists (the pass over the logits, HBM-bound), stage 1 = per-class NMS (instruction-bound).  A
 * pipeline can enqueue them on different streams -- ordered by an event -- so that the NMS shares the SMs
 * with an HBM-bound kernel of another branch (ssdgeom/pipeline.py).  out_row_ml float [B*A,2] / out_row_negbg
 * float [B*A] (both or neither, stage 0): per-prior softmax statistics for ssdg_multibox_loss_fused. */
SSDG_API int ssdg_detect_stage(int32_t stage, const float* pred_cls, const float* pred_box, const void* priors,
                int32_t prior_dtype, int64_t batch, int32_t n_priors, int32_t n_classes,
                float score_thresh, int32_t top_k, float iou_thresh, int32_t* out_kept,
                int32_t* out_count, float* out_kept_score, float* out_boxes, float* out_probs,
                float head_thresh, float* head_score, int32_t* head_cls, uint8_t* head_mask,
                float* out_row_ml, float* out_row_negbg, void* workspace, size_t workspace_bytes,
                void* stream);

/* Per-class NMS on caller-supplied scores and decoded boxes (the second stage alone):
 *   probs float [B,A,C] (16-byte aligned), boxes float [B,A,4]. */
SSDG_API int ssdg_nms(const float* probs, const float* boxes, int64_t batch, int32_t n_priors,
             int32_t n_classes, float score_thresh, int32_t top_k, float iou_thresh,
             int32_t* out_kept, int32_t* out_count, float* out_kept_score, void* workspace,
             size_t workspace_bytes, void* stream);

/* ---- A11: detection evaluation ---------------------------------------------------------------------------
 * The reference has no evaluation code.  COCO's AP (pycocotools COCOeval.evaluateImg + accumulate, iouType "bbox",
 * area range "all", no crowd / ignore flags) over the kept lists of ssdg_detect, accumulated on the device over
 * batches and data-parallel ranks (spec: tests/coco_eval_oracle.py; PARITY UNPINNED against pycocotools on pixel
 * boxes, bit-exact against that restatement).
 *   detections of (image, class c): the first min(count, max_dets) entries of the kept list (already in score desc,
 *     prior asc order); ground truth of (image, c): the image's CSR rows whose class (gt_cls truncated to int32, as
 *     ssdg_match_encode) is c, in row order.
 *   IoU in float64 from the exactly promoted float32 cxcywh boxes: x0 = cx - 0.5w, x1 = cx + 0.5w (y alike),
 *     iw = min(x1) - max(x0), ih alike, 0 unless iw > 0 and ih > 0, else inter / ((wd*hd + wg*hg) - inter).
 *   matching at threshold t: visit the detections in order; best = min(t, 1 - 1e-10); over the unmatched ground
 *     truth rows in order, skip iou < best, else best = iou and m = row (the last of equal IoUs wins); m >= 0 is a TP.
 * Each image has a GLOBAL index image_base + i, unique over batches and ranks, that orders equal scores.
 *
 * State (caller-owned device memory, 256-byte aligned, ssdg_eval_state_bytes bytes; K = n_classes - 1,
 * M = max_images, D = max_dets):
 *   int32 header[64]  [0] GT rows with a class outside [0, K)  [1] images with more GT rows than max_gt
 *                     [2] slots written more than once (set by finalize)  [3] kept prior indices outside [0, A)
 *   uint32 flags[K][M][D]  bits 0..15: TP at threshold k, bit 16: present
 *   int32 n_gt[K][M]       ground-truth rows per (class, image)
 *   int64 keys[K][M][D]    score_bits << 32 | (0xFFFFFFFF - (image << 10 | rank)); 0 = empty
 * One fixed slot per (class, global image, rank) with exactly one writer: no global atomics on the slots,
 * deterministic, and re-adding a batch with the same image_base overwrites it.  12 bytes per slot: COCO val
 * (5 000 images, 80 classes, 100 detections) takes 480 MB.
 * Limits: max_images < 2^22, max_dets <= 1024 and <= top_k, K*M*D < 2^31, n_thresholds <= 16, max_gt <= 2048,
 * n_recall <= 256.
 *
 * Data parallel: every slot is written by one rank and zero on the others, so summing the two buffers of
 * ssdg_eval_exchange over the ranks (ssdg_comm_allreduce_sum: which 0 as SSDG_I64, which 1 as SSDG_I32) is an
 * all-gather.  A slot written by two ranks carries its present bit into bit 17: finalize reports it (header[2]).
 *
 * Finalize (once per evaluation, leaves the state unchanged): records of class c in (score desc, global image asc,
 * rank asc) order; tp / fp cumulative sums as integers; rc = tp / n_gt, pr = tp / ((fp + tp) + 2^-52), pr made
 * non-increasing from the right; precision[t][r][c] = pr[searchsorted_left(rc, recall_thresholds[r])], 0 past the
 * last detection; recall[t][c] = rc[-1] (0 without detections); classes without ground truth: -1 in both.
 * Outputs: precision f64[T][R][K], recall f64[T][K], n_gt i64[K], n_det i64[K] (device).
 * Workspace: ssdg_eval_finalize_workspace_bytes (the sorted copy of the slots plus the sort's temporary storage;
 * the size query needs a CUDA device).
 */
SSDG_API size_t ssdg_eval_state_bytes(int32_t n_classes, int64_t max_images, int32_t max_dets,
                                      int32_t n_thresholds);   /* 0: arguments out of range */
SSDG_API int ssdg_eval_reset(void* state, size_t state_bytes, void* stream);
SSDG_API int ssdg_eval_accumulate(const int32_t* kept, const int32_t* count, const float* kept_score, int32_t top_k,
                         const float* boxes /* [B,A,4], 16-byte aligned */, int32_t batch, int32_t n_priors,
                         int32_t n_classes, const float* gt_boxes, const float* gt_cls, const int32_t* gt_offsets,
                         int32_t max_gt, const double* iou_thresholds /* host */, int32_t n_thresholds,
                         int32_t max_dets, int64_t image_base, int64_t max_images, void* state, size_t state_bytes,
                         void* stream);
SSDG_API int ssdg_eval_exchange(void* state, int32_t n_classes, int64_t max_images, int32_t max_dets, int32_t which,
                       void** out_ptr, int64_t* out_count);
/* Synchronous: status bits of the state (1: GT class out of range, 2: an image with more GT rows than max_gt,
 * 4: a slot written by more than one rank -- known after ssdg_eval_finalize, 8: a kept prior index out of range). */
SSDG_API int ssdg_eval_status(const void* state, int32_t* status, void* stream);
SSDG_API size_t ssdg_eval_finalize_workspace_bytes(int32_t n_classes, int64_t max_images, int32_t max_dets);
SSDG_API int ssdg_eval_finalize(void* state, size_t state_bytes, int32_t n_classes, int64_t max_images,
                       int32_t max_dets, int32_t n_thresholds, const double* recall_thresholds /* host */,
                       int32_t n_recall, double* out_precision, double* out_recall, int64_t* out_n_gt,
                       int64_t* out_n_det, void* workspace, size_t workspace_bytes, void* stream);

/* ---- A12: per-image keep_top_k -----------------------------------------------------------------------------
 * The reference has no post-processing beyond the score head.  The final detections of each image (the original
 * SSD's DetectionOutput keep_top_k, torchvision's detections_per_img): the kept lists of ssdg_detect /
 * ssdg_detect_stage / ssdg_nms ranked across classes and capped at keep_top_k = K (spec: tests/keep_top_k_oracle.py;
 * PARITY UNPINNED like A9).
 *   candidates of image b: the first clamp(count[b][c], 0, top_k) entries of every class list c (score
 *     non-increasing, as those entry points write them), ranked by kept_score descending (compared as floats:
 *     -0 == +0), then class ascending, then position in the list ascending; the first min(K, total) are kept.
 *   The survivors of every class form a prefix of its list, so out_count is itself a count array:
 *     (kept, out_count, kept_score, boxes) goes unchanged to everything that reads kept lists (ssdg_eval_accumulate).
 * Outputs (K slots per image, in rank order):
 *   out_prior int32 [B,K]   prior index (-1 padded)      out_class int32 [B,K]  foreground class in [0, C-1) (-1 padded)
 *   out_score float [B,K]   kept_score (0 padded)        out_box   float [B,K,4] or NULL: decoded cxcywh of the
 *     prior from `boxes` [B,A,4] (needs boxes and n_priors = A; 0 padded, and 0 for a prior index outside [0, A),
 *     which is never dereferenced)
 *   out_n int32 [B]  detections per image             out_count int32 [B,C-1] or NULL: survivors per class list
 * No workspace.  Limits: 1 <= keep_top_k <= 1024, top_k <= 1024, n_classes <= 2048, the batch limit of ssdg_detect.
 * boxes and out_box 16-byte aligned.  Lists that are not score-sorted are outside the contract (nothing outside the
 * arrays is read or written for them either).
 */
SSDG_API int ssdg_detect_keep_top_k(const int32_t* kept, const int32_t* count, const float* kept_score, int32_t top_k,
                                    const float* boxes /* [B,A,4] decoded, 16-byte aligned, or NULL */,
                                    int64_t batch, int32_t n_priors, int32_t n_classes, int32_t keep_top_k,
                                    int32_t* out_prior /* [B,K], -1 padded */, int32_t* out_class /* [B,K], -1 padded */,
                                    float* out_score /* [B,K], 0 padded */, float* out_box /* [B,K,4] or NULL, 0 padded */,
                                    int32_t* out_n /* [B] */, int32_t* out_count /* [B,C-1] or NULL */, void* stream);

/* ---- A13: SSD training augmentation ---------------------------------------------------------------------------
 * The reference's loader only resizes and normalises.  The SSD paper's augmentation of a batch already on the device
 * (spec: tests/augment_oracle.py; PARITY UNPINNED against torchvision 0.26 like A9, every discrete output bit-exact
 * against that restatement): torchvision's RandomZoomOut(fill, side_range=(side_lo, side_hi), p=zoom_p) ->
 * RandomIoUCrop(min_scale, max_scale, min_aspect, max_aspect, min_ious, trials) -> RandomHorizontalFlip(flip_p), then
 * a bilinear resize back to height x width.  Images float32 [B,H,W,3] (one size for the batch); ground truth as
 * ssdg_match_encode reads it: boxes float32 [rows,4] relative cxcywh, cls float32 [rows], offsets int32 [B+1].
 *
 * Random numbers: Philox4x32-10 (Random123), key = seed, counter = (g lo, g hi, stream, index) with g = image_base + b
 *   the global image index; a draw is u = (x >> 8) * 2^-24 (float32 in [0,1)).
 *     stream 0, index 0: zoom gate, zoom r, pad left, pad top      stream 0, index 1: flip gate
 *     stream 1, index q: the option of crop round q, (x0 * n_options) >> 32
 *     stream 2+q, index t: trial t of round q (scale w, scale h, left, top)
 *   Every draw has a fixed address: an image's result depends only on (seed, g, configuration).
 * Decisions (torchvision's float32 arithmetic where it decides an integer; p, side_lo, min_scale, fl32(side_hi -
 * side_lo), fl32(max_scale - min_scale) are rounded to float32 as torch does):
 *   a gate applies iff u < p.  Zoom: r = side_lo + u*(side_hi - side_lo), canvas_w = trunc(W*r), pad_left =
 *     trunc((canvas_w - W)*u) (float32 products), the same for h / top.
 *   crop round q: option m = min_ious[...]; m >= 1 means no crop.  Trial t: new_w = trunc(canvas_w * (min_scale +
 *     u*(max_scale - min_scale))), the same for h; it fails when new_h or new_w is 0 or new_w/new_h (float64) is outside
 *     [min_aspect, max_aspect]; left = trunc((canvas_w - new_w)*u), top alike.  Rows are tested in float64 from the
 *     exactly promoted inputs: pixel corners (cx -/+ 0.5w)*W + pad; a row is within iff left < 0.5(x0+x1) < left+new_w
 *     and the same in y (strict); the trial succeeds iff some within row has !(iou < m), iou by torchvision's box_iou
 *     formula (a NaN IoU passes, as torch.max propagates it).  The first successful trial by index ends the round.
 *   Deviations from torchvision: at most max_rounds rounds, then the image is not cropped and its record says so
 *   (torchvision loops until it draws a 1.0 option); n_options = 0 disables the crop; centres and IoU in float64.
 * Kept rows: with a crop, the within rows in input order, shifted by (left, top), clamped to [0,new_w] x [0,new_h],
 *   relative cxcywh of the crop; without one, every row affine-mapped only (not clamped).  A flip maps cx -> 1 - cx.
 *   Float64, rounded once to float32.  Labels travel with their rows (no SanitizeBoundingBoxes).  Rows are only ever
 *   dropped, so a max_gt bound of the input bounds the output for ssdg_match_encode.
 * Outputs of ssdg_augment_boxes (rows = gt_offsets[B]):
 *   out_boxes float32 [rows,4]  out_cls float32 [rows]  out_offsets int32 [B+1]  (rows past out_offsets[B]: 0)
 *   out_src_row int32 [rows]    input row of each output row (-1 past out_offsets[B])
 *   out_transform int32 [B,SSDG_AUG_RECORD]: canvas w, canvas h, pad left, pad top, crop left, top, w, h (the whole
 *     canvas without a crop), flip, rounds drawn (0 when n_options == 0, -1 when the cap was hit)
 *   No workspace.  Limits: max_gt <= 2048 (rows beyond it are read from global memory, not an error), n_options <= 16,
 *   height, width <= 16384, side_hi <= 64.  Argument errors (SSDG_ERR_ARG: nulls, p outside [0,1], 1 <= side_lo <=
 *   side_hi, 0 <= min_scale <= max_scale <= 1, 0 < min_aspect <= max_aspect, trials >= 1, max_rounds >= 1, a NaN option;
 *   SSDG_ERR_ALIGN: boxes not 16-byte aligned, other arrays not 4-byte aligned) return before any CUDA call.
 * ssdg_augment_images: output pixel (i,j) samples the crop [left, left+w) x [top, top+h) of a virtual canvas that is
 *   fill[c] (host float[3]) except where the image is pasted at (pad left, pad top), bilinear with align_corners=False
 *   and no antialiasing (F.interpolate's source x = max(0, (j+0.5)*(w/W) - 0.5) in float32, upper neighbour clamped to
 *   w-1); a flip reads column W-1-j.  It reads only the record, so a record can be replayed.  images and out_images
 *   must not overlap.
 */
#define SSDG_AUG_RECORD 10
SSDG_API int ssdg_augment_boxes(const float* gt_boxes, const float* gt_cls, const int32_t* gt_offsets, int32_t batch,
                                int32_t max_gt, int32_t height, int32_t width, uint64_t seed, int64_t image_base,
                                double zoom_p, double side_lo, double side_hi, const double* min_ious /* host */,
                                int32_t n_options, double min_scale, double max_scale, double min_aspect,
                                double max_aspect, int32_t trials, int32_t max_rounds, double flip_p, float* out_boxes,
                                float* out_cls, int32_t* out_offsets, int32_t* out_src_row, int32_t* out_transform,
                                void* stream);
SSDG_API int ssdg_augment_images(const float* images, const int32_t* transform, int32_t batch, int32_t height,
                                 int32_t width, const float* fill /* host float[3] */, float* out_images, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSDGEOM_H_ */
