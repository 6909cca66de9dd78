/*
 * sln_b200.h -- C ABI of libsln_b200.so: the B200 (sm_100a) implementation of the
 * SLN-Amodal detection-head hot path.
 *
 * This is the drop-in boundary.  It replaces the reference's dead pytorch-0.4
 * cffi builds:
 *     roialign/roi_align/src/crop_and_resize.h:1-16       (crop_and_resize_forward/backward)
 *     roialign/roi_align/src/crop_and_resize_gpu.h:1-16   (crop_and_resize_gpu_forward/backward)
 *     nms/src/nms.h / nms/src/nms_cuda.h                  (cpu_nms / gpu_nms)
 * and adds entry points for the Python-level functions of the same path
 * (proposal_layer, pyramid_roi_align, the layer codec, the EDT) and of the steps either side
 * of it (SURVEY.md section 8(f): detection / RPN targets, image and layer resize, RPN output
 * re-layout, mask paste, COCO run-length encoding).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *     parameter name ends in `_host`;
 *   - the caller owns every buffer, including outputs and workspace; the library
 *     never allocates, frees or retains a pointer past the call and has no global
 *     state besides a thread-local error string;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     nothing synchronises with the host (counts are returned in device memory);
 *   - return value: SLN_OK or a negative SLN_ERR_* code; sln_last_error_string()
 *     describes the last failure on the calling thread.  The library never exits
 *     the process (the reference printf+exit(-1)s: crop_and_resize.c:39-42,
 *     crop_and_resize_kernel.cu:186-191);
 *   - boxes are (y1, x1, y2, x2); crop boxes are normalised to [0,1] over
 *     (H-1, W-1) exactly as the reference (crop_and_resize.c:44-56).
 */
#ifndef SLN_B200_H
#define SLN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SLN_API __attribute__((visibility("default")))
#else
#define SLN_API
#endif

#define SLN_OK              0
#define SLN_ERR_ARG        (-1)  /* null pointer, negative size, unsupported value   */
#define SLN_ERR_LAYOUT     (-2)  /* unsupported layout combination / misaligned ptr   */
#define SLN_ERR_WORKSPACE  (-3)  /* workspace too small (see *_workspace_bytes)       */
#define SLN_ERR_CUDA       (-4)  /* a CUDA runtime call or kernel launch failed       */

#define SLN_LAYOUT_NCHW 0        /* [B,C,H,W] contiguous                              */
#define SLN_LAYOUT_NHWC 1        /* [B,H,W,C] contiguous (torch channels_last)        */

#define SLN_DTYPE_F32  0         /* element type of the *_ex crop entry points: float  */
#define SLN_DTYPE_BF16 1         /* bfloat16                                          */
#define SLN_DTYPE_F16  2         /* IEEE half                                         */

/* ---- library ---------------------------------------------------------- */
SLN_API int         sln_version(void);                 /* 10000*major + 100*minor + patch   */
SLN_API const char *sln_last_error_string(void);       /* thread-local, never NULL          */
/* sm_count / cc (major*10+minor) / opt-in smem per block / L2 bytes of the current device. */
SLN_API int         sln_device_info(int *sm_count, int *cc, size_t *smem_optin, size_t *l2_bytes);

/* ---- RoIAlign: crop_and_resize ---------------------------------------- *
 * Replaces crop_and_resize_[gpu_]forward (crop_and_resize.c:115-154,
 * crop_and_resize_gpu.c:7-37).  image f32 [B,C,H,W] in `layout`; boxes f32 [N,4];
 * box_ind i32 [N]; crops f32 [N,C,ph,pw] in the SAME layout family (NCHW -> NCHW,
 * NHWC -> [N,ph,pw,C]).  Every output element is written (no pre-zeroing needed).
 * Rows whose box_ind is outside [0,B) are written as zeros, like the reference GPU
 * kernel (crop_and_resize_kernel.cu:34-38); the CPU reference exits instead.       */
SLN_API int sln_crop_and_resize_fwd(const float *image, int B, int C, int H, int W, int layout,
                            const float *boxes, const int *box_ind, int N,
                            int ph, int pw, float extrapolation_value,
                            float *crops, void *stream);

/* Replaces crop_and_resize_[gpu_]backward (crop_and_resize.c:157-252,
 * crop_and_resize_gpu.c:40-69).  grads f32 [N,C,ph,pw] and grad_image f32 [B,C,H,W]
 * in `layout` (NHWC only in this version; NCHW callers convert with
 * sln_nchw_to_nhwc / sln_nhwc_to_nchw).  Deterministic: no atomics; every
 * destination pixel sums its contributions in the reference's serial order
 * (box, y, x, tap).  flags = 0: each term is fma(wy*wx, g, sum) -- within 1 ulp
 * per term of the reference, bit-reproducible run to run.  flags = SLN_BWD_EXACT:
 * each term is rounded exactly like crop_and_resize.c:241-247, which makes the
 * result bit-identical to the reference CPU backward (about 3x the arithmetic).
 * grad_image is fully written (zeros included); no memset needed.                 */
#define SLN_BWD_EXACT 1          /* flags bit: round every product/sum like crop_and_resize.c:241-247 */
/* sln_pyramid_crop_bwd only -- planning ahead.  The backward's ROI lists depend on the boxes, not on the gradients, so
 * they can be built while the FORWARD of the same ROIs runs (on another stream of the caller's):
 *   SLN_BWD_PLAN_ONLY : build the lists in `workspace` and return; grads may be NULL, grad_maps_host[l] only need to be
 *                       non-NULL (nothing is read or written through them).
 *   SLN_BWD_PLANNED   : `workspace` holds the lists of a PLAN_ONLY call with the same boxes, box_ind, level, N, C, ph, pw,
 *                       B and map sizes (a plan can be used any number of times): the three prep launches are skipped.
 * The lists do not depend on the gradients' alignment, so this works for every shape: the PLANNED call picks the
 * gather kernel from its own pointers.                                                                              */
#define SLN_BWD_PLAN_ONLY 2
#define SLN_BWD_PLANNED 4
SLN_API size_t sln_crop_and_resize_bwd_workspace_bytes(int N, int B, int ph, int pw);
SLN_API int sln_crop_and_resize_bwd(const float *grads, const float *boxes, const int *box_ind, int N,
                            int C, int ph, int pw,
                            float *grad_image, int B, int H, int W, int layout, int flags,
                            void *workspace, size_t workspace_bytes, void *stream);

/* Multi-level (FPN) variant for pyramid_roi_align (modal/modals.py:20-110): one
 * launch crops every ROI from the level named by level[i] in {0..n_levels-1} and
 * writes crops in the ORIGINAL ROI order (removes the reference's per-level
 * nonzero/cat/sort, modals.py:70-108).  maps_host / H_host / W_host are HOST arrays
 * of n_levels (<= 8) device pointers / sizes.  NHWC only.                           */
SLN_API int sln_pyramid_crop_fwd(const float *const *maps_host, const int *H_host, const int *W_host,
                         int n_levels, int B, int C,
                         const float *boxes, const int *box_ind, const int *level, int N,
                         int ph, int pw, float extrapolation_value,
                         float *crops, void *stream);
/* Backward of the above for ALL levels in one call: grads f32 [N,ph,pw,C] (NHWC) are
 * routed by level[i] into grad_maps_host[level[i]] (NHWC [B,H_l,W_l,C], fully written).
 * One prep pass + one gather kernel cover every level.  Same determinism / flags contract
 * as sln_crop_and_resize_bwd.                                                          */
SLN_API size_t sln_pyramid_crop_bwd_workspace_bytes(int N, int B, int n_levels, int ph, int pw);
SLN_API int sln_pyramid_crop_bwd(const float *grads, const float *boxes, const int *box_ind, const int *level,
                         int N, int C, int ph, int pw,
                         float *const *grad_maps_host, const int *H_host, const int *W_host, int n_levels,
                         int B, int flags, void *workspace, size_t workspace_bytes, void *stream);

/* FPN level of each ROI (modal/modals.py:53-64): level_out[i] = clamp(round(4 + log2(sqrt(h*w) / (224 / sqrt(H*W)))),
 * 2, 5) - 2, evaluated with the same fp32 operation sequence as the reference's torch expression on a CUDA tensor.
 * boxes f32 [N,4] normalised (y1,x1,y2,x2), 16-byte aligned; level_out i32 [N] in 0..3 (P2..P5).               */
SLN_API int sln_roi_levels(const float *boxes, int N, int image_h, int image_w, int *level_out, void *stream);

/* ---- RoIAlign on 2-byte maps (bf16 / fp16, e.g. under mixed precision) ------- *
 * The four crop entry points above with an element type: `dtype` (SLN_DTYPE_*) names the type of the maps, crops,
 * grads and grad maps of the call (one type for all of them); boxes stay f32 and indices i32.  SLN_DTYPE_F32 is
 * exactly the call without the suffix.  For a 2-byte type the kernels widen every element to f32 (exact), run the
 * f32 operation sequence with f32 accumulators, and round each result once to nearest even: a crop or gradient map
 * is bit-identical to the f32 call on the widened inputs, rounded to the type (NaN payloads aside).  The
 * extrapolation value is rounded the same way.
 *   forward : NHWC only (any C; 16-byte vectors when C % 8 == 0 and the pointers allow).  SLN_ERR_LAYOUT for NCHW:
 *             convert with sln_nchw_to_nhwc_b16, or widen and use the f32 NCHW kernel.
 *   backward: the bulk-async kernel only -- C % 8 == 0, ph and pw <= 32, grads and grad maps 16-byte aligned;
 *             SLN_ERR_LAYOUT otherwise (widen, run the f32 call and round: same bits).  SLN_BWD_PLAN_ONLY /
 *             SLN_BWD_PLANNED work as for f32, and a plan depends neither on the dtype nor on the shape's gather
 *             kernel: a PLAN_ONLY call of any dtype serves PLANNED calls of every dtype with the same boxes and
 *             sizes, including the f32 call of that widening fallback.                                            */
SLN_API int sln_crop_and_resize_fwd_ex(int dtype, const void *image, int B, int C, int H, int W, int layout,
                               const float *boxes, const int *box_ind, int N, int ph, int pw,
                               float extrapolation_value, void *crops, void *stream);
SLN_API int sln_crop_and_resize_bwd_ex(int dtype, const void *grads, const float *boxes, const int *box_ind, int N,
                               int C, int ph, int pw, void *grad_image, int B, int H, int W, int layout, int flags,
                               void *workspace, size_t workspace_bytes, void *stream);
SLN_API int sln_pyramid_crop_fwd_ex(int dtype, const void *const *maps_host, const int *H_host, const int *W_host,
                            int n_levels, int B, int C, const float *boxes, const int *box_ind, const int *level,
                            int N, int ph, int pw, float extrapolation_value, void *crops, void *stream);
SLN_API int sln_pyramid_crop_bwd_ex(int dtype, const void *grads, const float *boxes, const int *box_ind,
                            const int *level, int N, int C, int ph, int pw, void *const *grad_maps_host,
                            const int *H_host, const int *W_host, int n_levels, int B, int flags,
                            void *workspace, size_t workspace_bytes, void *stream);

/* Layout converters (f32; the _b16 forms move any 2-byte type).  src and dst must not alias.                    */
SLN_API int sln_nchw_to_nhwc(const float *src, float *dst, int B, int C, int H, int W, void *stream);
SLN_API int sln_nhwc_to_nchw(const float *src, float *dst, int B, int C, int H, int W, void *stream);
SLN_API int sln_nchw_to_nhwc_b16(const uint16_t *src, uint16_t *dst, int B, int C, int H, int W, void *stream);
SLN_API int sln_nhwc_to_nchw_b16(const uint16_t *src, uint16_t *dst, int B, int C, int H, int W, void *stream);

/* ---- NMS --------------------------------------------------------------- *
 * Replaces cpu_nms (nms/src/nms.c:4-69) + the pth_nms front end (nms/pth_nms.py:5-24)
 * and gpu_nms (nms/src/nms_cuda.c:17-67).  dets f32 [n,5] rows (c0,c1,c2,c3,score)
 * (the reference passes y1,x1,y2,x2 -- the overlap test is symmetric in the axes).
 * Semantics are the CPU extension's, bit for bit: areas = (c3-c1+1)*(c2-c0+1) and
 * the "+1" intersection, un-fused fp32, IEEE divide, suppress when ovr >= thresh.
 * Visiting order: score descending, index ascending among ties (stable).
 * class_ids (i32 [n]) may be NULL; if given, boxes only suppress boxes of the same
 * class (the per-class loop of refine_detections, modal/Functions.py:506-525, in
 * one call).  Outputs: keep i64 [min(n,max_keep)] = indices into dets in visiting
 * order; *num_keep (device i32).  max_keep <= 0 means n.  Everything stays on the
 * device; there is no host round trip (the reference copies the whole mask to the
 * host and scans it there, nms_cuda.c:33-58).                                       */
SLN_API size_t sln_nms_workspace_bytes(int n);
SLN_API int sln_nms(const float *dets, const int *class_ids, int n, float thresh, int max_keep,
            int64_t *keep, int *num_keep, void *workspace, size_t workspace_bytes,
            void *stream);
/* Same call with a `flags` word and an optional report of the path taken.  Two device pipelines produce
 * the identical result: a sparse one (boxes binned by centre, exact pair tests on neighbouring cells only,
 * in-CTA fixed point) used when 65 <= n <= 65535, thresh >= 0.05 and the boxes are finite, ordered
 * (c2 >= c0, c3 >= c1) and within +-32768; and the dense 64x64-tile bit-matrix pipeline, which also takes over
 * (decided on the device, no host round trip) when the sparse one meets more than 16 n overlapping pairs.
 * SLN_NMS_DENSE_ONLY forces the dense pipeline.  *path_out (device i32, may be NULL) receives 1 when the
 * sparse pipeline produced the result, else 0.                                                        */
#define SLN_NMS_DENSE_ONLY 1
/* SLN_NMS_SPARSE_ONLY: launch the sparse pipeline alone (3 kernels instead of 6).  If the input turns out to be
 * outside its contract *num_keep is set to -1 and `keep` is undefined: call again with SLN_NMS_DENSE_ONLY.  For
 * callers that read num_keep on the host anyway (the reference's nms() does, pth_nms.py:24); ignored when the
 * sparse pipeline is not attempted at all (then the dense one runs as usual).                           */
#define SLN_NMS_SPARSE_ONLY 2
SLN_API int sln_nms_ex(const float *dets, const int *class_ids, int n, float thresh, int max_keep, int flags,
               int64_t *keep, int *num_keep, int *path_out, void *workspace, size_t workspace_bytes,
               void *stream);
/* B independent problems of n boxes each in one call: dets f32 [B,n,5], class_ids i32 [B,n] (or NULL: class-agnostic).
 * keep i64 [B,mk] with mk = max_keep when 0 < max_keep <= n, else n; num_keep device i32 [B]; path_out device i32 [B]
 * (may be NULL).  For every b, keep[b, :num_keep[b]], num_keep[b] and path_out[b] are bit-identical to sln_nms_ex on
 * problem b alone with the same class_ids, thresh, max_keep and flags.  Each sparse stage is one launch for all B
 * problems (one cluster per problem); the dense pipeline is launched per problem and returns at once where that
 * problem's sparse pass succeeded.  No host sync, graph capturable.  SLN_NMS_DENSE_ONLY is honoured;
 * SLN_NMS_SPARSE_ONLY is rejected with SLN_ERR_ARG (it needs a host retry).  B == 0 and n == 0 are valid.        */
SLN_API size_t sln_nms_batched_workspace_bytes(int B, int n);
SLN_API int sln_nms_batched(const float *dets, const int *class_ids, int B, int n, float thresh, int max_keep, int flags,
                    int64_t *keep, int *num_keep, int *path_out, void *workspace, size_t workspace_bytes,
                    void *stream);

/* ---- refine_detections, elementwise front --------------------------------- *
 * Replaces the ~25 small torch kernels at the top of refine_detections (modal/Functions.py:453-493): per ROI the
 * argmax class (first maximum), class-specific deltas * std_dev (:436-450), apply_box_deltas (:77-98), scale to
 * pixels, clip to `window` (y1,x1,y2,x2) (:423-433), round half-to-even (:485) and the keep filter `class_id > 0 [and
 * score >= min_confidence]` (min_confidence == 0 disables the score test, :490).
 * rois f32 [N,4] normalised, probs f32 [N,K], deltas f32 [N,K,4]  ->  dets f32 [N,5] (y1,x1,y2,x2,score) and
 * cls_nms i32 [N], ready for sln_nms: filtered-out boxes carry score -inf and a unique negative class, so the
 * class-aware NMS returns them at the tail of its output; *n_excluded (device i32) counts them.  class_ids i32 [N] =
 * the argmax class of every ROI.                                                                        */
SLN_API int sln_refine_decode(const float *rois, const float *probs, const float *deltas, int N, int K,
                      const float *std_dev_host, float img_h, float img_w, const float *window_host,
                      float min_confidence, float *dets, int *cls_nms, int *class_ids, int *n_excluded,
                      void *stream);

/* ---- refine_detections, selection without NMS ------------------------------- *
 * The reference's shipped default (config.py:78 `USE_NMS = False`; modal/Functions.py:526-546): of the ROIs whose
 * argmax class is not background keep the `max_keep` (100, hard-coded at :530-532) best by score, in descending score
 * order; score ties go to the lower ROI index.  dets / class_ids are sln_refine_decode's outputs (run with
 * min_confidence = 0: this branch has no score filter).  Writes rows [0, min(max_keep, N - *n_excluded)) of
 * result f32 [max_keep,6] = (y1,x1,y2,x2,class_id,score) and keep i64 [max_keep] (ROI indices); later rows are not
 * touched.  One launch, no host sync.                                                                      */
SLN_API int sln_refine_topk(const float *dets, const int *class_ids, int N, int max_keep, float *result,
                    int64_t *keep, void *stream);
/* B images of N rows each in one launch: dets f32 [B,N,5], class_ids i32 [B,N] -> result f32 [B,max_keep,6], keep i64
 * [B,max_keep] (row indices within the image) and num_det device i32 [B] = min(max_keep, rows of the image with
 * class_id > 0 and score > -inf).  Image b's rows [0, num_det[b]) are what sln_refine_topk writes for that image alone;
 * later rows are not touched.  No host sync.                                                                   */
SLN_API int sln_refine_topk_batched(const float *dets, const int *class_ids, int B, int N, int max_keep, float *result,
                            int64_t *keep, int *num_det, void *stream);

/* ---- refine_detections, per-class NMS branch, B images ------------------------- *
 * The step after sln_nms_batched (run on sln_refine_decode's dets f32 [B,N,5] and cls_nms i32 [B,N] with
 * DETECTION_NMS_THRESHOLD and max_keep = D): nms_keep i64 [B,nms_max_keep], nms_num_keep device i32 [B] are its outputs.
 * Writes result f32 [B,D,6] = (y1,x1,y2,x2,class_id,score) with class_id from class_ids i32 [B,N], keep i64 [B,D] (row
 * indices within the image) and num_det device i32 [B] = min(D, survivors with a finite score); rows at and beyond
 * num_det[b] are zero.  Rows below num_det[b] are the first D rows of the single-image branch (sln_nms_ex on that image
 * without max_keep, filtered rows dropped): greedy NMS's first D survivors do not depend on where it stops.  One launch,
 * no host sync.                                                                                                     */
SLN_API int sln_refine_nms_emit_batched(const float *dets, const int *class_ids, int B, int N, const int64_t *nms_keep,
                                const int *nms_num_keep, int nms_max_keep, int D, float *result, int64_t *keep,
                                int *num_det, void *stream);

/* ---- detection targets (SURVEY 8(f)-1) -------------------------------------- *
 * sln_bbox_overlaps replaces bbox_overlaps (modal/Functions.py:184-218): IoU of boxes1 [N,4] against boxes2 [G,4]
 * (y1,x1,y2,x2; no "+1"; every operation rounded separately; 0/0 -> NaN).  Any of the three outputs may be NULL:
 * overlaps f32 [N,G]; iou_max f32 [N] and argmax i32 [N] = torch.max(overlaps, dim=1) (first maximum; NaN wins), the
 * two reductions detection_target_layer takes from the matrix (:277, :297).
 * sln_box_refinement replaces utils.box_refinement (utils.py:96-117) for M box pairs; std_dev_host (4 floats, may be
 * NULL) additionally divides the result by BBOX_STD_DEV (Functions.py:309-313).                           */
SLN_API int sln_bbox_overlaps(const float *boxes1, int N, const float *boxes2, int G, float *overlaps,
                      float *iou_max, int *argmax, void *stream);
SLN_API int sln_box_refinement(const float *box, const float *gt_box, int M, const float *std_dev_host, float *out,
                       void *stream);

/* Mask targets of detection_target_layer (modal/Functions.py:327-346, SURVEY row A12): for positive ROI p,
 * out[p, l] = round(crop_and_resize(gt_masks[l, assignment[p]], boxes[p], mh x mw, extrapolation 0)), sampled straight
 * from the u8 planes (the reference converts every assigned 1-MiB plane to float first).  gt_masks u8 [L,G,H,W],
 * assignment i32 [P], boxes f32 [P,4] normalised -> out f32 [P,L,mh,mw].  Same tap arithmetic as sln_crop_and_resize_fwd. */
SLN_API int sln_mask_targets(const uint8_t *gt_masks, int L, int G, int H, int W, const int *assignment,
                     const float *boxes, int P, int mh, int mw, float *out, void *stream);

/* detection_target_layer for B images, the two device halves around the host's sampling.
 * sln_target_match_batched: proposals f32 [B,R,4], num_proposals device i32 [B] (NULL: all R rows) -> per row codes u8
 * [B,R] (bit 0 = positive, iou_max >= 0.5; bit 1 = negative-eligible, iou_max < 0.5 and, in an image with a crowd GT row
 * (class < 0), crowd_iou_max < 0.001; a NaN iou_max is neither, as in the reference; 0 past num_proposals[b]) and argmax
 * i32 [B,R] = the first maximum's row in gt_boxes[b].  Candidates: the first num_gt_host[b] rows of gt_boxes f32 [B,G,4]
 * / gt_class_ids i32 [B,G], only those with class > 0 in a crowd image.  num_gt_host is passed by value in the kernel's
 * parameters (B <= 512).  Same IoU arithmetic as sln_bbox_overlaps.  One launch.
 * sln_detection_targets_emit_batched: after sampling, sel i32 [B,T] (proposal rows, positives first), num_positive /
 * num_rois i32 [B] and, per image, mask_planes[b] = device address of its u8 masks [L, mask_g[b], H, W] (device
 * arrays).  Writes the whole padded output: rois f32 [B,T,4], class_ids i32 [B,T], deltas f32 [B,T,4] (divided by
 * std_dev_host when not NULL), masks f32 [B,T,L,mh,mw]; positive rows as sln_box_refinement / sln_mask_targets compute
 * them (the mask box in the GT box's frame when use_mini_mask), negative rows the proposal with class 0 and zeros, rows
 * past num_rois[b] zeros.  One launch.                                                                          */
SLN_API int sln_target_match_batched(const float *proposals, int B, int R, const int *num_proposals,
                             const float *gt_boxes, const int *gt_class_ids, int G, const int *num_gt_host,
                             uint8_t *codes, int *argmax, void *stream);
SLN_API int sln_detection_targets_emit_batched(const float *proposals, int B, int R, const int *argmax,
                                       const float *gt_boxes, const int *gt_class_ids, int G, const int *sel,
                                       const int *num_positive, const int *num_rois,
                                       const uint8_t *const *mask_planes, const int *mask_g, int T, int L, int H,
                                       int W, int mh, int mw, const float *std_dev_host, int use_mini_mask,
                                       float *rois, int *class_ids, float *deltas, float *masks, void *stream);

/* Overlap reductions of build_rpn_targets (modal/Functions.py:773-792; SURVEY 8(f)-2) in float64, without the
 * [A,G] matrix: anchor_iou_max f64 [A] and anchor_argmax i32 [A] = max / first argmax over the GT boxes of every anchor,
 * gt_argmax i32 [G] = first argmax over the anchors of every GT box (numpy rules: NaN is the maximum).  Any output may
 * be NULL (crowd boxes only need anchor_iou_max, :769-770).  anchors f64 [A,4], gt_boxes f64 [G,4], 32-byte aligned.  */
SLN_API size_t sln_rpn_overlap_workspace_bytes(int G);     /* needed when gt_argmax is asked for */
SLN_API int sln_rpn_overlap_reductions(const double *anchors, int A, const double *gt_boxes, int G,
                               double *anchor_iou_max, int *anchor_argmax, int *gt_argmax, void *workspace,
                               size_t workspace_bytes, void *stream);

/* Tight bounding boxes of M binary u8 planes [M,H,W] (utils.extract_bboxes, utils.py:28-49, before its random jitter):
 * boxes i32 [M,4] = (y1, x1, y2, x2) with y2 / x2 exclusive, zeros for an empty plane.                       */
SLN_API int sln_plane_bboxes(const uint8_t *planes, int M, int H, int W, int *boxes, void *stream);

/* ---- COCO run-length codec (SURVEY 8(f)-3) ---------------------------------- *
 * sln_rle_encode replaces rleEncode (cocoapi/common/maskApi.c:32-41): masks u8 [n][a] in the memory order to encode
 * (pycocotools encodes column-major planes), counts u32 [n][cap], m_out i32 [n] = number of runs of mask i (the runs
 * alternate, starting with the possibly empty run of zeros), or -m when m > cap (nothing is written for that mask).
 * sln_rle_to_string is a HOST helper (no CUDA): rleToString (maskApi.c:204-216) of one count list into `out`; returns
 * the string length, or -(needed capacity) when cap is too small.                                          */
SLN_API int sln_rle_encode(const uint8_t *masks, int n, long long a, uint32_t *counts, int cap, int *m_out, void *stream);
SLN_API long long sln_rle_to_string(const uint32_t *counts, long long m, char *out, long long cap);
/* sln_rle_to_string on the device for n count lists counts u32 [n][cap] of m[i] runs each (a list with m[i] <= 0 or
 * > cap gets an empty string): the strings packed in list order into `strings` (no terminators), str_off / str_len
 * i32 [n], *str_total = total bytes.  strings_cap >= 7 * cap * n and < 2^31.  Three launches, no host sync.       */
SLN_API int sln_rle_strings(const uint32_t *counts, int n, int cap, const int *m, int *str_off, int *str_len,
                    int *str_total, char *strings, long long strings_cap, void *stream);

/* Mask paste after the path (SURVEY 8(f)-3): utils.unmold_mask (utils.py:447-465) for N detections in one launch.
 * masks f32 [N,mh,mw] (the head's small masks), boxes i32 [N,4] = (y1,x1,y2,x2) in image pixels, y2 / x2 exclusive,
 * out u8 [N,H,W].  Per detection: scipy.misc.bytescale (min/max stretch to u8, float32), Pillow's 8-bit bilinear
 * resample to (y2-y1, x2-x1) -- what scipy.misc.imresize(interp='bilinear') runs, bit-identical --, v/255 >= 0.5, paste
 * into a zero image.  A box that is empty or not inside [0,H]x[0,W] pastes nothing (the reference drops zero-area
 * detections first, model.py:786-795, and its paste raises on a box outside the image).  mh, mw <= 256.          */
SLN_API int sln_unmold_masks(const float *masks, int N, int mh, int mw, const int *boxes, int H, int W,
                     uint8_t *out, void *stream);

/* Batched evaluation tail: MaskRCNN.unmold_detections (model.py:747-806) + COCO RLE (amodal_train.py:371-400) for B
 * images of D detection rows, from box-sized masks: no H x W plane is written.  detections f32 [B,D,6] contiguous,
 * (y1,x1,y2,x2,class_id,score); mrcnn_mask f32 [B,D,mh,mw,K] read through mask_strides_host (5 element strides, any
 * layout); H_host / W_host: B image sizes; scale_shift_host f64 [B,4] = (h_scale, w_scale, window[0], window[1]) as
 * the reference computes them.  Per image: the padding cut (first row with class 0), class collapse to 1, astype(int32)
 * of (box - shift) * scale in float64, the keep rule of unmold_detections, compaction in order.  Outputs, rows at and
 * beyond num_kept[b] zero: boxes i32 [B,D,4], class_ids i32 [B,D], scores f32 [B,D], src_row i32 [B,D] (detection row
 * of each kept box), num_kept i32 [B] (-1: a row before the cut names a class outside the K mask channels, where the
 * reference raises).  Per kept mask, m_out [B,D] = number of runs of the column-major H x W plane, or -m when m > cap
 * (nothing written; 0 for rows past num_kept), and its rleToString string at strings[str_off : str_off + str_len]
 * (packed in row order, no terminator; *str_total bytes in all).  strings_cap >= 7 * cap * B * D.  Five launches for
 * any B and D, no host sync, graph capturable.  B <= 512.  B == 0 and D == 0 are valid.                        */
SLN_API size_t sln_unmold_rle_batched_workspace_bytes(int B, int D, const int *H_host, const int *W_host, int cap);
SLN_API int sln_unmold_rle_batched(const float *detections, int B, int D, const float *mrcnn_mask, int mh, int mw,
                           int K, const long long *mask_strides_host, const int *H_host, const int *W_host,
                           const double *scale_shift_host, int cap, int *boxes, int *class_ids, float *scores,
                           int *src_row, int *num_kept, int *m_out, int *str_off, int *str_len, int *str_total,
                           char *strings, long long strings_cap, void *workspace, size_t workspace_bytes,
                           void *stream);

/* Image resize in front of the path (SURVEY 8(f)-2): utils.resize_image (utils.py:301-356) squashes the uint8 image to
 * (max_dim, max_dim) with scipy.misc.imresize = Pillow's 8-bit bilinear resample per band (triangle filter of support
 * max(1, in/out), 22-bit fixed-point coefficients, horizontal pass first with an 8-bit intermediate) -- reproduced bit
 * for bit.  src u8 [h,w,C] (interleaved channels), out u8 [H2,W2,C]; three launches, workspace from the query below. */
SLN_API size_t sln_resize_image_workspace_bytes(int h, int w, int C, int H2, int W2);
SLN_API int sln_resize_image_u8(const uint8_t *src, int h, int w, int C, int H2, int W2, uint8_t *out, void *workspace,
                        size_t workspace_bytes, void *stream);

/* Nearest-neighbour zoom / flip of n u8 planes as a gather (utils.resize_layer, utils.py:358-362; np.fliplr,
 * Functions.py:712-715): dst[p][y][x] = src[p][iy[y]][ix[x]], 0 where an index is negative.  iy i32 [H2], ix i32 [W2] on
 * the device, computed by the caller with scipy.ndimage.zoom's float64 rule (sln_amodal_b200/targets.py).          */
SLN_API int sln_gather_planes(const uint8_t *src, int n, int H, int W, const int *iy, const int *ix, int H2, int W2,
                      uint8_t *dst, void *stream);

/* ---- RPN output re-layout (SURVEY 8(f)-4) ------------------------------------- *
 * Replaces, for all pyramid levels at once, the per-level permute(0,2,3,1).contiguous().view + Softmax(dim=2) of
 * RPN.forward (modal/modals.py:388-412) and the concatenation over levels of MaskRCNN.predict (model.py:553-563).
 * logits[l] f32 [B,2a,H_l,W_l], bbox[l] f32 [B,4a,H_l,W_l] (host arrays of n_levels device pointers; layout =
 * SLN_LAYOUT_NCHW, or SLN_LAYOUT_NHWC for channels_last conv outputs); a = anchors per location.  With
 * A = a * sum_l H_l*W_l:  out_logits f32 [B,A,2], out_probs f32 [B,A,2] = softmax over the last axis, out_bbox f32
 * [B,A,4]; row (y*W_l + x)*a + k of level l, value j <- channel 2k+j (4k+j).  Any output (and either input list) may
 * be NULL.  sln_rpn_unpack_grads is the backward of the two copies: it writes every element of d_logits[l] / d_bbox[l]
 * (same shapes and layout as the inputs) from g_logits [B,A,2] / g_bbox [B,A,4] (a NULL gradient writes zeros).     */
SLN_API int sln_rpn_pack(const float *const *logits, const float *const *bbox, const int *heights, const int *widths,
                 int n_levels, int B, int a, int layout, float *out_logits, float *out_probs, float *out_bbox,
                 void *stream);
SLN_API int sln_rpn_unpack_grads(const float *g_logits, const float *g_bbox, const int *heights, const int *widths,
                         int n_levels, int B, int a, int layout, float *const *d_logits, float *const *d_bbox,
                         void *stream);

/* ---- proposal_layer ----------------------------------------------------- *
 * Replaces proposal_layer (modal/Functions.py:114-178) for one image:
 * fg score = probs[:,1]; deltas *= std_dev; top `pre_nms_limit` anchors by score
 * (stable); apply_box_deltas (:77-98); clip to [0,0,img_h,img_w] (:101-111);
 * NMS(nms_thresh); first `proposal_count` survivors; divide by [h,w,h,w].
 * probs f32 [A,2], deltas f32 [A,4], anchors f32 [A,4] (pixels).
 * out_boxes f32 [proposal_count,4] (rows >= *num_out are zero-filled);
 * *num_out device i32.  std_dev_host: 4 host floats.                               */
SLN_API size_t sln_proposal_workspace_bytes(int A, int pre_nms_limit);
SLN_API int sln_proposal_layer(const float *probs, const float *deltas, const float *anchors, int A,
                       int pre_nms_limit, int proposal_count, float nms_thresh,
                       const float *std_dev_host, float img_h, float img_w,
                       float *out_boxes, int *num_out,
                       void *workspace, size_t workspace_bytes, void *stream);
/* B images per call, one launch per stage for all of them (the dense NMS fallback aside: it is launched per image and
 * returns at once where that image's sparse pass succeeded).  probs f32 [B,A,2], deltas f32 [B,A,4], anchors f32 [A,4]
 * shared by all images; out_boxes f32 [B,proposal_count,4], num_out device i32 [B].  For every image b, out_boxes[b] and
 * num_out[b] are bit-identical to sln_proposal_layer on that image alone, zero padding included.  No host sync, graph
 * capturable; B == 0 and proposal_count == 0 are valid.  Workspace: B copies of the single-image one.          */
SLN_API size_t sln_proposal_batched_workspace_bytes(int B, int A, int pre_nms_limit);
SLN_API int sln_proposal_layer_batched(const float *probs, const float *deltas, const float *anchors, int B, int A,
                               int pre_nms_limit, int proposal_count, float nms_thresh,
                               const float *std_dev_host, float img_h, float img_w,
                               float *out_boxes, int *num_out,
                               void *workspace, size_t workspace_bytes, void *stream);

/* ---- sem-dist target encoding ------------------------------------------- *
 * Layer codec: replaces AmodalDataset.load_layer2 (amodal_train.py:236-271) and the
 * codec helpers it drives (modal/Functions.py:1012-1095).  label u64 [B,H,W] (bit i =
 * object i visible, bit 32+i = object i occluded) -> out u8 [B,n_max,L,H,W]
 * (planes of objects >= n_obj are zero), n_obj i32 [B] (not clamped to n_max).
 * scratch: 2*B u32 words of device memory (overwritten).                            */
SLN_API int sln_layer_decode(const uint64_t *label, int B, int H, int W, int L, int n_max,
                     uint8_t *out, int *n_obj, uint32_t *scratch, void *stream);

/* Exact squared Euclidean distance transform (absent from the reference; see
 * DESIGN.md): maps u8 [M,H,W] -> out i32 [M,H,W] = squared distance to the nearest
 * ZERO pixel of the same map, (H+W)^2 where a map has no zero pixel.
 * Shapes with W % 32 == 0, W <= 1024, H <= 2048 and 16-byte aligned pointers take the
 * banded kernels (lower envelopes per 32-row band, no row-distance buffer; workspace:
 * 34 u32 stack slots per 32 rows + two words per (band, column) + a tile list, about
 * 4.5 bytes per pixel, contents undefined before and after the call); every other
 * shape takes the row pass + whole-column envelope kernels.  The environment variable
 * SLN_EDT_IMPL=legacy forces the latter (A/B).                                      */
SLN_API size_t sln_edt_workspace_bytes(int M, int H, int W);
SLN_API int sln_edt_sq(const uint8_t *maps, int M, int H, int W, int32_t *out,
               void *workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SLN_B200_H */
