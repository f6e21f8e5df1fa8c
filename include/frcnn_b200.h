/*
 * frcnn_b200 -- C ABI of the B200-native region-proposal / target-assignment /
 * NMS / RoI-layer hot path.
 *
 * The reference (Kelicious/faster_rcnn) is pure Python + numpy and has no FFI
 * layer of its own; its boundary is the Python functions listed below.  Each
 * entry point names the reference code it replaces (file:line under
 * /root/reference/faster_rcnn).  The Python package `faster_rcnn_b200` binds
 * these symbols with ctypes and re-exposes the reference's signatures
 * (see INTEGRATION.md).
 *
 * Conventions
 *  - every function returns FRCNN_OK (0) or a negative frcnn_status; nothing
 *    throws or aborts.  frcnn_last_error(h) gives a message for the last failure
 *    on that handle.
 *  - all data pointers are DEVICE pointers unless the parameter name ends in
 *    `_host`.  The caller owns every buffer.  Work is enqueued on `stream`
 *    (a cudaStream_t passed as void*) and is asynchronous.
 *  - one handle per (host thread, device); handles are not thread-safe.  A
 *    handle owns a scratch arena that grows on demand (growing synchronises the
 *    stream; call frcnn_reserve() up front to avoid that, e.g. before CUDA-graph
 *    capture).  The arena is shared by all calls on the handle: calls on one
 *    stream are ordered by the stream; a call on a DIFFERENT stream than the
 *    previous call first makes its stream wait (device-side event) for the work
 *    the handle enqueued on the previous stream, so two streams never use the
 *    scratch concurrently -- use one handle per stream for real concurrency.  A
 *    stream under CUDA-graph capture is exempt: capture on a private handle.
 *  - deviation from SURVEY.md 8b: there is no frcnn_workspace_bytes() and no
 *    `*_host` convenience variant.  Scratch is the handle's arena (pre-sized with
 *    frcnn_reserve), and the host<->device copies of the drop-in layer are done
 *    by the Python binding through pinned staging buffers (runtime.py).
 *  - boxes are [x1, y1, x2, y2]; a "batch" is a set of independent images laid
 *    out contiguously (image-major).  Flat anchor index = (y*C + x)*A + a.
 *  - arithmetic follows the reference bit for bit where it is integer / IEEE
 *    (+1 area convention and f64 ratio in NMS, f32 no-FMA IoU in labelling);
 *    the decode evaluates numpy's own float32 exp kernel (np_expf); float64
 *    log/exp in regression targets and post-processing follow the device libm
 *    (<= 1 ulp after the float32 store, DESIGN.md).
 */
#ifndef FRCNN_B200_H
#define FRCNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FRCNN_API __attribute__((visibility("default")))
#else
#define FRCNN_API
#endif

#define FRCNN_ABI_VERSION 1
#define FRCNN_MAX_ANCHORS 64       /* anchors per location */
#define FRCNN_MAX_GT 256           /* GT boxes per image   */
#define FRCNN_NMS_MAX_SORTED 22528 /* nms_i16: max n when scores arrive strictly descending */
#define FRCNN_NMS_MAX_UNSORTED 16384 /* nms_i16: max n when the kernel has to sort        */
#define FRCNN_NMS_F64_MAX 4096     /* nms_f64: max boxes per segment */

typedef enum {
  FRCNN_OK = 0,
  FRCNN_ERR_INVALID = -1,     /* bad argument */
  FRCNN_ERR_CUDA = -2,        /* CUDA runtime error (message in frcnn_last_error) */
  FRCNN_ERR_UNSUPPORTED = -3, /* size beyond what the kernels support */
  FRCNN_ERR_NOMEM = -4
} frcnn_status;

typedef enum { FRCNN_ROI_RESIZE = 0, FRCNN_ROI_MAX = 1 } frcnn_roi_mode;
typedef enum { FRCNN_ROI_I16 = 0, FRCNN_ROI_I32 = 1, FRCNN_ROI_F32 = 2 } frcnn_roi_dtype;

typedef struct frcnn_handle frcnn_handle;

/* ---- lifetime ---------------------------------------------------------- */
FRCNN_API int frcnn_abi_version(void);
FRCNN_API int frcnn_create(frcnn_handle** out, int device);
FRCNN_API void frcnn_destroy(frcnn_handle* h);
FRCNN_API const char* frcnn_last_error(frcnn_handle* h);
/* Pre-size the scratch arena (bytes). */
FRCNN_API int frcnn_reserve(frcnn_handle* h, size_t bytes);
/* Number of kernels this handle has launched so far (for bench accounting). */
FRCNN_API long long frcnn_launch_count(frcnn_handle* h);

/* ---- K-a: proposals = anchors + delta decode + sanitize + validity + top-k
 * Replaces det_util._get_rois (det_util.py:370-380), _get_anchor_coords
 * (:162-175), util.transform_np_inplace (util.py:111-142),
 * _sanitize_boxes_inplace (det_util.py:179-192), _get_valid_box_idxs
 * (:196-205) and the sort/truncate/int16 cast of det_util.py:68-76 / :147-155.
 *   regr  [batch,R,C,4A] f32   cls [batch,R,C,A] f32
 *   anchor_hw_host [A][2] int32 pixel [height,width] (util.get_anchors); the
 *   library applies `// stride` itself.
 *   out_boxes [batch,k,4] i16, out_scores [batch,k] f32, out_index [batch,k]
 *   i32 (flat anchor index), out_count [batch] i32.  Order: score descending,
 *   ties by descending anchor index; rows >= count are zero / index -1.
 *   dense_boxes (optional, may be NULL) [batch,R*C*A,4] f32 receives every
 *   decoded+sanitized box (the return value of _get_rois).
 *   Capacity: k <= 32768 (FRCNN_ERR_UNSUPPORTED above); any float scores are
 *   ranked exactly, the fast path is tuned for scores in [2^-32, 1). */
FRCNN_API int frcnn_decode_topk(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                      const int32_t* anchor_hw_host, int rows, int cols, int n_anchors,
                      int stride, int k, int batch, int16_t* out_boxes, float* out_scores,
                      int32_t* out_index, int32_t* out_count, float* dense_boxes);

/* ---- K-b: greedy NMS, int16 boxes (RPN stage)
 * Replaces det_util.nms (det_util.py:209-256) for int16 boxes.
 *   boxes [batch,n_max,4] i16, scores [batch,n_max] f32, n [batch] i32 (device;
 *   NULL = n_max for every image).  Visit order = (score desc, position desc),
 *   predicate = f64(inter/union) <= thresh keeps, +1 areas, stop at max_boxes.
 *   keep_index [batch,max_boxes] i32 positions into the image's rows (pick
 *   order, -1 padded), keep_count [batch]; keep_boxes [batch,max_boxes,4] i16
 *   and keep_scores [batch,max_boxes] f32 are optional (NULL to skip).
 *   Capacity: n <= FRCNN_NMS_MAX_UNSORTED for arbitrary scores; up to
 *   FRCNN_NMS_MAX_SORTED only when an image's scores arrive STRICTLY descending
 *   (the output of frcnn_decode_topk; equal neighbours count as unsorted).  An
 *   image that violates this gets keep_count = -1 and an all -1 keep_index
 *   (device-side flag, the call itself still returns FRCNN_OK). */
FRCNN_API int frcnn_nms_i16(frcnn_handle* h, void* stream, const int16_t* boxes, const float* scores,
                  const int32_t* n, int n_max, int batch, double thresh, int max_boxes,
                  int32_t* keep_index, int32_t* keep_count, int16_t* keep_boxes,
                  float* keep_scores);

/* ---- K-b': greedy NMS, float64 boxes, segmented (per-class stage)
 * Replaces det_util.nms as called from voc_dets.py:76 (all-f64 arithmetic).
 *   boxes [total,4] f64, scores [total] f32, seg_offsets [n_seg+1] i32
 *   (device).  keep_index [n_seg,out_stride] i32 relative to the segment
 *   start, keep_count [n_seg]. */
FRCNN_API int frcnn_nms_f64(frcnn_handle* h, void* stream, const double* boxes, const float* scores,
                  const int32_t* seg_offsets, int n_seg, int max_seg_len, double thresh,
                  int max_boxes, int out_stride, int32_t* keep_index, int32_t* keep_count);

/* ---- fused proposal stage: K-a feeding K-b without leaving the device.
 * Replaces DetTrainingManager.get_det_inputs / _process up to nms
 * (det_util.py:63-77, :136-158).  out_rois [batch,max_boxes,4] i16,
 * out_scores [batch,max_boxes] f32, out_count [batch] i32.
 * min(k, R*C*A) <= FRCNN_NMS_MAX_UNSORTED: tied scores make the top-k list
 * "unsorted" for K-b, and the fused call has no way to report K-b's flag. */
FRCNN_API int frcnn_proposals(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                    const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride,
                    int k, double thresh, int max_boxes, int batch, int16_t* out_rois,
                    float* out_scores, int32_t* out_count);

/* ---- mixed-size batches (the *_ragged entries and frcnn_clip_rois)
 * Images whose feature maps differ in size share one PADDED layout: rows x cols are the largest
 * extents of the batch (or any larger map) and extents [batch,2] i32 (device) holds every image's own
 * (rows_b, cols_b), clamped on the device to [0,rows] x [0,cols].  For every image the result equals the
 * uniform call on the cropped inputs [:rows_b, :cols_b], laid out in the padded layout: padding cells of
 * every output are zero and padding cells of the inputs are never read.  An image with a zero extent
 * gets no proposals and all-zero labels.
 *   decode_topk_ragged: out_index is the image's OWN flat index (y*cols_b + x)*A + a; dense_boxes must
 *   be NULL (FRCNN_ERR_INVALID otherwise).
 *   label_anchors_ragged: can_use / is_pos / bbreg in the padded [batch,rows*cols*A] layout, counts as
 *   frcnn_label_anchors; frcnn_pack_rpn_targets takes the result unchanged (the ranks of the usable
 *   anchors are those of the cropped call).
 *   clip_rois: rois [batch,n_rois,4] (roi_dtype) -> out (same layout, may alias rois), truncated to int
 *   like the RoI layer and clamped to x1,y1 >= 0, x2 <= cols_b, y2 <= rows_b (extents below 0 count
 *   as 0); the RoI layer entries then take the padded feature map [batch,rows,cols,C], whose own clamp
 *   completes the clamp of the extents, and see the cropped call's crops.  Max mode's int32 arg-max
 *   y*W + x then refers to the PADDED width W. */
FRCNN_API int frcnn_decode_topk_ragged(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                                       const int32_t* anchor_hw_host, int rows, int cols, int n_anchors,
                                       int stride, int k, int batch, const int32_t* extents,
                                       int16_t* out_boxes, float* out_scores, int32_t* out_index,
                                       int32_t* out_count, float* dense_boxes);
FRCNN_API int frcnn_proposals_ragged(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                                     const int32_t* anchor_hw_host, int rows, int cols, int n_anchors,
                                     int stride, int k, double thresh, int max_boxes, int batch,
                                     const int32_t* extents, int16_t* out_rois, float* out_scores,
                                     int32_t* out_count);
FRCNN_API int frcnn_label_anchors_ragged(frcnn_handle* h, void* stream, const float* gt, const int32_t* n_gt,
                                         const int32_t* img_wh, int g_max, int rows, int cols,
                                         int n_anchors, const int32_t* anchor_hw_host, int stride,
                                         int batch, const int32_t* extents, uint8_t* can_use,
                                         uint8_t* is_pos, float* bbreg, int32_t* counts);
FRCNN_API int frcnn_clip_rois(frcnn_handle* h, void* stream, const void* rois, int roi_dtype, int n_rois,
                              int batch, const int32_t* extents, void* out);

/* ---- K-c: RPN anchor labelling
 * Replaces RpnTrainingManager._process (rpn_util.py:54-103) incl.
 * _get_all_anchor_coords (:276-298), _get_out_of_bounds_idxs (:302-310),
 * util.cross_ious (util.py:146-177) and util.get_reg_params (:180-206).
 *   gt [batch,g_max,4] f32 pixel corners, n_gt [batch] i32, img_wh [batch,2]
 *   i32 (width,height).  can_use/is_pos [batch,N] u8, bbreg [batch,N,4] f32,
 *   counts [batch,2] i32 = (#pos&can_use, #neg&can_use) before sampling. */
FRCNN_API int frcnn_label_anchors(frcnn_handle* h, void* stream, const float* gt, const int32_t* n_gt,
                        const int32_t* img_wh, int g_max, int rows, int cols, int n_anchors,
                        const int32_t* anchor_hw_host, int stride, int batch, uint8_t* can_use,
                        uint8_t* is_pos, float* bbreg, int32_t* counts);

/* ---- T6/T7: apply host-drawn sampling and pack Keras y_true tensors
 * Replaces _apply_sampling (rpn_util.py:324-350) and the tail of
 * RpnTrainingManager.rpn_y_true (rpn_util.py:124-140).
 *   off_pos / off_neg (device, may be NULL): the values the reference draws with
 *   random.sample(range(num_pos), ..) / random.sample(range(num_neg), ..), i.e. RANKS
 *   among the image's usable positives / negatives in ascending anchor order (counts
 *   come from frcnn_label_anchors); off_*_offsets [batch+1] i32 delimit each image's
 *   slice.  The anchors at those ranks get can_use = 0 (in place, like the reference),
 *   then y_class [batch,R,C,2A] u8 = [can_use | is_pos] and y_bbreg [batch,R,C,8A] f32 =
 *   [repeat(is_pos & can_use, 4) | targets] are written.  bbreg and y_bbreg must be
 *   16-byte aligned (FRCNN_ERR_INVALID otherwise). */
FRCNN_API int frcnn_pack_rpn_targets(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos,
                                     const float* bbreg, const int32_t* off_pos,
                                     const int32_t* off_pos_offsets, const int32_t* off_neg,
                                     const int32_t* off_neg_offsets, int rows, int cols, int n_anchors,
                                     int batch, uint8_t* y_class, float* y_bbreg);

/* ---- K-c': detector RoI labelling
 * Replaces det_util._rois_to_truth (det_util.py:310-334),
 * _one_hot_encode_bbreg (:338-354) and _one_hot_encode_cls (:358-366).
 *   rois [batch,n_max,4] i16, n_roi [batch] (NULL = n_max), gt [batch,g_max,4]
 *   f64 in FEATURE units (pixel corner * (1/stride), python-float precision),
 *   gt_cls [batch,g_max] i32, n_gt [batch], n_classes incl. 'bg' (= last).
 *   Outputs are compacted to the eligible rows (max IoU >= 0.1), order kept:
 *   out_rois [batch,n_max,4] i16, out_cls [batch,n_max,K] i32 one-hot,
 *   out_bbreg [batch,n_max,8(K-1)] f32, out_src [batch,n_max] i32 (row of the
 *   input RoI, optional), out_count [batch]. */
FRCNN_API int frcnn_label_rois(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* n_roi,
                     int n_max, const double* gt, const int32_t* gt_cls, const int32_t* n_gt,
                     int g_max, int n_classes, int batch, int16_t* out_rois, int32_t* out_cls,
                     float* out_bbreg, int32_t* out_src, int32_t* out_count);

/* ---- K-d: RoI layer forward / backward
 * Replaces custom_layers.RoiResizeConv.call (custom_layers.py:35-56) and its
 * TF autodiff gradient.  mode RESIZE = crop + TF-1.3 legacy bilinear resize
 * (reference behaviour); mode MAX = max pooling (north-star addition).
 *   feat [batch,H,W,C] f32 channels-last, rois [batch,N,4] (dtype per
 *   roi_dtype, truncated to int like K.cast(...,'int32'); x2/y2 exclusive),
 *   out [batch,N,P,P,C] f32, argmax [batch,N,P,P,C] i32 (MAX mode only).
 *   Backward: grad_out like out; grad_feat [batch,H,W,C] f32 is overwritten. */
FRCNN_API int frcnn_roi_fwd(frcnn_handle* h, void* stream, int mode, const float* feat, int height,
                  int width, int channels, const void* rois, int roi_dtype, int n_rois, int pool,
                  int batch, float* out, int32_t* argmax);
FRCNN_API int frcnn_roi_bwd(frcnn_handle* h, void* stream, int mode, const float* grad_out,
                  const void* rois, int roi_dtype, const int32_t* argmax, int height, int width,
                  int channels, int n_rois, int pool, int batch, float* grad_feat);

/* Max mode with a ONE-BYTE arg-max (training fast path: 5 instead of 8 bytes per pooled element leave the forward and
 * enter the backward).  argmax_u8 [batch,N,P,P,C] u8 = (dy << 4) | dx of the first maximum relative to the bin's first
 * cell (row floor(ph*h/P), column floor(pw*w/P) of the crop); outputs are identical to frcnn_roi_fwd(MAX), and
 * y1 + floor(ph*h/P) + dy, x1 + floor(pw*w/P) + dx is the cell frcnn_roi_fwd reports as a flat index.  Available when
 * frcnn_roi_compact_supported() returns 1: channels % 4 == 0, pool <= 8 and ceil(H/pool)+1, ceil(W/pool)+1 <= 16 (every
 * bin fits 16 x 16 cells) and n_rois < 65536; otherwise FRCNN_ERR_UNSUPPORTED -- use the int32 entry points. */
FRCNN_API int frcnn_roi_compact_supported(int height, int width, int channels, int pool);
FRCNN_API int frcnn_roi_max_fwd_compact(frcnn_handle* h, void* stream, const float* feat, int height, int width,
                              int channels, const void* rois, int roi_dtype, int n_rois, int pool, int batch,
                              float* out, uint8_t* argmax_u8);
FRCNN_API int frcnn_roi_max_bwd_compact(frcnn_handle* h, void* stream, const float* grad_out, const void* rois,
                              int roi_dtype, const uint8_t* argmax_u8, int height, int width, int channels,
                              int n_rois, int pool, int batch, float* grad_feat);

/* ---- K-e: detector post-processing
 * Replaces the loops of voc_dets.get_dets (voc_dets.py:51-86): per-row argmax
 * class, f64 decode (util.transform, util.py:55-74), x stride, per-class f64
 * NMS, rescale + half-even rounding.
 *   rois [batch,M,4] i16, out_cls [batch,M,K] f32, out_reg [batch,M,4(K-1)]
 *   f32, resize_ratio [batch] f64, n_rows [batch] i32 (device, may be NULL = M):
 *   rows >= n_rows[b] are ignored (fixed-shape batches; frcnn_pad_rois gives the
 *   count the reference's batching would have run).  det_boxes [batch,M,4] i32, det_probs
 *   [batch,M] f32, det_cls [batch,M] i32, det_count [batch]; order = classes by
 *   first appearance, rows in NMS pick order.  out_reg's columns 4c..4c+3 belong
 *   to class c, so with bg_index != K-1 class K-1 has none: rows whose arg-max
 *   is K-1 are then dropped like 'bg' rows. */
FRCNN_API int frcnn_det_postprocess(frcnn_handle* h, void* stream, const int16_t* rois, const float* out_cls,
                          const float* out_reg, const double* resize_ratio, const int32_t* n_rows,
                          int m_rows, int n_classes, int bg_index, int stride, double det_threshold,
                          double nms_thresh, int max_boxes, int batch, int32_t* det_boxes,
                          float* det_probs, int32_t* det_cls, int32_t* det_count);

/* ---- stand-alone helpers behind the reference's module-level functions ------------------ */

/* util.cross_ious (util.py:146-177): iou [n, n_gt] f32, no +1 convention, float32 op order of
 * the reference.  boxes [n,4] int16 (box_dtype FRCNN_ROI_I16; areas wrap in int16 like numpy's)
 * or float32 (FRCNN_ROI_F32); gt [n_gt,4] f32. */
FRCNN_API int frcnn_cross_ious(frcnn_handle* h, void* stream, const void* boxes, int box_dtype, int n,
                     const float* gt, int n_gt, float* iou);

/* util.transform_np_inplace (util.py:111-142) when decode != 0, then
 * det_util._sanitize_boxes_inplace (det_util.py:179-192) when sanitize_cols/rows > 0.
 * boxes [n,4] f32 are updated in place; deltas [n,4] f32 = (tx,ty,tw,th) already divided by
 * BBREG_MULTIPLIERS. */
FRCNN_API int frcnn_box_transform(frcnn_handle* h, void* stream, float* boxes, const float* deltas, int n,
                        int decode, int sanitize_cols, int sanitize_rows);

/* Anchor boxes [rows,cols,A,4] f32.  pixel_space == 0: det_util._get_anchor_coords
 * (det_util.py:162-175), centre = cell index, `stride` ignored, dims used as given.
 * pixel_space != 0: rpn_util._get_all_anchor_coords (rpn_util.py:276-298), centre =
 * int(stride * (cell + 0.5)). */
FRCNN_API int frcnn_anchor_grid(frcnn_handle* h, void* stream, const int32_t* anchor_hw_host, int n_anchors,
                      int rows, int cols, int stride, int pixel_space, float* out);

/* det_util._get_valid_box_idxs (det_util.py:196-205): ascending indices of boxes [n,4] f32
 * with x2 > x1 and y2 > y1; out_index [n] i32, out_count [1] i32. */
FRCNN_API int frcnn_valid_boxes(frcnn_handle* h, void* stream, const float* boxes, int n, int32_t* out_index,
                      int32_t* out_count);

/* RoI batching rule of voc_dets.get_dets (voc_dets.py:37-46): the detector takes `group` RoIs at
 * a time and the last batch is padded with copies of its first RoI.  rois [batch,n_max,4] i16,
 * count [batch] -> out [batch,m_out,4] i16 with m_out >= n_max rounded up to `group`; rows past
 * the padded length are the empty box [0,0,0,0]; out_rows [batch] = count (clamped to 0..n_max)
 * rounded up. */
FRCNN_API int frcnn_pad_rois(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* count,
                             int n_max, int group, int m_out, int batch, int16_t* out, int32_t* out_rows);

/* Mini-batch gather of DetTrainingManager.get_training_input (det_util.py:119-125) for a batch of images:
 * rois [batch,n_max,4] i16, y_cls [batch,n_max,K] i32, y_tr [batch,n_max,8(K-1)] f32 are frcnn_label_rois's
 * outputs, index [batch,n_samples] i32 the host-drawn sample rows (det_util._get_det_samples, numpy's legacy RNG);
 * index -1 (image without an eligible RoI: the reference returns 4 x None) yields zero rows.
 * out_rois [batch,n_samples,4], out_cls [batch,n_samples,K], out_tr [batch,n_samples,8(K-1)]. */
FRCNN_API int frcnn_gather_det_samples(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* y_cls,
                                       const float* y_tr, const int32_t* index, int n_max, int n_classes,
                                       int n_samples, int batch, int16_t* out_rois, int32_t* out_cls, float* out_tr);

/* ---- masked losses fused with the path's own targets (widening row, SURVEY.md 8f-2)
 * Replaces loss_functions.py:15-48 (cls_loss_rpn, bbreg_loss_rpn) and :51-76 (bbreg_loss_det,
 * cls_loss_det), i.e. the Keras-backend expressions with binary_crossentropy / categorical_crossentropy
 * of Keras 2.0.8 on TF 1.3.  loss [batch,2] receives the scalar Keras reports per output
 * (RPN: class, box; detector: class, box); grad_* (optional, may be NULL) receive its gradient
 * with respect to the predictions.
 *   RPN: can_use / is_pos [batch,N] u8 and bbreg [batch,N,4] f32 are the UNPACKED labels
 *   (frcnn_label_anchors + sampling), cls_pred [batch,N] f32 (sigmoid outputs, (R,C,A) order),
 *   reg_pred [batch,N,4] f32.  The mask of the RPN box loss multiplies the summed smooth-L1
 *   like the reference does (loss_functions.py:40-46).
 *   Detector: y_class [batch,M,K] i32 one-hot, y_transform [batch,M,8(K-1)] f32 = [labels|targets]
 *   (frcnn_label_rois), cls_pred [batch,M,K] f32, reg_pred [batch,M,4(K-1)] f32. */
FRCNN_API int frcnn_rpn_losses(frcnn_handle* h, void* stream, const uint8_t* can_use, const uint8_t* is_pos,
                               const float* bbreg, const float* cls_pred, const float* reg_pred,
                               int n_per_image, int batch, float* loss, float* grad_cls, float* grad_reg);
/* RPN losses of a mixed-size batch: the inputs of frcnn_rpn_losses in the padded [batch,rows*cols*n_anchors] layout
 * ((R,C,A) order), extents [batch,2] i32 (device) = each image's own (rows_b, cols_b), clamped to [0,rows] x [0,cols].
 * loss[b] and the gradients of image b equal frcnn_rpn_losses on the cropped inputs [:rows_b, :cols_b] bit for bit
 * (the box loss's mean(mask) runs over the image's own rows_b*cols_b*A anchors).  Padding cells are never read; their
 * gradients are written as zero.  An image with a zero extent gets loss (0, 0) and zero gradients (the uniform entry
 * rejects n_per_image = 0). */
FRCNN_API int frcnn_rpn_losses_ragged(frcnn_handle* h, void* stream, const uint8_t* can_use, const uint8_t* is_pos,
                                      const float* bbreg, const float* cls_pred, const float* reg_pred, int rows,
                                      int cols, int n_anchors, int batch, const int32_t* extents, float* loss,
                                      float* grad_cls, float* grad_reg);
FRCNN_API int frcnn_det_losses(frcnn_handle* h, void* stream, const int32_t* y_class,
                               const float* y_transform, const float* cls_pred, const float* reg_pred,
                               int m_rows, int n_classes, int batch, float* loss, float* grad_cls,
                               float* grad_reg);

/* ---- VOC detection evaluation (widening row, SURVEY.md 8f-3)
 * Replaces the matching loop of eval_dets.voc_eval (eval_dets.py:75-116) and its precision /
 * recall / 11-point AP arithmetic (eval_dets.py:118-125, voc_ap :8-19) for one class.
 *   det_boxes [n_dets,4] f64 sorted by descending confidence; img_det_offsets [n_images+1] +
 *   img_det_rank [n_dets]: CSR listing, per image, the ranks of its detections in ascending order;
 *   gt_boxes [n_gt,4] f64 / gt_difficult [n_gt] u8 grouped by image with img_gt_offsets [n_images+1].
 *   IoU uses the devkit's +1 convention in float64; tp / fp [n_dets] f64 are indexed by rank.
 *   frcnn_voc_pr_ap: rec / prec [n_dets] f64 and ap [1] f64 = sum over thresholds [n_thresholds] f64
 *   (device) of max(prec[rec >= t]) / n_thresholds (0 where no element qualifies). */
FRCNN_API int frcnn_voc_match(frcnn_handle* h, void* stream, const double* det_boxes,
                              const int32_t* img_det_offsets, const int32_t* img_det_rank,
                              const double* gt_boxes, const uint8_t* gt_difficult,
                              const int32_t* img_gt_offsets, int n_images, int n_dets, int n_gt,
                              double ovthresh, double* tp, double* fp);
FRCNN_API int frcnn_voc_pr_ap(frcnn_handle* h, void* stream, const double* tp, const double* fp, int n_dets,
                              double npos, const double* thresholds, int n_thresholds, double* rec,
                              double* prec, double* ap);

/* ---- SURVEY 8f-4: host-side input pipeline on the device
 * Pixels of shapes.Image.data (shapes.py:19-29: cv2.resize(INTER_CUBIC) then cv2.flip(img, 1) when `flip`) for a
 * batch of equally sized uint8 images [batch,H,W,channels] (BGR as cv2.imread returns them).  OpenCV's generic
 * fixed-point bicubic (A = -0.75, x2048 short coefficients, (sum + 2^21) >> 22): within one grey level of cv2.resize.
 *   out_u8 [batch,dst_h,dst_w,channels] and / or out_f32 (same shape, float32 = pixel - mean_host[c], the mean
 *   subtraction of resnet.preprocess / vgg.preprocess, resnet.py:64-75; mean_host = `channels` doubles on the HOST,
 *   NULL = zeros) -- either may be NULL. */
FRCNN_API int frcnn_image_resize_cubic(frcnn_handle* h, void* stream, const uint8_t* src, int src_height, int src_width,
                             int channels, int dst_height, int dst_width, int flip, int batch,
                             const double* mean_host, uint8_t* out_u8, float* out_f32);

/* The same for a batch of DIFFERENTLY sized sources, each resized to its own size, in one launch.
 *   src: uint8 images [src_h_b, src_w_b, channels] packed back to back; src_offsets [batch] i64 byte offsets into it,
 *   src_bytes = size of the buffer.  geom [batch,4] i32 = (src_h_b, src_w_b, dst_h_b, dst_w_b), flip [batch] u8 (NULL =
 *   no mirror; else image b is mirrored within its own width where flip[b] != 0); all three on the device and never
 *   read on the host, so one captured graph serves every mix of sizes up to its padded shape.
 *   out_u8 / out_f32 [batch,dst_height,dst_width,channels] (either may be NULL; mean_host as above): out[b, :dst_h_b,
 *   :dst_w_b] equals frcnn_image_resize_cubic on image b alone bit for bit; every other element is written as zero.
 *   dst_h_b / dst_w_b are clamped to [0,dst_height] x [0,dst_width].  An image whose source size is not positive or
 *   whose bytes do not lie within [0, src_bytes) is written as zeros and none of its bytes are read. */
FRCNN_API int frcnn_image_resize_cubic_ragged(frcnn_handle* h, void* stream, const uint8_t* src, const int64_t* src_offsets,
                                              long long src_bytes, const int32_t* geom, const uint8_t* flip, int channels,
                                              int dst_height, int dst_width, int batch, const double* mean_host,
                                              uint8_t* out_u8, float* out_f32);

/* GT boxes of a resized / mirrored image (shapes.py:93-101 Box.resize, :292-300 horizontal_flip): boxes
 * [batch,n_max,4] f64 corners, n_box [batch] i32 (NULL = n_max), ratio [batch] f64, flip_width [batch] f64 (NULL or a
 * negative entry = not mirrored; else the width the box is mirrored about) -> out [batch,n_max,4] f64; float64 like
 * the reference's Python floats, rows >= n_box zeroed. */
FRCNN_API int frcnn_gt_transform(frcnn_handle* h, void* stream, const double* boxes, const int32_t* n_box, int n_max,
                       int batch, const double* ratio, const double* flip_width, double* out);

/* ---- training mini-batch draws on the device (counter-based RNG)
 * The opt-in alternative to the host draws that replay the reference's MT19937 streams (frcnn_pack_rpn_targets'
 * rank lists, frcnn_gather_det_samples' host-drawn index): the same sampling RULE, a different stream, no host round
 * trip, and the calls can be captured in a CUDA graph.
 *   state [2] i64 (device) = (seed, offset), read and never written: the caller advances offset by `batch` after a
 *   call (ops.sample_rpn_ / ops.sample_det do, stream-ordered).  Image b draws from
 *     word(j, tag) = word j & 3 of curand_Philox4x32_10(ctr = (j >> 2, img_lo, img_hi, tag), key = (seed_lo, seed_hi))
 *   with img = offset + b (64-bit), tag 0 = RPN anchor keys, 1 = detector RoI keys, 2 = detector draws with
 *   replacement.  Integer arithmetic only: oracle/sample_oracle.py reproduces every result bit for bit.
 *
 * RPN (rule of rpn_util.py:324-350): P = usable positives (can_use && is_pos), Q = usable negatives, sizes from
 *   counts [batch,2] (frcnn_label_anchors*'s output).  keep_p = min(|P|, max_pos), keep_q = min(|Q|, sample_size -
 *   keep_p) (the reference's 128 / 256).  In each category the kept anchors are the `keep` ones with the smallest
 *   (word(i, 0), i); every other anchor of the category gets can_use = 0 in place; is_pos and bbreg are untouched.  The
 *   kept set is a uniformly random subset of the size the reference keeps, i.e. the distribution of the reference's
 *   switch-off of a uniformly random complement.  i is the anchor's flat index on the image's OWN map,
 *   (y*cols_b + x)*A + a, so the ragged entry equals the uniform entry on each cropped map; padding is not touched.
 *   Requires 0 <= max_pos <= sample_size.
 *
 * Detector (rule of det_util.py:260-306): per image the rows r < n_rows[b] (clamped to n_max) of frcnn_label_rois'
 *   output, is_pos [batch,n_max] u8; P = rows with is_pos, Q = the other rows, S = n_samples, want_pos = S / 4.
 *   Positives: all of P if |P| < want_pos, else the want_pos rows with the smallest (word(r, 1), r).
 *   want_neg = S - #chosen positives.  |Q| >= want_neg: the want_neg rows of Q with the smallest (word(r, 1), r).
 *   0 < |Q| < want_neg: draws with replacement Q[(uint64(word(t, 2)) * |Q|) >> 32], t = 0..want_neg-1, Q ascending
 *   (each row's probability is off from 1/|Q| by at most |Q| / 2^32).  |Q| = 0: the reference's tiling of P,
 *   P[t % |P|].  Rows chosen without replacement are written in ascending row order, positives first; draws with
 *   replacement in draw order.  out_index [batch,n_samples] i32 (frcnn_gather_det_samples' index), out_has [batch] u8;
 *   an image without an eligible row gets an all -1 row and out_has = 0.  n_max <= 4096 (FRCNN_ERR_UNSUPPORTED above). */
FRCNN_API int frcnn_sample_rpn(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos,
                               const int32_t* counts, int n_per_image, int max_pos, int sample_size,
                               const int64_t* state, int batch);
FRCNN_API int frcnn_sample_rpn_ragged(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos,
                                      const int32_t* counts, int rows, int cols, int n_anchors, const int32_t* extents,
                                      int max_pos, int sample_size, const int64_t* state, int batch);
FRCNN_API int frcnn_sample_det(frcnn_handle* h, void* stream, const uint8_t* is_pos, const int32_t* n_rows, int n_max,
                               int n_samples, const int64_t* state, int batch, int32_t* out_index, uint8_t* out_has);

#ifdef __cplusplus
}
#endif
#endif /* FRCNN_B200_H */
