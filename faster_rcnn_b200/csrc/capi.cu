// extern "C" boundary of libfrcnn_b200.so (declared in include/frcnn_b200.h): argument checks,
// the per-handle scratch arena and the dispatch to the kernel launchers of the other TUs.
#include <new>

#include "roi_common.cuh"

namespace frcnn {

// launchers (one per kernel family)
int launch_decode_topk(frcnn_handle*, cudaStream_t, const float*, const float*, const AnchorTable&, int, int, int,
                       int, int16_t*, float*, int32_t*, int32_t*, float*, const int32_t*);
int launch_nms_i16(frcnn_handle*, cudaStream_t, const int16_t*, const float*, const int32_t*, int, int, double, int,
                   int32_t*, int32_t*, int16_t*, float*);
int launch_nms_f64(frcnn_handle*, cudaStream_t, const double*, const float*, const int32_t*, int, int, double, int,
                   int, int32_t*, int32_t*);
int launch_label_anchors(frcnn_handle*, cudaStream_t, const float*, const int32_t*, const int32_t*, int,
                         const AnchorTable&, int, int, int, int, uint8_t*, uint8_t*, float*, int32_t*, const int32_t*);
int launch_pack_rpn(frcnn_handle*, cudaStream_t, uint8_t*, const uint8_t*, const float*, const int32_t*,
                    const int32_t*, const int32_t*, const int32_t*, int, int, int, int, uint8_t*, float*);
int launch_label_rois(frcnn_handle*, cudaStream_t, const int16_t*, const int32_t*, int, const double*,
                      const int32_t*, const int32_t*, int, int, int, int16_t*, int32_t*, float*, int32_t*, int32_t*);
int launch_roi_fwd(frcnn_handle*, cudaStream_t, int, const float*, int, int, int, const void*, int, int, int, int,
                   float*, int32_t*, int);
int launch_roi_bwd(frcnn_handle*, cudaStream_t, int, const float*, const void*, int, const int32_t*, int, int, int,
                   int, int, int, float*, int);
int launch_det_postprocess(frcnn_handle*, cudaStream_t, const int16_t*, const float*, const float*, const double*,
                           const int32_t*, int, int, int, int, double, double, int, int, int32_t*, float*, int32_t*, int32_t*);

int launch_cross_ious(frcnn_handle*, cudaStream_t, const void*, int, int, const float*, int, float*);
int launch_box_transform(frcnn_handle*, cudaStream_t, float*, const float*, int, int, int, int);
int launch_anchor_grid(frcnn_handle*, cudaStream_t, const AnchorTable&, int, int, int, int, float*);
int launch_valid_boxes(frcnn_handle*, cudaStream_t, const float*, int, int32_t*, int32_t*);
int launch_gather_det_samples(frcnn_handle*, cudaStream_t, const int16_t*, const int32_t*, const float*, const int32_t*,
                              int, int, int, int, int, int16_t*, int32_t*, float*);
int launch_clip_rois(frcnn_handle*, cudaStream_t, const void*, int, int, int, const int32_t*, void*);
int launch_pad_rois(frcnn_handle*, cudaStream_t, const int16_t*, const int32_t*, int, int, int, int, int16_t*,
                    int32_t*);

int launch_rpn_losses(frcnn_handle*, cudaStream_t, const uint8_t*, const uint8_t*, const float*, const float*,
                      const float*, int, int, float*, float*, float*);
int launch_rpn_losses_ragged(frcnn_handle*, cudaStream_t, const uint8_t*, const uint8_t*, const float*, const float*,
                             const float*, int, int, int, int, const int32_t*, float*, float*, float*);
int launch_det_losses(frcnn_handle*, cudaStream_t, const int32_t*, const float*, const float*, const float*, int, int,
                      int, float*, float*, float*);

int launch_voc_match(frcnn_handle*, cudaStream_t, const double*, const int32_t*, const int32_t*, const double*,
                     const uint8_t*, const int32_t*, int, double, uint8_t*, double*, double*);
int launch_voc_pr_ap(frcnn_handle*, cudaStream_t, const double*, const double*, int, double, const double*, int, double*,
                     double*, double*);

int launch_image_resize(frcnn_handle*, cudaStream_t, const uint8_t*, int, int, int, int, int, int, int, const double*,
                        uint8_t*, float*);
int launch_image_resize_ragged(frcnn_handle*, cudaStream_t, const uint8_t*, const int64_t*, long long, const int32_t*,
                               const uint8_t*, int, int, int, int, const double*, uint8_t*, float*);
int jpeg_inspect(const uint8_t*, long long, int32_t*);
int launch_jpeg_decode(frcnn_handle*, cudaStream_t, const uint8_t*, const uint8_t*, const int64_t*, const int64_t*, int,
                       uint8_t*, const int64_t*, long long, int32_t*);
int launch_gt_transform(frcnn_handle*, cudaStream_t, const double*, const int32_t*, int, int, const double*, const double*,
                        double*);
int launch_sample_rpn(frcnn_handle*, cudaStream_t, uint8_t*, const uint8_t*, const int32_t*, int, int, int, int,
                      const int32_t*, int, int, const int64_t*, int);
int launch_sample_det(frcnn_handle*, cudaStream_t, const uint8_t*, const int32_t*, int, int, const int64_t*, int, int32_t*,
                      uint8_t*);

// ---- scratch arena -------------------------------------------------------------------------
// Bump allocator over one device block.  Every public entry point starts with arena_reset();
// the launchers then carve their workspaces with arena_get().  When a call needs more than the
// block holds, an overflow block is chained (never freed mid-call: kernels already enqueued may
// still use the old one) and the next arena_reset() synchronises the stream and merges them.
int arena_reset(frcnn_handle* h, cudaStream_t stream) {
  if (h->n_overflow > 0) {
    FRCNN_CUDA(h, cudaStreamSynchronize(stream));
    size_t total = h->arena_bytes;
    for (int i = 0; i < h->n_overflow; ++i) {
      total += h->overflow_bytes[i];
      cudaFree(h->overflow[i]);
    }
    h->n_overflow = 0;
    if (h->arena) cudaFree(h->arena);
    h->arena = nullptr;
    h->arena_bytes = 0;
    FRCNN_CUDA(h, cudaMalloc(&h->arena, total));
    h->arena_bytes = total;
  }
  h->arena_used = 0;
  return FRCNN_OK;
}

int arena_get(frcnn_handle* h, cudaStream_t stream, size_t bytes, void** out) {
  (void)stream;
  bytes = align_up(bytes ? bytes : 1, 256);
  if (h->arena_used + bytes <= h->arena_bytes) {
    *out = static_cast<char*>(h->arena) + h->arena_used;
    h->arena_used += bytes;
    return FRCNN_OK;
  }
  if (h->n_overflow >= FRCNN_MAX_OVERFLOW) return fail(h, FRCNN_ERR_NOMEM, "arena: too many overflow blocks%s%s");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return fail(h, FRCNN_ERR_NOMEM, "arena: cudaMalloc failed: %s%s", cudaGetErrorString(e));
  h->overflow[h->n_overflow] = p;
  h->overflow_bytes[h->n_overflow] = bytes;
  h->n_overflow++;
  *out = p;
  return FRCNN_OK;
}

int host_staging(frcnn_handle* h, cudaStream_t stream, size_t bytes) {
  (void)stream;
  if (h->pinned_used) FRCNN_CUDA(h, cudaEventSynchronize(h->pinned_done));
  if (bytes > h->pinned_bytes) {
    if (h->pinned) cudaFreeHost(h->pinned);
    h->pinned = nullptr;
    h->pinned_bytes = 0;
    FRCNN_CUDA(h, cudaMallocHost(&h->pinned, bytes));
    h->pinned_bytes = bytes;
  }
  h->pinned_used = 1;
  return FRCNN_OK;
}

// The scratch arena is per handle and is reused by every call.  Calls on ONE stream are ordered by the stream.  When a
// call arrives on a different stream than the previous call, the new stream first waits (on the device) for
// everything already enqueued on the previous stream, so kernels of the two calls can never share scratch
// concurrently.  A stream that is being captured is left alone (cross-stream dependencies would leak into the
// capture): captured sequences run on a private handle (pipeline.GraphedRun).
int stream_handover(frcnn_handle* h, cudaStream_t st) {
  if (h->last_stream_set && h->last_stream != st) {
    cudaStreamCaptureStatus a = cudaStreamCaptureStatusNone, b = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &a);
    cudaStreamIsCapturing(h->last_stream, &b);
    if (a == cudaStreamCaptureStatusNone && b == cudaStreamCaptureStatusNone) {
      FRCNN_CUDA(h, cudaEventRecord(h->handover, h->last_stream));
      FRCNN_CUDA(h, cudaStreamWaitEvent(st, h->handover, 0));
    }
  }
  h->last_stream = st;
  h->last_stream_set = 1;
  return FRCNN_OK;
}

static int make_table(frcnn_handle* h, const int32_t* anchor_hw_host, int n_anchors, int divide_by, AnchorTable* tab) {
  if (!anchor_hw_host || n_anchors <= 0 || n_anchors > FRCNN_MAX_ANCHORS)
    return fail(h, FRCNN_ERR_INVALID, "anchor table: need 1..FRCNN_MAX_ANCHORS [height,width] rows%s%s");
  tab->n = n_anchors;
  for (int a = 0; a < n_anchors; ++a) {
    tab->h[a] = floordiv(anchor_hw_host[2 * a], divide_by);       // det_util.py:374 `anchor_dims // stride`
    tab->w[a] = floordiv(anchor_hw_host[2 * a + 1], divide_by);
  }
  return FRCNN_OK;
}

}  // namespace frcnn

using namespace frcnn;

#define FRCNN_REQUIRE(h, cond, msg)                                          \
  do {                                                                       \
    if (!(cond)) return frcnn::fail((h), FRCNN_ERR_INVALID, "%s%s", msg);    \
  } while (0)

#define FRCNN_ENTER(h, stream_void)                                          \
  if (!(h)) return FRCNN_ERR_INVALID;                                        \
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_void);             \
  {                                                                          \
    cudaError_t e_ = cudaSetDevice((h)->device);                             \
    if (e_ != cudaSuccess) return frcnn::fail((h), FRCNN_ERR_CUDA, "cudaSetDevice: %s%s", cudaGetErrorString(e_)); \
    int rc_ = frcnn::stream_handover((h), st);                               \
    if (rc_) return rc_;                                                     \
    rc_ = frcnn::arena_reset((h), st);                                       \
    if (rc_) return rc_;                                                     \
  }

extern "C" {

int frcnn_abi_version(void) { return FRCNN_ABI_VERSION; }

int frcnn_create(frcnn_handle** out, int device) {
  if (!out) return FRCNN_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return FRCNN_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return FRCNN_ERR_CUDA;
  frcnn_handle* h = new (std::nothrow) frcnn_handle();
  if (!h) return FRCNN_ERR_NOMEM;
  memset(h, 0, sizeof(*h));
  h->device = device;
  int major = 0;
  cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetAttribute(&h->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (major != 10) {   // the library carries sm_100a code only
    delete h;
    return FRCNN_ERR_UNSUPPORTED;
  }
  if (cudaEventCreateWithFlags(&h->handover, cudaEventDisableTiming) != cudaSuccess) {
    delete h;
    return FRCNN_ERR_CUDA;
  }
  if (cudaEventCreateWithFlags(&h->pinned_done, cudaEventDisableTiming) != cudaSuccess) {
    cudaEventDestroy(h->handover);
    delete h;
    return FRCNN_ERR_CUDA;
  }
  *out = h;
  return FRCNN_OK;
}

void frcnn_destroy(frcnn_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (int i = 0; i < h->n_overflow; ++i) cudaFree(h->overflow[i]);
  if (h->arena) cudaFree(h->arena);
  if (h->handover) cudaEventDestroy(h->handover);
  if (h->pinned_used) cudaEventSynchronize(h->pinned_done);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->pinned_done) cudaEventDestroy(h->pinned_done);
  delete h;
}

const char* frcnn_last_error(frcnn_handle* h) { return h ? h->err : "null handle"; }

int frcnn_reserve(frcnn_handle* h, size_t bytes) {
  if (!h) return FRCNN_ERR_INVALID;
  FRCNN_CUDA(h, cudaSetDevice(h->device));
  if (bytes <= h->arena_bytes && h->n_overflow == 0) return FRCNN_OK;
  FRCNN_CUDA(h, cudaDeviceSynchronize());
  for (int i = 0; i < h->n_overflow; ++i) cudaFree(h->overflow[i]);
  h->n_overflow = 0;
  if (bytes > h->arena_bytes) {
    if (h->arena) cudaFree(h->arena);
    h->arena = nullptr;
    h->arena_bytes = 0;
    FRCNN_CUDA(h, cudaMalloc(&h->arena, align_up(bytes, 256)));
    h->arena_bytes = align_up(bytes, 256);
  }
  h->arena_used = 0;
  return FRCNN_OK;
}

long long frcnn_launch_count(frcnn_handle* h) { return h ? h->launches : 0; }

static int decode_topk_entry(frcnn_handle* h, cudaStream_t st, const float* regr, const float* cls,
                             const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                             int batch, const int32_t* extents, int16_t* out_boxes, float* out_scores,
                             int32_t* out_index, int32_t* out_count, float* dense_boxes) {
  FRCNN_REQUIRE(h, regr && cls && out_boxes && out_scores && out_index && out_count, "decode_topk: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && stride > 0 && k > 0 && batch > 0, "decode_topk: non-positive size");
  FRCNN_REQUIRE(h, rows <= 32767 && cols <= 32767, "decode_topk: map larger than int16 coordinates");
  AnchorTable tab;
  int rc = make_table(h, anchor_hw_host, n_anchors, stride, &tab);
  if (rc) return rc;
  return launch_decode_topk(h, st, regr, cls, tab, rows, cols, k, batch, out_boxes, out_scores, out_index,
                            out_count, dense_boxes, extents);
}

int frcnn_decode_topk(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                      const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                      int batch, int16_t* out_boxes, float* out_scores, int32_t* out_index,
                      int32_t* out_count, float* dense_boxes) {
  FRCNN_ENTER(h, stream);
  return decode_topk_entry(h, st, regr, cls, anchor_hw_host, rows, cols, n_anchors, stride, k, batch, nullptr,
                           out_boxes, out_scores, out_index, out_count, dense_boxes);
}

int frcnn_decode_topk_ragged(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                             const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                             int batch, const int32_t* extents, int16_t* out_boxes, float* out_scores,
                             int32_t* out_index, int32_t* out_count, float* dense_boxes) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, extents, "decode_topk_ragged: null extents");
  FRCNN_REQUIRE(h, !dense_boxes, "decode_topk_ragged: dense_boxes must be NULL");
  return decode_topk_entry(h, st, regr, cls, anchor_hw_host, rows, cols, n_anchors, stride, k, batch, extents,
                           out_boxes, out_scores, out_index, out_count, nullptr);
}

int frcnn_nms_i16(frcnn_handle* h, void* stream, const int16_t* boxes, const float* scores, const int32_t* n,
                  int n_max, int batch, double thresh, int max_boxes, int32_t* keep_index, int32_t* keep_count,
                  int16_t* keep_boxes, float* keep_scores) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && scores && keep_index && keep_count, "nms_i16: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && batch > 0 && max_boxes > 0, "nms_i16: non-positive size");
  return launch_nms_i16(h, st, boxes, scores, n, n_max, batch, thresh, max_boxes, keep_index, keep_count,
                        keep_boxes, keep_scores);
}

int frcnn_nms_f64(frcnn_handle* h, void* stream, const double* boxes, const float* scores,
                  const int32_t* seg_offsets, int n_seg, int max_seg_len, double thresh, int max_boxes,
                  int out_stride, int32_t* keep_index, int32_t* keep_count) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && scores && seg_offsets && keep_index && keep_count, "nms_f64: null pointer");
  FRCNN_REQUIRE(h, n_seg > 0 && max_seg_len > 0 && max_boxes > 0 && out_stride > 0, "nms_f64: non-positive size");
  FRCNN_REQUIRE(h, out_stride >= (max_boxes < max_seg_len ? max_boxes : max_seg_len),
                "nms_f64: out_stride smaller than min(max_boxes, max_seg_len)");
  return launch_nms_f64(h, st, boxes, scores, seg_offsets, n_seg, max_seg_len, thresh, max_boxes, out_stride,
                        keep_index, keep_count);
}

static int proposals_entry(frcnn_handle* h, cudaStream_t st, const float* regr, const float* cls,
                           const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                           double thresh, int max_boxes, int batch, const int32_t* extents, int16_t* out_rois,
                           float* out_scores, int32_t* out_count) {
  FRCNN_REQUIRE(h, regr && cls && out_rois && out_scores && out_count, "proposals: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && stride > 0 && k > 0 && batch > 0 && max_boxes > 0,
                "proposals: non-positive size");
  FRCNN_REQUIRE(h, rows <= 32767 && cols <= 32767, "proposals: map larger than int16 coordinates");
  AnchorTable tab;
  int rc = make_table(h, anchor_hw_host, n_anchors, stride, &tab);
  if (rc) return rc;
  const long long n_all = (long long)rows * cols * n_anchors;
  const int kk = (int)(k < n_all ? k : n_all);
  if (kk > FRCNN_NMS_MAX_UNSORTED)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "proposals: k above FRCNN_NMS_MAX_UNSORTED (use decode_topk + nms_i16)%s%s");
  void *tb = nullptr, *ts = nullptr, *ti = nullptr, *tc = nullptr, *ki = nullptr;
  if ((rc = arena_get(h, st, (size_t)batch * kk * 8, &tb))) return rc;
  if ((rc = arena_get(h, st, (size_t)batch * kk * 4, &ts))) return rc;
  if ((rc = arena_get(h, st, (size_t)batch * kk * 4, &ti))) return rc;
  if ((rc = arena_get(h, st, (size_t)batch * 4, &tc))) return rc;
  if ((rc = arena_get(h, st, (size_t)batch * max_boxes * 4, &ki))) return rc;
  rc = launch_decode_topk(h, st, regr, cls, tab, rows, cols, kk, batch, static_cast<int16_t*>(tb),
                          static_cast<float*>(ts), static_cast<int32_t*>(ti), static_cast<int32_t*>(tc), nullptr, extents);
  if (rc) return rc;
  return launch_nms_i16(h, st, static_cast<int16_t*>(tb), static_cast<float*>(ts), static_cast<int32_t*>(tc), kk,
                        batch, thresh, max_boxes, static_cast<int32_t*>(ki), out_count, out_rois, out_scores);
}

int frcnn_proposals(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                    const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                    double thresh, int max_boxes, int batch, int16_t* out_rois, float* out_scores,
                    int32_t* out_count) {
  FRCNN_ENTER(h, stream);
  return proposals_entry(h, st, regr, cls, anchor_hw_host, rows, cols, n_anchors, stride, k, thresh, max_boxes, batch,
                         nullptr, out_rois, out_scores, out_count);
}

int frcnn_proposals_ragged(frcnn_handle* h, void* stream, const float* regr, const float* cls,
                           const int32_t* anchor_hw_host, int rows, int cols, int n_anchors, int stride, int k,
                           double thresh, int max_boxes, int batch, const int32_t* extents, int16_t* out_rois,
                           float* out_scores, int32_t* out_count) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, extents, "proposals_ragged: null extents");
  return proposals_entry(h, st, regr, cls, anchor_hw_host, rows, cols, n_anchors, stride, k, thresh, max_boxes, batch,
                         extents, out_rois, out_scores, out_count);
}

static int label_anchors_entry(frcnn_handle* h, cudaStream_t st, const float* gt, const int32_t* n_gt,
                               const int32_t* img_wh, int g_max, int rows, int cols, int n_anchors,
                               const int32_t* anchor_hw_host, int stride, int batch, const int32_t* extents,
                               uint8_t* can_use, uint8_t* is_pos, float* bbreg, int32_t* counts) {
  FRCNN_REQUIRE(h, gt && n_gt && img_wh && can_use && is_pos && bbreg && counts, "label_anchors: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && stride > 0 && batch > 0, "label_anchors: non-positive size");
  FRCNN_REQUIRE(h, g_max > 0 && g_max <= FRCNN_MAX_GT, "label_anchors: g_max must be 1..FRCNN_MAX_GT");
  AnchorTable tab;
  int rc = make_table(h, anchor_hw_host, n_anchors, 1, &tab);
  if (rc) return rc;
  return launch_label_anchors(h, st, gt, n_gt, img_wh, g_max, tab, rows, cols, stride, batch, can_use, is_pos,
                              bbreg, counts, extents);
}

int frcnn_label_anchors(frcnn_handle* h, void* stream, const float* gt, const int32_t* n_gt, const int32_t* img_wh,
                        int g_max, int rows, int cols, int n_anchors, const int32_t* anchor_hw_host, int stride,
                        int batch, uint8_t* can_use, uint8_t* is_pos, float* bbreg, int32_t* counts) {
  FRCNN_ENTER(h, stream);
  return label_anchors_entry(h, st, gt, n_gt, img_wh, g_max, rows, cols, n_anchors, anchor_hw_host, stride, batch,
                             nullptr, can_use, is_pos, bbreg, counts);
}

int frcnn_label_anchors_ragged(frcnn_handle* h, void* stream, const float* gt, const int32_t* n_gt,
                               const int32_t* img_wh, int g_max, int rows, int cols, int n_anchors,
                               const int32_t* anchor_hw_host, int stride, int batch, const int32_t* extents,
                               uint8_t* can_use, uint8_t* is_pos, float* bbreg, int32_t* counts) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, extents, "label_anchors_ragged: null extents");
  return label_anchors_entry(h, st, gt, n_gt, img_wh, g_max, rows, cols, n_anchors, anchor_hw_host, stride, batch,
                             extents, can_use, is_pos, bbreg, counts);
}

int frcnn_clip_rois(frcnn_handle* h, void* stream, const void* rois, int roi_dtype, int n_rois, int batch,
                    const int32_t* extents, void* out) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, rois && extents && out, "clip_rois: null pointer");
  FRCNN_REQUIRE(h, roi_dtype >= FRCNN_ROI_I16 && roi_dtype <= FRCNN_ROI_F32, "clip_rois: unknown roi dtype");
  FRCNN_REQUIRE(h, n_rois > 0 && batch > 0 && batch <= 65535, "clip_rois: bad size");
  return launch_clip_rois(h, st, rois, roi_dtype, n_rois, batch, extents, out);
}

int frcnn_pack_rpn_targets(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos,
                           const float* bbreg, const int32_t* off_pos, const int32_t* off_pos_offsets,
                           const int32_t* off_neg, const int32_t* off_neg_offsets, int rows, int cols,
                           int n_anchors, int batch, uint8_t* y_class, float* y_bbreg) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, can_use && is_pos && bbreg && y_class && y_bbreg, "pack_rpn_targets: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && n_anchors > 0 && batch > 0, "pack_rpn_targets: bad size");
  FRCNN_REQUIRE(h, (!off_pos || off_pos_offsets) && (!off_neg || off_neg_offsets),
                "pack_rpn_targets: a rank list needs its offsets array");
  return launch_pack_rpn(h, st, can_use, is_pos, bbreg, off_pos, off_pos_offsets, off_neg, off_neg_offsets, rows,
                         cols, n_anchors, batch, y_class, y_bbreg);
}

int frcnn_label_rois(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* n_roi, int n_max,
                     const double* gt, const int32_t* gt_cls, const int32_t* n_gt, int g_max, int n_classes,
                     int batch, int16_t* out_rois, int32_t* out_cls, float* out_bbreg, int32_t* out_src,
                     int32_t* out_count) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, rois && gt && gt_cls && n_gt && out_rois && out_cls && out_bbreg && out_count,
                "label_rois: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && batch > 0 && n_classes >= 2, "label_rois: bad size");
  FRCNN_REQUIRE(h, g_max > 0 && g_max <= FRCNN_MAX_GT, "label_rois: g_max must be 1..FRCNN_MAX_GT");
  return launch_label_rois(h, st, rois, n_roi, n_max, gt, gt_cls, n_gt, g_max, n_classes, batch, out_rois,
                           out_cls, out_bbreg, out_src, out_count);
}

int frcnn_roi_fwd(frcnn_handle* h, void* stream, int mode, const float* feat, int height, int width, int channels,
                  const void* rois, int roi_dtype, int n_rois, int pool, int batch, float* out, int32_t* argmax) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, feat && rois && out, "roi_fwd: null pointer");
  FRCNN_REQUIRE(h, mode == FRCNN_ROI_RESIZE || mode == FRCNN_ROI_MAX, "roi_fwd: unknown mode");
  FRCNN_REQUIRE(h, mode != FRCNN_ROI_MAX || argmax, "roi_fwd: MAX mode needs an argmax buffer");
  FRCNN_REQUIRE(h, roi_dtype >= FRCNN_ROI_I16 && roi_dtype <= FRCNN_ROI_F32, "roi_fwd: unknown roi dtype");
  FRCNN_REQUIRE(h, height > 0 && width > 0 && channels > 0 && n_rois > 0 && pool > 0 && batch > 0,
                "roi_fwd: non-positive size");
  FRCNN_REQUIRE(h, batch <= 65535, "roi_fwd: batch > 65535");
  return launch_roi_fwd(h, st, mode, feat, height, width, channels, rois, roi_dtype, n_rois, pool, batch, out,
                        argmax, 0);
}

int frcnn_roi_compact_supported(int height, int width, int channels, int pool) {
  return roi_compact_supported(height, width, channels, pool) && pool <= 8 ? 1 : 0;
}

int frcnn_roi_max_fwd_compact(frcnn_handle* h, void* stream, const float* feat, int height, int width, int channels,
                              const void* rois, int roi_dtype, int n_rois, int pool, int batch, float* out,
                              uint8_t* argmax_u8) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, feat && rois && out && argmax_u8, "roi_max_fwd_compact: null pointer");
  FRCNN_REQUIRE(h, roi_dtype >= FRCNN_ROI_I16 && roi_dtype <= FRCNN_ROI_F32, "roi_max_fwd_compact: unknown roi dtype");
  FRCNN_REQUIRE(h, height > 0 && width > 0 && channels > 0 && n_rois > 0 && pool > 0 && batch > 0 && batch <= 65535,
                "roi_max_fwd_compact: bad size");
  return launch_roi_fwd(h, st, FRCNN_ROI_MAX, feat, height, width, channels, rois, roi_dtype, n_rois, pool, batch, out,
                        reinterpret_cast<int32_t*>(argmax_u8), 1);
}

int frcnn_roi_max_bwd_compact(frcnn_handle* h, void* stream, const float* grad_out, const void* rois, int roi_dtype,
                              const uint8_t* argmax_u8, int height, int width, int channels, int n_rois, int pool,
                              int batch, float* grad_feat) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, grad_out && rois && grad_feat && argmax_u8, "roi_max_bwd_compact: null pointer");
  FRCNN_REQUIRE(h, roi_dtype >= FRCNN_ROI_I16 && roi_dtype <= FRCNN_ROI_F32, "roi_max_bwd_compact: unknown roi dtype");
  FRCNN_REQUIRE(h, height > 0 && width > 0 && channels > 0 && n_rois > 0 && pool > 0 && batch > 0 && batch <= 65535,
                "roi_max_bwd_compact: bad size");
  return launch_roi_bwd(h, st, FRCNN_ROI_MAX, grad_out, rois, roi_dtype, reinterpret_cast<const int32_t*>(argmax_u8), height,
                        width, channels, n_rois, pool, batch, grad_feat, 1);
}

int frcnn_roi_bwd(frcnn_handle* h, void* stream, int mode, const float* grad_out, const void* rois, int roi_dtype,
                  const int32_t* argmax, int height, int width, int channels, int n_rois, int pool, int batch,
                  float* grad_feat) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, grad_out && rois && grad_feat, "roi_bwd: null pointer");
  FRCNN_REQUIRE(h, mode == FRCNN_ROI_RESIZE || mode == FRCNN_ROI_MAX, "roi_bwd: unknown mode");
  FRCNN_REQUIRE(h, mode != FRCNN_ROI_MAX || argmax, "roi_bwd: MAX mode needs the forward argmax");
  FRCNN_REQUIRE(h, roi_dtype >= FRCNN_ROI_I16 && roi_dtype <= FRCNN_ROI_F32, "roi_bwd: unknown roi dtype");
  FRCNN_REQUIRE(h, height > 0 && width > 0 && channels > 0 && n_rois > 0 && pool > 0 && batch > 0,
                "roi_bwd: non-positive size");
  FRCNN_REQUIRE(h, batch <= 65535, "roi_bwd: batch > 65535");
  return launch_roi_bwd(h, st, mode, grad_out, rois, roi_dtype, argmax, height, width, channels, n_rois, pool,
                        batch, grad_feat, 0);
}

int frcnn_det_postprocess(frcnn_handle* h, void* stream, const int16_t* rois, const float* out_cls,
                          const float* out_reg, const double* resize_ratio, const int32_t* n_rows, int m_rows, int n_classes,
                          int bg_index, int stride, double det_threshold, double nms_thresh, int max_boxes,
                          int batch, int32_t* det_boxes, float* det_probs, int32_t* det_cls, int32_t* det_count) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, rois && out_cls && out_reg && resize_ratio && det_boxes && det_probs && det_cls && det_count,
                "det_postprocess: null pointer");
  FRCNN_REQUIRE(h, m_rows > 0 && n_classes >= 2 && stride > 0 && max_boxes > 0 && batch > 0,
                "det_postprocess: bad size");
  return launch_det_postprocess(h, st, rois, out_cls, out_reg, resize_ratio, n_rows, m_rows, n_classes, bg_index, stride,
                                det_threshold, nms_thresh, max_boxes, batch, det_boxes, det_probs, det_cls,
                                det_count);
}

int frcnn_cross_ious(frcnn_handle* h, void* stream, const void* boxes, int box_dtype, int n, const float* gt,
                     int n_gt, float* iou) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && gt && iou, "cross_ious: null pointer");
  FRCNN_REQUIRE(h, box_dtype == FRCNN_ROI_I16 || box_dtype == FRCNN_ROI_F32, "cross_ious: boxes must be int16 or float32");
  FRCNN_REQUIRE(h, n > 0 && n_gt > 0, "cross_ious: non-positive size");
  FRCNN_REQUIRE(h, (reinterpret_cast<uintptr_t>(gt) & 15) == 0 && (reinterpret_cast<uintptr_t>(boxes) & 7) == 0,
                "cross_ious: misaligned pointer");
  return launch_cross_ious(h, st, boxes, box_dtype, n, gt, n_gt, iou);
}

int frcnn_box_transform(frcnn_handle* h, void* stream, float* boxes, const float* deltas, int n, int decode,
                        int sanitize_cols, int sanitize_rows) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && (deltas || !decode), "box_transform: null pointer");
  FRCNN_REQUIRE(h, n > 0, "box_transform: non-positive size");
  FRCNN_REQUIRE(h, (sanitize_cols > 0) == (sanitize_rows > 0), "box_transform: give both sanitize_cols and sanitize_rows or neither");
  return launch_box_transform(h, st, boxes, deltas, n, decode, sanitize_cols, sanitize_rows);
}

int frcnn_anchor_grid(frcnn_handle* h, void* stream, const int32_t* anchor_hw_host, int n_anchors, int rows,
                      int cols, int stride, int pixel_space, float* out) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, out, "anchor_grid: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && stride > 0, "anchor_grid: non-positive size");
  AnchorTable tab;
  int rc = make_table(h, anchor_hw_host, n_anchors, 1, &tab);
  if (rc) return rc;
  return launch_anchor_grid(h, st, tab, rows, cols, stride, pixel_space, out);
}

int frcnn_valid_boxes(frcnn_handle* h, void* stream, const float* boxes, int n, int32_t* out_index,
                      int32_t* out_count) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && out_index && out_count, "valid_boxes: null pointer");
  FRCNN_REQUIRE(h, n >= 0, "valid_boxes: negative size");
  return launch_valid_boxes(h, st, boxes, n, out_index, out_count);
}

int frcnn_pad_rois(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* count, int n_max, int group,
                   int m_out, int batch, int16_t* out, int32_t* out_rows) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, rois && count && out && out_rows, "pad_rois: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && group > 0 && batch > 0 && batch <= 65535, "pad_rois: bad size");
  FRCNN_REQUIRE(h, m_out >= (n_max + group - 1) / group * group, "pad_rois: m_out smaller than n_max rounded up to the group size");
  return launch_pad_rois(h, st, rois, count, n_max, group, m_out, batch, out, out_rows);
}

int frcnn_gather_det_samples(frcnn_handle* h, void* stream, const int16_t* rois, const int32_t* y_cls, const float* y_tr,
                             const int32_t* index, int n_max, int n_classes, int n_samples, int batch,
                             int16_t* out_rois, int32_t* out_cls, float* out_tr) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, rois && y_cls && y_tr && index && out_rois && out_cls && out_tr, "gather_det_samples: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && n_classes >= 2 && n_samples > 0 && batch > 0 && batch <= 65535,
                "gather_det_samples: bad size");
  return launch_gather_det_samples(h, st, rois, y_cls, y_tr, index, n_max, n_classes, 8 * (n_classes - 1), n_samples,
                                   batch, out_rois, out_cls, out_tr);
}

int frcnn_rpn_losses(frcnn_handle* h, void* stream, const uint8_t* can_use, const uint8_t* is_pos, const float* bbreg,
                     const float* cls_pred, const float* reg_pred, int n_per_image, int batch, float* loss,
                     float* grad_cls, float* grad_reg) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, can_use && is_pos && bbreg && cls_pred && reg_pred && loss, "rpn_losses: null pointer");
  FRCNN_REQUIRE(h, n_per_image > 0 && batch > 0, "rpn_losses: non-positive size");
  FRCNN_REQUIRE(h, ((reinterpret_cast<uintptr_t>(bbreg) | reinterpret_cast<uintptr_t>(reg_pred) |
                     reinterpret_cast<uintptr_t>(grad_reg)) & 15) == 0, "rpn_losses: box arrays must be 16-byte aligned");
  return launch_rpn_losses(h, st, can_use, is_pos, bbreg, cls_pred, reg_pred, n_per_image, batch, loss, grad_cls, grad_reg);
}

int frcnn_rpn_losses_ragged(frcnn_handle* h, void* stream, const uint8_t* can_use, const uint8_t* is_pos,
                            const float* bbreg, const float* cls_pred, const float* reg_pred, int rows, int cols,
                            int n_anchors, int batch, const int32_t* extents, float* loss, float* grad_cls,
                            float* grad_reg) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, can_use && is_pos && bbreg && cls_pred && reg_pred && extents && loss, "rpn_losses_ragged: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && n_anchors > 0 && batch > 0 && batch <= 65535, "rpn_losses_ragged: bad size");
  FRCNN_REQUIRE(h, (long long)rows * cols * n_anchors < (1LL << 31), "rpn_losses_ragged: map too large");
  FRCNN_REQUIRE(h, ((reinterpret_cast<uintptr_t>(bbreg) | reinterpret_cast<uintptr_t>(reg_pred) |
                     reinterpret_cast<uintptr_t>(grad_reg)) & 15) == 0, "rpn_losses_ragged: box arrays must be 16-byte aligned");
  return launch_rpn_losses_ragged(h, st, can_use, is_pos, bbreg, cls_pred, reg_pred, rows, cols, n_anchors, batch, extents,
                                  loss, grad_cls, grad_reg);
}

int frcnn_det_losses(frcnn_handle* h, void* stream, const int32_t* y_class, const float* y_transform,
                     const float* cls_pred, const float* reg_pred, int m_rows, int n_classes, int batch, float* loss,
                     float* grad_cls, float* grad_reg) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, y_class && y_transform && cls_pred && reg_pred && loss, "det_losses: null pointer");
  FRCNN_REQUIRE(h, m_rows > 0 && n_classes >= 2 && batch > 0, "det_losses: bad size");
  return launch_det_losses(h, st, y_class, y_transform, cls_pred, reg_pred, m_rows, n_classes, batch, loss, grad_cls,
                           grad_reg);
}

int frcnn_voc_match(frcnn_handle* h, void* stream, const double* det_boxes, const int32_t* img_det_offsets,
                    const int32_t* img_det_rank, const double* gt_boxes, const uint8_t* gt_difficult,
                    const int32_t* img_gt_offsets, int n_images, int n_dets, int n_gt, double ovthresh, double* tp,
                    double* fp) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, img_det_offsets && img_gt_offsets && tp && fp, "voc_match: null pointer");
  FRCNN_REQUIRE(h, n_images > 0 && n_dets >= 0 && n_gt >= 0, "voc_match: bad size");
  FRCNN_REQUIRE(h, (n_dets == 0 || (det_boxes && img_det_rank)) && (n_gt == 0 || (gt_boxes && gt_difficult)),
                "voc_match: null pointer");
  if (n_dets == 0) return FRCNN_OK;
  void* taken = nullptr;
  int rc = arena_get(h, st, (size_t)(n_gt > 0 ? n_gt : 1), &taken);
  if (rc) return rc;
  return launch_voc_match(h, st, det_boxes, img_det_offsets, img_det_rank, gt_boxes, gt_difficult, img_gt_offsets,
                          n_images, ovthresh, static_cast<uint8_t*>(taken), tp, fp);
}

int frcnn_voc_pr_ap(frcnn_handle* h, void* stream, const double* tp, const double* fp, int n_dets, double npos,
                    const double* thresholds, int n_thresholds, double* rec, double* prec, double* ap) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, ap && thresholds && n_thresholds > 0, "voc_pr_ap: null pointer");
  FRCNN_REQUIRE(h, n_dets >= 0 && (n_dets == 0 || (tp && fp && rec && prec)), "voc_pr_ap: null pointer");
  return launch_voc_pr_ap(h, st, tp, fp, n_dets, npos, thresholds, n_thresholds, rec, prec, ap);
}

int frcnn_image_resize_cubic(frcnn_handle* h, void* stream, const uint8_t* src, int src_height, int src_width,
                             int channels, int dst_height, int dst_width, int flip, int batch,
                             const double* mean_host, uint8_t* out_u8, float* out_f32) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, src && (out_u8 || out_f32), "image_resize_cubic: null pointer");
  FRCNN_REQUIRE(h, src_height > 0 && src_width > 0 && dst_height > 0 && dst_width > 0 && batch > 0 && batch <= 65535,
                "image_resize_cubic: bad size");
  FRCNN_REQUIRE(h, channels >= 1 && channels <= 4, "image_resize_cubic: 1..4 channels");
  FRCNN_REQUIRE(h, (long long)src_height * src_width * channels < (1LL << 31) && (dst_height + 7) / 8 <= 65535,
                "image_resize_cubic: image too large");
  return launch_image_resize(h, st, src, src_height, src_width, channels, dst_height, dst_width, flip, batch, mean_host,
                             out_u8, out_f32);
}

int frcnn_image_resize_cubic_ragged(frcnn_handle* h, void* stream, const uint8_t* src, const int64_t* src_offsets,
                                    long long src_bytes, const int32_t* geom, const uint8_t* flip, int channels,
                                    int dst_height, int dst_width, int batch, const double* mean_host, uint8_t* out_u8,
                                    float* out_f32) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, src && src_offsets && geom && (out_u8 || out_f32), "image_resize_cubic_ragged: null pointer");
  FRCNN_REQUIRE(h, src_bytes >= 0 && dst_height > 0 && dst_width > 0 && batch > 0 && batch <= 65535,
                "image_resize_cubic_ragged: bad size");
  FRCNN_REQUIRE(h, channels >= 1 && channels <= 4, "image_resize_cubic_ragged: 1..4 channels");
  FRCNN_REQUIRE(h, (dst_height + 31) / 32 <= 65535 && (long long)dst_width + dst_height < (1LL << 31),
                "image_resize_cubic_ragged: image too large");
  return launch_image_resize_ragged(h, st, src, src_offsets, src_bytes, geom, flip, channels, dst_height, dst_width, batch,
                                    mean_host, out_u8, out_f32);
}

int frcnn_jpeg_inspect(const uint8_t* file_host, long long n_bytes, int32_t* hw_host) {
  return jpeg_inspect(file_host, n_bytes, hw_host);
}

int frcnn_jpeg_decode(frcnn_handle* h, void* stream, const uint8_t* files_host, const uint8_t* files,
                      const int64_t* file_offsets_host, const int64_t* file_bytes_host, int batch, uint8_t* out,
                      const int64_t* out_offsets, long long out_bytes, int32_t* status) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, files_host && files && file_offsets_host && file_bytes_host && out && out_offsets && status,
                "jpeg_decode: null pointer");
  FRCNN_REQUIRE(h, batch > 0 && batch <= 65535 && out_bytes >= 0, "jpeg_decode: bad size");
  return launch_jpeg_decode(h, st, files_host, files, file_offsets_host, file_bytes_host, batch, out, out_offsets,
                            out_bytes, status);
}

int frcnn_gt_transform(frcnn_handle* h, void* stream, const double* boxes, const int32_t* n_box, int n_max, int batch,
                       const double* ratio, const double* flip_width, double* out) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, boxes && ratio && out, "gt_transform: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && batch > 0 && batch <= 65535, "gt_transform: bad size");
  return launch_gt_transform(h, st, boxes, n_box, n_max, batch, ratio, flip_width, out);
}

static int sample_rpn_entry(frcnn_handle* h, cudaStream_t st, uint8_t* can_use, const uint8_t* is_pos, const int32_t* counts,
                            int rows, int cols, int n_anchors, const int32_t* extents, int max_pos, int sample_size,
                            const int64_t* state, int batch) {
  FRCNN_REQUIRE(h, can_use && is_pos && counts && state, "sample_rpn: null pointer");
  FRCNN_REQUIRE(h, rows > 0 && cols > 0 && n_anchors > 0 && batch > 0, "sample_rpn: non-positive size");
  FRCNN_REQUIRE(h, (long long)rows * cols * n_anchors < (1LL << 31), "sample_rpn: map too large");
  FRCNN_REQUIRE(h, max_pos >= 0 && sample_size >= max_pos, "sample_rpn: need 0 <= max_pos <= sample_size");
  return launch_sample_rpn(h, st, can_use, is_pos, counts, rows * cols * n_anchors, rows, cols, n_anchors, extents, max_pos,
                           sample_size, state, batch);
}

int frcnn_sample_rpn(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos, const int32_t* counts,
                     int n_per_image, int max_pos, int sample_size, const int64_t* state, int batch) {
  FRCNN_ENTER(h, stream);
  return sample_rpn_entry(h, st, can_use, is_pos, counts, 1, n_per_image, 1, nullptr, max_pos, sample_size, state, batch);
}

int frcnn_sample_rpn_ragged(frcnn_handle* h, void* stream, uint8_t* can_use, const uint8_t* is_pos, const int32_t* counts,
                            int rows, int cols, int n_anchors, const int32_t* extents, int max_pos, int sample_size,
                            const int64_t* state, int batch) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, extents, "sample_rpn_ragged: null extents");
  return sample_rpn_entry(h, st, can_use, is_pos, counts, rows, cols, n_anchors, extents, max_pos, sample_size, state,
                          batch);
}

int frcnn_sample_det(frcnn_handle* h, void* stream, const uint8_t* is_pos, const int32_t* n_rows, int n_max, int n_samples,
                     const int64_t* state, int batch, int32_t* out_index, uint8_t* out_has) {
  FRCNN_ENTER(h, stream);
  FRCNN_REQUIRE(h, is_pos && n_rows && state && out_index && out_has, "sample_det: null pointer");
  FRCNN_REQUIRE(h, n_max > 0 && n_samples > 0 && batch > 0, "sample_det: non-positive size");
  return launch_sample_det(h, st, is_pos, n_rows, n_max, n_samples, state, batch, out_index, out_has);
}

}  // extern "C"
