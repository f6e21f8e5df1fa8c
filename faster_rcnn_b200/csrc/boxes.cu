// Stand-alone box helpers behind the reference's module-level functions.  The fused kernels in
// proposals.cu / label.cu are the hot path; these exist so that every helper the reference
// exposes (and its notebooks/tests call directly) runs on the device too.
//
//   cross_ious_kernel     util.cross_ious          util.py:146-177   (N,G) float32, no +1
//   box_transform_kernel  util.transform_np_inplace util.py:111-142  and/or
//                         det_util._sanitize_boxes_inplace det_util.py:179-192
//   anchor_grid_kernel    det_util._get_anchor_coords det_util.py:162-175 (feature space) or
//                         rpn_util._get_all_anchor_coords rpn_util.py:276-298 (pixel space)
//   valid_boxes_kernel    det_util._get_valid_box_idxs det_util.py:196-205 (ordered compaction)
#include "common.cuh"

namespace frcnn {

// One thread per (box, GT) element: consecutive threads write consecutive floats of the IoU row.
template <bool I16>
__global__ void __launch_bounds__(256)
cross_ious_kernel(const void* __restrict__ boxes, int n, const float* __restrict__ gt, int g_count,
                  float* __restrict__ iou) {
  const size_t e = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= (size_t)n * g_count) return;
  // 32-bit division whenever the matrix has fewer than 2^32 elements (a 64-bit division is ~100 instructions)
  int i, g;
  if (((unsigned long long)n * (unsigned)g_count >> 32) == 0ull) {
    i = (int)((unsigned)e / (unsigned)g_count);
    g = (int)((unsigned)e - (unsigned)i * (unsigned)g_count);
  } else {
    i = (int)(e / g_count);
    g = (int)(e % g_count);
  }
  float x1, y1, x2, y2, a_area;
  if (I16) {
    const short* p = reinterpret_cast<const short*>(boxes) + 4 * (size_t)i;
    x1 = (float)p[0]; y1 = (float)p[1]; x2 = (float)p[2]; y2 = (float)p[3];
    a_area = (float)((int)(short)((p[2] - p[0]) * (p[3] - p[1])));   // int16 product wraps like numpy's
  } else {
    const float4 b = ldg_f4(reinterpret_cast<const float*>(boxes) + 4 * (size_t)i);
    x1 = b.x; y1 = b.y; x2 = b.z; y2 = b.w;
    a_area = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
  }
  const float4 t = ldg_f4(gt + 4 * (size_t)g);
  const float g_area = __fmul_rn(__fsub_rn(t.z, t.x), __fsub_rn(t.w, t.y));
  const float w = np_max(0.0f, __fsub_rn(np_min(x2, t.z), np_max(x1, t.x)));
  const float h = np_max(0.0f, __fsub_rn(np_min(y2, t.w), np_max(y1, t.y)));
  const float inter = __fmul_rn(w, h);
  iou[e] = __fdiv_rn(inter, __fsub_rn(__fadd_rn(a_area, g_area), inter));
}

__global__ void __launch_bounds__(256)
box_transform_kernel(float4* __restrict__ boxes, const float4* __restrict__ deltas, int n, int decode,
                     int cols, int rows) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  float4 b = boxes[i];
  float x = b.x, y = b.y, x2 = b.z, y2 = b.w;
  if (decode) {
    const float4 t = deltas[i];
    float w = __fsub_rn(x2, x), h = __fsub_rn(y2, y);
    x = __fadd_rn(x, __fdiv_rn(w, 2.0f));
    y = __fadd_rn(y, __fdiv_rn(h, 2.0f));
    x = __fadd_rn(x, __fmul_rn(t.x, w));
    y = __fadd_rn(y, __fmul_rn(t.y, h));
    w = __fmul_rn(w, np_expf(t.z));
    h = __fmul_rn(h, np_expf(t.w));
    x = __fsub_rn(x, __fdiv_rn(w, 2.0f));
    y = __fsub_rn(y, __fdiv_rn(h, 2.0f));
    x = rintf(x); y = rintf(y); w = rintf(w); h = rintf(h);
    x2 = __fadd_rn(w, x);
    y2 = __fadd_rn(h, y);
  }
  if (cols > 0) {
    x2 = np_max(__fadd_rn(x, 1.0f), x2);
    y2 = np_max(__fadd_rn(y, 1.0f), y2);
    x = np_max(0.0f, x);
    y = np_max(0.0f, y);
    x2 = np_min((float)(cols - 1), x2);
    y2 = np_min((float)(rows - 1), y2);
  }
  boxes[i] = make_float4(x, y, x2, y2);
}

__global__ void __launch_bounds__(256)
anchor_grid_kernel(AnchorTable tab, int rows, int cols, int stride, int pixel_space, float4* __restrict__ out) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  const int n = rows * cols * tab.n;
  if (i >= n) return;
  const int a = i % tab.n, loc = i / tab.n;
  int cx = loc % cols, cy = loc / cols;
  if (pixel_space) {   // int(stride * (c + 0.5)), rpn_util.py:184-189
    cx = (int)((double)stride * ((double)cx + 0.5));
    cy = (int)((double)stride * ((double)cy + 0.5));
  }
  const int x1 = cx - floordiv(tab.w[a], 2), y1 = cy - floordiv(tab.h[a], 2);
  out[i] = make_float4((float)x1, (float)y1, (float)(x1 + tab.w[a]), (float)(y1 + tab.h[a]));
}

// single CTA, order-preserving stream compaction of the indices with x2 > x1 and y2 > y1
__global__ void __launch_bounds__(1024)
valid_boxes_kernel(const float4* __restrict__ boxes, int n, int* __restrict__ out_index, int* __restrict__ out_count) {
  __shared__ int warp_tot[32];
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int start = 0; start < n; start += 1024) {
    const int i = start + tid;
    bool ok = false;
    if (i < n) {
      const float4 b = boxes[i];
      ok = (b.z > b.x) && (b.w > b.y);
    }
    const unsigned ball = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) warp_tot[warp] = __popc(ball);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    if (ok) out_index[before + __popc(ball & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (tid == 0) {
      int add = 0;
      for (int w = 0; w < 32; ++w) add += warp_tot[w];
      s_base += add;
    }
    __syncthreads();
  }
  if (tid == 0) *out_count = s_base;
}

// voc_dets.py:37-46: RoIs go to the detector in batches of `group`; the last batch is padded with
// copies of ITS first RoI.  rows < ceil(count/group)*group are real or padding rows, the rest of
// the fixed-size output is the empty box [0,0,0,0] (an empty crop, ignored downstream).
__global__ void __launch_bounds__(256)
pad_rois_kernel(const unsigned long long* __restrict__ rois, const int* __restrict__ count, int n_max, int group,
                int m_out, unsigned long long* __restrict__ out, int* __restrict__ out_rows) {
  const int img = blockIdx.y;
  const int r = blockIdx.x * 256 + threadIdx.x;
  const int n = min(max(count[img], 0), n_max);               // a negative count is an empty list: rows = 0
  const int rows = (n + group - 1) / group * group;
  if (r == 0) out_rows[img] = rows;
  if (r >= m_out) return;
  unsigned long long v = 0ull;
  if (r < n) v = rois[(size_t)img * n_max + r];
  else if (r < rows) v = rois[(size_t)img * n_max + (rows - group)];
  out[(size_t)img * m_out + r] = v;
}

int launch_pad_rois(frcnn_handle* h, cudaStream_t stream, const int16_t* rois, const int32_t* count, int n_max,
                    int group, int m_out, int batch, int16_t* out, int32_t* out_rows) {
  dim3 grid((m_out + 255) / 256, batch);
  pad_rois_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const unsigned long long*>(rois), count, n_max, group,
                                           m_out, reinterpret_cast<unsigned long long*>(out), out_rows);
  FRCNN_LAUNCH_CHECK(h, "pad_rois_kernel");
  return FRCNN_OK;
}

// Mini-batch gather of DetTrainingManager.get_training_input (det_util.py:119-125: rois[sampled_idxs],
// y_class_num[sampled_idxs], y_transform[sampled_idxs]) for a batch of images: one CTA per (sample, image) copies the
// three labelled rows index[img][s] points at; index -1 (image without eligible RoI) writes zero rows.
__global__ void __launch_bounds__(128)
gather_det_samples_kernel(const unsigned long long* __restrict__ rois, const int* __restrict__ y_cls,
                          const float* __restrict__ y_tr, const int* __restrict__ index, int n_max, int k, int t,
                          int n_samples, unsigned long long* __restrict__ out_rois, int* __restrict__ out_cls,
                          float* __restrict__ out_tr) {
  const int s = blockIdx.x, img = blockIdx.y;
  const int src = __ldg(index + (size_t)img * n_samples + s);
  const bool live = src >= 0 && src < n_max;
  const size_t in_row = (size_t)img * n_max + (live ? src : 0), out_row = (size_t)img * n_samples + s;
  if (threadIdx.x == 0) out_rois[out_row] = live ? __ldg(rois + in_row) : 0ull;
  for (int i = threadIdx.x; i < k; i += 128) out_cls[out_row * k + i] = live ? __ldg(y_cls + in_row * k + i) : 0;
  for (int i = threadIdx.x; i < t; i += 128) out_tr[out_row * t + i] = live ? __ldg(y_tr + in_row * t + i) : 0.f;
}

int launch_gather_det_samples(frcnn_handle* h, cudaStream_t stream, const int16_t* rois, const int32_t* y_cls,
                              const float* y_tr, const int32_t* index, int n_max, int k, int t, int n_samples, int batch,
                              int16_t* out_rois, int32_t* out_cls, float* out_tr) {
  dim3 grid(n_samples, batch);
  gather_det_samples_kernel<<<grid, 128, 0, stream>>>(reinterpret_cast<const unsigned long long*>(rois), y_cls, y_tr, index,
                                                     n_max, k, t, n_samples,
                                                     reinterpret_cast<unsigned long long*>(out_rois), out_cls, out_tr);
  FRCNN_LAUNCH_CHECK(h, "gather_det_samples_kernel");
  return FRCNN_OK;
}

int launch_cross_ious(frcnn_handle* h, cudaStream_t stream, const void* boxes, int dtype, int n, const float* gt,
                      int g, float* iou) {
  const size_t total = (size_t)n * g;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (dtype == FRCNN_ROI_I16)
    cross_ious_kernel<true><<<blocks, 256, 0, stream>>>(boxes, n, gt, g, iou);
  else
    cross_ious_kernel<false><<<blocks, 256, 0, stream>>>(boxes, n, gt, g, iou);
  FRCNN_LAUNCH_CHECK(h, "cross_ious_kernel");
  return FRCNN_OK;
}

int launch_box_transform(frcnn_handle* h, cudaStream_t stream, float* boxes, const float* deltas, int n, int decode,
                         int cols, int rows) {
  box_transform_kernel<<<(n + 255) / 256, 256, 0, stream>>>(reinterpret_cast<float4*>(boxes),
                                                           reinterpret_cast<const float4*>(deltas), n, decode, cols, rows);
  FRCNN_LAUNCH_CHECK(h, "box_transform_kernel");
  return FRCNN_OK;
}

int launch_anchor_grid(frcnn_handle* h, cudaStream_t stream, const AnchorTable& tab, int rows, int cols, int stride,
                       int pixel_space, float* out) {
  const int n = rows * cols * tab.n;
  anchor_grid_kernel<<<(n + 255) / 256, 256, 0, stream>>>(tab, rows, cols, stride, pixel_space,
                                                         reinterpret_cast<float4*>(out));
  FRCNN_LAUNCH_CHECK(h, "anchor_grid_kernel");
  return FRCNN_OK;
}

int launch_valid_boxes(frcnn_handle* h, cudaStream_t stream, const float* boxes, int n, int32_t* out_index,
                       int32_t* out_count) {
  valid_boxes_kernel<<<1, 1024, 0, stream>>>(reinterpret_cast<const float4*>(boxes), n, out_index, out_count);
  FRCNN_LAUNCH_CHECK(h, "valid_boxes_kernel");
  return FRCNN_OK;
}

// RoIs of a padded batch clamped to each image's own map: rois [batch][n][4] (int16 / int32 / float32, truncated to int
// like load_crop, roi_common.cuh), extents [batch][2] (rows, cols).  x1, y1 >= 0 and x2 <= cols_b, y2 <= rows_b; the RoI
// layer's own clamp to the padded map (load_crop) then completes the clamp of the extents to that map and leaves the
// crop a call on the image's own map takes, so no kernel reads a padding cell.  out may alias rois.
template <typename T>
__global__ void __launch_bounds__(256)
clip_rois_kernel(const T* rois, int n, const int* __restrict__ extents, T* out) {
  const int img = blockIdx.y, r = blockIdx.x * 256 + threadIdx.x;
  if (r >= n) return;
  const int rows_b = max(extents[2 * img], 0), cols_b = max(extents[2 * img + 1], 0);
  const size_t o = ((size_t)img * n + r) * 4;
  const int x1 = (int)rois[o], y1 = (int)rois[o + 1], x2 = (int)rois[o + 2], y2 = (int)rois[o + 3];
  out[o] = (T)max(x1, 0);
  out[o + 1] = (T)max(y1, 0);
  out[o + 2] = (T)min(x2, cols_b);
  out[o + 3] = (T)min(y2, rows_b);
}

int launch_clip_rois(frcnn_handle* h, cudaStream_t stream, const void* rois, int dtype, int n, int batch,
                     const int32_t* extents, void* out) {
  dim3 grid((n + 255) / 256, batch);
  if (dtype == FRCNN_ROI_I16)
    clip_rois_kernel<short><<<grid, 256, 0, stream>>>(static_cast<const short*>(rois), n, extents,
                                                     static_cast<short*>(out));
  else if (dtype == FRCNN_ROI_I32)
    clip_rois_kernel<int><<<grid, 256, 0, stream>>>(static_cast<const int*>(rois), n, extents,
                                                   static_cast<int*>(out));
  else
    clip_rois_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(rois), n, extents,
                                                     static_cast<float*>(out));
  FRCNN_LAUNCH_CHECK(h, "clip_rois_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
