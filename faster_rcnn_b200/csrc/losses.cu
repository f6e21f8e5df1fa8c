// Masked RPN / detector losses fused with the hot path's own targets (SURVEY.md 8f-2).
//
// Replaces loss_functions.py:15-76 (Keras-backend expressions on TF 1.3).  The RPN kernel reads the
// UNPACKED labels (can_use, is_pos, bbreg -- what label_anchors / apply_sampling leave on the device), so the
// Keras y_true layouts never have to be materialised; the detector kernel reads y_class_num / y_transform as
// label_rois emits them.  Each kernel returns the scalar Keras reports for the output (mean of the loss
// tensor) and, optionally, its gradient with respect to the prediction.
//
//   binary_crossentropy (Keras 2.0.8, TF backend): p = clip(p, 1e-7, 1-1e-7); x = log(p/(1-p));
//       bce = max(x,0) - x*z + log1p(exp(-|x|))
//   smooth-L1: 0.5*d^2 if |d| <= 1 else |d| - 0.5
//   categorical_crossentropy: p /= sum(p); p = clip(p, 1e-7, 1-1e-7); -sum(t*log(p))
// Quirk kept (loss_functions.py:40-46): the RPN box loss applies its mask OUTSIDE the sum:
//       loss tensor = mask * (10 * S_all / 2400), reported value = mean(mask) * 10 * S_all / 2400.
//
// One CTA per image; element math in float32, reductions in float64 with a fixed tree (deterministic).
#include "common.cuh"

namespace frcnn {

constexpr int LOSS_THREADS = 1024;    // one CTA per image: its warps have to hide the log / exp chains themselves

// deterministic block sum of `K` doubles per thread; result valid in every thread
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double* scratch /* [K][LOSS_THREADS/32] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], d);
    if (lane == 0) scratch[k * (LOSS_THREADS / 32) + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double s = 0.0;
    for (int w = 0; w < LOSS_THREADS / 32; ++w) s += scratch[k * (LOSS_THREADS / 32) + w];
    v[k] = s;
  }
  __syncthreads();
}

__device__ __forceinline__ float smooth_l1(float d) {
  const float a = fabsf(d);
  return a <= 1.0f ? 0.5f * a * a : a - 0.5f;
}
__device__ __forceinline__ float smooth_l1_grad(float d) { return fabsf(d) <= 1.0f ? d : (d > 0.f ? 1.0f : -1.0f); }

// can_use / is_pos [B,N] u8, bbreg [B,N,4] f32, cls_pred [B,N] f32, reg_pred [B,N,4] f32
// loss [B,2] = (cls_loss_rpn, bbreg_loss_rpn); grad_cls [B,N], grad_reg [B,N,4] optional
__global__ void __launch_bounds__(LOSS_THREADS)
rpn_losses_kernel(const unsigned char* __restrict__ can_use, const unsigned char* __restrict__ is_pos,
                  const float4* __restrict__ bbreg, const float* __restrict__ cls_pred,
                  const float4* __restrict__ reg_pred, int n, float* __restrict__ loss,
                  float* __restrict__ grad_cls, float4* __restrict__ grad_reg) {
  __shared__ double scratch[3 * (LOSS_THREADS / 32)];
  const int img = blockIdx.x, tid = threadIdx.x;
  const size_t base = (size_t)img * n;
  const float eps = 1e-7f, one_m_eps = 1.0f - 1e-7f;
  double acc[3] = {0.0, 0.0, 0.0};                 // sum sel*bce, sum smooth-L1 over ALL anchors, #(pos & use)
  for (int i = tid; i < n; i += LOSS_THREADS) {
    const bool use = can_use[base + i] != 0, pos = is_pos[base + i] != 0;
    const float p_raw = cls_pred[base + i];
    const float p = fminf(fmaxf(p_raw, eps), one_m_eps);
    const float x = logf(p / (1.0f - p));
    const float z = pos ? 1.0f : 0.0f;
    const float bce = fmaxf(x, 0.0f) - x * z + log1pf(expf(-fabsf(x)));
    if (use) acc[0] += (double)bce;
    const float4 t = bbreg[base + i], q = reg_pred[base + i];
    acc[1] += (double)smooth_l1(t.x - q.x) + (double)smooth_l1(t.y - q.y) + (double)smooth_l1(t.z - q.z) +
              (double)smooth_l1(t.w - q.w);
    if (use && pos) acc[2] += 1.0;
    if (grad_cls) {
      const bool inside = p_raw >= eps && p_raw <= one_m_eps;          // clip_by_value passes the gradient inside only
      grad_cls[base + i] = (use && inside) ? (p - z) / (p * (1.0f - p)) / 256.0f : 0.0f;
    }
  }
  block_sum<3>(acc, scratch);
  const float mean_sel = (float)(acc[2] / (double)n);                 // mean of repeat(is_pos & can_use, 4)
  if (tid == 0) {
    loss[2 * img + 0] = (float)acc[0] / 256.0f;
    loss[2 * img + 1] = mean_sel * (10.0f * (float)acc[1] / 2400.0f);
  }
  if (grad_reg) {
    const float scale = mean_sel * (10.0f / 2400.0f);
    for (int i = tid; i < n; i += LOSS_THREADS) {
      const float4 t = bbreg[base + i], q = reg_pred[base + i];
      grad_reg[base + i] = make_float4(-scale * smooth_l1_grad(t.x - q.x), -scale * smooth_l1_grad(t.y - q.y),
                                       -scale * smooth_l1_grad(t.z - q.z), -scale * smooth_l1_grad(t.w - q.w));
    }
  }
}

// The same losses on a padded batch: inputs [B, rows*cols*A] with image b's own map (rows_b, cols_b) = extents[b]
// (clamped to the padded map).  Threads walk the image's OWN flat index i = ((y*cols_b + x)*A + a) with the thread
// mapping of rpn_losses_kernel, so every partial sum, the reduction and mean_sel = #sel / n_b are those of the call on
// the cropped inputs: loss[b] and both gradients equal it bit for bit.  Padding is never read; its gradients are zero.
// An empty extent gives loss (0, 0) and zero gradients.  One CTA per SM, as rpn_losses_kernel: left free, ptxas aims at
// two and spills at 32 registers.
__global__ void __launch_bounds__(LOSS_THREADS, 1)
rpn_losses_ragged_kernel(const unsigned char* __restrict__ can_use, const unsigned char* __restrict__ is_pos,
                         const float4* __restrict__ bbreg, const float* __restrict__ cls_pred,
                         const float4* __restrict__ reg_pred, int rows, int cols, int n_anchors,
                         const int* __restrict__ extents, float* __restrict__ loss, float* __restrict__ grad_cls,
                         float4* __restrict__ grad_reg) {
  __shared__ double scratch[3 * (LOSS_THREADS / 32)];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int rows_b = min(max(extents[2 * img], 0), rows), cols_b = min(max(extents[2 * img + 1], 0), cols);
  const int n = rows * cols * n_anchors, n_b = rows_b * cols_b * n_anchors, row_b = cols_b * n_anchors;
  const int row = cols * n_anchors;
  const size_t base = (size_t)img * n;
  const float eps = 1e-7f, one_m_eps = 1.0f - 1e-7f;
  double acc[3] = {0.0, 0.0, 0.0};
  for (int i = tid; i < n_b; i += LOSS_THREADS) {
    const int y = i / row_b;
    const size_t j = base + (size_t)y * row + (i - y * row_b);      // the same cell and anchor in the padded layout
    const bool use = can_use[j] != 0, pos = is_pos[j] != 0;
    const float p = fminf(fmaxf(cls_pred[j], eps), one_m_eps);
    const float x = logf(p / (1.0f - p));
    const float z = pos ? 1.0f : 0.0f;
    const float bce = fmaxf(x, 0.0f) - x * z + log1pf(expf(-fabsf(x)));
    if (use) acc[0] += (double)bce;
    const float4 t = bbreg[j], q = reg_pred[j];
    acc[1] += (double)smooth_l1(t.x - q.x) + (double)smooth_l1(t.y - q.y) + (double)smooth_l1(t.z - q.z) +
              (double)smooth_l1(t.w - q.w);
    if (use && pos) acc[2] += 1.0;
  }
  block_sum<3>(acc, scratch);
  const float mean_sel = n_b > 0 ? (float)(acc[2] / (double)n_b) : 0.0f;
  if (tid == 0) {
    loss[2 * img + 0] = (float)acc[0] / 256.0f;
    loss[2 * img + 1] = mean_sel * (10.0f * (float)acc[1] / 2400.0f);
  }
  if (!grad_cls && !grad_reg) return;
  const float scale = mean_sel * (10.0f / 2400.0f);
  for (int j = tid; j < n; j += LOSS_THREADS) {                     // padded index: every output element once
    const int y = j / row, k = j - y * row;
    const size_t e = base + j;
    if (y >= rows_b || k >= row_b) {
      if (grad_cls) grad_cls[e] = 0.0f;
      if (grad_reg) grad_reg[e] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      continue;
    }
    if (grad_cls) {
      const bool use = can_use[e] != 0, pos = is_pos[e] != 0;
      const float p_raw = cls_pred[e];
      const float p = fminf(fmaxf(p_raw, eps), one_m_eps);
      const float z = pos ? 1.0f : 0.0f;
      const bool inside = p_raw >= eps && p_raw <= one_m_eps;
      grad_cls[e] = (use && inside) ? (p - z) / (p * (1.0f - p)) / 256.0f : 0.0f;
    }
    if (grad_reg) {
      const float4 t = bbreg[e], q = reg_pred[e];
      grad_reg[e] = make_float4(-scale * smooth_l1_grad(t.x - q.x), -scale * smooth_l1_grad(t.y - q.y),
                                -scale * smooth_l1_grad(t.z - q.z), -scale * smooth_l1_grad(t.w - q.w));
    }
  }
}

// y_class [B,M,K] i32 one-hot, y_transform [B,M,8Kf] f32 = [labels | targets], cls_pred [B,M,K], reg_pred [B,M,4Kf]
// loss [B,2] = (cls_loss_det, bbreg_loss_det); grads optional
__global__ void __launch_bounds__(LOSS_THREADS)
det_losses_kernel(const int* __restrict__ y_class, const float* __restrict__ y_transform,
                  const float* __restrict__ cls_pred, const float* __restrict__ reg_pred, int m, int k,
                  float* __restrict__ loss, float* __restrict__ grad_cls, float* __restrict__ grad_reg) {
  __shared__ double scratch[3 * (LOSS_THREADS / 32)];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int kf4 = 4 * (k - 1);
  const int* yc = y_class + (size_t)img * m * k;
  const float* yt = y_transform + (size_t)img * m * 2 * kf4;
  const float* pc = cls_pred + (size_t)img * m * k;
  const float* pr = reg_pred + (size_t)img * m * kf4;
  const float eps = 1e-7f, one_m_eps = 1.0f - 1e-7f;
  double acc[3] = {0.0, 0.0, 0.0};                 // sum mask*sl1, sum (1e-4 + mask), sum of per-row cross entropies
  for (int e = tid; e < m * kf4; e += LOSS_THREADS) {
    const int r = e / kf4, c = e - r * kf4;
    const float mask = yt[(size_t)r * 2 * kf4 + c];
    const float x = yt[(size_t)r * 2 * kf4 + kf4 + c] - pr[e];
    acc[0] += (double)(mask * smooth_l1(x));
    acc[1] += (double)(1e-4f + mask);
  }
  for (int r = tid; r < m; r += LOSS_THREADS) {    // one thread per row: K is small (21)
    float s = 0.0f;
    for (int c = 0; c < k; ++c) s += pc[(size_t)r * k + c];
    float ce = 0.0f, tsum_in = 0.0f;
    for (int c = 0; c < k; ++c) {
      const float t = (float)yc[(size_t)r * k + c];
      const float y_raw = pc[(size_t)r * k + c] / s;
      const float y = fminf(fmaxf(y_raw, eps), one_m_eps);
      ce -= t * logf(y);
      if (y_raw >= eps && y_raw <= one_m_eps) tsum_in += t;
    }
    acc[2] += (double)ce;
    if (grad_cls) {
      for (int c = 0; c < k; ++c) {
        const float t = (float)yc[(size_t)r * k + c];
        const float p = pc[(size_t)r * k + c];
        const float y_raw = p / s;
        const bool inside = y_raw >= eps && y_raw <= one_m_eps;
        grad_cls[(size_t)img * m * k + (size_t)r * k + c] = ((inside ? -t / p : 0.0f) + tsum_in / s) / (float)m;
      }
    }
  }
  block_sum<3>(acc, scratch);
  const float den = (float)acc[1];                 // K.sum(1e-4 + mask)
  if (tid == 0) {
    loss[2 * img + 0] = (float)(acc[2] / (double)m);
    loss[2 * img + 1] = (float)acc[0] / den;
  }
  if (grad_reg) {
    for (int e = tid; e < m * kf4; e += LOSS_THREADS) {
      const int r = e / kf4, c = e - r * kf4;
      const float mask = yt[(size_t)r * 2 * kf4 + c];
      const float x = yt[(size_t)r * 2 * kf4 + kf4 + c] - pr[e];
      grad_reg[(size_t)img * m * kf4 + e] = -mask * smooth_l1_grad(x) / den;
    }
  }
}

int launch_rpn_losses(frcnn_handle* h, cudaStream_t stream, const uint8_t* can_use, const uint8_t* is_pos,
                      const float* bbreg, const float* cls_pred, const float* reg_pred, int n, int batch, float* loss,
                      float* grad_cls, float* grad_reg) {
  rpn_losses_kernel<<<batch, LOSS_THREADS, 0, stream>>>(can_use, is_pos, reinterpret_cast<const float4*>(bbreg), cls_pred,
                                                       reinterpret_cast<const float4*>(reg_pred), n, loss, grad_cls,
                                                       reinterpret_cast<float4*>(grad_reg));
  FRCNN_LAUNCH_CHECK(h, "rpn_losses_kernel");
  return FRCNN_OK;
}

int launch_rpn_losses_ragged(frcnn_handle* h, cudaStream_t stream, const uint8_t* can_use, const uint8_t* is_pos,
                             const float* bbreg, const float* cls_pred, const float* reg_pred, int rows, int cols,
                             int n_anchors, int batch, const int32_t* extents, float* loss, float* grad_cls,
                             float* grad_reg) {
  rpn_losses_ragged_kernel<<<batch, LOSS_THREADS, 0, stream>>>(
      can_use, is_pos, reinterpret_cast<const float4*>(bbreg), cls_pred, reinterpret_cast<const float4*>(reg_pred), rows,
      cols, n_anchors, extents, loss, grad_cls, reinterpret_cast<float4*>(grad_reg));
  FRCNN_LAUNCH_CHECK(h, "rpn_losses_ragged_kernel");
  return FRCNN_OK;
}

int launch_det_losses(frcnn_handle* h, cudaStream_t stream, const int32_t* y_class, const float* y_transform,
                      const float* cls_pred, const float* reg_pred, int m, int k, int batch, float* loss, float* grad_cls,
                      float* grad_reg) {
  det_losses_kernel<<<batch, LOSS_THREADS, 0, stream>>>(y_class, y_transform, cls_pred, reg_pred, m, k, loss, grad_cls,
                                                       grad_reg);
  FRCNN_LAUNCH_CHECK(h, "det_losses_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
