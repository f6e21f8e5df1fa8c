// Shared device helpers of the RoI layer kernels (roi.cu forward, roi_bwd.cu backward).
#pragma once
#include "common.cuh"

namespace frcnn {

// largest pool size of the vectorised kernels: the forward's per-CTA tap table and the backward's 32-bit masks
constexpr int ROI_MAX_TABLE_P = 32;

// true when the one-byte arg-max format can describe every bin of an H x W map pooled to P x P (roi.cu)
bool roi_compact_supported(int H, int W, int C, int P);

struct Crop { int x1, y1, w, h; };   // clipped to the map; w,h <= 0 means empty

__device__ __forceinline__ Crop load_crop(const void* rois, int dtype, size_t idx, int W, int H) {
  int x1, y1, x2, y2;
  if (dtype == FRCNN_ROI_I16) {
    const short* p = reinterpret_cast<const short*>(rois) + idx * 4;
    x1 = p[0]; y1 = p[1]; x2 = p[2]; y2 = p[3];
  } else if (dtype == FRCNN_ROI_I32) {
    const int* p = reinterpret_cast<const int*>(rois) + idx * 4;
    x1 = p[0]; y1 = p[1]; x2 = p[2]; y2 = p[3];
  } else {
    const float* p = reinterpret_cast<const float*>(rois) + idx * 4;
    x1 = (int)p[0]; y1 = (int)p[1]; x2 = (int)p[2]; y2 = (int)p[3];   // K.cast(.., 'int32') truncates
  }
  x1 = max(x1, 0); y1 = max(y1, 0); x2 = min(x2, W); y2 = min(y2, H);
  return Crop{x1, y1, x2 - x1, y2 - y1};
}

struct Tap { int lo, hi; float lerp; };
__device__ __forceinline__ Tap axis_tap(int i, float scale, int in_size) {
  const float src = (float)i * scale;
  Tap t;
  t.lo = (int)src;
  t.hi = min(t.lo + 1, in_size - 1);
  t.lerp = src - (float)t.lo;
  return t;
}

// Blackwell packed fp32 (add/mul/fma.rn.f32x2 -> FADD2 / FMUL2 / FFMA2): two IEEE-rounded float32 results per
// instruction on an aligned register pair, i.e. half the issue slots for the same arithmetic.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long sub2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

}  // namespace frcnn
