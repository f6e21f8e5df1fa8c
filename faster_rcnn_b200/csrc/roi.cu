// K-d: RoI layer (custom_layers.py:35-56) forward, channels-last.  The backward is in roi_bwd.cu.
//
// All int<->float conversions and divisions of the layer (they run on the 16-lane XU pipe) happen once per
// (RoI, output index) as "tap records" that the forward CTA builds for its RoI in shared memory in its prologue.
//
// Forward (both modes): one CTA per (RoI, 256-channel block, image); a thread owns four
// consecutive channels (128-bit loads/stores), walks the PxP outputs and streams them out with
// evict-first stores.  The feature map (9.8 MB at 38x63x1024) stays L2-resident, the P*P*C
// outputs (401 MB at N=2000) are the HBM stream.  Values that two consecutive outputs share are
// carried in registers instead of being fetched twice: the interpolated bottom row (or the right
// taps, for crops taller than wide) in resize mode, the boundary row of two bins in max mode.
//
// RESIZE mode = TF-1.3 legacy bilinear (align_corners=False, no half-pixel offset):
//   scale = in/float(out); src = i*scale; lo = (int)src; hi = min(lo+1, in-1); lerp = src-lo
//   top = tl + (tr-tl)*lx; bottom = bl + (br-bl)*lx; out = top + (bottom-top)*ly
// MAX mode: bin rows y1+floor(ph*h/P) .. y1+ceil((ph+1)*h/P)-1, first maximum in row-major scan.
// This TU is compiled with -fmad=false so that a*b+c keeps two roundings like the CPU oracle.
#include "roi_common.cuh"

namespace frcnn {

// a + (b - a) * t with three roundings per element like numpy / TF's CPU kernel.  The subtraction and the product are
// packed; the final addition stays scalar because ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (a
// single rounding) even with -fmad=false, which would break the bit-exact forward.  8 instead of 12 instructions.
__device__ __forceinline__ float4 lerp4(float4 a, float4 b, float t) {
  const unsigned long long tt = pack2(t, t);
  const unsigned long long p0 = mul2(sub2(pack2(b.x, b.y), pack2(a.x, a.y)), tt);
  const unsigned long long p1 = mul2(sub2(pack2(b.z, b.w), pack2(a.z, a.w)), tt);
  float px, py, pz, pw;
  unpack2(p0, px, py);
  unpack2(p1, pz, pw);
  return make_float4(__fadd_rn(a.x, px), __fadd_rn(a.y, py), __fadd_rn(a.z, pz), __fadd_rn(a.w, pw));
}

__device__ __forceinline__ float4 scale4(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }

// one tap record of RoI crop `k` for output index p: the source taps (resize) or bin bounds (max) of both axes in
// ABSOLUTE map coordinates
//   resize: (ylo | yhi << 16, bits(ylerp), xlo | xhi << 16, bits(xlerp))
//   max:    (ya  | yb  << 16, 0,           xa  | xb  << 16, 0)   [a, b) bounds
template <int MODE>
__device__ __forceinline__ int4 make_tap(const Crop& k, int p, int P) {
  if (k.w <= 0 || k.h <= 0) return make_int4(0, 0, 0, 0);
  if (MODE == FRCNN_ROI_RESIZE) {
    const Tap ty = axis_tap(p, (float)k.h / (float)P, k.h), tx = axis_tap(p, (float)k.w / (float)P, k.w);
    return make_int4((k.y1 + ty.lo) | ((k.y1 + ty.hi) << 16), __float_as_int(ty.lerp),
                     (k.x1 + tx.lo) | ((k.x1 + tx.hi) << 16), __float_as_int(tx.lerp));
  }
  const int ya = k.y1 + (p * k.h) / P, yb = k.y1 + ((p + 1) * k.h + P - 1) / P;
  const int xa = k.x1 + (p * k.w) / P, xb = k.x1 + ((p + 1) * k.w + P - 1) / P;
  return make_int4(ya | (yb << 16), 0, xa | (xb << 16), 0);
}

// 64-thread CTAs (256 channels): measured 1-7 % faster than 256-thread CTAs at every batch size (finer-grained CTAs,
// 23 instead of 5 resident per SM at 44 registers -> 46 instead of 40 warps, shorter tail at 2000 RoIs x 1 image).
constexpr int ROI_FWD_THREADS = 64;

// Forward: one CTA per (RoI, 256-channel block, image); a thread owns four consecutive channels.
// COMPACT (max mode only): the arg-max is stored as ONE BYTE per element, (dy << 4) | dx relative to the bin's first
// cell, instead of the int32 flat cell index: 5 instead of 8 bytes per pooled element leave the kernel (and enter the
// backward).  Bins are at most ceil(H/P)+1 cells high / wide; the launcher takes this path only when that is <= 16.
template <int MODE, bool COMPACT = false>
__global__ void __launch_bounds__(ROI_FWD_THREADS)
roi_fwd_kernel(const float* __restrict__ feat, int H, int W, int C, const void* __restrict__ rois, int dtype,
               int N, int P, int ph_groups, float* __restrict__ out, int* __restrict__ argmax) {
  __shared__ int4 s_tap[ROI_MAX_TABLE_P];
  __shared__ int4 s_xoff[ROI_MAX_TABLE_P];
  __shared__ int4 s_crop;
  const int r = blockIdx.x, img = blockIdx.z;
  const size_t roi = (size_t)img * N + r;
  // the CTA's own tap table: P threads do all int<->float conversions / divisions of this RoI once
  if (threadIdx.x <= P && threadIdx.x <= ROI_MAX_TABLE_P) {
    const Crop k = load_crop(rois, dtype, roi, W, H);
    if (threadIdx.x < P) {
      const int4 t = make_tap<MODE>(k, threadIdx.x, P);
      s_tap[threadIdx.x] = t;
      s_xoff[threadIdx.x] = make_int4((t.z & 0xffff) * C * 4, (t.z >> 16) * C * 4, t.w, 0);
    } else {
      s_crop = make_int4(k.x1, k.y1, k.w, k.h);
    }
  }
  __syncthreads();
  // blockIdx.y = channel block * ph_groups + group: small max-mode launches (2000 RoIs of ONE image are 2.7 waves of
  // CTAs) are cut into two row groups per RoI so that the last wave is fuller; everything else uses one group.
  const int cblock = blockIdx.y / ph_groups, grp = blockIdx.y - cblock * ph_groups;
  const int ph0 = grp * P / ph_groups, ph1 = (grp + 1) * P / ph_groups;
  const int c = (cblock * ROI_FWD_THREADS + threadIdx.x) * 4;
  if (c >= C) return;
  const float* f = feat + (size_t)img * H * W * C + c;
  const size_t obase = (roi * P * P) * C + c;
  if (s_crop.z <= 0 || s_crop.w <= 0) {   // TF would raise on an empty crop; we emit zeros
    for (int b = ph0 * P; b < ph1 * P; ++b) {
      st_cs_f4(out + obase + (size_t)b * C, make_float4(0.f, 0.f, 0.f, 0.f));
      if (MODE == FRCNN_ROI_MAX && !COMPACT) st_cs_i4(argmax + obase + (size_t)b * C, make_int4(0, 0, 0, 0));
      if (MODE == FRCNN_ROI_MAX && COMPACT) __stcs(reinterpret_cast<unsigned*>(reinterpret_cast<unsigned char*>(argmax) + obase + (size_t)b * C), 0u);
    }
    return;
  }
  const size_t row_stride = (size_t)W * C;
  const size_t row_bytes = row_stride * 4;
  if (MODE == FRCNN_ROI_RESIZE) {
    // Loop order pw (outer) / ph (inner): the x taps of a column stay in registers (byte offsets from the row pointer;
    // the per-output address arithmetic was 38 of the 80 SASS instructions of the first version, and this kernel
    // runs into the 1000 W power cap in sustained operation, so instructions are energy), and when the source row of
    // this output's top taps is the row of the previous output's bottom taps (crops lower than 2P rows) the already
    // interpolated bottom value is carried over instead of being loaded and interpolated again -- identical
    // arithmetic on identical inputs, so the result is bit for bit the same.
    const char* fb = reinterpret_cast<const char*>(f);
    if (s_crop.w <= s_crop.z) {                     // crop height <= width: more row reuse than column reuse
      for (int pw = 0; pw < P; ++pw) {
        const int4 tx = s_xoff[pw];                 // (byte offset of xlo, of xhi, bits(lx), -), unsigned 32-bit
        const float lx = __int_as_float(tx.z);
        const unsigned bl_off = (unsigned)tx.x, bh_off = (unsigned)tx.y;
        float* o = out + obase + ((size_t)ph0 * P + pw) * C;
        float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
        int carry_row = -1;
        for (int ph = ph0; ph < ph1; ++ph, o += (size_t)P * C) {
          const int4 ty = s_tap[ph];
          const int ylo = ty.x & 0xffff, yhi = ty.x >> 16;
          const char* row_hi = fb + (size_t)yhi * row_bytes;
          float4 top;
          if (ylo == carry_row) {                   // warp-uniform
            top = carry;
          } else {
            const char* row_lo = fb + (size_t)ylo * row_bytes;
            top = lerp4(ldg_f4(reinterpret_cast<const float*>(row_lo + bl_off)),
                        ldg_f4(reinterpret_cast<const float*>(row_lo + bh_off)), lx);
          }
          const float4 bot = lerp4(ldg_f4(reinterpret_cast<const float*>(row_hi + bl_off)),
                                   ldg_f4(reinterpret_cast<const float*>(row_hi + bh_off)), lx);
          st_cs_f4(o, lerp4(top, bot, __int_as_float(ty.y)));
          carry = bot;
          carry_row = yhi;
        }
      }
    } else {                                        // taller than wide: ph outer, the right taps become the next left taps
      for (int ph = ph0; ph < ph1; ++ph) {
        const int4 ty = s_tap[ph];
        const char* row_lo = fb + (size_t)(ty.x & 0xffff) * row_bytes;
        const char* row_hi = fb + (size_t)(ty.x >> 16) * row_bytes;
        const float ly = __int_as_float(ty.y);
        float* o = out + obase + (size_t)ph * P * C;
        float4 ctop = make_float4(0.f, 0.f, 0.f, 0.f), cbot = ctop;
        unsigned carry_off = 0xffffffffu;
        for (int pw = 0; pw < P; ++pw, o += C) {
          const int4 tx = s_xoff[pw];
          const float lx = __int_as_float(tx.z);
          const unsigned bl_off = (unsigned)tx.x, bh_off = (unsigned)tx.y;
          float4 tl, bl;
          if (bl_off == carry_off) {                // warp-uniform
            tl = ctop;
            bl = cbot;
          } else {
            tl = ldg_f4(reinterpret_cast<const float*>(row_lo + bl_off));
            bl = ldg_f4(reinterpret_cast<const float*>(row_hi + bl_off));
          }
          const float4 tr = ldg_f4(reinterpret_cast<const float*>(row_lo + bh_off));
          const float4 br = ldg_f4(reinterpret_cast<const float*>(row_hi + bh_off));
          st_cs_f4(o, lerp4(lerp4(tl, tr, lx), lerp4(bl, br, lx), ly));
          ctop = tr;
          cbot = br;
          carry_off = bh_off;
        }
      }
    }
  } else {
    // MAX mode.  For one column of bins (pw) the thread walks the crop's rows ONCE, top to bottom: every row segment
    // [xa, xb) is reduced to its first maximum (a row tracker), merged into the bin that is open (strict '>' keeps the
    // earlier row on ties = first maximum in row-major order), and when a bin ends on this row it is stored and the
    // next bin -- which starts on the same row whenever (ph+1)*h is not a multiple of P, or repeats it when h < P --
    // is seeded from the same row tracker.  The row scan is specialised on the segment width (1..4 cells cover every
    // RoI up to 21 cells wide), so the loads of a segment are issued together and there is no inner loop: the first
    // version of this branch spent 52 instructions per visited cell, 40 of them loop set-up and address arithmetic
    // for segments of two or three cells (ncu: IMAD 35 %, LDG 1.9 % of the instruction mix).
    const char* fb = reinterpret_cast<const char*>(f);
    const unsigned cell_bytes = (unsigned)C * 4u;
    const int y_begin = s_tap[ph0].x & 0xffff;
    for (int pw = 0; pw < P; ++pw) {
      const int xa = s_tap[pw].z & 0xffff, bw = (s_tap[pw].z >> 16) - xa;
      const char* rowp = fb + ((size_t)y_begin * W + xa) * cell_bytes;
      int cell0 = y_begin * W + xa;
      int ph = ph0;
      int yb = s_tap[ph].x >> 16;
      float* o = out + obase + (size_t)(ph0 * P + pw) * C;
      int* oa = argmax + obase + (size_t)(ph0 * P + pw) * C;
      unsigned char* oc = reinterpret_cast<unsigned char*>(argmax) + obase + (size_t)(ph0 * P + pw) * C;   // COMPACT
      float4 best = make_float4(0.f, 0.f, 0.f, 0.f);
      int4 arg = make_int4(0, 0, 0, 0);
      bool open = false;
      int ya_open = y_begin;                          // first row of the open bin (COMPACT: dy is relative to it)
      for (int y = y_begin; ph < ph1; ++y, rowp += row_bytes, cell0 += W) {
        float4 rb;
        int4 ra;
        if (!open) ya_open = y;
        const int code0 = COMPACT ? ((y - ya_open) << 4) : cell0;      // arg value of the segment's first cell
#define FRCNN_ROW_STEP(J)                                                                    \
  {                                                                                          \
    const int cj_ = code0 + (J);                                                             \
    if (v_[J].x > rb.x) { rb.x = v_[J].x; ra.x = cj_; }                                      \
    if (v_[J].y > rb.y) { rb.y = v_[J].y; ra.y = cj_; }                                      \
    if (v_[J].z > rb.z) { rb.z = v_[J].z; ra.z = cj_; }                                      \
    if (v_[J].w > rb.w) { rb.w = v_[J].w; ra.w = cj_; }                                      \
  }
#define FRCNN_ROW_SCAN(BW)                                                                   \
  {                                                                                          \
    float4 v_[BW];                                                                           \
    _Pragma("unroll") for (int j = 0; j < BW; ++j)                                           \
      v_[j] = ldg_f4(reinterpret_cast<const float*>(rowp + j * cell_bytes));                 \
    rb = v_[0];                                                                              \
    ra = make_int4(code0, code0, code0, code0);                                              \
    _Pragma("unroll") for (int j = 1; j < BW; ++j) FRCNN_ROW_STEP(j)                         \
  }
        if (bw == 2) FRCNN_ROW_SCAN(2)
        else if (bw == 3) FRCNN_ROW_SCAN(3)
        else if (bw == 1) FRCNN_ROW_SCAN(1)
        else if (bw == 4) FRCNN_ROW_SCAN(4)
        else {                                        // wide segments: four cells at a time
          FRCNN_ROW_SCAN(4)
          for (int x = 4; x < bw; ++x) {
            const float4 v1 = ldg_f4(reinterpret_cast<const float*>(rowp + x * cell_bytes));
            const int cj_ = code0 + x;
            if (v1.x > rb.x) { rb.x = v1.x; ra.x = cj_; }
            if (v1.y > rb.y) { rb.y = v1.y; ra.y = cj_; }
            if (v1.z > rb.z) { rb.z = v1.z; ra.z = cj_; }
            if (v1.w > rb.w) { rb.w = v1.w; ra.w = cj_; }
          }
        }
#undef FRCNN_ROW_SCAN
#undef FRCNN_ROW_STEP
        if (!open) {                                  // warp-uniform
          best = rb;
          arg = ra;
          open = true;
        } else {
          if (rb.x > best.x) { best.x = rb.x; arg.x = ra.x; }
          if (rb.y > best.y) { best.y = rb.y; arg.y = ra.y; }
          if (rb.z > best.z) { best.z = rb.z; arg.z = ra.z; }
          if (rb.w > best.w) { best.w = rb.w; arg.w = ra.w; }
        }
        while (y == yb - 1) {                         // the open bin ends on this row
          st_cs_f4(o, best);
          if (COMPACT) {
            __stcs(reinterpret_cast<unsigned*>(oc), (unsigned)arg.x | ((unsigned)arg.y << 8) | ((unsigned)arg.z << 16) | ((unsigned)arg.w << 24));
          } else {
            st_cs_i4(oa, arg);
          }
          o += (size_t)P * C;
          oa += (size_t)P * C;
          oc += (size_t)P * C;
          if (++ph == ph1) break;
          const int t = s_tap[ph].x;
          yb = t >> 16;
          if ((t & 0xffff) <= y) {                    // the next bin starts on (or repeats) this row
            best = rb;
            arg = COMPACT ? make_int4(ra.x & 15, ra.y & 15, ra.z & 15, ra.w & 15) : ra;      // dy = 0 in the new bin
            ya_open = y;
          } else {
            open = false;
            break;
          }
        }
      }
    }
  }
}

// scalar-channel fallback for C % 4 != 0 (not a performance path)
template <int MODE>
__global__ void roi_fwd_scalar_kernel(const float* __restrict__ feat, int H, int W, int C,
                                      const void* __restrict__ rois, int dtype, int N, int P,
                                      float* __restrict__ out, int* __restrict__ argmax) {
  const int r = blockIdx.x, img = blockIdx.z;
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const Crop k = load_crop(rois, dtype, (size_t)img * N + r, W, H);
  const float* f = feat + (size_t)img * H * W * C + c;
  const size_t obase = (((size_t)img * N + r) * P * P) * C + c;
  if (k.w <= 0 || k.h <= 0) {
    for (int b = 0; b < P * P; ++b) { out[obase + (size_t)b * C] = 0.f; if (MODE == FRCNN_ROI_MAX) argmax[obase + (size_t)b * C] = 0; }
    return;
  }
  const float ys = (float)k.h / (float)P, xs = (float)k.w / (float)P;
  for (int ph = 0; ph < P; ++ph) {
    for (int pw = 0; pw < P; ++pw) {
      const size_t o = obase + (size_t)(ph * P + pw) * C;
      if (MODE == FRCNN_ROI_RESIZE) {
        const Tap ty = axis_tap(ph, ys, k.h), tx = axis_tap(pw, xs, k.w);
        const float tl = f[((size_t)(k.y1 + ty.lo) * W + k.x1 + tx.lo) * C], tr = f[((size_t)(k.y1 + ty.lo) * W + k.x1 + tx.hi) * C];
        const float bl = f[((size_t)(k.y1 + ty.hi) * W + k.x1 + tx.lo) * C], br = f[((size_t)(k.y1 + ty.hi) * W + k.x1 + tx.hi) * C];
        const float top = tl + (tr - tl) * tx.lerp, bot = bl + (br - bl) * tx.lerp;
        out[o] = top + (bot - top) * ty.lerp;
      } else {
        const int ya = k.y1 + (ph * k.h) / P, yb = k.y1 + ((ph + 1) * k.h + P - 1) / P;
        const int xa = k.x1 + (pw * k.w) / P, xb = k.x1 + ((pw + 1) * k.w + P - 1) / P;
        float best = f[((size_t)ya * W + xa) * C];
        int arg = ya * W + xa;
        for (int y = ya; y < yb; ++y)
          for (int x = xa; x < xb; ++x) {
            const float v = f[((size_t)y * W + x) * C];
            if (v > best) { best = v; arg = y * W + x; }
          }
        out[o] = best;
        argmax[o] = arg;
      }
    }
  }
}

// true when the one-byte arg-max format can describe every bin of an H x W map pooled to P x P
bool roi_compact_supported(int H, int W, int C, int P) {
  return C % 4 == 0 && P >= 1 && P <= ROI_MAX_TABLE_P && (H + P - 1) / P + 1 <= 16 && (W + P - 1) / P + 1 <= 16;
}

int launch_roi_fwd(frcnn_handle* h, cudaStream_t stream, int mode, const float* feat, int H, int W, int C,
                   const void* rois, int dtype, int N, int P, int batch, float* out, int32_t* argmax, int compact) {
  if (compact && (mode != FRCNN_ROI_MAX || !roi_compact_supported(H, W, C, P) || (reinterpret_cast<uintptr_t>(argmax) & 3)))
    return fail(h, FRCNN_ERR_UNSUPPORTED, "roi_fwd: compact arg-max needs max mode, C %% 4 == 0 and bins of at most 16 x 16 cells%s%s");
  if (C % 4 == 0 && P <= ROI_MAX_TABLE_P && H < 32768 && W < 32768 && (long long)W * C < (1LL << 29) &&
      (reinterpret_cast<uintptr_t>(feat) % 16 == 0) &&
      (reinterpret_cast<uintptr_t>(out) % 16 == 0) &&
      (mode != FRCNN_ROI_MAX || compact || reinterpret_cast<uintptr_t>(argmax) % 16 == 0)) {
    const int cblocks = (C / 4 + ROI_FWD_THREADS - 1) / ROI_FWD_THREADS;
    // max mode, fewer than 8 waves of CTAs (20 resident per SM): split every RoI into two row groups (same-box A/B at
    // 2000 RoIs x 1 image: 0.252 ms with one group, 0.236 with two or three, 0.265 with P groups -- more groups break
    // the boundary-row carry-over; resize mode got slower with any split and keeps one)
    const long long ctas = (long long)N * cblocks * batch;
    const int ph_groups = (mode == FRCNN_ROI_MAX && P >= 2 && ctas < 8LL * 20 * h->sm_count) ? 2 : 1;
    dim3 grid(N, cblocks * ph_groups, batch);
    if (mode == FRCNN_ROI_RESIZE)
      roi_fwd_kernel<FRCNN_ROI_RESIZE><<<grid, ROI_FWD_THREADS, 0, stream>>>(feat, H, W, C, rois, dtype, N, P, ph_groups, out, argmax);
    else if (compact)
      roi_fwd_kernel<FRCNN_ROI_MAX, true><<<grid, ROI_FWD_THREADS, 0, stream>>>(feat, H, W, C, rois, dtype, N, P, ph_groups, out, argmax);
    else
      roi_fwd_kernel<FRCNN_ROI_MAX><<<grid, ROI_FWD_THREADS, 0, stream>>>(feat, H, W, C, rois, dtype, N, P, ph_groups, out, argmax);
  } else {
    if (compact) return fail(h, FRCNN_ERR_UNSUPPORTED, "roi_fwd: compact arg-max needs 16-byte aligned buffers%s%s");
    dim3 grid(N, (C + 127) / 128, batch);
    if (mode == FRCNN_ROI_RESIZE)
      roi_fwd_scalar_kernel<FRCNN_ROI_RESIZE><<<grid, 128, 0, stream>>>(feat, H, W, C, rois, dtype, N, P, out, argmax);
    else
      roi_fwd_scalar_kernel<FRCNN_ROI_MAX><<<grid, 128, 0, stream>>>(feat, H, W, C, rois, dtype, N, P, out, argmax);
  }
  FRCNN_LAUNCH_CHECK(h, "roi_fwd_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
