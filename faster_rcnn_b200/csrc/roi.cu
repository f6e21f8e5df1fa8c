// K-d: RoI layer (custom_layers.py:35-56) forward and backward, channels-last.
//
// All int<->float conversions and divisions of the layer (they run on the 16-lane XU pipe) happen once per
// (RoI, output index) as "tap records": the forward CTA builds its RoI's records in shared memory in its
// prologue, the backward launches a tiny pre-kernel that writes them for all RoIs (every cell needs them).
//
// Forward (both modes): one CTA per (RoI, 256-channel block, image); a thread owns four
// consecutive channels (128-bit loads/stores), walks the PxP outputs and streams them out with
// evict-first stores.  The feature map (9.8 MB at 38x63x1024) stays L2-resident, the P*P*C
// outputs (401 MB at N=2000) are the HBM stream.  Values that two consecutive outputs share are
// carried in registers instead of being fetched twice: the interpolated bottom row (or the right
// taps, for crops taller than wide) in resize mode, the boundary row of two bins in max mode.
//
// Backward (both modes): cell-stationary gather, one warp per dX cell accumulating in registers
// (four warps per cell, each a quarter of the RoIs, for small resize-mode launches).
// Both walk RoIs in index order and, inside a RoI, bins in (ph, pw, tap) order, so every addition
// into a given dX element happens in one fixed order: no atomics, bit-reproducible run to run.
// (oracle/roi_oracle.py sums each RoI into a private crop first, like TF's slice-gradient +
// AddN, so resize-mode gradients agree to float32 round-off, not bit for bit; max mode is exact.)
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

// ---------------------------------------------------------------------------------------
// per-launch RoI tables (tiny pre-kernel): the crop of every RoI and, per output index p, the
// source taps (resize) or bin bounds (max) of both axes in ABSOLUTE map coordinates.  All integer
// <-> float conversions and divisions of the layer happen here, once per (RoI, p), instead of
// once per (RoI, p, channel block) in the streaming kernels (they run on the 16-lane XU pipe).
//   crops[roi]      = (x1, y1, w, h)
//   taps[roi*P + p] = resize: (ylo | yhi << 16, bits(ylerp), xlo | xhi << 16, bits(xlerp))
//                     max:    (ya  | yb  << 16, 0,           xa  | xb  << 16, 0)   [a, b) bounds
// ---------------------------------------------------------------------------------------
// one tap record of RoI crop `k` for output index p (see the table layout above)
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

template <int MODE>
__global__ void __launch_bounds__(256)
roi_table_kernel(const void* __restrict__ rois, int dtype, int n_total, int W, int H, int P,
                 int4* __restrict__ crops, int4* __restrict__ taps) {
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (idx >= n_total * (P + 1)) return;
  const int roi = idx / (P + 1), p = idx - roi * (P + 1);
  const Crop k = load_crop(rois, dtype, (size_t)roi, W, H);
  if (p == P) {
    crops[roi] = make_int4(k.x1, k.y1, k.w, k.h);
    return;
  }
  taps[(size_t)roi * P + p] = make_tap<MODE>(k, p, P);
}

// 64-thread CTAs (256 channels): measured 1-7 % faster than 256-thread CTAs at every batch size (finer-grained CTAs,
// 23 instead of 5 resident per SM at 44 registers -> 46 instead of 40 warps, shorter tail at 2000 RoIs x 1 image).
constexpr int ROI_FWD_THREADS = 64;
constexpr int ROI_MAX_TABLE_P = 32;     // table-driven kernels support pool sizes up to 32

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

// ---------------------------------------------------------------------------------------
// backward, resize mode: cell-stationary gather, one warp per dX cell
//
// A warp owns one feature-map cell (y, x) for up to 1024 channels (lane l holds float4 channel
// blocks l, l+32, ...) and accumulates in registers -- no shared memory, no atomics, one store.
// It walks the RoIs 32 at a time (lane <-> RoI containment test, ballot), and for every RoI whose
// crop contains the cell the lanes compute the P y-taps and P x-taps in parallel (lane <-> tap
// index); two ballots give the bins whose taps land on this cell.  Each matching (ph, pw) bin is
// one coalesced dY row read (512 B per channel block) scaled by (g*wy)*wx.  Contributions are
// added in ascending (roi, ph, pw, TL/TR/BL/BR) order, so the result is bit-reproducible.
// dY rows are shared by the <= 4 neighbouring cells they touch; neighbouring cells sit in the
// same CTA (x direction) or the same wave (y direction), so the re-reads hit L1 / L2, not DRAM.
// ---------------------------------------------------------------------------------------
// 4-warp CTAs: a CTA slot is only recycled when its slowest warp is done (cells differ in the number of RoIs that
// cover them), and with 8 warps per CTA only 18 of the 24 resident warp slots were busy (ncu); 4 and 2 warps per CTA
// both measured 1.06 ms against 1.13-1.20 ms (resize), 2.47 against 2.62-2.69 ms (max) at C1 x 64 images.
constexpr int CW_WARPS = 4;
// Measured and rejected (profiles/): queueing the contributions per warp in shared memory and streaming
// them with a two-deep software pipeline (2.1 ms vs 1.34 ms at C1 x 64 images): separating the integer
// "collect" phase from the load phase removes the overlap that independent warps get for free.

template <int CPB>
__device__ __forceinline__ void cell_accumulate(int yc, int xc, float wy1, float wx1, const float4 (&g)[CPB],
                                                float4 (&acc)[CPB]) {
  const float wy0 = 1.0f - wy1, wx0 = 1.0f - wx1;
  // Taps in the order TL, TR, BL, BR.  The four conditions are warp-uniform and sit outside the channel
  // loop (4 branches per bin).  The tap weight wy*wx is formed once per bin and applied with one (packed, FFMA2) FMA per
  // element pair: resize-mode gradients are a tolerance comparison anyway (fixed but different summation order
  // than TF's slice-grad + AddN; TF's own GPU kernel uses atomics), and this cuts the FP instruction count 3x.
#define FRCNN_CELL_ACCUM(WY, WX)                                                              \
  {                                                                                            \
    const float wgt = __fmul_rn(WY, WX);                                                       \
    const unsigned long long ww = pack2(wgt, wgt);                                             \
    _Pragma("unroll") for (int j = 0; j < CPB; ++j) {                                          \
      unpack2(fma2(pack2(g[j].x, g[j].y), ww, pack2(acc[j].x, acc[j].y)), acc[j].x, acc[j].y);  \
      unpack2(fma2(pack2(g[j].z, g[j].w), ww, pack2(acc[j].z, acc[j].w)), acc[j].z, acc[j].w);  \
    }                                                                                          \
  }
  if ((yc & 1) && (xc & 1)) FRCNN_CELL_ACCUM(wy0, wx0)
  if ((yc & 1) && (xc & 2)) FRCNN_CELL_ACCUM(wy0, wx1)
  if ((yc & 2) && (xc & 1)) FRCNN_CELL_ACCUM(wy1, wx0)
  if ((yc & 2) && (xc & 2)) FRCNN_CELL_ACCUM(wy1, wx1)
#undef FRCNN_CELL_ACCUM
}

// FULL: the CTA's CPB*128 channels all exist (C % (CPB*128) == 0): no per-load channel guards.  The per-bin
// bookkeeping matters: in the first version of this loop 85 of the ~130 SASS instructions per bin were guards,
// register zeroing and 64-bit address arithmetic (ncu source page), so the row address is kept as a per-RoI
// pointer plus a 32-bit (ph, pw) offset.
// RS > 1 (small launches, e.g. 2000 RoIs of ONE image): RS warps share a cell, each walks a contiguous 1/RS of the
// RoI chunks, and the partial sums are added in part order through shared memory.  With one image the launch is a
// single wave whose duration is the longest chain (the busiest cells see twice the average number of RoIs); the
// split shortens that chain RS-fold (0.335 -> 0.246 ms at 2000 RoIs x 1 image; RS = 2 / 8 and 512-channel warps were
// measured too: 0.31 / 0.24 ms -- beyond RS = 4 the launch is bound by resident warps x bytes in flight, not by the
// longest chain).  The summation order is still fixed (deterministic), just not the RS = 1 order.
template <int CPB, bool FULL, int G, int RS, int WARPS = (RS > 1 ? RS : CW_WARPS)>
__global__ void __launch_bounds__(WARPS * 32, (RS == 1 && CPB == 8) ? 768 / (WARPS * 32) : 0)      // 24 warps per SM need <= 80 registers
roi_bwd_resize_cell_kernel(const float* __restrict__ gout, const int4* __restrict__ crops,
                           const int4* __restrict__ taps, int H, int W, int C, int N, int P,
                           float* __restrict__ gfeat) {
  __shared__ float4 s_part[RS > 1 ? WARPS * CPB * 32 : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int part = warp % RS;
  const int cell_raw = blockIdx.x * (WARPS / RS) + warp / RS;
  const bool live = cell_raw < H * W;
  if (RS == 1 && !live) return;                     // warp-uniform; the RS = 1 kernel has no block-level barrier
  const int cell = live ? cell_raw : 0;
  const int img = blockIdx.z;
  const int y = cell / W, x = cell - y * W;
  const int cbase = blockIdx.y * (CPB * 128) + 4 * lane;
  const float* g_lane = gout + (size_t)img * N * P * P * C + cbase;
  const int4* crop_img = crops + (size_t)img * N;
  const int4* tap_img = taps + (size_t)img * N * P;
  const int row_floats = P * C;
  const int sub = lane / G, p = lane % G;
  float4 acc[CPB];
#pragma unroll
  for (int j = 0; j < CPB; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);

  // The kernel is occupancy-sensitive (80 registers at CPB = 8): prefetching the next chunk's crops and the next
  // covering RoI's tap record one step ahead costs 32 registers and was slower (1.59 ms vs 1.25 ms, profiles/README.md).
  const int chunks = (N + 31) / 32, per_part = (chunks + RS - 1) / RS;
  const int w_begin = RS == 1 ? 0 : part * per_part * 32;
  const int w_end = RS == 1 ? N : (live ? min(N, (part + 1) * per_part * 32) : 0);
  for (int w0 = w_begin; w0 < w_end; w0 += 32) {
    const int r = w0 + lane;
    bool inside = false;
    if (r < w_end) {
      const int4 k = __ldg(crop_img + r);
      inside = k.z > 0 && k.w > 0 && x >= k.x && x < k.x + k.z && y >= k.y && y < k.y + k.w;
    }
    unsigned m = __ballot_sync(0xffffffffu, inside);
    while (m) {
      // Up to 32/G covering RoIs per pass: lane = G*sub + p looks at tap p (both axes) of the sub-th covering RoI;
      // code bit0 = "lo tap is this cell", bit1 = "hi tap is this cell".  One table load and two ballots serve
      // four RoIs when P <= 8 (the per-RoI scan was 40 % of this kernel's instructions).
      int b = -1;
      {
        unsigned mm = m;
#pragma unroll
        for (int i = 0; i < 32 / G; ++i) {
          const int bi = mm ? __ffs(mm) - 1 : -1;
          if (sub == i) b = bi;
          mm &= mm - 1;
        }
        m = mm;
      }
      int ycode = 0, xcode = 0;
      int lyb = 0, lxb = 0;
      if (b >= 0 && p < P) {
        const int4 t = __ldg(tap_img + (w0 + b) * P + p);
        ycode = ((t.x & 0xffff) == y ? 1 : 0) | ((t.x >> 16) == y ? 2 : 0);
        xcode = ((t.z & 0xffff) == x ? 1 : 0) | ((t.z >> 16) == x ? 2 : 0);
        lyb = t.y;
        lxb = t.w;
      }
      const unsigned by = __ballot_sync(0xffffffffu, ycode != 0);
      const unsigned bx = __ballot_sync(0xffffffffu, xcode != 0);
#pragma unroll
      for (int i = 0; i < 32 / G; ++i) {
        unsigned my = G == 32 ? by : (by >> (G * i % 32)) & ((1u << (G % 32)) - 1u);
        const unsigned mx = G == 32 ? bx : (bx >> (G * i % 32)) & ((1u << (G % 32)) - 1u);
        if (my == 0u || mx == 0u) continue;
        const int bb = __shfl_sync(0xffffffffu, b, G * i % 32);
        const float* g_roi = g_lane + (size_t)(w0 + bb) * P * row_floats;
        while (my) {
          const int ph = __ffs(my) - 1;
          my &= my - 1;
          const int yc = __shfl_sync(0xffffffffu, ycode, G * i % 32 + ph);
          const int wyb = __shfl_sync(0xffffffffu, lyb, G * i % 32 + ph);
          const int ph_off = ph * row_floats;
          unsigned mxx = mx;
          while (mxx) {
            const int pw = __ffs(mxx) - 1;
            mxx &= mxx - 1;
            const int xc = __shfl_sync(0xffffffffu, xcode, G * i % 32 + pw);
            const int wxb = __shfl_sync(0xffffffffu, lxb, G * i % 32 + pw);
            const float* row = g_roi + (ph_off + pw * C);
            float4 g[CPB];
#pragma unroll
            for (int j = 0; j < CPB; ++j)
              g[j] = (FULL || cbase + j * 128 < C) ? ldg_f4(row + j * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
            cell_accumulate<CPB>(yc, xc, __int_as_float(wyb), __int_as_float(wxb), g, acc);
          }
        }
      }
    }
  }
  if (RS > 1) {
#pragma unroll
    for (int j = 0; j < CPB; ++j) s_part[(warp * CPB + j) * 32 + lane] = acc[j];
    __syncthreads();
    if (part != 0 || !live) return;
#pragma unroll
    for (int q = 1; q < RS; ++q)
#pragma unroll
      for (int j = 0; j < CPB; ++j) {
        const float4 v = s_part[((warp + q) * CPB + j) * 32 + lane];
        acc[j].x += v.x; acc[j].y += v.y; acc[j].z += v.z; acc[j].w += v.w;
      }
  }
  float* dst = gfeat + ((size_t)img * H * W + cell) * C + cbase;
#pragma unroll
  for (int j = 0; j < CPB; ++j)
    if (cbase + j * 128 < C) *reinterpret_cast<float4*>(dst + j * 128) = acc[j];
}

// ---------------------------------------------------------------------------------------
// backward, max mode: the same cell-stationary gather.  A bin (ph, pw) of a RoI can route its
// gradient to this cell only if the bin covers it, so the warp visits the covering bins in
// ascending (roi, ph, pw) order, reads the bin's arg-max row (int4 per lane and channel block),
// and adds dY where the arg-max equals this cell -- the order of oracle roi_max_bwd, bit for bit.
// The arg-max row of a bin is re-read by every cell the bin covers (L2 hits); dY is read only by
// the lanes whose channels actually selected this cell.
// (A shared-memory tile-ownership kernel with per-tile work lists was the first version: 11.9 ms at
// C1 x 64 images against 2.x ms for this one -- serial LDS/FADD/STS chains and 8 warps per SM.)
// ---------------------------------------------------------------------------------------
// The kernel waits on its arg-max / dY round trips (ncu: issue 26 %, long-scoreboard stalls 17 per issue), so resident
// warps buy throughput: the 512-channel variant used for small launches is capped at 64 registers (4 CTAs per SM;
// 2000 RoIs x 1 image: 0.54 -> 0.36 ms).  The same cap on the 1024-channel variant spills and was 5 % slower at 8 images.
template <int CPB, bool FULL, int G>
__global__ void __launch_bounds__(CW_WARPS * 32, CPB == 8 ? 0 : 1024 / (CW_WARPS * 32))
roi_bwd_max_cell_kernel(const float* __restrict__ gout, const int* __restrict__ argmax,
                        const int4* __restrict__ crops, const int4* __restrict__ taps, int H, int W, int C, int N,
                        int P, float* __restrict__ gfeat) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cell = blockIdx.x * CW_WARPS + warp;
  if (cell >= H * W) return;
  const int img = blockIdx.z;
  const int y = cell / W, x = cell - y * W;
  const int cbase = blockIdx.y * (CPB * 128) + 4 * lane;
  const size_t img_off = (size_t)img * N * P * P * C + cbase;
  const float* g_lane = gout + img_off;
  const int* a_lane = argmax + img_off;
  const int4* crop_img = crops + (size_t)img * N;
  const int4* tap_img = taps + (size_t)img * N * P;
  const int row_floats = P * C;
  const int sub = lane / G, p = lane % G;

  float4 acc[CPB];
#pragma unroll
  for (int j = 0; j < CPB; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);

  for (int w0 = 0; w0 < N; w0 += 32) {
    const int r = w0 + lane;
    bool inside = false;
    if (r < N) {
      const int4 k = __ldg(crop_img + r);
      inside = k.z > 0 && k.w > 0 && x >= k.x && x < k.x + k.z && y >= k.y && y < k.y + k.w;
    }
    unsigned m = __ballot_sync(0xffffffffu, inside);
    while (m) {
      // 32/G covering RoIs per pass, lane = G*sub + p (see the resize kernel)
      int b = -1;
      {
        unsigned mm = m;
#pragma unroll
        for (int i = 0; i < 32 / G; ++i) {
          const int bi = mm ? __ffs(mm) - 1 : -1;
          if (sub == i) b = bi;
          mm &= mm - 1;
        }
        m = mm;
      }
      bool hy = false, hx = false;
      if (b >= 0 && p < P) {
        const int4 t = __ldg(tap_img + (w0 + b) * P + p);
        hy = y >= (t.x & 0xffff) && y < (t.x >> 16);
        hx = x >= (t.z & 0xffff) && x < (t.z >> 16);
      }
      const unsigned by = __ballot_sync(0xffffffffu, hy);
      const unsigned bx = __ballot_sync(0xffffffffu, hx);
#pragma unroll
      for (int i = 0; i < 32 / G; ++i) {
        unsigned my = G == 32 ? by : (by >> (G * i % 32)) & ((1u << (G % 32)) - 1u);
        const unsigned mx = G == 32 ? bx : (bx >> (G * i % 32)) & ((1u << (G % 32)) - 1u);
        if (my == 0u || mx == 0u) continue;
        const int bb = __shfl_sync(0xffffffffu, b, G * i % 32);
        const size_t roi_off = (size_t)(w0 + bb) * P * row_floats;
        const float* g_roi = g_lane + roi_off;
        const int* a_roi = a_lane + roi_off;
        while (my) {
          const int ph = __ffs(my) - 1;
          my &= my - 1;
          const int ph_off = ph * row_floats;
          unsigned mxx = mx;
          while (mxx) {
            const int pw = __ffs(mxx) - 1;
            mxx &= mxx - 1;
            const int o = ph_off + pw * C;
            // arg-max and dY rows are requested together (no dependent second round trip); a lane whose
            // channels did not select this cell simply drops its dY values
            int4 a[CPB];
            float4 g[CPB];
#pragma unroll
            for (int j = 0; j < CPB; ++j) {
              const bool live = FULL || cbase + j * 128 < C;
              a[j] = live ? __ldg(reinterpret_cast<const int4*>(a_roi + o + j * 128)) : make_int4(-1, -1, -1, -1);
              g[j] = live ? ldg_f4(g_roi + o + j * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < CPB; ++j) {
              if (a[j].x == cell) acc[j].x += g[j].x;
              if (a[j].y == cell) acc[j].y += g[j].y;
              if (a[j].z == cell) acc[j].z += g[j].z;
              if (a[j].w == cell) acc[j].w += g[j].w;
            }
          }
        }
      }
    }
  }
  float* dst = gfeat + ((size_t)img * H * W + cell) * C + cbase;
#pragma unroll
  for (int j = 0; j < CPB; ++j)
    if (cbase + j * 128 < C) *reinterpret_cast<float4*>(dst + j * 128) = acc[j];
}

// ---------------------------------------------------------------------------------------
// backward, scalar-channel fallback (C % 4 != 0 or pool sizes beyond the work-list capacity): 8x8 tile,
// one channel per thread, every CTA scans all RoIs.  Not a performance path.
// ---------------------------------------------------------------------------------------
constexpr int BWD_TILE = 8;          // 8x8 cells
constexpr int BWD_CH = 512;          // channels per CTA = threads per CTA

template <int MODE>
__global__ void __launch_bounds__(BWD_CH, 1)
roi_bwd_scalar_kernel(const float* __restrict__ gout, const void* __restrict__ rois, int dtype,
               const int* __restrict__ argmax, int H, int W, int C, int N, int P, int tiles_x,
               float* __restrict__ gfeat) {
  extern __shared__ float acc[];     // [BWD_TILE*BWD_TILE][BWD_CH]
  const int tile = blockIdx.x, img = blockIdx.z;
  const int ty0 = (tile / tiles_x) * BWD_TILE, tx0 = (tile % tiles_x) * BWD_TILE;
  const int ty1 = min(ty0 + BWD_TILE, H), tx1 = min(tx0 + BWD_TILE, W);
  const int c = blockIdx.y * BWD_CH + threadIdx.x;
  const bool live = c < C;
  for (int i = 0; i < BWD_TILE * BWD_TILE; ++i) acc[i * BWD_CH + threadIdx.x] = 0.f;

  const float* g_img = gout + (size_t)img * N * P * P * C + c;
  const int* a_img = (MODE == FRCNN_ROI_MAX) ? argmax + (size_t)img * N * P * P * C + c : nullptr;

  for (int r = 0; r < N; ++r) {
    const Crop k = load_crop(rois, dtype, (size_t)img * N + r, W, H);
    if (k.w <= 0 || k.h <= 0) continue;
    if (k.x1 >= tx1 || k.x1 + k.w <= tx0 || k.y1 >= ty1 || k.y1 + k.h <= ty0) continue;   // CTA-uniform
    const float* g_roi = g_img + (size_t)r * P * P * C;
    if (MODE == FRCNN_ROI_RESIZE) {
      const float ys = (float)k.h / (float)P, xs = (float)k.w / (float)P;
      for (int ph = 0; ph < P; ++ph) {
        const Tap ty = axis_tap(ph, ys, k.h);
        const int ylo = k.y1 + ty.lo, yhi = k.y1 + ty.hi;
        const bool rlo = ylo >= ty0 && ylo < ty1, rhi = yhi >= ty0 && yhi < ty1;
        if (!rlo && !rhi) continue;
        const float wy1 = ty.lerp, wy0 = 1.0f - ty.lerp;
        for (int pw = 0; pw < P; ++pw) {
          const Tap tx = axis_tap(pw, xs, k.w);
          const int xlo = k.x1 + tx.lo, xhi = k.x1 + tx.hi;
          const bool clo = xlo >= tx0 && xlo < tx1, chi = xhi >= tx0 && xhi < tx1;
          if (!clo && !chi) continue;
          const float g = live ? __ldg(g_roi + (size_t)(ph * P + pw) * C) : 0.f;
          const float wx1 = tx.lerp, wx0 = 1.0f - tx.lerp;
          // order TL, TR, BL, BR; weight product (g*wy)*wx as in ResizeBilinearGrad
          if (rlo && clo) acc[((ylo - ty0) * BWD_TILE + (xlo - tx0)) * BWD_CH + threadIdx.x] += g * wy0 * wx0;
          if (rlo && chi) acc[((ylo - ty0) * BWD_TILE + (xhi - tx0)) * BWD_CH + threadIdx.x] += g * wy0 * wx1;
          if (rhi && clo) acc[((yhi - ty0) * BWD_TILE + (xlo - tx0)) * BWD_CH + threadIdx.x] += g * wy1 * wx0;
          if (rhi && chi) acc[((yhi - ty0) * BWD_TILE + (xhi - tx0)) * BWD_CH + threadIdx.x] += g * wy1 * wx1;
        }
      }
    } else {
      for (int ph = 0; ph < P; ++ph) {
        const int ya = k.y1 + (ph * k.h) / P, yb = k.y1 + ((ph + 1) * k.h + P - 1) / P;
        if (ya >= ty1 || yb <= ty0) continue;
        for (int pw = 0; pw < P; ++pw) {
          const int xa = k.x1 + (pw * k.w) / P, xb = k.x1 + ((pw + 1) * k.w + P - 1) / P;
          if (xa >= tx1 || xb <= tx0) continue;
          if (!live) continue;
          const size_t o = (size_t)r * P * P * C + (size_t)(ph * P + pw) * C;
          const int cell = __ldg(a_img + o);
          const int ay = cell / W, ax = cell - ay * W;
          if (ay >= ty0 && ay < ty1 && ax >= tx0 && ax < tx1)
            acc[((ay - ty0) * BWD_TILE + (ax - tx0)) * BWD_CH + threadIdx.x] += __ldg(g_img + o);
        }
      }
    }
  }
  if (!live) return;
  float* dst = gfeat + (size_t)img * H * W * C + c;
  for (int y = ty0; y < ty1; ++y)
    for (int x = tx0; x < tx1; ++x)
      dst[((size_t)y * W + x) * C] = acc[((y - ty0) * BWD_TILE + (x - tx0)) * BWD_CH + threadIdx.x];
}

// builds the per-launch RoI tables in the handle's scratch arena
static int build_tables(frcnn_handle* h, cudaStream_t stream, int mode, const void* rois, int dtype, int n_total,
                        int W, int H, int P, int4** crops, int4** taps) {
  void *pc = nullptr, *pt = nullptr;
  int rc = arena_get(h, stream, (size_t)n_total * sizeof(int4), &pc);
  if (rc) return rc;
  if ((rc = arena_get(h, stream, (size_t)n_total * P * sizeof(int4), &pt))) return rc;
  *crops = static_cast<int4*>(pc);
  *taps = static_cast<int4*>(pt);
  const int blocks = (int)(((size_t)n_total * (P + 1) + 255) / 256);
  if (mode == FRCNN_ROI_RESIZE)
    roi_table_kernel<FRCNN_ROI_RESIZE><<<blocks, 256, 0, stream>>>(rois, dtype, n_total, W, H, P, *crops, *taps);
  else
    roi_table_kernel<FRCNN_ROI_MAX><<<blocks, 256, 0, stream>>>(rois, dtype, n_total, W, H, P, *crops, *taps);
  FRCNN_LAUNCH_CHECK(h, "roi_table_kernel");
  return FRCNN_OK;
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

bool roi_bwd_blk_eligible(int mode, int H, int W, int C, int N, int P);
int launch_roi_bwd_blk(frcnn_handle*, cudaStream_t, int, const float*, const void*, int, const int32_t*, int, int, int,
                       int, int, int, float*, int);

int launch_roi_bwd(frcnn_handle* h, cudaStream_t stream, int mode, const float* gout, const void* rois, int dtype,
                   const int32_t* argmax, int H, int W, int C, int N, int P, int batch, float* gfeat, int compact) {
  if (compact) {
    const bool ok = mode == FRCNN_ROI_MAX && roi_compact_supported(H, W, C, P) && roi_bwd_blk_eligible(mode, H, W, C, N, P) &&
                    (reinterpret_cast<uintptr_t>(gout) % 16 == 0) && (reinterpret_cast<uintptr_t>(gfeat) % 16 == 0) &&
                    (reinterpret_cast<uintptr_t>(argmax) % 4 == 0);
    if (!ok) return fail(h, FRCNN_ERR_UNSUPPORTED, "roi_bwd: compact arg-max needs max mode, C %% 4 == 0, pool <= 8 and bins of at most 16 x 16 cells%s%s");
    return launch_roi_bwd_blk(h, stream, mode, gout, rois, dtype, argmax, H, W, C, N, P, batch, gfeat, 1);
  }
  const bool aligned = (reinterpret_cast<uintptr_t>(gout) % 16 == 0) && (reinterpret_cast<uintptr_t>(gfeat) % 16 == 0) &&
                       (mode != FRCNN_ROI_MAX || reinterpret_cast<uintptr_t>(argmax) % 16 == 0);
  if (aligned && roi_bwd_blk_eligible(mode, H, W, C, N, P))
    return launch_roi_bwd_blk(h, stream, mode, gout, rois, dtype, argmax, H, W, C, N, P, batch, gfeat, 0);
  if (C % 4 == 0 && aligned && P <= ROI_MAX_TABLE_P && H < 32768 && W < 32768) {
    int4 *crops = nullptr, *taps = nullptr;
    int rc = build_tables(h, stream, mode, rois, dtype, batch * N, W, H, P, &crops, &taps);
    if (rc) return rc;
    const int blocks128 = (C + 127) / 128;
    // channel blocks per warp: 8 (one warp per cell at C = 1024) when the launch has enough cells to fill
    // the GPU, else 4 so that a single image still yields >= 32 warps per SM
    int cpb = blocks128 >= 8 ? 8 : (blocks128 >= 4 ? 4 : (blocks128 >= 2 ? 2 : 1));
    // resize mode, fewer than ~4 waves of warps and enough RoI chunks to share: four warps per cell (RS = 4)
    const long long cell_warps = (long long)H * W * batch * ((blocks128 + cpb - 1) / cpb);
    const bool split = mode == FRCNN_ROI_RESIZE && P <= 8 && cell_warps < 8LL * h->sm_count * 24 && N >= 256;
    if (!split && cpb == 8 && (long long)H * W * batch < 2LL * h->sm_count * 32) cpb = 4;
    const int cells_per_cta = split ? 1 : CW_WARPS;        // split: one cell per 4-warp CTA
    dim3 grid((H * W + cells_per_cta - 1) / cells_per_cta, (blocks128 + cpb - 1) / cpb, batch);
#define FRCNN_LAUNCH_CELL(CPB)                                                                                      \
  if (mode == FRCNN_ROI_RESIZE) {                                                                                   \
    if (split && C % (CPB * 128) == 0)                                                                              \
      roi_bwd_resize_cell_kernel<CPB, true, 8, 4><<<grid, 4 * 32, 0, stream>>>(gout, crops, taps, H, W, C, N, P, gfeat); \
    else if (split)                                                                                                 \
      roi_bwd_resize_cell_kernel<CPB, false, 8, 4><<<grid, 4 * 32, 0, stream>>>(gout, crops, taps, H, W, C, N, P, gfeat); \
    else if (C % (CPB * 128) == 0 && P <= 8)                                                                        \
      roi_bwd_resize_cell_kernel<CPB, true, 8, 1><<<grid, CW_WARPS * 32, 0, stream>>>(gout, crops, taps, H, W, C, N, P, gfeat);  \
    else if (P <= 8)                                                                                                \
      roi_bwd_resize_cell_kernel<CPB, false, 8, 1><<<grid, CW_WARPS * 32, 0, stream>>>(gout, crops, taps, H, W, C, N, P, gfeat); \
    else                                                                                                            \
      roi_bwd_resize_cell_kernel<CPB, false, 32, 1><<<grid, CW_WARPS * 32, 0, stream>>>(gout, crops, taps, H, W, C, N, P, gfeat); \
  } else if (C % (CPB * 128) == 0 && P <= 8)                                                                        \
    roi_bwd_max_cell_kernel<CPB, true, 8><<<grid, CW_WARPS * 32, 0, stream>>>(gout, argmax, crops, taps, H, W, C, N, P, gfeat); \
  else if (P <= 8)                                                                                                  \
    roi_bwd_max_cell_kernel<CPB, false, 8><<<grid, CW_WARPS * 32, 0, stream>>>(gout, argmax, crops, taps, H, W, C, N, P, gfeat); \
  else                                                                                                              \
    roi_bwd_max_cell_kernel<CPB, false, 32><<<grid, CW_WARPS * 32, 0, stream>>>(gout, argmax, crops, taps, H, W, C, N, P, gfeat);
    if (cpb == 8) { FRCNN_LAUNCH_CELL(8) } else if (cpb == 4) { FRCNN_LAUNCH_CELL(4) } else if (cpb == 2) { FRCNN_LAUNCH_CELL(2) } else { FRCNN_LAUNCH_CELL(1) }
#undef FRCNN_LAUNCH_CELL
    FRCNN_LAUNCH_CHECK(h, "roi_bwd_cell_kernel");
    return FRCNN_OK;
  }
  const int tiles_x = (W + BWD_TILE - 1) / BWD_TILE, tiles_y = (H + BWD_TILE - 1) / BWD_TILE;
  dim3 grid(tiles_x * tiles_y, (C + BWD_CH - 1) / BWD_CH, batch);
  const size_t smem = (size_t)BWD_TILE * BWD_TILE * BWD_CH * sizeof(float);
  if (mode == FRCNN_ROI_RESIZE) {
    FRCNN_CUDA(h, cudaFuncSetAttribute(roi_bwd_scalar_kernel<FRCNN_ROI_RESIZE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    roi_bwd_scalar_kernel<FRCNN_ROI_RESIZE><<<grid, BWD_CH, smem, stream>>>(gout, rois, dtype, argmax, H, W, C, N, P, tiles_x, gfeat);
  } else {
    FRCNN_CUDA(h, cudaFuncSetAttribute(roi_bwd_scalar_kernel<FRCNN_ROI_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    roi_bwd_scalar_kernel<FRCNN_ROI_MAX><<<grid, BWD_CH, smem, stream>>>(gout, rois, dtype, argmax, H, W, C, N, P, tiles_x, gfeat);
  }
  FRCNN_LAUNCH_CHECK(h, "roi_bwd_scalar_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
