// K-c: training-target assignment.
//
//  label_anchors_kernel   anchor x GT IoU (float32, reference op order, no FMA), per-anchor
//                         max/argmax in registers, per-GT max/argmax with redux.sync warp
//                         reductions + one packed 64-bit atomicMax per (warp, GT); writes the
//                         threshold-rule labels and regression targets directly.
//  label_gt_fixup_kernel  "best anchor of every GT is positive" rule (rpn_util.py:76-82).
//  count_kernel           #pos&can_use / #neg&can_use per image (needed by host-side sampling).
//  apply_sampling_kernel  host-drawn switch-offs by rank (rpn_util.py:324-350).
//  pack_rpn_kernel        Keras y_true layouts (rpn_util.py:125-140).
//  label_rois_kernel      RoI x GT labelling, compaction, one-hot class / bbreg targets
//                         (det_util.py:310-366).
//
// IoU (util.py:146-177): area1 = (x2-x1)*(y2-y1); inter = max(0,min(x2)-max(x1)) *
// max(0,min(y2)-max(y1)); iou = inter / ((area1 + area2) - inter); all float32, IEEE division.
// np.argmax = FIRST maximum on both axes.
#include "common.cuh"

namespace frcnn {

constexpr int LBL_THREADS = 256;

struct __align__(8) BoxI16 { short x1, y1, x2, y2; };

__device__ __forceinline__ float iou_f32(float ax1, float ay1, float ax2, float ay2, float a_area,
                                         float gx1, float gy1, float gx2, float gy2, float g_area) {
  const float w = np_max(0.0f, __fsub_rn(np_min(ax2, gx2), np_max(ax1, gx1)));
  const float h = np_max(0.0f, __fsub_rn(np_min(ay2, gy2), np_max(ay1, gy1)));
  const float inter = __fmul_rn(w, h);
  const float uni = __fsub_rn(__fadd_rn(a_area, g_area), inter);
  return __fdiv_rn(inter, uni);
}

__device__ __forceinline__ void pixel_anchor(int i, const AnchorTable& tab, int cols, int stride,
                                             int& x1, int& y1, int& x2, int& y2) {
  const int a = i % tab.n, loc = i / tab.n;
  const int cx = loc % cols, cy = loc / cols;
  // int(stride * (c + 0.5)) for non-negative values: exact in double (rpn_util.py:184-189)
  const int px = (int)((double)stride * ((double)cx + 0.5));
  const int py = (int)((double)stride * ((double)cy + 0.5));
  x1 = px - (tab.w[a] >> 1);
  y1 = py - (tab.h[a] >> 1);
  x2 = x1 + tab.w[a];
  y2 = y1 + tab.h[a];
}

// RPN regression target (util.py:180-206 + rpn_util.py:93): anchor corners are exact ints,
// GT corners float32; GT centre/size are formed in float32 then everything is float64;
// the x[10,10,5,5] happens in float64 before the store to float32.
__device__ __forceinline__ float4 rpn_bbreg(int ax1, int ay1, int ax2, int ay2, float gx1, float gy1,
                                            float gx2, float gy2) {
  const double gcx = (double)__fadd_rn(gx2, gx1) / 2.0, gcy = (double)__fadd_rn(gy2, gy1) / 2.0;
  const double gw = (double)__fsub_rn(gx2, gx1), gh = (double)__fsub_rn(gy2, gy1);
  const double acx = (double)(ax2 + ax1) / 2.0, acy = (double)(ay2 + ay1) / 2.0;
  const double aw = (double)(ax2 - ax1), ah = (double)(ay2 - ay1);
  const double tx = __ddiv_rn(__dsub_rn(gcx, acx), aw), ty = __ddiv_rn(__dsub_rn(gcy, acy), ah);
  const double tw = log(__ddiv_rn(gw, aw)), th = log(__ddiv_rn(gh, ah));
  return make_float4((float)__dmul_rn(10.0, tx), (float)__dmul_rn(10.0, ty),
                     (float)__dmul_rn(5.0, tw), (float)__dmul_rn(5.0, th));
}

// A warp takes ONE anchor shape and a patch of 8 x 4 feature cells, so its 32 anchors fill a small rectangle of the
// image (anchor size + 112 x 48 pixels at stride 16) and a GT box that misses that rectangle is skipped for the whole
// warp with four compares: every IoU of the warp would be +0 (GT area > 0 is checked, so the union is positive), which
// changes neither the row maximum (starts at 0, strict '>') nor the column maximum (only IoU > 0 is recorded).  With one
// thread per flat anchor index a warp held all nine shapes of 3.5 cells and its rectangle was the largest anchor's.
// best_gt [batch, g_max] u64 = (iou_bits << 32) | ~anchor_index, zero-initialised by the caller (IoU >= 0 so float
// bits order like unsigned ints).  Lanes are in anchor-index order (cell row-major inside the patch), which the
// "lowest anchor index on ties" rule below relies on.
constexpr int LBL_PATCH_W = 8, LBL_PATCH_H = 4;
//
// RAGGED: the batch is padded to one rows x cols map and `extents` [batch][2] (rows, cols) gives each image's own map,
// clamped to the padded one.  Only cells inside it are live; padding cells get can_use = is_pos = 0 and bbreg = 0.  The
// patches are the same 8 x 4 tiles as in a call on the image's own map, the padded flat index is monotone in the
// image's own one, so the per-GT arg-max (lowest index on ties) picks the same anchor, and the ranks that
// pack_rpn_targets counts among usable anchors are unchanged.  `extents` is unused when RAGGED is false.
template <bool RAGGED>
__global__ void __launch_bounds__(LBL_THREADS)
label_anchors_kernel(const float* __restrict__ gt_all, const int* __restrict__ n_gt_all,
                     const int* __restrict__ img_wh, int g_max, AnchorTable tab, int rows, int cols,
                     int stride, int n, unsigned char* __restrict__ can_use,
                     unsigned char* __restrict__ is_pos, float4* __restrict__ bbreg,
                     unsigned long long* __restrict__ best_gt, const int* __restrict__ extents) {
  __shared__ float4 s_gt[FRCNN_MAX_GT];
  __shared__ float s_garea[FRCNN_MAX_GT];
  const int img = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
  const int G = min(n_gt_all[img], g_max);
  const float* gt = gt_all + (size_t)img * g_max * 4;
  for (int g = tid; g < G; g += LBL_THREADS) {
    const float4 b = make_float4(gt[4 * g], gt[4 * g + 1], gt[4 * g + 2], gt[4 * g + 3]);
    s_gt[g] = b;
    s_garea[g] = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  }
  __syncthreads();

  const int patches_x = (cols + LBL_PATCH_W - 1) / LBL_PATCH_W, patches_y = (rows + LBL_PATCH_H - 1) / LBL_PATCH_H;
  const int gw = blockIdx.x * (LBL_THREADS / 32) + (tid >> 5);      // (patch, anchor shape), shape fastest
  const int a = gw % tab.n, patch = gw / tab.n;
  if (patch >= patches_x * patches_y) return;                       // whole warp
  const int py = patch / patches_x, px = patch - py * patches_x;
  const int cx = px * LBL_PATCH_W + (lane & (LBL_PATCH_W - 1)), cy = py * LBL_PATCH_H + lane / LBL_PATCH_W;
  int rows_b = rows, cols_b = cols;
  if (RAGGED) {
    rows_b = min(max(extents[2 * img], 0), rows);
    cols_b = min(max(extents[2 * img + 1], 0), cols);
  }
  const bool live = cx < cols_b && cy < rows_b;
  const bool pad_cell = RAGGED && !live && cx < cols && cy < rows;
  const size_t o_own = (size_t)img * n + (size_t)(cy * cols + cx) * tab.n + a;
  if (RAGGED && (px * LBL_PATCH_W >= cols_b || py * LBL_PATCH_H >= rows_b)) {     // whole patch outside the image
    if (pad_cell) { is_pos[o_own] = 0; can_use[o_own] = 0; bbreg[o_own] = make_float4(0.f, 0.f, 0.f, 0.f); }
    return;
  }
  // a lane outside the map computes on the patch's first cell (inside by construction) and stores nothing
  const int ccx = live ? cx : px * LBL_PATCH_W, ccy = live ? cy : py * LBL_PATCH_H;
  const int i = (ccy * cols + ccx) * tab.n + a;
  // int(stride * (c + 0.5)) for non-negative values: exact in double (rpn_util.py:184-189)
  const int pcx = (int)((double)stride * ((double)ccx + 0.5)), pcy = (int)((double)stride * ((double)ccy + 0.5));
  const int x1 = pcx - (tab.w[a] >> 1), y1 = pcy - (tab.h[a] >> 1), x2 = x1 + tab.w[a], y2 = y1 + tab.h[a];
  const float fx1 = (float)x1, fy1 = (float)y1, fx2 = (float)x2, fy2 = (float)y2;
  const float a_area = __fmul_rn(__fsub_rn(fx2, fx1), __fsub_rn(fy2, fy1));
  // the warp's rectangle (integer pixel corners; min / max over the lanes)
  const int wx1 = __reduce_min_sync(0xffffffffu, x1), wy1 = __reduce_min_sync(0xffffffffu, y1);
  const int wx2 = __reduce_max_sync(0xffffffffu, x2), wy2 = __reduce_max_sync(0xffffffffu, y2);
  const float bx1 = (float)wx1, by1 = (float)wy1, bx2 = (float)wx2, by2 = (float)wy2;

  float best = 0.0f;      // np.amax over a row of the (N,G) matrix; G == 0 cannot happen (guarded on the host)
  int best_g = 0;
  bool first = true;
  for (int g = 0; g < G; ++g) {
    const float4 b = s_gt[g];
    const float g_area = s_garea[g];
    // no overlap with any anchor of the warp (min(x2) - max(x1) <= 0 or the same in y for every lane), finite GT
    // corners and a positive union: all 32 IoUs are +0
    if (g_area > 0.0f && (!(fminf(bx2, b.z) > fmaxf(bx1, b.x)) || !(fminf(by2, b.w) > fmaxf(by1, b.y))) &&
        isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w)) {
      first = false;      // the row maximum so far is >= 0 and '>' is strict: nothing to update
      continue;
    }
    const float v = iou_f32(fx1, fy1, fx2, fy2, a_area, b.x, b.y, b.z, b.w, g_area);
    if (first || v > best) { best = v; best_g = g; first = false; }   // strict '>' keeps the first maximum
    // per-GT maximum over anchors, lowest anchor index on ties
    const unsigned bits = live ? __float_as_uint(v) : 0u;
    const unsigned wmax = __reduce_max_sync(0xffffffffu, bits);
    if (wmax != 0u) {
      const unsigned who = __ballot_sync(0xffffffffu, live && bits == wmax);
      if (lane == (__ffs(who) - 1)) {
        const unsigned long long key = ((unsigned long long)wmax << 32) | (unsigned)(~(unsigned)i);
        atomicMax(best_gt + (size_t)img * g_max + g, key);
      }
    }
  }
  if (!live) {
    if (pad_cell) { is_pos[o_own] = 0; can_use[o_own] = 0; bbreg[o_own] = make_float4(0.f, 0.f, 0.f, 0.f); }
    return;
  }

  const int W = img_wh[2 * img], H = img_wh[2 * img + 1];
  const bool oob = (x1 < 0) || (y1 < 0) || (x2 >= W) || (y2 >= H);
  const bool pos = best > 0.7f;                 // rpn_util.py:75 compared in float32
  const bool neg = !pos && best < 0.3f;         // rpn_util.py:95
  const size_t o = (size_t)img * n + i;
  is_pos[o] = pos;
  can_use[o] = (pos || neg) && !oob;
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  if (pos) {
    const float4 b = s_gt[best_g];
    t = rpn_bbreg(x1, y1, x2, y2, b.x, b.y, b.z, b.w);
  }
  bbreg[o] = t;
}

// one thread per (GT, image): the arg-max anchor of every GT with max IoU > 0 becomes positive.
__global__ void label_gt_fixup_kernel(const float* __restrict__ gt_all, const int* __restrict__ n_gt_all,
                                      const int* __restrict__ img_wh, int g_max, AnchorTable tab,
                                      int cols, int stride, int n,
                                      const unsigned long long* __restrict__ best_gt,
                                      unsigned char* __restrict__ can_use,
                                      unsigned char* __restrict__ is_pos, float4* __restrict__ bbreg) {
  const int img = blockIdx.y;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int G = min(n_gt_all[img], g_max);
  if (g >= G) return;
  const unsigned long long key = best_gt[(size_t)img * g_max + g];
  if ((key >> 32) == 0ull) return;              // max IoU == 0 (rpn_util.py:77)
  const int i = (int)(~(unsigned)(key & 0xffffffffull));
  int x1, y1, x2, y2;
  pixel_anchor(i, tab, cols, stride, x1, y1, x2, y2);
  const float fx1 = (float)x1, fy1 = (float)y1, fx2 = (float)x2, fy2 = (float)y2;
  const float a_area = __fmul_rn(__fsub_rn(fx2, fx1), __fsub_rn(fy2, fy1));
  const float* gt = gt_all + (size_t)img * g_max * 4;
  // regression target goes to the anchor's OWN best GT (rpn_util.py:90), recomputed here
  float best = 0.f;
  int best_g = 0;
  for (int q = 0; q < G; ++q) {
    const float gx1 = gt[4 * q], gy1 = gt[4 * q + 1], gx2 = gt[4 * q + 2], gy2 = gt[4 * q + 3];
    const float v = iou_f32(fx1, fy1, fx2, fy2, a_area, gx1, gy1, gx2, gy2,
                            __fmul_rn(__fsub_rn(gx2, gx1), __fsub_rn(gy2, gy1)));
    if (q == 0 || v > best) { best = v; best_g = q; }
  }
  const int W = img_wh[2 * img], H = img_wh[2 * img + 1];
  const bool oob = (x1 < 0) || (y1 < 0) || (x2 >= W) || (y2 >= H);
  const size_t o = (size_t)img * n + i;
  // several GTs may share one arg-max anchor: every writer stores identical values
  is_pos[o] = 1;
  can_use[o] = !oob;
  bbreg[o] = rpn_bbreg(x1, y1, x2, y2, gt[4 * best_g], gt[4 * best_g + 1], gt[4 * best_g + 2], gt[4 * best_g + 3]);
}

__global__ void __launch_bounds__(LBL_THREADS)
count_kernel(const unsigned char* __restrict__ can_use, const unsigned char* __restrict__ is_pos, int n,
             int* __restrict__ counts) {
  const int img = blockIdx.y;
  const int i = blockIdx.x * LBL_THREADS + threadIdx.x;
  bool p = false, q = false;
  if (i < n) {
    const size_t o = (size_t)img * n + i;
    p = can_use[o] && is_pos[o];
    q = can_use[o] && !is_pos[o];
  }
  const int np_ = __popc(__ballot_sync(0xffffffffu, p)), nq = __popc(__ballot_sync(0xffffffffu, q));
  if ((threadIdx.x & 31) == 0) {
    if (np_) atomicAdd(counts + 2 * img, np_);
    if (nq) atomicAdd(counts + 2 * img + 1, nq);
  }
}

// Host-drawn sampling (rpn_util.py:324-350): one CTA per image.  off_pos / off_neg hold RANKS --
// positions among the image's usable positives / negatives in ascending anchor order, i.e. the
// values random.sample(range(num_pos|num_neg), ...) returned -- and the anchors at those ranks get
// can_use = 0.  Ranks are staged as bitmaps in shared memory; an ordered ballot scan over the
// anchors recovers every anchor's rank.  Both rank sets refer to the flags as they were on entry.
constexpr int SMP_THREADS = 1024;
__global__ void __launch_bounds__(SMP_THREADS)
apply_sampling_kernel(unsigned char* __restrict__ can_use_all, const unsigned char* __restrict__ is_pos_all, int n,
                      const int* __restrict__ off_pos, const int* __restrict__ off_pos_offsets,
                      const int* __restrict__ off_neg, const int* __restrict__ off_neg_offsets, int words) {
  extern __shared__ unsigned smp_bits[];
  unsigned* pos_bits = smp_bits;
  unsigned* neg_bits = smp_bits + words;
  __shared__ int tot_p[SMP_THREADS / 32], tot_q[SMP_THREADS / 32];
  __shared__ int base_p, base_q;
  const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = off_pos ? off_pos_offsets[img] : 0, p1 = off_pos ? off_pos_offsets[img + 1] : 0;
  const int q0 = off_neg ? off_neg_offsets[img] : 0, q1 = off_neg ? off_neg_offsets[img + 1] : 0;
  if (p1 <= p0 && q1 <= q0) return;                 // nothing to switch off in this image (CTA-uniform)
  for (int i = tid; i < 2 * words; i += SMP_THREADS) smp_bits[i] = 0u;
  if (tid == 0) { base_p = 0; base_q = 0; }
  __syncthreads();
  for (int j = p0 + tid; j < p1; j += SMP_THREADS) {
    const int r = off_pos[j];
    if (r >= 0 && r < n) atomicOr(&pos_bits[r >> 5], 1u << (r & 31));
  }
  for (int j = q0 + tid; j < q1; j += SMP_THREADS) {
    const int r = off_neg[j];
    if (r >= 0 && r < n) atomicOr(&neg_bits[r >> 5], 1u << (r & 31));
  }
  __syncthreads();
  unsigned char* can_use = can_use_all + (size_t)img * n;
  const unsigned char* is_pos = is_pos_all + (size_t)img * n;
  const unsigned below = (1u << lane) - 1u;
  for (int start = 0; start < n; start += SMP_THREADS) {
    const int i = start + tid;
    bool p = false, q = false;
    if (i < n) {
      const bool cu = can_use[i] != 0, ip = is_pos[i] != 0;
      p = cu && ip;
      q = cu && !ip;
    }
    const unsigned bp = __ballot_sync(0xffffffffu, p), bq = __ballot_sync(0xffffffffu, q);
    if (lane == 0) { tot_p[warp] = __popc(bp); tot_q[warp] = __popc(bq); }
    __syncthreads();
    int rp = base_p, rq = base_q;
    for (int w = 0; w < warp; ++w) { rp += tot_p[w]; rq += tot_q[w]; }
    rp += __popc(bp & below);
    rq += __popc(bq & below);
    if (p && ((pos_bits[rp >> 5] >> (rp & 31)) & 1u)) can_use[i] = 0;
    if (q && ((neg_bits[rq >> 5] >> (rq & 31)) & 1u)) can_use[i] = 0;
    __syncthreads();
    if (tid == 0) {
      int ap = 0, aq = 0;
      for (int w = 0; w < SMP_THREADS / 32; ++w) { ap += tot_p[w]; aq += tot_q[w]; }
      base_p += ap;
      base_q += aq;
    }
    __syncthreads();
  }
}

// one thread per anchor: two 16-byte stores into the cell's y_bbreg row (the selector repeated four times, the four
// targets) and two bytes into its y_class row.  The first version ran one thread per float of y_bbreg with a 64-bit
// division and modulo by 8A each: 0.125 ms per 128 images for 143 MB, six times the HBM time.
__global__ void __launch_bounds__(LBL_THREADS)
pack_rpn_kernel(const unsigned char* __restrict__ can_use, const unsigned char* __restrict__ is_pos,
                const float4* __restrict__ bbreg, int n_loc, int A, unsigned char* __restrict__ y_class,
                float4* __restrict__ y_bbreg) {
  const int img = blockIdx.y;
  const unsigned t = blockIdx.x * LBL_THREADS + threadIdx.x;      // anchor inside the image
  if (t >= (unsigned)n_loc * (unsigned)A) return;
  const unsigned loc = t / (unsigned)A, a = t - loc * (unsigned)A;
  const size_t anchor = (size_t)img * n_loc * A + t, cell = (size_t)img * n_loc + loc;
  const unsigned char cu = can_use[anchor], ip = is_pos[anchor];
  const float sel = (cu && ip) ? 1.0f : 0.0f;                     // np.repeat(sel, 4, axis=2)
  float4* row = y_bbreg + cell * 2 * A;                           // 8A floats per cell
  row[a] = make_float4(sel, sel, sel, sel);
  row[A + a] = bbreg[anchor];
  unsigned char* crow = y_class + cell * 2 * A;
  crow[a] = cu;
  crow[A + a] = ip;
}

// ------------------------------------------------------------------------------------------
// Detector RoI labelling: one CTA per image.
// ------------------------------------------------------------------------------------------
// 1024 threads per image: the kernel is one CTA per image (order-preserving compaction), so its latency chains -- 50
// dependent IoU divisions per RoI, float64 log for the positives -- need the warps of one CTA to overlap them
// (0.134 ms per 128 images x 2000 RoIs with 256 threads).
constexpr int LR_THREADS = 1024;

__global__ void __launch_bounds__(LR_THREADS)
label_rois_kernel(const BoxI16* __restrict__ rois_all, const int* __restrict__ n_roi_all, int n_max,
                  const double* __restrict__ gt_all, const int* __restrict__ gt_cls_all,
                  const int* __restrict__ n_gt_all, int g_max, int K, BoxI16* __restrict__ out_rois,
                  int* __restrict__ out_cls, float* __restrict__ out_bbreg, int* __restrict__ out_src,
                  int* __restrict__ out_count) {
  __shared__ float4 s_gt[FRCNN_MAX_GT];
  __shared__ float s_garea[FRCNN_MAX_GT];
  __shared__ int s_warp_tot[LR_THREADS / 32];
  __shared__ int s_base;
  __shared__ int s_row_cls[LR_THREADS];                       // class | positive << 16 of the chunk's eligible rows
  __shared__ float4 s_row_tg[LR_THREADS];                     // their four regression targets
  const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = n_roi_all ? min(n_roi_all[img], n_max) : n_max;
  const int G = min(n_gt_all[img], g_max);
  const double* gt64 = gt_all + (size_t)img * g_max * 4;
  const int* gcls = gt_cls_all + (size_t)img * g_max;
  const BoxI16* rois = rois_all + (size_t)img * n_max;
  const int kfg = K - 1;
  for (int g = tid; g < G; g += LR_THREADS) {
    const float4 b = make_float4((float)gt64[4 * g], (float)gt64[4 * g + 1], (float)gt64[4 * g + 2], (float)gt64[4 * g + 3]);
    s_gt[g] = b;                                              // util.py:229-239: f64 -> f32 copy
    s_garea[g] = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  }
  if (tid == 0) s_base = 0;
  __syncthreads();

  for (int start = 0; start < n; start += LR_THREADS) {
    const int i = start + tid;
    bool elig = false, pos = false;
    int best_g = 0;
    BoxI16 r = {0, 0, 0, 0};
    if (i < n && G > 0) {
      r = rois[i];
      // int16 areas are exact integers (no wrap below 181x181 cells); widened to f32 by the add
      const float fx1 = (float)r.x1, fy1 = (float)r.y1, fx2 = (float)r.x2, fy2 = (float)r.y2;
      const float a_area = (float)((int)(short)((r.x2 - r.x1) * (r.y2 - r.y1)));
      float best = 0.f;
      for (int g = 0; g < G; ++g) {
        const float4 b = s_gt[g];
        const float v = iou_f32(fx1, fy1, fx2, fy2, a_area, b.x, b.y, b.z, b.w, s_garea[g]);
        if (g == 0 || v > best) { best = v; best_g = g; }
      }
      elig = best >= 0.1f;                                    // det_util.py:318 (float32 compare)
      pos = best >= 0.5f;                                     // det_util.py:321
    }
    // order-preserving compaction
    const unsigned ball = __ballot_sync(0xffffffffu, elig);
    if (lane == 0) s_warp_tot[warp] = __popc(ball);
    __syncthreads();
    int before = s_base;
    for (int wv = 0; wv < warp; ++wv) before += s_warp_tot[wv];
    const int row = before + __popc(ball & ((1u << lane) - 1u));
    // The thread keeps only the row's label record in shared memory; the K + 8(K-1) output words of every row of the
    // chunk are then written by the whole CTA, coalesced (128-bit stores for y_transform).  One thread filling its
    // own 724-byte row word by word reached 9 % of the HBM write bandwidth.
    int cls_of_row = K - 1;                                   // 'bg'
    float4 tg4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (elig) {
      const size_t o = (size_t)img * n_max + row;
      out_rois[o] = r;
      if (out_src) out_src[o] = i;
      if (pos) {
        cls_of_row = gcls[best_g];
        // det_util.py:346-352: get_reg_params(roi int16, GT float64) in float64, stored to f32,
        // then multiplied by [10,10,5,5] in float32.
        const double gx1 = gt64[4 * best_g], gy1 = gt64[4 * best_g + 1], gx2 = gt64[4 * best_g + 2], gy2 = gt64[4 * best_g + 3];
        const double gcx = __ddiv_rn(__dadd_rn(gx2, gx1), 2.0), gcy = __ddiv_rn(__dadd_rn(gy2, gy1), 2.0);
        const double gw = __dsub_rn(gx2, gx1), gh = __dsub_rn(gy2, gy1);
        const double acx = (double)(short)(r.x2 + r.x1) / 2.0, acy = (double)(short)(r.y2 + r.y1) / 2.0;
        const double aw = (double)(short)(r.x2 - r.x1), ah = (double)(short)(r.y2 - r.y1);
        const float tx = (float)__ddiv_rn(__dsub_rn(gcx, acx), aw), ty = (float)__ddiv_rn(__dsub_rn(gcy, acy), ah);
        const float tw = (float)log(__ddiv_rn(gw, aw)), th = (float)log(__ddiv_rn(gh, ah));
        tg4 = make_float4(__fmul_rn(tx, 10.f), __fmul_rn(ty, 10.f), __fmul_rn(tw, 5.f), __fmul_rn(th, 5.f));
      }
      s_row_cls[row - s_base] = cls_of_row | (pos ? 0x10000 : 0);
      s_row_tg[row - s_base] = tg4;
    }
    __syncthreads();
    {
      int chunk_rows = 0;
      for (int wv = 0; wv < LR_THREADS / 32; ++wv) chunk_rows += s_warp_tot[wv];
      const size_t row0 = (size_t)img * n_max + s_base;
      int* oc = out_cls + row0 * K;
      for (int w = tid; w < chunk_rows * K; w += LR_THREADS) {
        const int rr = w / K, c = w - rr * K;
        oc[w] = (c == (s_row_cls[rr] & 0xffff)) ? 1 : 0;       // one-hot, 'bg' = last class (det_util.py:358-366)
      }
      const int f4_per_row = 2 * kfg;                          // [4(K-1) labels | 4(K-1) targets] as float4 per class
      const bool vec = (reinterpret_cast<uintptr_t>(out_bbreg) & 15) == 0;
      float* ob = out_bbreg + row0 * 8 * kfg;
      for (int w = tid; w < chunk_rows * f4_per_row; w += LR_THREADS) {
        const int rr = w / f4_per_row, q = w - rr * f4_per_row;
        const int rec = s_row_cls[rr];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rec & 0x10000) {                                   // positive row (det_util.py:338-354)
          if (q == (rec & 0xffff)) v = make_float4(1.f, 1.f, 1.f, 1.f);
          else if (q - kfg == (rec & 0xffff)) v = s_row_tg[rr];
        }
        if (vec) {
          reinterpret_cast<float4*>(ob)[w] = v;
        } else {
          ob[4 * w] = v.x; ob[4 * w + 1] = v.y; ob[4 * w + 2] = v.z; ob[4 * w + 3] = v.w;
        }
      }
    }
    __syncthreads();
    if (tid == 0) {
      int add = 0;
      for (int wv = 0; wv < LR_THREADS / 32; ++wv) add += s_warp_tot[wv];
      s_base += add;
    }
    __syncthreads();
  }
  if (tid == 0) out_count[img] = s_base;
}

// ------------------------------------------------------------------------------------------
int launch_label_anchors(frcnn_handle* h, cudaStream_t stream, const float* gt, const int32_t* n_gt,
                         const int32_t* img_wh, int g_max, const AnchorTable& tab, int rows, int cols,
                         int stride, int batch, uint8_t* can_use, uint8_t* is_pos, float* bbreg,
                         int32_t* counts, const int32_t* extents) {
  const int n = rows * cols * tab.n;
  void* ws = nullptr;
  const size_t best_bytes = (size_t)batch * g_max * sizeof(unsigned long long);
  int rc = arena_get(h, stream, best_bytes, &ws);
  if (rc) return rc;
  auto* best = reinterpret_cast<unsigned long long*>(ws);
  FRCNN_CUDA(h, cudaMemsetAsync(best, 0, best_bytes, stream));
  FRCNN_CUDA(h, cudaMemsetAsync(counts, 0, (size_t)batch * 2 * sizeof(int), stream));
  const int patches = ((cols + LBL_PATCH_W - 1) / LBL_PATCH_W) * ((rows + LBL_PATCH_H - 1) / LBL_PATCH_H);
  dim3 grid((patches * tab.n + LBL_THREADS / 32 - 1) / (LBL_THREADS / 32), batch);
  auto kernel = extents ? label_anchors_kernel<true> : label_anchors_kernel<false>;
  kernel<<<grid, LBL_THREADS, 0, stream>>>(gt, n_gt, img_wh, g_max, tab, rows, cols, stride, n, can_use, is_pos,
                                           reinterpret_cast<float4*>(bbreg), best, extents);
  FRCNN_LAUNCH_CHECK(h, "label_anchors_kernel");
  dim3 g2((g_max + 63) / 64, batch);
  label_gt_fixup_kernel<<<g2, 64, 0, stream>>>(gt, n_gt, img_wh, g_max, tab, cols, stride, n, best, can_use,
                                              is_pos, reinterpret_cast<float4*>(bbreg));
  FRCNN_LAUNCH_CHECK(h, "label_gt_fixup_kernel");
  count_kernel<<<grid, LBL_THREADS, 0, stream>>>(can_use, is_pos, n, counts);
  FRCNN_LAUNCH_CHECK(h, "count_kernel");
  return FRCNN_OK;
}

int launch_pack_rpn(frcnn_handle* h, cudaStream_t stream, uint8_t* can_use, const uint8_t* is_pos,
                    const float* bbreg, const int32_t* off_pos, const int32_t* off_pos_offsets,
                    const int32_t* off_neg, const int32_t* off_neg_offsets, int rows, int cols, int A,
                    int batch, uint8_t* y_class, float* y_bbreg) {
  const int n_loc = rows * cols;
  if (off_pos || off_neg) {
    const int n = n_loc * A;
    const int words = (n + 31) / 32;
    const size_t smem = (size_t)2 * words * sizeof(unsigned);
    if (smem + 1024 > (size_t)h->max_smem_optin)
      return fail(h, FRCNN_ERR_UNSUPPORTED, "pack_rpn_targets: too many anchors per image for the rank bitmaps%s%s");
    if (smem > 48 * 1024)
      FRCNN_CUDA(h, cudaFuncSetAttribute(apply_sampling_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    apply_sampling_kernel<<<batch, SMP_THREADS, smem, stream>>>(can_use, is_pos, n, off_pos, off_pos_offsets, off_neg,
                                                               off_neg_offsets, words);
    FRCNN_LAUNCH_CHECK(h, "apply_sampling_kernel");
  }
  if ((reinterpret_cast<uintptr_t>(bbreg) | reinterpret_cast<uintptr_t>(y_bbreg)) & 15u)
    return fail(h, FRCNN_ERR_INVALID, "pack_rpn_targets: bbreg and y_bbreg must be 16-byte aligned%s%s");
  const unsigned per_img = (unsigned)n_loc * (unsigned)A;
  pack_rpn_kernel<<<dim3((per_img + LBL_THREADS - 1) / LBL_THREADS, batch), LBL_THREADS, 0, stream>>>(
      can_use, is_pos, reinterpret_cast<const float4*>(bbreg), n_loc, A, y_class, reinterpret_cast<float4*>(y_bbreg));
  FRCNN_LAUNCH_CHECK(h, "pack_rpn_kernel");
  return FRCNN_OK;
}

int launch_label_rois(frcnn_handle* h, cudaStream_t stream, const int16_t* rois, const int32_t* n_roi,
                      int n_max, const double* gt, const int32_t* gt_cls, const int32_t* n_gt, int g_max,
                      int K, int batch, int16_t* out_rois, int32_t* out_cls, float* out_bbreg,
                      int32_t* out_src, int32_t* out_count) {
  label_rois_kernel<<<batch, LR_THREADS, 0, stream>>>(reinterpret_cast<const BoxI16*>(rois), n_roi, n_max, gt,
                                                      gt_cls, n_gt, g_max, K,
                                                      reinterpret_cast<BoxI16*>(out_rois), out_cls, out_bbreg,
                                                      out_src, out_count);
  FRCNN_LAUNCH_CHECK(h, "label_rois_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
