// K-b: greedy NMS.  One CTA per image (int16 RPN boxes) or per segment (float64 per-class
// boxes); the whole problem lives in shared memory.
//
// Algorithm (work-efficient form of the bitmask NMS):
//   1. order: visit candidates by (score desc, position desc) -- the order
//      `np.argsort(probs, kind='stable')` consumed from the back gives (det_util.py:231-236).
//      If the scores already arrive strictly descending (the output of K-a) the order is the
//      identity and the box array is pulled into shared memory with one 1-D TMA bulk copy
//      (cp.async.bulk + mbarrier); otherwise 64-bit keys are bitonic-sorted in shared memory
//      and the boxes are gathered into the same buffer.
//   2. sweep in tiles of 64 candidates: (a) each candidate of the tile is tested against the
//      kept list (shared memory, broadcast reads), warp ballots build the 64-bit
//      "suppressed by kept" mask; (b) the 64x64 intra-tile IoU matrix is reduced to 64-bit row
//      masks; (c) one thread resolves the tile serially over set bits only and appends the
//      survivors to the kept list.  Only kept x candidate pairs are ever tested
//      (<= n*max_boxes instead of n^2/2) and the sweep stops at max_boxes (det_util.py:253-254).
//
// Predicate (det_util.py:243-251): areas with the +1 convention, ratio = inter/union in
// float64, candidate survives iff ratio <= thresh.  For int16 boxes inter and union are exact
// integers; a float32 band test decides the clear cases and only |inter - t*union| tiny falls
// through to the IEEE float64 division, so the decision is identical to numpy's.
#include <cooperative_groups.h>

#include <math.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace frcnn {

constexpr int NMS_THREADS = 512;
constexpr int NMS_TILE = 64;

struct __align__(8) BoxI16 { short x1, y1, x2, y2; };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// exact int16 pair test; a = kept box, b = candidate.  returns true if b is suppressed.
__device__ __forceinline__ bool suppressed_i16(int ax1, int ay1, int ax2, int ay2, int a_area,
                                               int bx1, int by1, int bx2, int by2, int b_area,
                                               float t_f, double t, bool zero_survives) {
  const int iw = min(ax2, bx2) - max(ax1, bx1) + 1;
  const int ih = min(ay2, by2) - max(ay1, by1) + 1;
  const int inter = (iw > 0 && ih > 0) ? iw * ih : 0;
  const int uni = a_area + b_area - inter;
  if (uni > 0) {
    if (inter == 0) return !zero_survives;
    const float fi = (float)inter, fu = (float)uni;
    const float d = __fmaf_rn(-t_f, fu, fi);               // inter - t*union, ~1e-7 relative
    const float band = 1e-4f * fu;
    if (d > band) return true;
    if (d < -band) return false;
  }
  const double ratio = __ddiv_rn((double)inter, (double)uni);   // IEEE, same as numpy true_divide
  return !(ratio <= t);
}

// Branch-free screening test in 64-bit fixed point: d = inter*2^32 - round(t*2^32)*union.  |d| > union
// decides (the rounding of t moves d by < union/2); anything inside the band is "uncertain" and is
// re-examined with the exact double division above.  Valid for 0 < t < 1 and 0 < union < 2^31.  A union <= 0
// (boxes with x2 < x1 - 1 or y2 < y1 - 1 have a negative area) would wrap the unsigned product, so it is
// "uncertain" too and the exact predicate decides it (inter / union <= t in float64, as numpy does).
// returns 1 = suppressed, 0 = survives, 2 = uncertain
__device__ __forceinline__ int screen_i16(int ax1, int ay1, int ax2, int ay2, int a_area, int bx1, int by1,
                                          int bx2, int by2, int b_area, unsigned long long t_fix) {
  const int iw = min(ax2, bx2) - max(ax1, bx1) + 1;
  const int ih = min(ay2, by2) - max(ay1, by1) + 1;
  const int inter = max(iw, 0) * max(ih, 0);
  const int uni = a_area + b_area - inter;
  const long long d = (long long)(((unsigned long long)(unsigned)inter << 32) - t_fix * (unsigned long long)(unsigned)uni);
  const long long band = (long long)uni;
  return uni <= 0 ? 2 : (d > band ? 1 : (d < -band ? 0 : 2));
}

// Thresholds that are a ratio of small integers (0.7 = 7/10 as a double: the RPN's value) need no fixed point and no
// band: with t_d = RN(p/q), RN(inter/union) <= t_d  <=>  inter*q <= p*union, exactly.  (If inter/union <= p/q the
// rounded quotient cannot exceed RN(p/q); if it is larger, it is larger by at least 1/(union*q) > 2^-41, hundreds of
// ulps above t_d, for union < 2^31 and q <= 1000.)  Two 64-bit products and one compare instead of the 12-instruction
// screening test: the candidate x kept tests are what the training configuration (12000 -> 2000) spends its time on.
// returns 1 = suppressed, 0 = survives, 2 = uncertain (union <= 0: degenerate boxes go to the exact predicate)
__device__ __forceinline__ int screen_rational(int ax1, int ay1, int ax2, int ay2, int a_area, int bx1, int by1,
                                               int bx2, int by2, int b_area, int p, int q) {
  const int iw = min(ax2, bx2) - max(ax1, bx1) + 1;
  const int ih = min(ay2, by2) - max(ay1, by1) + 1;
  const int inter = max(iw, 0) * max(ih, 0);
  const int uni = a_area + b_area - inter;
  const bool over = (long long)inter * q > (long long)uni * p;
  return uni > 0 ? (over ? 1 : 0) : 2;
}

// The same test with 32-bit products, for images whose boxes are small enough that no product can overflow
// (3 * maxdim^2 * max(p, q) < 2^31, checked once per image) and all valid (x2 >= x1, y2 >= y1: union > 0 always, no
// "uncertain" case).  The kept-list sweep is issue-bound, every instruction of the pair test counts, so it is folded:
// inter*q > (A + B - inter)*p  <=>  inter*(p+q) - A*p > B*p.  The kept list then stores -A*p instead of A and the
// candidate carries B*p: one IMAD and one compare after the intersection (12 ALU instructions per pair in all).
__device__ __forceinline__ bool screen_small_valid(int ax1, int ay1, int ax2, int ay2, int neg_ap, int bx1, int by1,
                                                   int bx2, int by2, int bp, int pq) {
  const int iw = min(ax2, bx2) - max(ax1, bx1) + 1;
  const int ih = min(ay2, by2) - max(ay1, by1) + 1;
  const int inter = max(iw, 0) * max(ih, 0);
  return inter * pq + neg_ap > bp;
}

// Thread-block clusters: an image may be given a cluster of CL CTAs (1, 2, 4, 8 or 16 SMs).  Every CTA
// holds the full candidate array, the kept list is dealt round-robin over the CTAs (kept j lives in CTA
// j % CL), each CTA tests the tile's 64 candidates against ITS share, the 64-bit partial masks are
// exchanged through distributed shared memory (one remote 8-byte store per peer) + one cluster barrier
// per tile, and every CTA then resolves the tile redundantly (identical inputs -> identical keep bits), so
// no second exchange is needed.  This cuts the dominant candidate x kept work of the training
// configuration (12000 -> 2000) by CL for a single image.
//
// Dynamic shared memory layout (bytes):
//   [0, buf_bytes)            sort keys (u64) then, in place, boxes in visit order (8 B each)
//   kept boxes int4[keep_local] ; kept area int[keep_local] ; kept slot (visit rank) int[max_keep]
__global__ void __launch_bounds__(NMS_THREADS, 1)
nms_i16_kernel(const BoxI16* __restrict__ boxes_all, const float* __restrict__ scores_all,
               const int* __restrict__ n_all, int n_max, double thresh, int max_boxes, int max_keep,
               int keep_local, int buf_elems, int cl, int rat_p, int rat_q, int* __restrict__ order_all,
               int* __restrict__ keep_index,
               int* __restrict__ keep_count, BoxI16* __restrict__ keep_boxes,
               float* __restrict__ keep_scores) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(smem);
  int4* kept_box = reinterpret_cast<int4*>(smem + (((size_t)buf_elems * 8 + 15) & ~(size_t)15));
  int* kept_area = reinterpret_cast<int*>(kept_box + keep_local);
  int* kept_slot = kept_area + keep_local;

  __shared__ __align__(8) unsigned long long mbar;
  __shared__ unsigned long long row_mask[NMS_TILE];
  __shared__ unsigned sup_part[NMS_THREADS / 32];
  __shared__ unsigned long long s_xpart[2][16];      // [tile parity][cluster rank] partial "suppressed by kept" masks
  __shared__ unsigned long long s_keepbits;
  __shared__ int s_unsorted, s_nkept, s_stop, s_maxdim, s_maxabs;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (cl > 1) ? (int)cluster.block_rank() : 0;
  const int img = blockIdx.x / cl, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = n_all ? min(n_all[img], n_max) : n_max;
  const BoxI16* boxes = boxes_all + (size_t)img * n_max;
  const float* scores = scores_all + (size_t)img * n_max;
  int* order = order_all + ((size_t)img * cl + rank) * n_max;     // per-CTA scratch (only rank 0's is read back)

  if (tid == 0) { s_unsorted = 0; s_nkept = 0; s_stop = 0; s_maxdim = 0; s_maxabs = 0; }
  __syncthreads();
  // distributed shared memory may only be touched once every CTA of the cluster is running
  if (cl > 1) cluster.sync();

  // ---- 1. visit order --------------------------------------------------------------------
  int bad = 0;
#pragma unroll 4
  for (int i = tid; i + 1 < n; i += NMS_THREADS) bad |= !(__ldg(scores + i) > __ldg(scores + i + 1));
  if (__any_sync(0xffffffffu, bad) && lane == 0) s_unsorted = 1;
  __syncthreads();
  const bool unsorted = s_unsorted != 0;

  if (!unsorted) {
    // identity order: 1-D TMA bulk copy of the contiguous box rows into shared memory
    const uint32_t bytes = (uint32_t)n * 8u;
    const bool tma_ok = (bytes % 16u == 0) && ((reinterpret_cast<uintptr_t>(boxes) & 15u) == 0) && n > 0;
    if (tma_ok) {
      if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      }
      __syncthreads();
      if (tid == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(buf)), "l"(boxes), "r"(bytes), "r"(smem_u32(&mbar)) : "memory");
      }
      // everyone waits on phase 0
      uint32_t done = 0;
      while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_u32(&mbar)) : "memory");
      }
    } else {
      for (int i = tid; i < n; i += NMS_THREADS) buf[i] = reinterpret_cast<const unsigned long long*>(boxes)[i];
    }
    __syncthreads();
  } else {
    int m = 1;
    while (m < n) m <<= 1;
    if (m > buf_elems) {
      // More than FRCNN_NMS_MAX_UNSORTED candidates that are NOT strictly descending (ties count): the power-of-two
      // sort buffer does not fit.  Fail safe instead of overrunning shared memory: keep_count = -1, nothing kept.
      // Every CTA of a cluster sees the same scores and takes this exit together.
      if (tid == 0 && rank == 0) keep_count[img] = -1;
      for (int i = tid; i < max_boxes && rank == 0; i += NMS_THREADS) keep_index[(size_t)img * max_boxes + i] = -1;
      return;
    }
    for (int i = tid; i < m; i += NMS_THREADS)
      buf[i] = (i < n) ? (((unsigned long long)mono_key(scores[i]) << 32) | (unsigned)i) : 0ull;
    // padding keys are 0: mono_key() of any real score is >= 1, so padding sorts last
    bitonic_sort_desc(buf, m);
    for (int base = 0; base < n; base += NMS_THREADS) {
      const int i = base + tid;
      if (i < n) {   // slot i is read and rewritten by the same thread: no hazard
        const int pos = (int)(unsigned)(buf[i] & 0xffffffffull);
        order[i] = pos;
        buf[i] = reinterpret_cast<const unsigned long long*>(boxes)[pos];
      }
    }
    __syncthreads();
  }
  const BoxI16* sorted = reinterpret_cast<const BoxI16*>(buf);

  // ---- 2. tiled sweep --------------------------------------------------------------------
  const float t_f = (float)thresh;
  const bool zero_survives = (0.0 <= thresh);
  const bool fast_ok = thresh > 1e-6 && thresh < 1.0;
  const unsigned long long t_fix = fast_ok ? (unsigned long long)__double2ll_rn(thresh * 4294967296.0) : 0ull;
  const int cand = tid & (NMS_TILE - 1);
  const int slice = tid >> 6;                       // NMS_THREADS / NMS_TILE = 8 slices of the kept list
  constexpr int SLICES = NMS_THREADS / NMS_TILE;

  // largest box edge of the image -> may the pair test use 32-bit products?
  {
    int md = 0, ac = 0;
    for (int i = tid; i < n; i += NMS_THREADS) {
      const BoxI16 b = sorted[i];
      md = max(md, max(abs(b.x2 - b.x1), abs(b.y2 - b.y1)) + 1);
      ac = max(ac, max(max(abs((int)b.x1), abs((int)b.y1)), max(abs((int)b.x2), abs((int)b.y2))));
      if (b.x1 < 0 || b.y1 < 0) ac = 1 << 20;                  // the packed forms below assume non-negative coordinates
      if (b.x2 < b.x1 || b.y2 < b.y1) md = 1 << 20;          // an invalid box switches both fast paths off
    }
    md = __reduce_max_sync(0xffffffffu, md);
    ac = __reduce_max_sync(0xffffffffu, ac);
    if (lane == 0) { atomicMax(&s_maxdim, md); atomicMax(&s_maxabs, ac); }
    if (tid < NMS_TILE) row_mask[tid] = 0ull;
  }
  __syncthreads();
  // An invalid box sets s_maxdim = 2^20, which fails the bound, so `small` also means every box is valid; kept_area then
  // holds -area * p (see screen_small_valid).
  const bool small = rat_q > 0 && 3.0 * (double)s_maxdim * (double)s_maxdim * (double)max(rat_p, rat_q) < 2147483647.0;
  // ... and with coordinates below 16000 both corner pairs live in one register each and the intersection is three
  // packed 16-bit DPX instructions: (-max x1, -max y1) = VIMNMX.S16x2 of the negated lows, (min x2+1, min y2+1) =
  // VIMNMX.S16x2, (iw, ih) = relu(sum) = VIADDMNMX.S16x2.RELU; 8 ALU instructions per pair.  kept_box then holds
  // (pack(-x1,-y1), pack(x2+1,y2+1), -area*p, -) -- one 128-bit load per pair and no kept_area load.
  const bool packed = small && s_maxabs < 16000;

  int parity = 0;
  for (int base = 0; base < n; base += NMS_TILE, parity ^= 1) {
    const int tile_n = min(NMS_TILE, n - base);
    const int nkept = s_nkept;
    const int nlocal = (nkept > rank) ? (nkept - rank + cl - 1) / cl : 0;     // kept j with j % cl == rank
    // (a) candidate vs this CTA's share of the kept list
    BoxI16 cb = {0, 0, 0, 0};
    if (cand < tile_n) cb = sorted[base + cand];
    const int bx1 = cb.x1, by1 = cb.y1, bx2 = cb.x2, by2 = cb.y2;
    const int b_area = (bx2 - bx1 + 1) * (by2 - by1 + 1);
    bool sup = false;
    if (fast_ok) {
      int flags = 0;                               // bit0: suppressed by some kept box, bit1: some test uncertain
      if (packed) {
        const int bp = b_area * rat_p, pq = rat_p + rat_q;
        const unsigned nb_lo = ((unsigned)(-bx1) & 0xffffu) | ((unsigned)(-by1) << 16);
        const unsigned b_hi = ((unsigned)(bx2 + 1) & 0xffffu) | ((unsigned)(by2 + 1) << 16);
        bool hit = false;
#pragma unroll 4
        for (int j = slice; j < nlocal; j += SLICES) {
          const int4 kb = kept_box[j];
          const unsigned d = __viaddmax_s16x2_relu(__vmins2((unsigned)kb.y, b_hi), __vmins2((unsigned)kb.x, nb_lo), 0u);
          hit |= (int)(d & 0xffffu) * (int)(d >> 16) * pq + kb.z > bp;
        }
        flags = hit ? 1 : 0;
      } else if (small) {
        const int bp = b_area * rat_p, pq = rat_p + rat_q;
        bool hit = false;
#pragma unroll 4
        for (int j = slice; j < nlocal; j += SLICES) {
          const int4 kb = kept_box[j];
          hit |= screen_small_valid(kb.x, kb.y, kb.z, kb.w, kept_area[j], bx1, by1, bx2, by2, bp, pq);
        }
        flags = hit ? 1 : 0;
      } else if (rat_q > 0) {
#pragma unroll 4
        for (int j = slice; j < nlocal; j += SLICES) {
          const int4 kb = kept_box[j];
          flags |= screen_rational(kb.x, kb.y, kb.z, kb.w, kept_area[j], bx1, by1, bx2, by2, b_area, rat_p, rat_q);
        }
      } else {
#pragma unroll 4
        for (int j = slice; j < nlocal; j += SLICES) {
          const int4 kb = kept_box[j];
          flags |= screen_i16(kb.x, kb.y, kb.z, kb.w, kept_area[j], bx1, by1, bx2, by2, b_area, t_fix);
        }
      }
      sup = (flags & 1) != 0;
      if (!sup && (flags & 2)) {                   // rare: redo this candidate's share with the exact predicate
        for (int j = slice; j < nlocal; j += SLICES) {
          const int4 kb = kept_box[j];
          sup |= suppressed_i16(kb.x, kb.y, kb.z, kb.w, kept_area[j], bx1, by1, bx2, by2, b_area, t_f, thresh, zero_survives);
        }
      }
    } else {
      for (int j = slice; j < nlocal; j += SLICES) {
        const int4 kb = kept_box[j];
        sup |= suppressed_i16(kb.x, kb.y, kb.z, kb.w, kept_area[j], bx1, by1, bx2, by2, b_area, t_f, thresh, zero_survives);
      }
    }
    const unsigned ball = __ballot_sync(0xffffffffu, sup);
    if (lane == 0) sup_part[warp] = ball;
    // (b) intra-tile row masks, triangular: only the 2016 pairs i < j exist.  Rows p and 63 - p together have 63 of them;
    // 16 threads share such a row pair, four pairs each, so every warp runs four pair tests per thread instead of the
    // eight (half of them masked off) of a square 64 x 64 mapping.
    {
      const int p = tid >> 4, e0 = (tid & 15) * 4, n1 = 63 - p;
      const BoxI16 a1 = sorted[base + min(p, tile_n - 1)], a2 = sorted[base + min(63 - p, tile_n - 1)];
      const int a1_area = (a1.x2 - a1.x1 + 1) * (a1.y2 - a1.y1 + 1), a2_area = (a2.x2 - a2.x1 + 1) * (a2.y2 - a2.y1 + 1);
      unsigned lo1 = 0, hi1 = 0, lo2 = 0, hi2 = 0;
      if (packed) {
        // Packed form (coordinates in [0, 16000), valid boxes): a box is two 32-bit words as it lies in memory,
        // lo = (x1, y1), hi = (x2, y2).  With w0 = ~lo = (-x1-1, -y1-1) and w1 = hi + (2, 2):
        //   (iw, ih) = relu(min(a.w1, c.w1) + min(a.w0, c.w0))      two VIMNMX.S16x2 + one VIADDMNMX.S16x2.RELU
        // and the areas come from hi - lo + (1, 1).  ~25 instructions per pair; letting the compiler work on the `short`
        // fields produced 16-bit min/max glued together with ~100 PRMT per pair (1440 cycles per tile, clock64).
        const int pq = rat_p + rat_q;
        const uint2* sb = reinterpret_cast<const uint2*>(sorted);
        const uint2 r1 = sb[base + min(p, tile_n - 1)], r2 = sb[base + min(63 - p, tile_n - 1)];
        const unsigned d1 = r1.y - r1.x + 0x00010001u, d2 = r2.y - r2.x + 0x00010001u;
        const int na1 = -((int)(d1 & 0xffffu) * (int)(d1 >> 16) * rat_p), na2 = -((int)(d2 & 0xffffu) * (int)(d2 >> 16) * rat_p);
        const unsigned a1w0 = ~r1.x, a1w1 = r1.y + 0x00020002u, a2w0 = ~r2.x, a2w1 = r2.y + 0x00020002u;
#pragma unroll
        for (int ee = 0; ee < 4; ++ee) {
          const int e = e0 + ee;
          const bool first = e < n1;
          const int j = first ? p + 1 + e : 64 - p + (e - n1);
          const bool valid = e < 63 && j < tile_n;
          const uint2 c = sb[base + min(j, tile_n - 1)];
          const unsigned dc = c.y - c.x + 0x00010001u;
          const int c_bp = (int)(dc & 0xffffu) * (int)(dc >> 16) * rat_p;
          const unsigned d = __viaddmax_s16x2_relu(__vmins2(first ? a1w1 : a2w1, c.y + 0x00020002u),
                                                   __vmins2(first ? a1w0 : a2w0, ~c.x), 0u);
          const bool hit = (int)(d & 0xffffu) * (int)(d >> 16) * pq + (first ? na1 : na2) > c_bp;
          const unsigned bit = (valid && hit) ? 1u << (j & 31) : 0u;
          const unsigned blo = j < 32 ? bit : 0u, bhi = j < 32 ? 0u : bit;
          lo1 |= first ? blo : 0u; hi1 |= first ? bhi : 0u;
          lo2 |= first ? 0u : blo; hi2 |= first ? 0u : bhi;
        }
      } else if (small) {
        const int pq = rat_p + rat_q;
        const int na1 = -(a1_area * rat_p), na2 = -(a2_area * rat_p);
#pragma unroll
        for (int ee = 0; ee < 4; ++ee) {
          const int e = e0 + ee;
          const bool first = e < n1;
          const int j = first ? p + 1 + e : 64 - p + (e - n1);
          const bool valid = e < 63 && j < tile_n;
          const BoxI16 c = sorted[base + min(j, tile_n - 1)];
          const int cx1 = c.x1, cy1 = c.y1, cx2 = c.x2, cy2 = c.y2;
          const int c_bp = (cx2 - cx1 + 1) * (cy2 - cy1 + 1) * rat_p;
          const bool hit = screen_small_valid(first ? (int)a1.x1 : (int)a2.x1, first ? (int)a1.y1 : (int)a2.y1, first ? (int)a1.x2 : (int)a2.x2,
                                              first ? (int)a1.y2 : (int)a2.y2, first ? na1 : na2, cx1, cy1, cx2, cy2, c_bp, pq);
          const unsigned bit = (valid && hit) ? 1u << (j & 31) : 0u;
          const unsigned blo = j < 32 ? bit : 0u, bhi = j < 32 ? 0u : bit;
          lo1 |= first ? blo : 0u; hi1 |= first ? bhi : 0u;
          lo2 |= first ? 0u : blo; hi2 |= first ? 0u : bhi;
        }
      } else {
#pragma unroll
      for (int ee = 0; ee < 4; ++ee) {
        const int e = e0 + ee;
        const bool first = e < n1;                     // pair of row p, else of row 63 - p
        const int j = first ? p + 1 + e : 64 - p + (e - n1);
        if (e < 63 && j < tile_n) {                    // i < j by construction
          const BoxI16 a = first ? a1 : a2;
          const int a_area = first ? a1_area : a2_area;
          const BoxI16 c = sorted[base + j];
          const int c_area = (c.x2 - c.x1 + 1) * (c.y2 - c.y1 + 1);
          bool hit;
          if (rat_q > 0) {
            const int r = screen_rational(a.x1, a.y1, a.x2, a.y2, a_area, c.x1, c.y1, c.x2, c.y2, c_area, rat_p, rat_q);
            hit = r == 1 || (r == 2 && suppressed_i16(a.x1, a.y1, a.x2, a.y2, a_area, c.x1, c.y1, c.x2, c.y2, c_area, t_f, thresh, zero_survives));
          } else {
            hit = suppressed_i16(a.x1, a.y1, a.x2, a.y2, a_area, c.x1, c.y1, c.x2, c.y2, c_area, t_f, thresh, zero_survives);
          }
          if (hit) {
            const unsigned bit = 1u << (j & 31);
            if (first) { if (j < 32) lo1 |= bit; else hi1 |= bit; }
            else       { if (j < 32) lo2 |= bit; else hi2 |= bit; }
          }
        }
      }
      }
      // hits are rare: OR them straight into the (zeroed) row masks.  The half-warp __reduce_or_sync this replaces
      // compiles to two serialised REDUX regions per call and cost 1100 cycles per tile (clock64).
      unsigned* rm32 = reinterpret_cast<unsigned*>(row_mask);
      if (lo1) atomicOr(rm32 + 2 * p, lo1);
      if (hi1) atomicOr(rm32 + 2 * p + 1, hi1);
      if (lo2) atomicOr(rm32 + 2 * (63 - p), lo2);
      if (hi2) atomicOr(rm32 + 2 * (63 - p) + 1, hi2);
    }
    __syncthreads();
    // exchange the partial masks inside the cluster (distributed shared memory)
    if (cl > 1) {
      if (tid < cl) {
        unsigned long long loc = 0ull;
#pragma unroll
        for (int s = 0; s < SLICES; ++s)
          loc |= (unsigned long long)sup_part[2 * s] | ((unsigned long long)sup_part[2 * s + 1] << 32);
        unsigned long long* remote = cluster.map_shared_rank(&s_xpart[parity][rank], tid);
        *remote = loc;
      }
      cluster.sync();
    }
    // (c) serial resolve over live bits only, by warp 0 with the row masks in registers
    if (warp == 0) {
      unsigned long long supk = 0ull;
      if (cl > 1) {
        for (int rk = 0; rk < cl; ++rk) supk |= s_xpart[parity][rk];
      } else {
#pragma unroll
        for (int s = 0; s < SLICES; ++s)
          supk |= (unsigned long long)sup_part[2 * s] | ((unsigned long long)sup_part[2 * s + 1] << 32);
      }
      const unsigned long long rm_lo = row_mask[lane], rm_hi = row_mask[lane + 32];
      unsigned long long alive = ~supk;
      if (tile_n < 64) alive &= (1ull << tile_n) - 1ull;
      // Only candidates whose row mask hits a live candidate can change the outcome; visiting just those, in
      // order, gives the greedy result (a row mask holds later candidates only).  With few overlaps inside a tile
      // (the inference setting: 300 of the first ~330 candidates survive) this is a handful of steps instead of 64
      // dependent ones -- the other 15 warps wait at the barrier below meanwhile (37 % of the kernel's stall samples).
      int room = max_boxes - nkept;
      const unsigned act_lo = __ballot_sync(0xffffffffu, ((alive >> lane) & 1ull) && (rm_lo & alive) != 0ull);
      const unsigned act_hi = __ballot_sync(0xffffffffu, ((alive >> (lane + 32)) & 1ull) && (rm_hi & alive) != 0ull);
      unsigned long long active = ((unsigned long long)act_hi << 32) | act_lo;
      while (active) {
        const int i = __ffsll((long long)active) - 1;
        active &= active - 1ull;
        const unsigned long long rlo = __shfl_sync(0xffffffffu, rm_lo, i & 31), rhi = __shfl_sync(0xffffffffu, rm_hi, i & 31);
        if ((alive >> i) & 1ull) alive &= ~((i < 32) ? rlo : rhi);
      }
      // survivors beyond the remaining room are not picked (the sweep stops there)
      unsigned long long keepbits = room > 0 ? alive : 0ull;
      if (room > 0 && __popcll(alive) > room) {
        const unsigned lo = (unsigned)alive, hi = (unsigned)(alive >> 32);
        const int nlo = __popc(lo);
        int last;                                   // position of the room-th live bit (room >= 1 here)
        if (room <= nlo) last = (int)__fns(lo, 0, room);
        else last = 32 + (int)__fns(hi, 0, room - nlo);
        keepbits = alive & ((last >= 63) ? ~0ull : ((1ull << (last + 1)) - 1ull));
      }
      room -= __popcll(keepbits);
      if (lane == 0) {
        s_keepbits = keepbits;
        s_nkept = nkept + __popcll(keepbits);
        if (room == 0) s_stop = 1;
      }
    }
    __syncthreads();
    const unsigned long long keepbits = s_keepbits;
    if (tid < NMS_TILE && ((keepbits >> tid) & 1ull)) {
      const int slot = nkept + __popcll(keepbits & ((1ull << tid) - 1ull));
      if (slot % cl == rank) {
        if (packed)                                               // tid < 64 => cand == tid
          kept_box[slot / cl] = make_int4((int)(((unsigned)(-bx1) & 0xffffu) | ((unsigned)(-by1) << 16)),
                                          (int)(((unsigned)(bx2 + 1) & 0xffffu) | ((unsigned)(by2 + 1) << 16)), -(b_area * rat_p), 0);
        else
          kept_box[slot / cl] = make_int4(bx1, by1, bx2, by2);
        kept_area[slot / cl] = small ? -(b_area * rat_p) : b_area;
      }
      kept_slot[slot] = base + tid;
    }
    if (tid < NMS_TILE) row_mask[tid] = 0ull;         // consumed by the resolve; the next tile ORs into it
    __syncthreads();
    if (s_stop) break;
  }
  if (cl > 1) cluster.sync();      // no CTA may exit while a peer can still write into its shared memory

  // ---- 3. outputs (rank 0) ---------------------------------------------------------------
  if (rank != 0) return;
  const int total = s_nkept;
  for (int r = tid; r < max_boxes; r += NMS_THREADS) {
    const size_t o = (size_t)img * max_boxes + r;
    if (r < total) {
      const int vr = kept_slot[r];
      const int pos = unsorted ? order[vr] : vr;
      keep_index[o] = pos;
      if (keep_boxes) keep_boxes[o] = sorted[vr];
      if (keep_scores) keep_scores[o] = scores[pos];
    } else {
      keep_index[o] = -1;
      if (keep_boxes) keep_boxes[o] = BoxI16{0, 0, 0, 0};
      if (keep_scores) keep_scores[o] = 0.0f;
    }
  }
  if (tid == 0) keep_count[img] = total;
}

int launch_nms_i16(frcnn_handle* h, cudaStream_t stream, const int16_t* boxes, const float* scores,
                   const int32_t* n, int n_max, int batch, double thresh, int max_boxes,
                   int32_t* keep_index, int32_t* keep_count, int16_t* keep_boxes, float* keep_scores) {
  if (n_max > FRCNN_NMS_MAX_SORTED)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "nms_i16: n_max exceeds FRCNN_NMS_MAX_SORTED%s%s");
  // The sort path needs a power-of-two buffer; above FRCNN_NMS_MAX_UNSORTED only pre-sorted input fits.
  int pow2 = 1;
  while (pow2 < n_max) pow2 <<= 1;
  const int buf_elems = (n_max <= FRCNN_NMS_MAX_UNSORTED) ? pow2 : n_max;
  const int max_keep = max_boxes < n_max ? max_boxes : n_max;
  // cluster size: spread one image over several SMs when the kept list is long (its tests dominate) and
  // the batch alone does not fill the GPU
  int cl = 1;
  if (max_keep >= 1024) {
    // measured: 16 (non-portable cluster size) at batch 1: 0.81 -> 0.74 ms at 12000 -> 2000; 2 at batch 64
    while (cl < 16 && (long long)batch * cl * 2 <= h->sm_count) cl <<= 1;
  } else if (max_keep >= 256) {
    // inference setting (8000 -> 300): the per-tile fixed phases dominate, a cluster buys little -- 58.2 / 59.1 / 55.3 /
    // 54.2 / 55.1 us with 1 / 2 / 4 / 8 / 16 CTAs on clustered scores, 25-27 us on uniform ones -- so take up to 8
    // while SMs are idle
    while (cl < 8 && (long long)batch * cl * 2 <= h->sm_count) cl <<= 1;
  }
  const int keep_local = (max_keep + cl - 1) / cl;
  const size_t smem = align_up((size_t)buf_elems * 8, 16) + (size_t)keep_local * (16 + 4) + (size_t)max_keep * 4 + 16;
  if (smem + 2048 > (size_t)h->max_smem_optin)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "nms_i16: n_max/max_boxes need more shared memory than one SM has%s%s");
  void* ws = nullptr;
  int rc = arena_get(h, stream, (size_t)batch * cl * n_max * sizeof(int), &ws);
  if (rc) return rc;
  FRCNN_CUDA(h, cudaFuncSetAttribute(nms_i16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (cl > 8) FRCNN_CUDA(h, cudaFuncSetAttribute(nms_i16_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(batch * cl));
  cfg.blockDim = dim3(NMS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cl;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // threshold as an exact ratio of small integers (0.7 -> 7/10), if it is one: see screen_rational
  int rat_p = 0, rat_q = 0;
  if (thresh > 1e-6 && thresh < 1.0) {
    for (int q = 2; q <= 1000 && rat_q == 0; ++q) {
      const double p = nearbyint(thresh * q);
      if (p >= 1.0 && p < (double)q && p / (double)q == thresh) { rat_p = (int)p; rat_q = q; }
    }
  }
  FRCNN_CUDA(h, cudaLaunchKernelEx(&cfg, nms_i16_kernel, reinterpret_cast<const BoxI16*>(boxes), scores, n, n_max, thresh,
                                   max_boxes, max_keep, keep_local, buf_elems, cl, rat_p, rat_q, reinterpret_cast<int*>(ws), keep_index,
                                   keep_count, reinterpret_cast<BoxI16*>(keep_boxes), keep_scores));
  FRCNN_LAUNCH_CHECK(h, "nms_i16_kernel");
  return FRCNN_OK;
}

// ------------------------------------------------------------------------------------------
// float64 segmented NMS (per-class stage, voc_dets.py:72-76).  All arithmetic in IEEE double,
// no FMA contraction (explicit _rn intrinsics), same expression order as det_util.py:230-249.
// ------------------------------------------------------------------------------------------
constexpr int NMS64_THREADS = 256;

__device__ __forceinline__ bool suppressed_f64(const double4& a, double a_area, const double4& b,
                                               double b_area, double t) {
  const double iw = fmax(0.0, __dadd_rn(__dsub_rn(fmin(a.z, b.z), fmax(a.x, b.x)), 1.0));
  const double ih = fmax(0.0, __dadd_rn(__dsub_rn(fmin(a.w, b.w), fmax(a.y, b.y)), 1.0));
  const double inter = __dmul_rn(iw, ih);
  const double uni = __dsub_rn(__dadd_rn(a_area, b_area), inter);
  return !(__ddiv_rn(inter, uni) <= t);
}

// Dynamic smem: keys u64[pow2] | sorted boxes double4[n] | area double[n] | alive flags
// Simple form: candidates are visited one at a time by the whole CTA (segments are small:
// <= 320 rows in the reference's post-processing), each kept box clears later candidates.
__global__ void __launch_bounds__(NMS64_THREADS)
nms_f64_kernel(const double* __restrict__ boxes_all, const float* __restrict__ scores_all,
               const int* __restrict__ seg_offsets, int max_seg_len, int pow2, double thresh,
               int max_boxes, int out_stride, int* __restrict__ keep_index, int* __restrict__ keep_count) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem);
  double4* sb = reinterpret_cast<double4*>(smem + (size_t)pow2 * 8);
  double* area = reinterpret_cast<double*>(sb + max_seg_len);
  unsigned char* dead = reinterpret_cast<unsigned char*>(area + max_seg_len);

  const int seg = blockIdx.x, tid = threadIdx.x;
  const int start = seg_offsets[seg];
  const int n = min(seg_offsets[seg + 1] - start, max_seg_len);
  const double* boxes = boxes_all + (size_t)start * 4;
  const float* scores = scores_all + start;

  int m = 1;
  while (m < n) m <<= 1;
  for (int i = tid; i < m; i += NMS64_THREADS)
    keys[i] = (i < n) ? (((unsigned long long)mono_key(scores[i]) << 32) | (unsigned)i) : 0ull;
  bitonic_sort_desc(keys, m);
  for (int i = tid; i < n; i += NMS64_THREADS) {
    const int pos = (int)(unsigned)(keys[i] & 0xffffffffull);
    const double4 b = make_double4(boxes[4 * pos], boxes[4 * pos + 1], boxes[4 * pos + 2], boxes[4 * pos + 3]);
    sb[i] = b;
    area[i] = __dmul_rn(__dadd_rn(__dsub_rn(b.z, b.x), 1.0), __dadd_rn(__dsub_rn(b.w, b.y), 1.0));
    dead[i] = 0;
  }
  __syncthreads();

  int cur = 0, kept = 0;
  while (true) {
    // next live candidate (all threads scan the same flags -> uniform result)
    while (cur < n && dead[cur]) ++cur;
    if (cur >= n) break;
    if (tid == 0) keep_index[(size_t)seg * out_stride + kept] = (int)(unsigned)(keys[cur] & 0xffffffffull);
    ++kept;
    if (kept >= max_boxes) break;
    const double4 a = sb[cur];
    const double a_area = area[cur];
    for (int j = cur + 1 + tid; j < n; j += NMS64_THREADS)
      if (!dead[j] && suppressed_f64(a, a_area, sb[j], area[j], thresh)) dead[j] = 1;
    ++cur;
    __syncthreads();
  }
  for (int r = kept + tid; r < out_stride; r += NMS64_THREADS) keep_index[(size_t)seg * out_stride + r] = -1;
  if (tid == 0) keep_count[seg] = kept;
}

int launch_nms_f64(frcnn_handle* h, cudaStream_t stream, const double* boxes, const float* scores,
                   const int32_t* seg_offsets, int n_seg, int max_seg_len, double thresh, int max_boxes,
                   int out_stride, int32_t* keep_index, int32_t* keep_count) {
  if (max_seg_len > FRCNN_NMS_F64_MAX)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "nms_f64: segment longer than FRCNN_NMS_F64_MAX%s%s");
  int pow2 = 4;   // >= 4 keeps the double4 array behind the keys 32-byte aligned
  while (pow2 < max_seg_len) pow2 <<= 1;
  const size_t smem = (size_t)pow2 * 8 + (size_t)max_seg_len * (32 + 8 + 1) + 64;
  FRCNN_CUDA(h, cudaFuncSetAttribute(nms_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nms_f64_kernel<<<n_seg, NMS64_THREADS, smem, stream>>>(boxes, scores, seg_offsets, max_seg_len, pow2,
                                                        thresh, max_boxes, out_stride, keep_index, keep_count);
  FRCNN_LAUNCH_CHECK(h, "nms_f64_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
