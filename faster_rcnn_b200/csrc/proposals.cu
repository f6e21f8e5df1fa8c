// K-a: anchors + delta decode + sanitize + validity filter + exact top-k in sorted order, ONE kernel.
//
// proposals_kernel: a thread-block cluster of `splits` CTAs per image (up to 16).
//   1. decode   every CTA decodes 1/splits of the image's anchors (regr 16 B + cls 4 B in; a 32-bit order-preserving
//               score word + an int16x4 box out, L2-resident; the sort key of an anchor is (score word << 32) | position)
//               and histograms its score words by a 2048-bucket monotone digit in shared memory;
//   2. exchange the per-CTA histograms are summed through distributed shared memory (reduce-scatter + all-gather, two
//               cluster barriers), so every CTA knows how many keys each bucket holds in the whole image;
//   3. slice    CTA r owns the ranks [r*k/splits, (r+1)*k/splits) of the descending order.  The buckets of its two
//               bounds follow from the histogram; ONE sweep over the image's score words (128-bit loads, a thread counts
//               its hits, one warp scan + one shared atomic per warp place them) collects the CANDIDATES: every key of
//               the buckets from the lower bound's to the upper bound's.  The two exact splitters are then found among
//               the candidates only (11-bit radix passes in shared memory, both selects share one packed histogram);
//   4. sort     candidates outside the splitters become zeros and sink; 256 threads sort M = 256*E keys held E per
//               thread in registers (bitonic network unrolled at compile time: strides < E are register swaps, < 32E
//               one shuffle per key, >= 32E one shared-memory exchange with alternating buffers = one barrier);
//   5. gather   boxes / scores / indices of the slice are written at their final ranks.  Slices need no merge.
// The bucket digit is the key's top 15 bits (sign, exponent, 6 mantissa bits) taken relative to 1.0 and clamped, i.e. 64
// buckets per octave over [2^-32, 1): objectness scores are sigmoid outputs, and the plain top-11-bit digit of round 1
// resolves them into four buckets per octave only (2700-key boundary buckets on uniform scores).  Scores outside the
// window land in the two clamped end buckets; a bound that falls into one of those, or candidates that outgrow the
// buffer (massive ties), take the fall-back: exact radix selects over all keys of the image (several sweeps).
// Round 1's pair decode_kernel + topk_kernel (global histogram, memset, two launches, three sweeps per slice, one
// key per thread in the sort) took 25 us for one image and 64 us for 64 (k = 8000, CUDA-graph replay); this kernel
// takes 14 us and 40 us.
//
// Reference semantics (file:line under /root/reference/faster_rcnn):
//   det_util.py:162-175 anchors (centre = cell index, x1 = x - w//2, x2 = x1 + w)
//   util.py:111-142     float32 decode, separate roundings (this TU is built with -fmad=false)
//   det_util.py:179-192 sanitize order, :196-205 validity, :68-76/:147-155 sort + top-k + int16
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace frcnn {

struct __align__(8) BoxI16 { short x1, y1, x2, y2; };

constexpr int TOPK_BITS = 11;                       // radix digit width
constexpr int TOPK_BINS = 1 << TOPK_BITS;
constexpr int TOPK_U = 8;                           // keys fetched per thread before any is consumed (hides the L2 latency)
constexpr int SORT_T = 256;                         // threads of a CTA that run the sorting network
constexpr int FINE_SHIFT = 49;                      // bucket digit = key bits 63..49 ...
constexpr int FINE_BASE = 0x5FC0 - (TOPK_BINS - 1); // ... minus this, clamped to [0, 2047]; 0x5FC0 = those bits of 1.0f
constexpr int MAX_SPLITS = 16;                      // cluster size limit (non-portable above 8)

__device__ __forceinline__ int fine_digit(unsigned long long key) {
  const int d = (int)(key >> FINE_SHIFT) - FINE_BASE;
  return min(max(d, 0), TOPK_BINS - 1);
}
__device__ __forceinline__ unsigned long long fine_prefix(int digit) {
  return (unsigned long long)(digit + FINE_BASE) << FINE_SHIFT;
}

// unsigned division by a launch-time constant (Granlund-Montgomery round-up form, exact for all 32-bit numerators)
struct FastDiv { unsigned m, s1, s2; };
static FastDiv make_fastdiv(unsigned d) {
  FastDiv f = {0u, 0u, 0u};
  if (d <= 1) return f;
  unsigned l = 0;
  while ((1ull << l) < d) ++l;
  f.m = (unsigned)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
  f.s1 = 1;
  f.s2 = l - 1;
  return f;
}
__device__ __forceinline__ unsigned fast_div(unsigned i, FastDiv f) {
  const unsigned t = __umulhi(f.m, i);
  return (t + ((i - t) >> f.s1)) >> f.s2;
}

// x / D by the reciprocal-and-residual form of div_const (common.cuh), without its range guard
template <int D>
__device__ __forceinline__ float div_const_core(float x) {
  const float c = 1.0f / (float)D;
  const float q0 = __fmul_rn(x, c);
  return __fmaf_rn(__fmaf_rn(-(float)D, q0, x), c, q0);
}

__device__ __forceinline__ void st_shared_u64(unsigned addr, unsigned long long v) {
  asm volatile("st.shared.b64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ int atom_shared_add(unsigned addr, int v) {
  int old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
  return old;
}

// block-wide inclusive scan of one value per thread with ONE barrier: every warp scans the warp totals itself.
// `warp_tot` is [2][32] shared, `phase` alternates between the halves so that back-to-back calls need no second barrier.
template <int THREADS>
__device__ __forceinline__ unsigned block_inclusive_scan(unsigned v, unsigned (*warp_tot)[32], int& phase) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned u = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += u;
  }
  if (lane == 31) warp_tot[phase][warp] = v;
  __syncthreads();
  unsigned w = lane < THREADS / 32 ? warp_tot[phase][lane] : 0u;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned u = __shfl_up_sync(0xffffffffu, w, d);
    if (lane >= d) w += u;
  }
  const unsigned before = __shfl_sync(0xffffffffu, w, (warp + 31) & 31);
  phase ^= 1;
  return v + (warp ? before : 0u);
}

// Suffix scan over a TOPK_BINS histogram (bins counted from the top) and up to two look-ups in it: the bin that holds
// the need-th largest element (1-based), written as out[3*s + {0,1,2}] = {bin, rank of that element inside the bin,
// size of the bin}.  PACKED: the histogram carries two 16-bit counts per word (select 0 in the low half, 1 in the high
// half; no half exceeds 65535 in total), otherwise both look-ups read the whole word.  Block-wide, ends with a barrier.
template <int THREADS, bool PACKED>
__device__ __forceinline__ void hist_lookup2(const unsigned* hh, int need0, bool use0, int need1, bool use1,
                                             unsigned (*warp_tot)[32], int& phase, int* out) {
  constexpr int BPT = TOPK_BINS / THREADS;
  const int tid = threadIdx.x;
  unsigned c[BPT], sum = 0u;
#pragma unroll
  for (int j = 0; j < BPT; ++j) { c[j] = hh[TOPK_BINS - 1 - BPT * tid - j]; sum += c[j]; }
  const unsigned incl = block_inclusive_scan<THREADS>(sum, warp_tot, phase);
  const unsigned excl = incl - sum;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    if (!(s ? use1 : use0)) continue;
    const int need = s ? need1 : need0;
    const int lo = PACKED ? (int)(s ? excl >> 16 : excl & 0xffffu) : (int)excl;
    const int hi = PACKED ? (int)(s ? incl >> 16 : incl & 0xffffu) : (int)incl;
    if (lo < need && need <= hi) {                   // exactly one thread
      int e = lo;
#pragma unroll
      for (int j = 0; j < BPT; ++j) {
        const int cj = PACKED ? (int)(s ? c[j] >> 16 : c[j] & 0xffffu) : (int)c[j];
        if (need > e && need <= e + cj) { out[3 * s] = TOPK_BINS - 1 - BPT * tid - j; out[3 * s + 1] = need - e; out[3 * s + 2] = cj; }
        e += cj;
      }
    }
  }
  __syncthreads();
}

// Fall-back: exact selection over all keys of the image, the key T with exactly `need` valid keys >= T (a key is the
// score word and, below it, the anchor's position; 0 < need <= number of valid keys).  MSB-first radix select, one sweep
// per 11-bit digit.
template <int THREADS>
__device__ unsigned long long radix_select_global(const unsigned* skeys, int n, int need, unsigned* hist,
                                                  unsigned (*warp_tot)[32], int& phase, int* s_out) {
  unsigned long long prefix = 0ull;
  int hi = 64;
  while (true) {
    const int bits = hi < TOPK_BITS ? hi : TOPK_BITS, shift = hi - bits;
    for (int i = threadIdx.x; i < TOPK_BINS; i += THREADS) hist[i] = 0u;
    __syncthreads();
    for (int base = 0; base < n; base += THREADS * TOPK_U) {
      unsigned kk[TOPK_U];
#pragma unroll
      for (int u = 0; u < TOPK_U; ++u) {
        const int i = base + u * THREADS + (int)threadIdx.x;
        kk[u] = (i < n) ? __ldcg(skeys + i) : 0u;
      }
#pragma unroll
      for (int u = 0; u < TOPK_U; ++u) {
        const unsigned long long key = ((unsigned long long)kk[u] << 32) | (unsigned)(base + u * THREADS + (int)threadIdx.x);
        if (kk[u] != 0u && (hi == 64 || (key >> hi) == (prefix >> hi)))
          atomicAdd(&hist[(unsigned)((key >> shift) & (unsigned long long)((1u << bits) - 1u))], 1u);
      }
    }
    __syncthreads();
    hist_lookup2<THREADS, false>(hist, need, true, 0, false, warp_tot, phase, s_out);
    const int d = s_out[0], rest = s_out[1], cnt = s_out[2];
    __syncthreads();
    prefix |= (unsigned long long)d << shift;
    need = rest;
    hi = shift;
    if (shift == 0 || cnt == rest) break;            // bucket taken whole: the low bits are free
  }
  return prefix;
}

// shared-memory slot of logical element e: one pad entry per E elements keeps the blocked register <-> shared
// transfers (thread t owns e = t*E .. t*E+E-1) at the 2-way minimum of 64-bit accesses
template <int E>
__device__ __forceinline__ int pad_slot(int e) { return E == 1 ? e : e + e / E; }

template <int THREADS>
__device__ __forceinline__ void sort_barrier() {
  if (THREADS == SORT_T) __syncthreads();
  else asm volatile("bar.sync 1, %0;" ::"n"(SORT_T) : "memory");
}

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// Bitonic sort, descending, of M = SORT_T * E keys held E per thread (thread t owns elements t*E .. t*E+E-1) by the first
// SORT_T threads of the CTA.  The network is unrolled at compile time: strides < E are register compare-exchanges,
// strides < 32E one shuffle per key, larger strides one shared-memory exchange per key (two buffers alternate, so a
// stage costs one barrier).  Per key and stage: fetch the partner, one 64-bit compare, one predicate, two selects.
template <int THREADS, int E>
__device__ __forceinline__ void bitonic_sort_regs(unsigned long long (&v)[E], unsigned long long* buf0,
                                                  unsigned long long* buf1, int tid) {
  constexpr int M = SORT_T * E;
  int which = 0;
#pragma unroll
  for (int size = 2; size <= M; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      if (stride >= E) {
        // partner element lives in thread tid ^ (stride / E), same register index
        const bool keep_max = (((tid * E) & stride) == 0) == (((tid * E) & size) == 0);
        unsigned long long other[E];
        if (stride / E < 32) {
#pragma unroll
          for (int i = 0; i < E; ++i) other[i] = __shfl_xor_sync(0xffffffffu, v[i], stride / E);
        } else {
          unsigned long long* buf = which ? buf1 : buf0;
          which ^= 1;
#pragma unroll
          for (int i = 0; i < E; ++i) buf[pad_slot<E>(tid * E + i)] = v[i];
          sort_barrier<THREADS>();
#pragma unroll
          for (int i = 0; i < E; ++i) other[i] = buf[pad_slot<E>((tid ^ (stride / E)) * E + i)];
        }
#pragma unroll
        for (int i = 0; i < E; ++i) {
          const bool take = (v[i] < other[i]) == keep_max;
          v[i] = take ? other[i] : v[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < E; ++i) {
          if ((i & stride) == 0) {
            const bool desc = size < E ? ((i & size) == 0) : (((tid * E) & size) == 0);
            const unsigned long long a = v[i], b = v[i | stride];
            const bool swap = (a < b) == desc;
            v[i] = swap ? b : a;
            v[i | stride] = swap ? a : b;
          }
        }
      }
    }
  }
}

struct ProposalArgs {
  const float* regr;
  const float* cls;
  int rows, cols, n, k, splits, w_cap;
  FastDiv div_a, div_cols;
  unsigned* skeys;                                   // workspace [batch][n_pad]: order-preserving score words, 0 = no box;
                                                     // a sort key is (score word << 32) | position
  int n_pad;                                         // n rounded up to a multiple of 4 (128-bit loads)
  BoxI16* boxes;                                     // workspace [batch][n]
  float4* dense;                                     // optional output
  BoxI16* out_boxes;
  float* out_scores;
  int* out_index;
  int* out_count;
};

// first / last value of the keys' high words that fall into bucket d (valid keys have a non-zero high word)
__device__ __forceinline__ unsigned bucket_first(int d) { return d <= 0 ? 1u : (unsigned)(d + FINE_BASE) << (FINE_SHIFT - 32); }
__device__ __forceinline__ unsigned bucket_last(int d) {
  return d >= TOPK_BINS - 1 ? 0xffffffffu : ((unsigned)(d + FINE_BASE + 1) << (FINE_SHIFT - 32)) - 1u;
}

// RAGGED: the images of the batch are padded to one (rows, cols) map and `extents` [batch][2] (rows, cols) gives each
// image's own map, clamped to the padded one.  Cells outside it are "no box" without a load of regr / cls, boxes are
// sanitized against the image's own map, and out_index is the image's own flat index (y * cols_b + x) * A + a.  The
// sort position stays the padded index, which is monotone in the image's own one, so ties resolve as in a call on the
// cropped map.  `extents` is unused when RAGGED is false.
template <int THREADS, int E, bool RAGGED>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 1 : 4)
proposals_kernel(const ProposalArgs p, const AnchorTable tab, const int* __restrict__ extents) {
  constexpr int M = SORT_T * E;                      // sort size (power of two), >= slice length
  extern __shared__ __align__(16) unsigned long long sbuf[];      // M + SORT_T sort entries, then the candidate buffer
  __shared__ unsigned hist_own[TOPK_BINS];           // this CTA's share of the bucket histogram; later the select passes'
  __shared__ unsigned hist[TOPK_BINS];               // bucket histogram of the whole image
  __shared__ unsigned warp_tot[2][32];
  __shared__ int s_count, s_sel[6], s_total;
  __shared__ int4 s_anchor[FRCNN_MAX_ANCHORS];       // (bits of float w, bits of float h, -(w >> 1), -(h >> 1)) in feature cells

  const int splits = p.splits, n = p.n, k = p.k;
  const int img = blockIdx.x / splits, part = blockIdx.x - img * splits;
  const int tid = threadIdx.x, lane = tid & 31;
  unsigned* skeys = p.skeys + (size_t)img * p.n_pad;
  BoxI16* boxes = p.boxes + (size_t)img * n;
  cg::cluster_group cluster = cg::this_cluster();
  int phase = 0;
  int rows_b = p.rows, cols_b = p.cols;
  if (RAGGED) {
    rows_b = min(max(extents[2 * img], 0), p.rows);
    cols_b = min(max(extents[2 * img + 1], 0), p.cols);
  }

  for (int i = tid; i < TOPK_BINS; i += THREADS) hist_own[i] = 0u;
  if (tid < tab.n)
    s_anchor[tid] = make_int4(__float_as_int((float)tab.w[tid]), __float_as_int((float)tab.h[tid]), -(tab.w[tid] >> 1), -(tab.h[tid] >> 1));
  if (tid == 0) s_count = 0;
  __syncthreads();

  // ---- 1. decode this CTA's share of the anchors ----
  {
    const int chunk = (p.n_pad + splits - 1) / splits;
    const int lo = part * chunk, hi = min(p.n_pad, lo + chunk);
    const float colmax = (float)(cols_b - 1), rowmax = (float)(rows_b - 1);
    for (int i = lo + tid; i < hi; i += THREADS) {
      if (i >= n) { skeys[i] = 0u; continue; }       // padding of the last 128-bit group
      if (RAGGED) {                                  // a cell outside the image: no box, its inputs are never read
        const unsigned loc = fast_div((unsigned)i, p.div_a);
        const unsigned cy = fast_div(loc, p.div_cols);
        if ((int)cy >= rows_b || (int)loc - (int)cy * p.cols >= cols_b) { skeys[i] = 0u; continue; }
      }
      const size_t g = (size_t)img * n + i;
      const float4 r = ldg_f4(p.regr + 4 * g);
      const float score = __ldg(p.cls + g);
      const unsigned loc = fast_div((unsigned)i, p.div_a);
      const int a = i - (int)loc * tab.n;
      const unsigned cy_i = fast_div(loc, p.div_cols);
      const int cx_i = (int)loc - (int)cy_i * p.cols;
      const int4 an = s_anchor[a];

      // anchors are integer valued -> exact in float32
      float x = (float)(cx_i + an.z);
      float y = (float)((int)cy_i + an.w);
      float w = __int_as_float(an.x);     // (x + aw) - x
      float hgt = __int_as_float(an.y);

      // deltas / [10, 10, 5, 5] (util.py:118-121): one range guard for the four, the generic division outside it
      float tx = div_const_core<10>(r.x), ty = div_const_core<10>(r.y);
      float tw = div_const_core<5>(r.z), th = div_const_core<5>(r.w);
      {
        const float ax = fabsf(r.x), ay = fabsf(r.y), az = fabsf(r.z), aw4 = fabsf(r.w);
        const float mn = fminf(fminf(ax, ay), fminf(az, aw4)), mx = fmaxf(fmaxf(ax, ay), fmaxf(az, aw4));
        if (!(mn > 1e-30f && mx < 1e30f)) {
          tx = __fdiv_rn(r.x, 10.0f); ty = __fdiv_rn(r.y, 10.0f);
          tw = __fdiv_rn(r.z, 5.0f); th = __fdiv_rn(r.w, 5.0f);
        }
      }

      x = __fadd_rn(x, __fmul_rn(w, 0.5f));          // w / 2.0: exact either way
      y = __fadd_rn(y, __fmul_rn(hgt, 0.5f));
      x = __fadd_rn(x, __fmul_rn(tx, w));
      y = __fadd_rn(y, __fmul_rn(ty, hgt));
      if (fabsf(tw) <= EXP_MID_LIMIT && fabsf(th) <= EXP_MID_LIMIT) {
        w = __fmul_rn(w, np_expf_mid(tw));
        hgt = __fmul_rn(hgt, np_expf_mid(th));
      } else {                                       // huge deltas, NaN
        w = __fmul_rn(w, np_expf(tw));
        hgt = __fmul_rn(hgt, np_expf(th));
      }
      x = __fsub_rn(x, __fmul_rn(w, 0.5f));
      y = __fsub_rn(y, __fmul_rn(hgt, 0.5f));
      x = rintf(x); y = rintf(y); w = rintf(w); hgt = rintf(hgt);     // np.round: half to even
      float x2 = __fadd_rn(w, x), y2 = __fadd_rn(hgt, y);

      x2 = np_max(__fadd_rn(x, 1.0f), x2);
      y2 = np_max(__fadd_rn(y, 1.0f), y2);
      x = np_max(0.0f, x);
      y = np_max(0.0f, y);
      x2 = np_min(colmax, x2);
      y2 = np_min(rowmax, y2);

      if (p.dense) p.dense[g] = make_float4(x, y, x2, y2);

      const bool valid = (x2 > x) && (y2 > y);
      unsigned skey = 0u;
      BoxI16 b = {0, 0, 0, 0};
      if (valid) {
        // the score word of a box is never 0 (the one score pattern that maps there, a NaN, shares its neighbour's word):
        // the sweep tests validity and bucket membership on this word alone
        skey = max(mono_key(score), 1u);
        b.x1 = (short)(int)x; b.y1 = (short)(int)y; b.x2 = (short)(int)x2; b.y2 = (short)(int)y2;
        atomicAdd(&hist_own[fine_digit((unsigned long long)skey << 32)], 1u);
      }
      skeys[i] = skey;
      boxes[i] = b;
    }
  }

  // ---- 2. bucket histogram of the whole image: reduce-scatter + all-gather through distributed shared memory ----
  if (splits > 1) {
    const int bpr = (TOPK_BINS + splits - 1) / splits;                 // bins summed by one CTA
    cluster.sync();                                  // also publishes the keys and boxes to the other CTAs of the image
    const int b_lo = part * bpr, b_hi = min(TOPK_BINS, b_lo + bpr);
    for (int b = b_lo + tid; b < b_hi; b += THREADS) {
      unsigned sum = 0u;
      for (int r = 0; r < splits; ++r) sum += cluster.map_shared_rank(hist_own, r)[b];
      hist[b] = sum;
    }
    cluster.sync();
    for (int b = tid; b < TOPK_BINS; b += THREADS) {
      const int owner = b / bpr;
      if (owner != part) hist[b] = cluster.map_shared_rank(hist, owner)[b];
    }
    cluster_arrive();                                // the matching wait is the last thing the CTA does: peers may
                                                     // still be reading this CTA's `hist`, which is read-only from here on
  } else {
    __syncthreads();
    for (int b = tid; b < TOPK_BINS; b += THREADS) hist[b] = hist_own[b];
  }
  __syncthreads();
  bool cluster_pending = splits > 1;

  // ---- 3. the slice: ranks [first, last) of the descending order ----
  const int first = (int)((long long)part * k / splits);
  const int slice_end = (int)((long long)(part + 1) * k / splits);
  // one scan serves both bounds; the look-ups need n_valid (= the scan's total), so they run on saved registers
  int da = TOPK_BINS, rest_a = 0, cnt_a = 0, db = -1, rest_b = 0, cnt_b = 0;
  int n_valid, m, last;
  {
    constexpr int BPT = TOPK_BINS / THREADS;
    unsigned c[BPT], sum = 0u;
#pragma unroll
    for (int j = 0; j < BPT; ++j) { c[j] = hist[TOPK_BINS - 1 - BPT * tid - j]; sum += c[j]; }
    const int incl = (int)block_inclusive_scan<THREADS>(sum, warp_tot, phase);
    const int excl = incl - (int)sum;
    if (tid == THREADS - 1) s_total = incl;
    __syncthreads();
    n_valid = s_total;
    m = min(k, n_valid);
    last = min(slice_end, m);
    if (first < last) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int need = s ? last : first;
        if (s ? (last >= n_valid) : (first <= 0)) continue;
        if (excl < need && need <= incl) {
          int e = excl;
#pragma unroll
          for (int j = 0; j < BPT; ++j) {
            const int cj = (int)c[j];
            if (need > e && need <= e + cj) { s_sel[3 * s] = TOPK_BINS - 1 - BPT * tid - j; s_sel[3 * s + 1] = need - e; s_sel[3 * s + 2] = cj; }
            e += cj;
          }
        }
      }
    }
    __syncthreads();
  }
  unsigned long long* cand = sbuf + (M + SORT_T);    // candidate buffer: the slice plus the keys of its boundary buckets
  unsigned* hist_sel = hist_own;                     // every peer finished reading hist_own before the second cluster barrier
  unsigned long long t_hi = ~0ull, t_lo = 1ull;
  bool done = first >= last;
  int n_cand = 0;
  if (!done) {
    const bool need_hi = first > 0, need_lo = last < n_valid;
    if (need_hi) { da = s_sel[0]; rest_a = s_sel[1]; cnt_a = s_sel[2]; }
    if (need_lo) { db = s_sel[3]; rest_b = s_sel[4]; cnt_b = s_sel[5]; }
    const bool one_bucket = da == db;
    bool sel_a = need_hi && rest_a != cnt_a;         // rest == cnt: the bucket goes to one side whole, nothing to select
    bool sel_b = need_lo && rest_b != cnt_b;
    // candidates = every key of the buckets [d_first .. d_last]: everything between the two bounds, the upper bound's
    // bucket if it has to be split (otherwise it belongs to the slices above whole), and the lower bound's bucket
    // (split, or this slice's whole)
    const int d_last = sel_a ? da : da - 1;
    const int d_first = need_lo ? db : 0;
    const int extra_a = sel_a ? rest_a : 0;                  // candidates above the slice
    const int extra_b = sel_b ? cnt_b - rest_b : 0;          // ... and below it
    n_cand = (last - first) + extra_a + extra_b;
    const bool clamped = (sel_a && (da == 0 || da == TOPK_BINS - 1)) || (sel_b && (db == 0 || db == TOPK_BINS - 1));
    if (need_hi) t_hi = fine_prefix(da);
    if (need_lo) t_lo = fine_prefix(db);
    if (!clamped && n_cand <= p.w_cap && d_first <= d_last) {
      done = true;
      const unsigned h_lo = bucket_first(d_first), h_span = bucket_last(d_last) - h_lo;
      // One sweep over the image's keys.  A thread counts the candidates among its TOPK_U keys, a warp scan and one
      // shared atomic per warp place them.  Two register batches alternate, so the next batch's L2 reads are in flight
      // while this one is placed.
      const unsigned cand_s = (unsigned)__cvta_generic_to_shared(cand);
      const unsigned count_s = (unsigned)__cvta_generic_to_shared(&s_count);
      const uint4* kp = reinterpret_cast<const uint4*>(skeys) + tid;
      const int n4 = p.n_pad >> 2;
      constexpr int U4 = TOPK_U / 2;                 // 128-bit loads per thread and batch: 4 * U4 keys
      constexpr int BATCH = THREADS * U4;            // in 128-bit groups
      auto load_batch = [&](uint4 (&dst)[U4], int base) {
        if (base + BATCH <= n4) {
#pragma unroll
          for (int u = 0; u < U4; ++u) dst[u] = __ldcg(kp + base + u * THREADS);
        } else {
#pragma unroll
          for (int u = 0; u < U4; ++u) dst[u] = (base + u * THREADS + tid < n4) ? __ldcg(kp + base + u * THREADS) : make_uint4(0u, 0u, 0u, 0u);
        }
      };
      auto place_batch = [&](const uint4 (&src)[U4], int base) {
        int mine = 0;
#pragma unroll
        for (int u = 0; u < U4; ++u) {               // a zero score word (no box) is below every range: h_lo >= 1
          mine += (src[u].x - h_lo <= h_span ? 1 : 0) + (src[u].y - h_lo <= h_span ? 1 : 0) +
                  (src[u].z - h_lo <= h_span ? 1 : 0) + (src[u].w - h_lo <= h_span ? 1 : 0);
        }
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, d);
          if (lane >= d) incl += v;
        }
        int wbase = 0;
        if (lane == 31 && incl) wbase = atom_shared_add(count_s, incl);
        unsigned addr = cand_s + 8u * (unsigned)(__shfl_sync(0xffffffffu, wbase, 31) + incl - mine);
        if (mine) {
#pragma unroll
          for (int u = 0; u < U4; ++u) {
            const unsigned pos = 4u * (unsigned)(base + u * THREADS + tid);
            if (src[u].x - h_lo <= h_span) { st_shared_u64(addr, ((unsigned long long)src[u].x << 32) | pos); addr += 8u; }
            if (src[u].y - h_lo <= h_span) { st_shared_u64(addr, ((unsigned long long)src[u].y << 32) | (pos + 1u)); addr += 8u; }
            if (src[u].z - h_lo <= h_span) { st_shared_u64(addr, ((unsigned long long)src[u].z << 32) | (pos + 2u)); addr += 8u; }
            if (src[u].w - h_lo <= h_span) { st_shared_u64(addr, ((unsigned long long)src[u].w << 32) | (pos + 3u)); addr += 8u; }
          }
        }
      };
      uint4 ka[U4], kb[U4];
      load_batch(ka, 0);
      for (int base = 0; base < n4; base += 2 * BATCH) {
        load_batch(kb, base + BATCH);
        place_batch(ka, base);
        if (base + BATCH >= n4) break;
        load_batch(ka, base + 2 * BATCH);
        place_batch(kb, base + BATCH);
      }
      __syncthreads();
      // both exact splitters in one set of passes over the candidates: select A counts in the low half of the
      // histogram words, select B in the high half
      unsigned long long pa = t_hi, pb = t_lo;
      int need_a = rest_a, need_b = rest_b;
      for (int hi = FINE_SHIFT; (sel_a || sel_b) && hi > 0;) {
        const int bits = hi < TOPK_BITS ? hi : TOPK_BITS, shift = hi - bits;
        for (int i = tid; i < TOPK_BINS; i += THREADS) hist_sel[i] = 0u;
        __syncthreads();
        for (int i = tid; i < n_cand; i += THREADS) {
          const unsigned long long key = cand[i];
          unsigned add = 0u;
          if (sel_a && (key >> hi) == (pa >> hi)) add = 1u;
          if (sel_b && (key >> hi) == (pb >> hi)) add += 0x10000u;
          if (add) atomicAdd(&hist_sel[(unsigned)((key >> shift) & (unsigned long long)((1u << bits) - 1u))], add);
        }
        __syncthreads();
        hist_lookup2<THREADS, true>(hist_sel, need_a, sel_a, need_b, sel_b, warp_tot, phase, s_sel);
        if (sel_a) {
          pa |= (unsigned long long)s_sel[0] << shift;
          need_a = s_sel[1];
          if (shift == 0 || s_sel[2] == need_a) sel_a = false;         // bucket taken whole: the low bits are free
        }
        if (sel_b) {
          pb |= (unsigned long long)s_sel[3] << shift;
          need_b = s_sel[4];
          if (shift == 0 || s_sel[5] == need_b) sel_b = false;
        }
        hi = shift;
        __syncthreads();
      }
      t_hi = pa;
      t_lo = pb;
    }
  }
  if (!done) {
    // fall-back: exact splitters by radix select over all keys (keys >= t_lo and < t_hi are exactly the ranks [first, last))
    if (cluster_pending) { cluster_wait(); cluster_pending = false; }   // `hist` is about to be reused
    const bool need_hi = first > 0, need_lo = last < n_valid;
    t_hi = ~0ull;
    t_lo = 1ull;
    if (need_hi) t_hi = radix_select_global<THREADS>(skeys, n, first, hist, warp_tot, phase, s_sel);
    if (need_lo) t_lo = radix_select_global<THREADS>(skeys, n, last, hist, warp_tot, phase, s_sel);
    if (tid == 0) s_count = 0;
    __syncthreads();
    for (int base = 0; base < n; base += THREADS * TOPK_U) {
      unsigned kk[TOPK_U];
#pragma unroll
      for (int u = 0; u < TOPK_U; ++u) {
        const int i = base + u * THREADS + tid;
        kk[u] = (i < n) ? __ldcg(skeys + i) : 0u;
      }
#pragma unroll
      for (int u = 0; u < TOPK_U; ++u) {
        const unsigned long long key = ((unsigned long long)kk[u] << 32) | (unsigned)(base + u * THREADS + tid);
        const bool take = kk[u] != 0u && key >= t_lo && (first == 0 || key < t_hi);
        const unsigned ballot = __ballot_sync(0xffffffffu, take);
        int wbase = 0;
        if (lane == 0 && ballot) wbase = atomicAdd(&s_count, __popc(ballot));
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        if (take) cand[wbase + __popc(ballot & ((1u << lane) - 1u))] = key;
      }
    }
    __syncthreads();
    n_cand = first < last ? last - first : 0;
  }

  // The candidates that are not of the slice (boundary-bucket keys beyond the splitters) become zeros, the smallest
  // key: they sink behind the slice.  More than M candidates (only when the boundary buckets are large) are compacted
  // through the sort buffer first.
  const bool in_first = first == 0;
  const unsigned long long* src = cand;
  if (n_cand > M) {
    src = sbuf;
    if (tid == 0) s_count = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n_cand; i0 += THREADS) {
      const int i = i0 + tid;
      const unsigned long long key = i < n_cand ? cand[i] : 0ull;
      const bool take = key != 0ull && key >= t_lo && (in_first || key < t_hi);
      const unsigned ballot = __ballot_sync(0xffffffffu, take);
      int wbase = 0;
      if (lane == 0 && ballot) wbase = atomicAdd(&s_count, __popc(ballot));
      wbase = __shfl_sync(0xffffffffu, wbase, 0);
      if (take) sbuf[wbase + __popc(ballot & ((1u << lane) - 1u))] = key;
    }
    __syncthreads();
    n_cand = s_count;                                // = last - first
  }
  const bool compacted = src == sbuf;
  __syncthreads();

  // ---- 4. sort on the first SORT_T threads ----
  if (tid < SORT_T) {
    unsigned long long v[E];
#pragma unroll
    for (int i = 0; i < E; ++i) {
      const int j = i * SORT_T + tid;                // any assignment of candidates to sort elements will do
      const unsigned long long key = j < n_cand ? src[j] : 0ull;
      v[i] = (key >= t_lo && (in_first || key < t_hi)) ? key : 0ull;
    }
    if (compacted) sort_barrier<THREADS>();      // the network's first exchange overwrites the buffer just read
    bitonic_sort_regs<THREADS, E>(v, sbuf, cand, tid);
    sort_barrier<THREADS>();                         // the last exchange may still be read from sbuf
#pragma unroll
    for (int i = 0; i < E; ++i) sbuf[pad_slot<E>(tid * E + i)] = v[i];
  }
  __syncthreads();

  // ---- 5. gather at the final ranks ----
  const float* cls = p.cls + (size_t)img * n;
  for (int r = first + tid; r < slice_end; r += THREADS) {
    const size_t o = (size_t)img * k + r;
    if (r < last) {
      const int idx = (int)(unsigned)(sbuf[pad_slot<E>(r - first)] & 0xffffffffull);
      const uint2 bw = __ldcg(reinterpret_cast<const uint2*>(boxes + idx));   // written by a peer CTA: L2, not the read-only path
      reinterpret_cast<uint2*>(p.out_boxes)[o] = bw;
      p.out_scores[o] = __ldg(cls + idx);
      if (RAGGED) {                                  // the image's own flat anchor index
        const unsigned loc = fast_div((unsigned)idx, p.div_a);
        const unsigned cy = fast_div(loc, p.div_cols);
        const int cx = (int)loc - (int)cy * p.cols;
        p.out_index[o] = ((int)cy * cols_b + cx) * tab.n + (idx - (int)loc * tab.n);
      } else {
        p.out_index[o] = idx;
      }
    } else {
      p.out_boxes[o] = BoxI16{0, 0, 0, 0};
      p.out_scores[o] = 0.0f;
      p.out_index[o] = -1;
    }
  }
  if (tid == 0 && part == 0) p.out_count[img] = m;
  if (cluster_pending) cluster_wait();               // no CTA may exit while a peer can still read its shared memory
}

// probe_only: configure the kernel for this (cluster size, shared memory) once per handle and report whether a cluster
// of that size can be resident at all; the answer is cached in the handle, so a steady-state call is one launch.
template <int THREADS, int E, bool RAGGED>
static int launch_proposals(frcnn_handle* h, cudaStream_t stream, const ProposalArgs& args, const AnchorTable& tab,
                            const int* extents, int batch, bool probe_only) {
  const size_t smem = (size_t)(SORT_T * E + SORT_T + args.w_cap) * sizeof(unsigned long long);
  auto kernel = proposals_kernel<THREADS, E, RAGGED>;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(batch * args.splits));
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)args.splits;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (probe_only) {
    constexpr int LOG_E = E == 1 ? 0 : E == 2 ? 1 : E == 4 ? 2 : 3;
    // cudaFuncSetAttribute is per kernel function: every instance has its own entry
    unsigned char& state = h->proposals_cfg[RAGGED ? 1 : 0][THREADS == 1024 ? 1 : 0][LOG_E][args.splits];
    if (state == 0) {
      FRCNN_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      if (args.splits > 8) FRCNN_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      int clusters = 0;
      cfg.gridDim = dim3((unsigned)args.splits);
      if (cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); clusters = 0; }
      state = clusters > 0 ? 1 : 2;
    }
    return state == 1 ? FRCNN_OK : FRCNN_ERR_UNSUPPORTED;
  }
  FRCNN_CUDA(h, cudaLaunchKernelEx(&cfg, kernel, args, tab, extents));
  FRCNN_LAUNCH_CHECK(h, "proposals_kernel");
  return FRCNN_OK;
}

template <int THREADS, bool RAGGED>
static int launch_proposals_e(frcnn_handle* h, cudaStream_t stream, const ProposalArgs& args, const AnchorTable& tab,
                              const int* extents, int batch, int e, bool probe_only) {
  switch (e) {
    case 1: return launch_proposals<THREADS, 1, RAGGED>(h, stream, args, tab, extents, batch, probe_only);
    case 2: return launch_proposals<THREADS, 2, RAGGED>(h, stream, args, tab, extents, batch, probe_only);
    case 4: return launch_proposals<THREADS, 4, RAGGED>(h, stream, args, tab, extents, batch, probe_only);
    default: return launch_proposals<THREADS, 8, RAGGED>(h, stream, args, tab, extents, batch, probe_only);
  }
}

template <bool RAGGED>
static int launch_proposals_cfg(frcnn_handle* h, cudaStream_t stream, const ProposalArgs& args, const AnchorTable& tab,
                                const int* extents, int batch, int e, bool wide, bool probe_only) {
  return wide ? launch_proposals_e<1024, RAGGED>(h, stream, args, tab, extents, batch, e, probe_only)
              : launch_proposals_e<256, RAGGED>(h, stream, args, tab, extents, batch, e, probe_only);
}

int launch_decode_topk(frcnn_handle* h, cudaStream_t stream, const float* regr, const float* cls,
                       const AnchorTable& tab, int rows, int cols, int k, int batch,
                       int16_t* out_boxes, float* out_scores, int32_t* out_index,
                       int32_t* out_count, float* dense_boxes, const int32_t* extents) {
  if (extents && dense_boxes) return fail(h, FRCNN_ERR_INVALID, "decode_topk: dense_boxes is not available with extents%s%s");
  const long long n_ll = (long long)rows * cols * tab.n;
  if (n_ll >= (1ll << 31)) return fail(h, FRCNN_ERR_UNSUPPORTED, "decode_topk: more than 2^31 anchors per image%s%s");
  const int n = (int)n_ll;
  if (k > MAX_SPLITS * SORT_T * 8)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "decode_topk: k above 32768 is not supported%s%s");
  const int n_pad = (n + 3) & ~3;
  const size_t key_bytes = align_up((size_t)batch * n_pad * sizeof(unsigned), 256);
  const size_t box_bytes = align_up((size_t)batch * n * sizeof(BoxI16), 256);
  void* ws = nullptr;
  int rc = arena_get(h, stream, key_bytes + box_bytes, &ws);
  if (rc) return rc;

  ProposalArgs args;
  args.regr = regr;
  args.cls = cls;
  args.rows = rows; args.cols = cols; args.n = n; args.k = k;
  args.div_a = make_fastdiv((unsigned)tab.n);
  args.div_cols = make_fastdiv((unsigned)cols);
  args.skeys = reinterpret_cast<unsigned*>(ws);
  args.n_pad = n_pad;
  args.boxes = reinterpret_cast<BoxI16*>(reinterpret_cast<char*>(ws) + key_bytes);
  args.dense = reinterpret_cast<float4*>(dense_boxes);
  args.out_boxes = reinterpret_cast<BoxI16*>(out_boxes);
  args.out_scores = out_scores;
  args.out_index = out_index;
  args.out_count = out_count;

  // CTAs per image (= cluster size): slices of at most 1000 ranks, sorted four keys per thread.  While the GPU has SMs to
  // spare the image is spread over the largest cluster (decode, sweep and sort all shrink per CTA: 17.7 -> 14.1 us at
  // one image, k = 8000); a small k still gets enough CTAs to decode the anchors in parallel.  One CTA per SM with 1024
  // threads while batch * splits fits the SM count, 256-thread CTAs (four or more per SM) beyond.
  int splits = (k + 999) / 1000;
  const int for_decode = (n + 4095) / 4096;
  if (splits < 8 && splits < for_decode) splits = for_decode < 8 ? for_decode : 8;
  if ((long long)batch * MAX_SPLITS <= h->sm_count && n >= 4096) splits = MAX_SPLITS;
  if (splits > MAX_SPLITS) splits = MAX_SPLITS;
  // Large batches run 256-thread CTAs, four per SM (three with 2048-key sorts).  When 1000-rank slices need a second
  // wave of CTAs but 2000-rank slices fit one, take those: half the sweeps, and no 30 %-full tail wave (64 images,
  // k = 12000: 61.8 -> 49.0 us at VOC shapes, 125.9 -> 91.3 us at KITTI's 64 k anchors; k = 8000 fits one wave as it is).
  {
    const int half = (k + 1999) / 2000;
    if ((long long)batch * splits > 4LL * h->sm_count && (long long)batch * half <= 3LL * h->sm_count && half >= 1) splits = half;
  }
  // 1000-rank slices number more than 16 above k = 16000, 2000-rank ones above k = 32000
  if (splits > MAX_SPLITS) splits = MAX_SPLITS;
  const bool wide = (long long)batch * splits <= h->sm_count;
  for (;; splits = (splits + 1) / 2) {
    const int slice = (k + splits - 1) / splits;
    int e = 1;
    while (SORT_T * e < slice) e <<= 1;
    if (e > 8) return fail(h, FRCNN_ERR_UNSUPPORTED, "decode_topk: k too large for the shared-memory sort%s%s");
    args.splits = splits;
    // a cluster of sixteen 1024-thread CTAs may not fit one GPC: try the narrow CTAs before giving up slices
    for (int attempt = 0; attempt < 2; ++attempt) {
      const bool w = attempt == 0 ? wide : false;
      if (attempt == 1 && !wide) break;
      args.w_cap = w ? 6144 : (e == 8 ? 3072 : 2560);   // >= M + SORT_T: the candidate buffer doubles as the sort's second exchange buffer
      auto run = extents ? launch_proposals_cfg<true> : launch_proposals_cfg<false>;
      if (run(h, stream, args, tab, extents, batch, e, w, true) == FRCNN_OK)
        return run(h, stream, args, tab, extents, batch, e, w, false);
    }
    if (splits == 1) return fail(h, FRCNN_ERR_UNSUPPORTED, "decode_topk: no cluster configuration fits this device%s%s");
  }
}

}  // namespace frcnn
