// Device-side training mini-batch draws with a counter-based RNG (opt-in alternative to the host draws that replay the
// reference's MT19937 streams).
//
//  sample_rpn_kernel<RAGGED>  256-anchor balancing of rpn_util.py:324-350: keeps the `keep` usable anchors of each
//                             category (positive / negative) with the smallest (u_i, i) and clears can_use of the rest.
//  sample_det_kernel          64-RoI mini-batch of det_util.py:260-306 over label_rois' rows -> (B,S) row index.
//
// Random words: curand_Philox4x32_10(ctr = (j >> 2, img_lo, img_hi, tag), key = (seed_lo, seed_hi)), word j & 3, with
// (seed, offset) read from a device int64[2] and img = offset + b, so a captured graph draws fresh samples whenever the
// caller advances the offset.  Keeping the `keep` smallest of i.i.d. uniform keys picks a uniformly random subset of that
// size, i.e. the distribution of the reference's switch-off of a uniformly random complement; only the stream differs.
// Selection is an exact radix select (4 passes of 8 bits over the 32-bit keys, keys recomputed per pass) with ties on
// equal keys broken by index through an ordered CTA scan: integer arithmetic only, so oracle/sample_oracle.py
// reproduces every result bit for bit.
#include <curand_philox4x32_x.h>

#include "common.cuh"

namespace frcnn {

constexpr int SAMPLE_THREADS = 1024;
constexpr int SAMPLE_DET_ROWS = 4;                                   // label_rois rows per thread, held in registers
constexpr int SAMPLE_DET_MAX = SAMPLE_THREADS * SAMPLE_DET_ROWS;     // n_max bound of sample_det_kernel
constexpr unsigned TAG_RPN = 0, TAG_DET = 1, TAG_DET_DRAW = 2;
enum { KEEP_ALL = 0, SELECT = 1, DROP_ALL = 2 };

struct PhiloxStream {
  uint2 key;
  unsigned img_lo, img_hi;
};

__device__ __forceinline__ PhiloxStream make_stream(const int64_t* state, int b) {
  const unsigned long long seed = (unsigned long long)state[0];
  const unsigned long long img = (unsigned long long)state[1] + (unsigned long long)b;
  PhiloxStream s;
  s.key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  s.img_lo = (unsigned)img;
  s.img_hi = (unsigned)(img >> 32);
  return s;
}

// words 4*group .. 4*group+3 of stream `tag`
__device__ __forceinline__ uint4 draw4(const PhiloxStream& s, unsigned group, unsigned tag) {
  return curand_Philox4x32_10(make_uint4(group, s.img_lo, s.img_hi, tag), s.key);
}

__device__ __forceinline__ unsigned word_of(const uint4& v, int w) {
  return w == 0 ? v.x : w == 1 ? v.y : w == 2 ? v.z : v.w;
}

// Radix select of the `keep` smallest keys of two categories at once.  After the four passes prefix[c] is the keep-th
// smallest key T of category c, and rem[c] of the eq[c] elements whose key equals T are kept (the lowest indices).
struct RadixSelect {
  int hist[2][256];
  unsigned prefix[2];
  int rem[2], mode[2], eq[2];
};

__device__ __forceinline__ void select_init(RadixSelect& s, int c, int total, int keep) {
  s.mode[c] = keep >= total ? KEEP_ALL : keep <= 0 ? DROP_ALL : SELECT;
  s.prefix[c] = 0u;
  s.rem[c] = keep;
  s.eq[c] = 0;
}

__device__ __forceinline__ unsigned select_mask(int shift) { return shift == 24 ? 0u : ~0u << (shift + 8); }

__device__ __forceinline__ void select_count(RadixSelect& s, int c, unsigned key, int shift, unsigned mask) {
  if (s.mode[c] == SELECT && (key & mask) == s.prefix[c]) atomicAdd(&s.hist[c][(key >> shift) & 255u], 1);
}

// Warp c resolves category c's byte at `shift` from the histogram; then the histogram is cleared.  Contains barriers:
// every thread of the CTA calls it.
__device__ void select_resolve(RadixSelect& s, int shift) {
  __syncthreads();
  const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (c < 2 && s.mode[c] == SELECT) {                   // warp-uniform
    int h[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { h[k] = s.hist[c][8 * lane + k]; sum += h[k]; }
    int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    const int total = __shfl_sync(0xffffffffu, inc, 31), rem = s.rem[c];
    if (total < rem) {                                  // fewer candidates than `keep` (counts above the category)
      if (lane == 0) s.mode[c] = KEEP_ALL;
    } else {
      const int owner = __ffs(__ballot_sync(0xffffffffu, inc >= rem)) - 1;
      if (lane == owner) {
        int before = inc - sum, k = 0;
        while (before + h[k] < rem) before += h[k++];
        s.prefix[c] |= (unsigned)(8 * lane + k) << shift;
        s.rem[c] = rem - before;
        s.eq[c] = h[k];
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 512; i += blockDim.x) (&s.hist[0][0])[i] = 0;
  __syncthreads();
}

// Is an element of category c with key u kept?  eq_rank = number of elements of the category with the same key and a
// lower index (only read when u equals the threshold).
__device__ __forceinline__ bool select_keeps(const RadixSelect& s, int c, unsigned u, int eq_rank) {
  if (s.mode[c] != SELECT) return s.mode[c] == KEEP_ALL;
  return u < s.prefix[c] || (u == s.prefix[c] && eq_rank < s.rem[c]);
}

// Exclusive scan over the CTA in thread order; *total = the CTA's sum.  Every thread calls it.
__device__ int block_excl_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  const int excl = x - v + (warp ? s_warp[warp - 1] : 0);
  *total = s_warp[SAMPLE_THREADS / 32 - 1];
  __syncthreads();
  return excl;
}

// One CTA per image.  Thread tid takes the groups of four consecutive anchors g = tid, tid + 1024, .. (one Philox call
// each).  RAGGED: anchor i is the image's own flat index (y*cols_b + x)*A + a and lives at (y*cols + x)*A + a of the
// padded layout; padding is never read or written.
template <bool RAGGED>
__global__ void __launch_bounds__(SAMPLE_THREADS)
sample_rpn_kernel(unsigned char* __restrict__ can_use_all, const unsigned char* __restrict__ is_pos_all,
                  const int* __restrict__ counts, int n, int rows, int cols, int A, const int* __restrict__ extents,
                  int max_pos, int sample_size, const int64_t* __restrict__ state) {
  __shared__ RadixSelect s;
  __shared__ int s_warp[SAMPLE_THREADS / 32];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int n_p = max(counts[2 * img], 0), n_q = max(counts[2 * img + 1], 0);
  const int keep_p = min(n_p, max_pos), keep_q = min(n_q, sample_size - keep_p);
  if (keep_p >= n_p && keep_q >= n_q) return;          // nothing to switch off (CTA-uniform)
  int n_b = n, cols_b = cols;
  if (RAGGED) {
    const int rows_b = min(max(extents[2 * img], 0), rows);
    cols_b = min(max(extents[2 * img + 1], 0), cols);
    n_b = rows_b * cols_b * A;
  }
  unsigned char* can_use = can_use_all + (size_t)img * n;
  const unsigned char* is_pos = is_pos_all + (size_t)img * n;
  const PhiloxStream st = make_stream(state, img);
  if (tid == 0) {
    select_init(s, 0, n_p, keep_p);
    select_init(s, 1, n_q, keep_q);
  }
  for (int i = tid; i < 512; i += SAMPLE_THREADS) (&s.hist[0][0])[i] = 0;
  __syncthreads();
  const int groups = (n_b + 3) >> 2;

  auto offset = [&](int i) -> int {
    if (!RAGGED) return i;
    const int loc = i / A, a = i - loc * A, y = loc / cols_b, x = loc - y * cols_b;
    return (y * cols + x) * A + a;
  };
  // category of anchor i: 0 = usable positive, 1 = usable negative, -1 = not usable
  auto category = [&](int i, int& off) -> int {
    off = offset(i);
    if (!can_use[off]) return -1;
    return is_pos[off] ? 0 : 1;
  };

  for (int shift = 24; shift >= 0; shift -= 8) {
    if (s.mode[0] == SELECT || s.mode[1] == SELECT) {  // CTA-uniform
      const unsigned mask = select_mask(shift);
      for (int g = tid; g < groups; g += SAMPLE_THREADS) {
        const uint4 u4 = draw4(st, (unsigned)g, TAG_RPN);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const int i = 4 * g + w;
          int off;
          const int c = i < n_b ? category(i, off) : -1;
          if (c >= 0) select_count(s, c, word_of(u4, w), shift, mask);
        }
      }
    }
    select_resolve(s, shift);
  }

  // final pass in index order: the ordered scan ranks equal keys by index
  int base0 = 0, base1 = 0;
  for (int g0 = 0; g0 < groups; g0 += SAMPLE_THREADS) {
    const int g = g0 + tid;
    uint4 u4 = make_uint4(0u, 0u, 0u, 0u);
    int cat[4], off[4], n_eq0 = 0, n_eq1 = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      cat[w] = -1;
      off[w] = 0;
    }
    if (g < groups) {
      u4 = draw4(st, (unsigned)g, TAG_RPN);
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const int i = 4 * g + w;
        if (i < n_b) cat[w] = category(i, off[w]);
        if (cat[w] >= 0 && s.mode[cat[w]] == SELECT && word_of(u4, w) == s.prefix[cat[w]]) {
          n_eq0 += cat[w] == 0;
          n_eq1 += cat[w] == 1;
        }
      }
    }
    int total;
    const int pre = block_excl_scan(n_eq0 | (n_eq1 << 16), s_warp, &total);
    int rank0 = base0 + (pre & 0xffff), rank1 = base1 + (pre >> 16);
    base0 += total & 0xffff;
    base1 += total >> 16;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const int c = cat[w];
      if (c < 0) continue;
      const unsigned u = word_of(u4, w);
      const bool keep = select_keeps(s, c, u, c ? rank1 : rank0);
      if (s.mode[c] == SELECT && u == s.prefix[c]) {
        rank0 += c == 0;
        rank1 += c == 1;
      }
      if (!keep) can_use[off[w]] = 0;
    }
  }
}

// One CTA per image; thread tid holds rows 4*tid .. 4*tid+3 (keys of one Philox call in registers).
__global__ void __launch_bounds__(SAMPLE_THREADS)
sample_det_kernel(const unsigned char* __restrict__ is_pos_all, const int* __restrict__ n_rows, int n_max, int S,
                  const int64_t* __restrict__ state, int* __restrict__ out_index, unsigned char* __restrict__ out_has) {
  __shared__ RadixSelect s;
  __shared__ int s_warp[SAMPLE_THREADS / 32];
  __shared__ int s_list[SAMPLE_DET_MAX];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int m = min(max(n_rows[img], 0), n_max);
  int* out = out_index + (size_t)img * S;
  if (m == 0) {                                        // no eligible RoI: the reference returns 4 x None
    for (int t = tid; t < S; t += SAMPLE_THREADS) out[t] = -1;
    if (tid == 0) out_has[img] = 0;
    return;
  }
  const PhiloxStream st = make_stream(state, img);
  const uint4 u4 = draw4(st, (unsigned)tid, TAG_DET);
  const unsigned char* is_pos = is_pos_all + (size_t)img * n_max;
  int cat[SAMPLE_DET_ROWS], n_p = 0, n_q = 0;
#pragma unroll
  for (int w = 0; w < SAMPLE_DET_ROWS; ++w) {
    const int r = SAMPLE_DET_ROWS * tid + w;
    cat[w] = r < m ? (is_pos[r] ? 0 : 1) : -1;
    n_p += cat[w] == 0;
    n_q += cat[w] == 1;
  }
  int total;
  const int pre_all = block_excl_scan(n_p | (n_q << 16), s_warp, &total);
  const int nP = total & 0xffff, nQ = total >> 16;
  const int want_pos = S / 4;
  const int kp = nP < want_pos ? nP : want_pos;
  const int want_neg = S - kp;
  if (tid == 0) {
    select_init(s, 0, nP, kp);
    select_init(s, 1, nQ, nQ >= want_neg ? want_neg : nQ);   // too few negatives: drawn with replacement below
  }
  for (int i = tid; i < 512; i += SAMPLE_THREADS) (&s.hist[0][0])[i] = 0;
  __syncthreads();
  for (int shift = 24; shift >= 0; shift -= 8) {
    if (s.mode[0] == SELECT || s.mode[1] == SELECT) {
      const unsigned mask = select_mask(shift);
#pragma unroll
      for (int w = 0; w < SAMPLE_DET_ROWS; ++w)
        if (cat[w] >= 0) select_count(s, cat[w], word_of(u4, w), shift, mask);
    }
    select_resolve(s, shift);
  }
  int n_eq = 0;                                        // packed: positives | negatives << 16
#pragma unroll
  for (int w = 0; w < SAMPLE_DET_ROWS; ++w)
    if (cat[w] >= 0 && s.mode[cat[w]] == SELECT && word_of(u4, w) == s.prefix[cat[w]]) n_eq += cat[w] ? 0x10000 : 1;
  const int pre_eq = block_excl_scan(n_eq, s_warp, &total);
  int eq_p = pre_eq & 0xffff, eq_q = pre_eq >> 16;
  bool keep[SAMPLE_DET_ROWS];
  int n_keep = 0;
#pragma unroll
  for (int w = 0; w < SAMPLE_DET_ROWS; ++w) {
    const int c = cat[w];
    keep[w] = false;
    if (c < 0 || (c == 1 && nQ < want_neg)) continue;
    const unsigned u = word_of(u4, w);
    keep[w] = select_keeps(s, c, u, c ? eq_q : eq_p);
    if (s.mode[c] == SELECT && u == s.prefix[c]) {
      eq_p += c == 0;
      eq_q += c == 1;
    }
    if (keep[w]) n_keep += c ? 0x10000 : 1;
  }
  const int pre_keep = block_excl_scan(n_keep, s_warp, &total);
  // rows chosen without replacement: ascending row order, positives first
  int at_p = pre_keep & 0xffff, at_q = kp + (pre_keep >> 16);
  // the ascending list of the category drawn from with replacement (negatives) or tiled (positives)
  const int list_cat = nQ > 0 ? 1 : 0;
  int at_list = list_cat ? pre_all >> 16 : pre_all & 0xffff;
#pragma unroll
  for (int w = 0; w < SAMPLE_DET_ROWS; ++w) {
    const int r = SAMPLE_DET_ROWS * tid + w;
    if (keep[w]) out[cat[w] ? at_q++ : at_p++] = r;
    if (cat[w] == list_cat) s_list[at_list++] = r;
  }
  if (nQ < want_neg) {                                 // CTA-uniform
    __syncthreads();
    for (int t = tid; t < want_neg; t += SAMPLE_THREADS) {
      int row;
      if (nQ > 0) {                                    // with replacement: Q[(v_t * |Q|) >> 32], bias <= |Q| / 2^32
        const unsigned v = word_of(draw4(st, (unsigned)t >> 2, TAG_DET_DRAW), t & 3);
        row = s_list[(unsigned)(((unsigned long long)v * (unsigned)nQ) >> 32)];
      } else {                                         // np.tile(pos, want_neg // |P| + 1)[:want_neg]
        row = s_list[t % nP];
      }
      out[kp + t] = row;
    }
  }
  if (tid == 0) out_has[img] = 1;
}

int launch_sample_rpn(frcnn_handle* h, cudaStream_t stream, uint8_t* can_use, const uint8_t* is_pos,
                      const int32_t* counts, int n, int rows, int cols, int A, const int32_t* extents, int max_pos,
                      int sample_size, const int64_t* state, int batch) {
  auto kernel = extents ? sample_rpn_kernel<true> : sample_rpn_kernel<false>;
  kernel<<<batch, SAMPLE_THREADS, 0, stream>>>(can_use, is_pos, counts, n, rows, cols, A, extents, max_pos, sample_size,
                                               state);
  FRCNN_LAUNCH_CHECK(h, "sample_rpn_kernel");
  return FRCNN_OK;
}

int launch_sample_det(frcnn_handle* h, cudaStream_t stream, const uint8_t* is_pos, const int32_t* n_rows, int n_max,
                      int n_samples, const int64_t* state, int batch, int32_t* out_index, uint8_t* out_has) {
  if (n_max > SAMPLE_DET_MAX)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "sample_det: n_max above 4096 rows per image%s%s");
  sample_det_kernel<<<batch, SAMPLE_THREADS, 0, stream>>>(is_pos, n_rows, n_max, n_samples, state, out_index, out_has);
  FRCNN_LAUNCH_CHECK(h, "sample_det_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
