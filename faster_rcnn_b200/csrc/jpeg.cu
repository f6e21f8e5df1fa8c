// Baseline JPEG decode on the device, bit-exact with cv2.imdecode(buf, IMREAD_COLOR) (libjpeg-turbo's ISLOW IDCT, fancy
// upsampling and table-driven YCbCr -> BGR).  oracle/jpeg_oracle.py is the sequential restatement the tests pin.
//
//   host:   parse every header up to its scan (bounds-checked: these bytes come from outside the program) and build
//           one descriptor blob (geometry, quantisation and Huffman tables, scratch layout), uploaded with one copy
//   1..3    jpeg_unstuff_{count,scan,write}_kernel: per-byte classification of the entropy-coded data (stuffed zero,
//           fill byte, RSTn, end marker), a scan and a compaction into one clean byte stream per image plus the byte
//           offset of every restart interval
//   4       jpeg_huffman_kernel: one CTA per image; every interval is cut into SUB_BITS-bit subsequences that are
//           decoded in parallel from a guessed state and re-decoded from their predecessor's exit state until no exit
//           state changes (self-synchronisation, Weissenberger & Schmidt, ICPP 2018; a predecessor whose chain met
//           corrupt data hands over the guess instead, so one wrong guess cannot travel along the stream); scans of the per-subsequence
//           block counts and DC sums place the blocks and the DC predictors, and a last pass writes the dequantised
//           coefficients [blocks][64] int16 in natural order with absolute DCs
//   5       jpeg_idct_kernel: jpeg_idct_islow per block into per-component sample planes
//   6       jpeg_color_kernel: upsampling (h2v1 / h2v2 / h1v2 fancy, replication) and ycc_rgb_convert into the
//           image's slot of the packed output
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace frcnn {

namespace {

constexpr int FAST_BITS = 9;
constexpr uint32_t SUB_BITS = 1024;       // subsequence length of the parallel Huffman decode
constexpr int CHUNK = 4096;               // bytes per CTA of the unstuffing kernels (256 threads x 16 bytes)
constexpr int HUFF_THREADS = 512;
constexpr uint32_t ST_ERR = 0xFFFFFFFFu;  // exit state of a chain that met corrupt data

// jpeg status of an image (frcnn_jpeg_decode's `status`)
constexpr int JS_OK = 0, JS_CORRUPT = -1, JS_TRUNCATED = -2, JS_RESTART = -3, JS_SLOT = -4;

struct HuffTab {                 // libjpeg's d_derived_tbl, plus a FAST_BITS lookup
  uint16_t fast[1 << FAST_BITS];  // (length << 8) | symbol for codes of <= FAST_BITS bits, 0 = longer / absent
  int32_t maxcode[18];            // largest code of each length, -1 if none
  int32_t valoff[18];             // symbol index = code + valoff[length]
  int32_t nval;
  uint8_t val[256];
};

struct Comp {
  int h, v, hx, vx;        // sampling factors and upsampling expansion (max / own)
  int dw, dh;              // libjpeg's downsampled_width / _height
  int pw;                  // sample plane width (pixels, a multiple of 8)
  int tq;
  long long plane_off;     // byte offset of the plane in the planes scratch
};

struct Img {
  long long scan_off, file_end;    // entropy-coded data: [scan_off, file_end) of the packed files
  long long coef_base;             // first block in the coefficient scratch
  int width, height, ncomp, bpm, mcux, mcuy, ri, n_iv, iv_base;
  int sub_base, sub_cap, chunk_base, n_chunks;
  int dc_tab[3], ac_tab[3];        // global table index per component
  int8_t blk_comp[10], blk_dy[10], blk_dx[10];
  uint16_t quant[3][64];           // natural order
  Comp comp[3];
  // written on the device by the unstuffing kernels (initial values come with the upload)
  long long end_pos;               // first byte of the marker that ends the scan
  uint32_t stream_len;             // clean bytes
  int n_rst;                       // RSTn markers seen before the end
};

struct SubRec {                    // exit state of one subsequence's decode and what it decoded
  uint32_t pos;                    // bit position (ST_ERR: corrupt)
  uint16_t blk, k;
  uint32_t count;                  // blocks ended
  int32_t dc[3];                   // DC differences per component
};

struct SubPre {                    // exclusive prefixes over an image's subsequences
  uint32_t count;
  int32_t dc[3];
};

__constant__ uint8_t c_natural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                      12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                      35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                      58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
const uint8_t h_natural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ---- host: header parse ----------------------------------------------------------------------------------------------
struct HostHuff {
  uint8_t counts[16];
  uint8_t val[256];
  int nval;
};

struct Parsed {
  int width, height, ncomp, dri;
  int id[3], h[3], v[3], tq[3], td[3], ta[3];
  uint16_t qt[4][64];        // natural order
  int qt_set, ht_set;        // bit masks: qt id, (class * 4 + id)
  HostHuff ht[8];
  long long scan;            // offset of the first entropy-coded byte
};

inline int rd16(const uint8_t* p) { return (p[0] << 8) | p[1]; }

// Orientation tag of an Exif payload (after "Exif\0\0"): 1 when absent, -1 when unreadable.
int exif_orientation(const uint8_t* p, long long n) {
  if (n < 8 || !((p[0] == 'I' && p[1] == 'I') || (p[0] == 'M' && p[1] == 'M'))) return -1;
  const bool le = p[0] == 'I';
  auto u16 = [&](long long o) { return le ? (p[o] | (p[o + 1] << 8)) : ((p[o] << 8) | p[o + 1]); };
  auto u32 = [&](long long o) {
    return le ? ((uint32_t)p[o] | ((uint32_t)p[o + 1] << 8) | ((uint32_t)p[o + 2] << 16) | ((uint32_t)p[o + 3] << 24))
              : (((uint32_t)p[o] << 24) | ((uint32_t)p[o + 1] << 16) | ((uint32_t)p[o + 2] << 8) | (uint32_t)p[o + 3]);
  };
  const long long off = u32(4);
  if (off + 2 > n) return -1;
  const int cnt = u16(off);
  for (int i = 0; i < cnt; ++i) {
    const long long q = off + 2 + 12LL * i;
    if (q + 12 > n) return -1;
    if (u16(q) == 0x0112) return u16(q + 2) == 3 ? u16(q + 8) : 1;
  }
  return 1;
}

// Returns FRCNN_OK, FRCNN_ERR_UNSUPPORTED or FRCNN_ERR_INVALID (rules in include/frcnn_b200.h, frcnn_jpeg_inspect).
int parse_header(const uint8_t* d, long long n, Parsed* P) {
  memset(P, 0, sizeof(*P));
  if (!d || n < 4 || d[0] != 0xFF || d[1] != 0xD8) return FRCNN_ERR_INVALID;
  long long pos = 2;
  bool jfif = false, have_frame = false;
  int adobe = -1;
  for (;;) {
    if (pos >= n || d[pos] != 0xFF) return FRCNN_ERR_INVALID;
    while (pos < n && d[pos] == 0xFF) ++pos;
    if (pos >= n) return FRCNN_ERR_INVALID;
    const int m = d[pos++];
    if (m == 0x01 || (m >= 0xD0 && m <= 0xD9)) return FRCNN_ERR_INVALID;
    if (pos + 2 > n) return FRCNN_ERR_INVALID;
    const long long len = rd16(d + pos);
    if (len < 2 || pos + len > n) return FRCNN_ERR_INVALID;
    const uint8_t* s = d + pos + 2;
    const long long sl = len - 2;
    pos += len;
    if (m == 0xC0 || m == 0xC1) {
      if (have_frame || sl < 6) return FRCNN_ERR_INVALID;
      if (s[0] != 8) return FRCNN_ERR_UNSUPPORTED;
      const int nc = s[5];
      if (sl != 6 + 3LL * nc) return FRCNN_ERR_INVALID;
      if (nc != 1 && nc != 3) return FRCNN_ERR_UNSUPPORTED;
      P->height = rd16(s + 1);
      P->width = rd16(s + 3);
      if (P->height == 0 || P->width == 0) return FRCNN_ERR_INVALID;
      P->ncomp = nc;
      for (int c = 0; c < nc; ++c) {
        P->id[c] = s[6 + 3 * c];
        P->h[c] = s[7 + 3 * c] >> 4;
        P->v[c] = s[7 + 3 * c] & 15;
        P->tq[c] = s[8 + 3 * c];
        if (P->h[c] < 1 || P->h[c] > 4 || P->v[c] < 1 || P->v[c] > 4 || P->tq[c] > 3) return FRCNN_ERR_INVALID;
      }
      have_frame = true;
    } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4) {
      return FRCNN_ERR_UNSUPPORTED;   // progressive, lossless, hierarchical, arithmetic (SOF9.., DAC)
    } else if (m == 0xC4) {
      long long q = 0;
      while (q < sl) {
        if (q + 17 > sl) return FRCNN_ERR_INVALID;
        const int tc = s[q] >> 4, th = s[q] & 15;
        if (tc > 1 || th > 3) return FRCNN_ERR_INVALID;
        HostHuff& t = P->ht[tc * 4 + th];
        int tot = 0;
        for (int i = 0; i < 16; ++i) tot += (t.counts[i] = s[q + 1 + i]);
        if (tot > 256 || q + 17 + tot > sl) return FRCNN_ERR_INVALID;
        memcpy(t.val, s + q + 17, tot);
        t.nval = tot;
        // canonical codes must fit their lengths (jpeg_make_d_derived_tbl); DC categories are at most 15
        long long code = 0;
        for (int l = 1; l <= 16; ++l) {
          code += t.counts[l - 1];
          if (code > (1LL << l)) return FRCNN_ERR_INVALID;
          code <<= 1;
        }
        if (tc == 0)
          for (int i = 0; i < tot; ++i)
            if (t.val[i] > 15) return FRCNN_ERR_INVALID;
        P->ht_set |= 1 << (tc * 4 + th);
        q += 17 + tot;
      }
    } else if (m == 0xDB) {
      long long q = 0;
      while (q < sl) {
        const int pq = s[q] >> 4, tq = s[q] & 15;
        if (pq > 1 || tq > 3 || q + 1 + 64LL * (pq + 1) > sl) return FRCNN_ERR_INVALID;
        for (int i = 0; i < 64; ++i)
          P->qt[tq][h_natural[i]] = pq ? (uint16_t)rd16(s + q + 1 + 2 * i) : s[q + 1 + i];
        P->qt_set |= 1 << tq;
        q += 1 + 64LL * (pq + 1);
      }
    } else if (m == 0xDD) {
      if (sl != 2) return FRCNN_ERR_INVALID;
      P->dri = rd16(s);
    } else if (m == 0xDC) {
      return FRCNN_ERR_UNSUPPORTED;   // DNL
    } else if (m == 0xE0) {
      if (sl >= 14 && !memcmp(s, "JFIF\0", 5)) jfif = true;
    } else if (m == 0xE1) {
      if (sl >= 6 && !memcmp(s, "Exif\0\0", 6)) {
        const int o = exif_orientation(s + 6, sl - 6);
        if (o != 0 && o != 1) return FRCNN_ERR_UNSUPPORTED;   // rotated (or unreadable): cv2.imread applies it
      }
    } else if (m == 0xEE) {
      if (sl >= 12 && !memcmp(s, "Adobe", 5)) adobe = s[11];
    } else if (m == 0xDA) {
      if (!have_frame) return FRCNN_ERR_INVALID;
      if (sl < 1 || sl != 4 + 2LL * s[0]) return FRCNN_ERR_INVALID;
      const int ns = s[0];
      if (ns != P->ncomp) return FRCNN_ERR_UNSUPPORTED;   // one scan must carry every component
      for (int i = 0; i < ns; ++i) {
        if (s[1 + 2 * i] != P->id[i]) return FRCNN_ERR_INVALID;
        P->td[i] = s[2 + 2 * i] >> 4;
        P->ta[i] = s[2 + 2 * i] & 15;
        if (P->td[i] > 3 || P->ta[i] > 3 || !(P->ht_set >> P->td[i] & 1) || !(P->ht_set >> (4 + P->ta[i]) & 1) ||
            !(P->qt_set >> P->tq[i] & 1))
          return FRCNN_ERR_INVALID;
      }
      if (s[1 + 2 * ns] != 0 || s[2 + 2 * ns] != 63 || s[3 + 2 * ns] != 0) return FRCNN_ERR_UNSUPPORTED;
      if (P->ncomp == 3) {
        // libjpeg's colour-space guess (jdapimin.c default_decompress_parms): JFIF, else Adobe's transform, else IDs
        const bool rgb = !jfif && (adobe >= 0 ? adobe == 0 : (P->id[0] == 'R' && P->id[1] == 'G' && P->id[2] == 'B'));
        if (rgb) return FRCNN_ERR_UNSUPPORTED;
        if (P->h[1] != 1 || P->v[1] != 1 || P->h[2] != 1 || P->v[2] != 1) return FRCNN_ERR_UNSUPPORTED;
        const int hv = P->h[0] * 10 + P->v[0];
        if (hv != 11 && hv != 21 && hv != 12 && hv != 22 && hv != 41) return FRCNN_ERR_UNSUPPORTED;
      }
      P->scan = pos;
      return FRCNN_OK;
    }
    // APPn / COM / anything else with a length: skipped
  }
}

void derive_table(const HostHuff& t, HuffTab* o) {
  memset(o, 0, sizeof(*o));
  int code = 0, k = 0;
  for (int l = 1; l <= 16; ++l) {
    o->valoff[l] = k - code;
    o->maxcode[l] = t.counts[l - 1] ? code + t.counts[l - 1] - 1 : -1;
    for (int i = 0; i < t.counts[l - 1]; ++i, ++k, ++code)
      if (l <= FAST_BITS)
        for (int f = code << (FAST_BITS - l); f < (code + 1) << (FAST_BITS - l); ++f)
          o->fast[f] = (uint16_t)((l << 8) | t.val[k]);
    code <<= 1;
  }
  o->maxcode[17] = 0x7FFFFFFF;
  o->nval = t.nval;
  memcpy(o->val, t.val, t.nval);
}

// ---- device helpers --------------------------------------------------------------------------------------------------
// Exclusive scan of one value per thread over the CTA (blockDim.x a multiple of 32); *total gets the CTA's sum.
template <typename T>
__device__ T block_scan_excl(T v, T* total) {
  __shared__ T warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  T x = v;
  for (int o = 1; o < 32; o <<= 1) {
    T y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  __syncthreads();
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  if (warp == 0) {
    T w = lane < nw ? warp_sums[lane] : T(0);
    for (int o = 1; o < 32; o <<= 1) {
      T y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < nw) warp_sums[lane] = w;
  }
  __syncthreads();
  const T before = (warp ? warp_sums[warp - 1] : T(0)) + x - v;
  *total = warp_sums[nw - 1];
  __syncthreads();
  return before;
}

// Byte classes of the entropy-coded data: bit 0 = kept, bit 1 = RSTn code byte, bit 2 = code byte of another marker.
__device__ __forceinline__ int byte_class(const uint8_t* f, long long i, long long lo, long long hi) {
  const int c = f[i];
  const int prev = i > lo ? f[i - 1] : 0;
  if (prev == 0xFF && c != 0xFF) {
    if (c == 0x00) return 0;                       // stuffed zero after a data 0xFF
    return (c >= 0xD0 && c <= 0xD7) ? 2 : 4;
  }
  if (c == 0xFF) return (i + 1 < hi && f[i + 1] == 0x00) ? 1 : 0;   // data 0xFF, or fill / marker prefix
  return 1;
}

__global__ void __launch_bounds__(256) jpeg_unstuff_count_kernel(const uint8_t* __restrict__ files, Img* imgs,
                                                                 const int2* __restrict__ chunks,
                                                                 uint32_t* __restrict__ chunk_sum) {
  const int2 ch = chunks[blockIdx.x];
  Img& d = imgs[ch.x];
  const long long c0 = d.scan_off + (long long)ch.y * CHUNK;
  const long long i0 = c0 + threadIdx.x * 16, hi = d.file_end;
  uint32_t kept = 0, rst = 0;
  for (long long i = i0; i < i0 + 16 && i < hi; ++i) {
    const int cl = byte_class(files, i, d.scan_off, hi);
    kept += cl & 1;
    rst += (cl >> 1) & 1;
    if (cl & 4) atomicMin(reinterpret_cast<unsigned long long*>(&d.end_pos), (unsigned long long)i);
  }
  uint32_t tot;
  block_scan_excl<uint32_t>(kept | (rst << 16), &tot);
  if (threadIdx.x == 0) chunk_sum[blockIdx.x] = tot;
}

// One CTA per image: exclusive prefixes of its chunks' (kept, rst) counts; the stream length defaults to every kept byte
// (a scan without an end marker runs to the end of the file).
__global__ void __launch_bounds__(256) jpeg_unstuff_scan_kernel(Img* imgs, const uint32_t* __restrict__ chunk_sum,
                                                                uint2* __restrict__ chunk_pre) {
  Img& d = imgs[blockIdx.x];
  uint32_t carry_k = 0, carry_r = 0;
  for (int b = 0; b < d.n_chunks; b += blockDim.x) {
    const int j = b + threadIdx.x;
    const uint32_t s = j < d.n_chunks ? chunk_sum[d.chunk_base + j] : 0u;
    uint32_t tk, tr;
    const uint32_t ek = block_scan_excl<uint32_t>(s & 0xFFFFu, &tk);
    const uint32_t er = block_scan_excl<uint32_t>(s >> 16, &tr);
    if (j < d.n_chunks) chunk_pre[d.chunk_base + j] = make_uint2(carry_k + ek, carry_r + er);
    carry_k += tk;
    carry_r += tr;
  }
  if (threadIdx.x == 0) d.stream_len = carry_k;
}

__global__ void __launch_bounds__(256) jpeg_unstuff_write_kernel(const uint8_t* __restrict__ files, Img* imgs,
                                                                 const int2* __restrict__ chunks,
                                                                 const uint2* __restrict__ chunk_pre,
                                                                 uint8_t* __restrict__ clean, uint32_t* __restrict__ iv_start) {
  const int2 ch = chunks[blockIdx.x];
  Img& d = imgs[ch.x];
  const long long c0 = d.scan_off + (long long)ch.y * CHUNK;
  const long long i0 = c0 + threadIdx.x * 16, hi = d.file_end, end = d.end_pos;
  int cls[16];
  uint32_t kept = 0, rst = 0;
#pragma unroll
  for (int t = 0; t < 16; ++t) {
    const long long i = i0 + t;
    cls[t] = i < hi ? byte_class(files, i, d.scan_off, hi) : 0;
    kept += cls[t] & 1;
    rst += (cls[t] >> 1) & 1;
  }
  uint32_t tot;
  const uint32_t ex = block_scan_excl<uint32_t>(kept | (rst << 16), &tot);
  uint32_t pk = chunk_pre[blockIdx.x].x + (ex & 0xFFFFu), pr = chunk_pre[blockIdx.x].y + (ex >> 16);
  uint8_t* out = clean + d.scan_off;
#pragma unroll
  for (int t = 0; t < 16; ++t) {
    const long long i = i0 + t;
    if (i >= end) break;
    if (cls[t] & 1) out[pk++] = files[i];
    if (cls[t] & 2) {
      if (pr + 1 < (uint32_t)d.n_iv) iv_start[d.iv_base + pr + 1] = pk;
      atomicMax(&d.n_rst, (int)pr + 1);
      ++pr;
    }
  }
  if (i0 <= end && end < i0 + 16 && end < hi) d.stream_len = pk;   // pk = kept bytes before the end marker
}

// ---- Huffman decode --------------------------------------------------------------------------------------------------
struct BitReader {
  const uint8_t* s;
  uint32_t n, next;
  uint64_t buf;
  int cnt;
  __device__ void init(const uint8_t* s_, uint32_t n_, uint32_t pos) {
    s = s_;
    n = n_;
    next = pos >> 3;
    buf = 0;
    cnt = 0;
    refill();
    buf <<= (pos & 7);
    cnt -= (pos & 7);
  }
  __device__ __forceinline__ void refill() {
    while (cnt <= 56) {
      const uint64_t b = next < n ? s[next] : 0u;   // zeros past the interval's end (never consumed: see run)
      ++next;
      buf |= b << (56 - cnt);
      cnt += 8;
    }
  }
};

__device__ __forceinline__ int huff_symbol(const HuffTab* t, uint32_t top16, int* len) {
  const uint32_t f = t->fast[top16 >> (16 - FAST_BITS)];
  if (f) {
    *len = f >> 8;
    return f & 0xFF;
  }
  for (int l = FAST_BITS + 1; l <= 16; ++l) {
    const int code = top16 >> (16 - l);
    if (code <= t->maxcode[l]) {
      const int idx = code + t->valoff[l];
      if (idx < 0 || idx >= t->nval) return -1;
      *len = l;
      return t->val[idx];
    }
  }
  return -1;
}

// Decode from (pos, blk, k) while pos < stop and fewer than max_blocks blocks have ended; a symbol that would reach past
// the interval's last bit stops the run before it.  WRITE = false: count ended blocks and sum DC differences per
// component.  WRITE = true: write dequantised coefficients of block `blk_out` on, DC made absolute with `dc`.
// Returns false on a code missing from its table or a coefficient index past 63.
template <bool WRITE>
__device__ bool run(const Img& d, const HuffTab* __restrict__ tabs, const uint8_t* s, uint32_t nbytes, uint32_t& pos,
                    int& blk, int& k, uint32_t stop, uint32_t max_blocks, uint32_t& nblk, int dc[3], int16_t* coef) {
  const uint32_t nbits = nbytes * 8u;
  BitReader r;
  r.init(s, nbytes, pos);
  while (pos < stop && nblk < max_blocks) {
    r.refill();
    const int comp = d.blk_comp[blk];
    const HuffTab* t = &tabs[k == 0 ? d.dc_tab[comp] : d.ac_tab[comp]];
    int len;
    const int sym = huff_symbol(t, (uint32_t)(r.buf >> 48), &len);
    if (sym < 0) {
      if (nbits - pos < 16) break;   // the lookup window reaches past the data: padding, not a code
      return false;
    }
    const int rr = k ? sym >> 4 : 0, ss = k ? sym & 15 : sym;
    if (pos + len + ss > nbits) break;
    const uint64_t rest = r.buf << len;
    const int raw = ss ? (int)(rest >> (64 - ss)) : 0;
    const int v = (ss && raw < (1 << (ss - 1))) ? raw - (1 << ss) + 1 : raw;
    r.buf = rest << ss;
    r.cnt -= len + ss;
    pos += len + ss;
    const uint16_t* q = d.quant[comp];
    if (k == 0) {
      dc[comp] += v;
      if (WRITE) coef[0] = (int16_t)((int16_t)dc[comp] * (int)q[0]);
      k = 1;
    } else if (ss) {
      if (k + rr > 63) return false;
      if (WRITE)
        for (int z = k; z < k + rr; ++z) coef[c_natural[z]] = 0;
      k += rr;
      if (WRITE) coef[c_natural[k]] = (int16_t)(v * (int)q[c_natural[k]]);
      ++k;
    } else if (rr == 15) {
      if (k + 16 > 64) return false;
      if (WRITE)
        for (int z = k; z < k + 16; ++z) coef[c_natural[z]] = 0;
      k += 16;
    } else {
      if (WRITE)
        for (int z = k; z < 64; ++z) coef[c_natural[z]] = 0;
      k = 64;
    }
    if (k >= 64) {
      k = 0;
      blk = blk + 1 == d.bpm ? 0 : blk + 1;
      ++nblk;
      if (WRITE) coef += 64;
    }
  }
  return true;
}

__device__ __forceinline__ uint32_t iv_bytes(const Img& d, const uint32_t* iv_start, int k) {
  const uint32_t a = iv_start[d.iv_base + k];
  const uint32_t b = k + 1 < d.n_iv ? iv_start[d.iv_base + k + 1] : d.stream_len;
  return b > a ? b - a : 0u;
}

__device__ SubRec decode_sub(const Img& d, const HuffTab* tabs, const uint8_t* clean, const uint32_t* iv_start, int k,
                             uint32_t local, uint32_t pos, int blk, int kk) {
  SubRec o;
  o.count = 0;
  o.dc[0] = o.dc[1] = o.dc[2] = 0;
  const uint32_t nb = iv_bytes(d, iv_start, k);
  const uint32_t stop = min((local + 1) * SUB_BITS, nb * 8u);
  const bool ok = run<false>(d, tabs, clean + d.scan_off + iv_start[d.iv_base + k], nb, pos, blk, kk, stop, 0xFFFFFFFFu,
                             o.count, o.dc, nullptr);
  o.pos = ok ? pos : ST_ERR;
  o.blk = (uint16_t)blk;
  o.k = (uint16_t)kk;
  return o;
}

__global__ void __launch_bounds__(HUFF_THREADS) jpeg_huffman_kernel(const Img* __restrict__ imgs,
                                                                    const HuffTab* __restrict__ tabs,
                                                                    const uint8_t* __restrict__ clean,
                                                                    uint32_t* __restrict__ iv_start,
                                                                    uint32_t* __restrict__ sub_off, uint32_t* __restrict__ sub_iv,
                                                                    SubRec* __restrict__ rec_a, SubRec* __restrict__ rec_b,
                                                                    uint8_t* __restrict__ chg_a, uint8_t* __restrict__ chg_b,
                                                                    SubPre* __restrict__ pre, int16_t* __restrict__ coef,
                                                                    const int64_t* __restrict__ out_offsets,
                                                                    long long out_bytes, int32_t* __restrict__ status) {
  const Img& d = imgs[blockIdx.x];
  __shared__ int s_flag[2];
  __shared__ int s_err;
  const int tid = threadIdx.x, nt = blockDim.x;
  {
    const long long o = out_offsets[blockIdx.x];
    if (o < 0 || o > out_bytes || out_bytes - o < 3LL * d.width * d.height) {
      if (tid == 0) status[blockIdx.x] = JS_SLOT;
      return;
    }
  }
  if (d.n_rst != d.n_iv - 1) {
    if (tid == 0) status[blockIdx.x] = JS_RESTART;
    return;
  }
  const int n_iv = d.n_iv;
  uint32_t* soff = sub_off + d.iv_base;
  // subsequences per interval and their offsets
  uint32_t carry = 0;
  for (int b = 0; b < n_iv; b += nt) {
    const int k = b + tid;
    const uint32_t ns = k < n_iv ? max(1u, (iv_bytes(d, iv_start, k) * 8u + SUB_BITS - 1) / SUB_BITS) : 0u;
    uint32_t tot;
    const uint32_t ex = block_scan_excl<uint32_t>(ns, &tot);
    if (k < n_iv) soff[k] = carry + ex;
    carry += tot;
  }
  const uint32_t n_sub = carry;
  if (tid == 0) s_err = 0;
  if (n_sub > (uint32_t)d.sub_cap) {   // cannot happen for a consistent layout; never write past the capacity
    if (tid == 0) status[blockIdx.x] = JS_CORRUPT;
    return;
  }
  __syncthreads();
  uint32_t* siv = sub_iv + d.sub_base;
  for (int k = tid; k < n_iv; k += nt) {
    const uint32_t a = soff[k], b = k + 1 < n_iv ? soff[k + 1] : n_sub;
    for (uint32_t j = a; j < b; ++j) siv[j] = k;
  }
  __syncthreads();
  SubRec* cur = rec_a + d.sub_base;
  SubRec* nxt = rec_b + d.sub_base;
  uint8_t* ccur = chg_a + d.sub_base;
  uint8_t* cnxt = chg_b + d.sub_base;
  // phase 1: every subsequence from a guessed state (its first bit, block 0, coefficient 0)
  for (uint32_t j = tid; j < n_sub; j += nt) {
    const int k = siv[j];
    const uint32_t local = j - soff[k];
    cur[j] = decode_sub(d, tabs, clean, iv_start, k, local, local * SUB_BITS, 0, 0);
    ccur[j] = 1;
  }
  // synchronisation: re-decode j from j-1's exit state while that changed; the fixed point is the sequential decode
  if (tid == 0) s_flag[0] = s_flag[1] = 0;
  int it = 0;
  for (;;) {
    __syncthreads();
    for (uint32_t j = tid; j < n_sub; j += nt) {
      const int k = siv[j];
      const uint32_t local = j - soff[k];
      SubRec r = cur[j];
      uint8_t ch = 0;
      if (local > 0 && ccur[j - 1]) {
        const SubRec p = cur[j - 1];
        SubRec q;
        // a predecessor that met corrupt data was a wrong guess (or the file is corrupt, which its own state shows
        // at the fixed point): restart from this subsequence's guess, so an error never travels along the stream
        if (p.pos == ST_ERR) q = decode_sub(d, tabs, clean, iv_start, k, local, local * SUB_BITS, 0, 0);
        else q = decode_sub(d, tabs, clean, iv_start, k, local, p.pos, p.blk, p.k);
        ch = q.pos != r.pos || q.blk != r.blk || q.k != r.k;
        r = q;
      }
      nxt[j] = r;
      cnxt[j] = ch;
      if (ch) s_flag[it & 1] = 1;
    }
    __syncthreads();
    const int any = s_flag[it & 1];
    if (tid == 0) s_flag[(it + 1) & 1] = 0;
    SubRec* t = cur; cur = nxt; nxt = t;
    uint8_t* tc = ccur; ccur = cnxt; cnxt = tc;
    ++it;
    if (!any) break;
    if (it > (int)n_sub + 1) {   // a fixed point is reached within n_sub iterations; never spin past that
      if (tid == 0) status[blockIdx.x] = JS_CORRUPT;
      return;
    }
  }
  // exclusive scans of block counts and DC sums (image-wide; interval-relative values subtract the first subsequence's)
  SubPre* P = pre + d.sub_base;
  uint32_t cc = 0;
  int cd0 = 0, cd1 = 0, cd2 = 0;
  for (uint32_t b = 0; b < n_sub; b += nt) {
    const uint32_t j = b + tid;
    SubRec r;
    if (j < n_sub) r = cur[j];
    else { r.pos = 0; r.count = 0; r.dc[0] = r.dc[1] = r.dc[2] = 0; }
    if (j < n_sub && r.pos == ST_ERR) s_err = JS_CORRUPT;
    uint32_t t0;
    int t1, t2, t3;
    const uint32_t e0 = block_scan_excl<uint32_t>(r.count, &t0);
    const int e1 = block_scan_excl<int>(r.dc[0], &t1);
    const int e2 = block_scan_excl<int>(r.dc[1], &t2);
    const int e3 = block_scan_excl<int>(r.dc[2], &t3);
    if (j < n_sub) {
      SubPre p;
      p.count = cc + e0;
      p.dc[0] = cd0 + e1;
      p.dc[1] = cd1 + e2;
      p.dc[2] = cd2 + e3;
      P[j] = p;
    }
    cc += t0;
    cd0 += t1;
    cd1 += t2;
    cd2 += t3;
  }
  __syncthreads();
  const int n_mcu = d.mcux * d.mcuy;
  for (int k = tid; k < n_iv; k += nt) {
    const uint32_t a = soff[k], b = k + 1 < n_iv ? soff[k + 1] : n_sub;
    const uint32_t got = (b < n_sub ? P[b].count : cc) - P[a].count;
    const uint32_t want = (uint32_t)min(d.ri, n_mcu - k * d.ri) * d.bpm;
    if (got < want) atomicMin(&s_err, JS_TRUNCATED);
  }
  __syncthreads();
  if (s_err) {
    if (tid == 0) status[blockIdx.x] = s_err;
    return;
  }
  // final pass: the coefficients
  for (uint32_t j = tid; j < n_sub; j += nt) {
    const int k = siv[j];
    const uint32_t first = soff[k], local = j - first;
    const uint32_t rel = P[j].count - P[first].count;
    const uint32_t want = (uint32_t)min(d.ri, n_mcu - k * d.ri) * d.bpm;
    if (rel >= want) continue;
    uint32_t pos = 0;
    int blk = 0, kk = 0;
    if (local > 0) {
      const SubRec p = cur[j - 1];
      pos = p.pos;
      blk = p.blk;
      kk = p.k;
    }
    int dc[3] = {P[j].dc[0] - P[first].dc[0], P[j].dc[1] - P[first].dc[1], P[j].dc[2] - P[first].dc[2]};
    const uint32_t nb = iv_bytes(d, iv_start, k);
    uint32_t nblk = 0;
    int16_t* out = coef + (d.coef_base + (long long)k * d.ri * d.bpm + rel) * 64;
    run<true>(d, tabs, clean + d.scan_off + iv_start[d.iv_base + k], nb, pos, blk, kk, min((local + 1) * SUB_BITS, nb * 8u),
              want - rel, nblk, dc, out);
  }
  if (tid == 0) status[blockIdx.x] = JS_OK;
}

// ---- IDCT, upsampling, colour ----------------------------------------------------------------------------------------
__device__ __forceinline__ void idct_1d(int in[8], int out[8], int shift) {
  const int z2 = in[2], z3 = in[6];
  int z1 = (z2 + z3) * 4433;
  const int tmp2 = z1 + z3 * -15137, tmp3 = z1 + z2 * 6270;
  const int tmp0e = (in[0] + in[4]) * 8192, tmp1e = (in[0] - in[4]) * 8192;
  const int tmp10 = tmp0e + tmp3, tmp13 = tmp0e - tmp3, tmp11 = tmp1e + tmp2, tmp12 = tmp1e - tmp2;
  int t0 = in[7], t1 = in[5], t2 = in[3], t3 = in[1];
  z1 = t0 + t3;
  int zz2 = t1 + t2, zz3 = t0 + t2, z4 = t1 + t3;
  const int z5 = (zz3 + z4) * 9633;
  t0 *= 2446;
  t1 *= 16819;
  t2 *= 25172;
  t3 *= 12299;
  z1 *= -7373;
  zz2 *= -20995;
  zz3 = zz3 * -16069 + z5;
  z4 = z4 * -3196 + z5;
  t0 += z1 + zz3;
  t1 += zz2 + z4;
  t2 += zz2 + zz3;
  t3 += z1 + z4;
  const int rnd = 1 << (shift - 1);
  out[0] = (tmp10 + t3 + rnd) >> shift;
  out[7] = (tmp10 - t3 + rnd) >> shift;
  out[1] = (tmp11 + t2 + rnd) >> shift;
  out[6] = (tmp11 - t2 + rnd) >> shift;
  out[2] = (tmp12 + t1 + rnd) >> shift;
  out[5] = (tmp12 - t1 + rnd) >> shift;
  out[3] = (tmp13 + t0 + rnd) >> shift;
  out[4] = (tmp13 - t0 + rnd) >> shift;
}

// libjpeg's post-IDCT range_limit[x & 1023]
__device__ __forceinline__ uint32_t range_limit(int x) { return (uint32_t)min(max((((x + 512) & 1023) - 512) + 128, 0), 255); }

__global__ void __launch_bounds__(128) jpeg_idct_kernel(const Img* __restrict__ imgs, const int16_t* __restrict__ coef,
                                                        const int32_t* __restrict__ status, uint8_t* __restrict__ planes) {
  const Img& d = imgs[blockIdx.y];
  if (status[blockIdx.y] != JS_OK) return;
  const long long nblocks = (long long)d.mcux * d.mcuy * d.bpm;
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblocks) return;
  const int m = (int)(b / d.bpm), i = (int)(b % d.bpm);
  const int c = d.blk_comp[i];
  const Comp& cp = d.comp[c];
  const int my = m / d.mcux, mx = m % d.mcux;
  const int by = d.bpm > 1 ? my * cp.v + d.blk_dy[i] : my, bx = d.bpm > 1 ? mx * cp.h + d.blk_dx[i] : mx;
  const int4* src = reinterpret_cast<const int4*>(coef + (d.coef_base + b) * 64);
  int ws[64];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int4 v = src[r];
    const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      ws[r * 8 + 2 * q] = (int)(int16_t)(w[q] & 0xFFFF);
      ws[r * 8 + 2 * q + 1] = (int)(int16_t)((uint32_t)w[q] >> 16);
    }
  }
  // pass 1: columns (CONST_BITS - PASS1_BITS = 11)
#pragma unroll
  for (int col = 0; col < 8; ++col) {
    int in[8], out[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) in[r] = ws[r * 8 + col];
    idct_1d(in, out, 11);
#pragma unroll
    for (int r = 0; r < 8; ++r) ws[r * 8 + col] = out[r];
  }
  // pass 2: rows (CONST_BITS + PASS1_BITS + 3 = 18), range limit, 8 bytes per row
  uint8_t* dst = planes + cp.plane_off + (long long)by * 8 * cp.pw + bx * 8;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    int out[8];
    idct_1d(&ws[r * 8], out, 18);
    uint2 pk;
    pk.x = range_limit(out[0]) | (range_limit(out[1]) << 8) | (range_limit(out[2]) << 16) | (range_limit(out[3]) << 24);
    pk.y = range_limit(out[4]) | (range_limit(out[5]) << 8) | (range_limit(out[6]) << 16) | (range_limit(out[7]) << 24);
    *reinterpret_cast<uint2*>(dst + (long long)r * cp.pw) = pk;
  }
}

// Sample of component c at output pixel (y, x) after libjpeg-turbo's upsampler (jdsample.c): full size, h2v1 / h2v2
// fancy (replication when downsampled_width <= 2), h1v2 fancy, int_upsample (4:1:1).  Context rows are clamped to
// [0, downsampled_height - 1] and columns to [0, downsampled_width - 1], libjpeg's edge rules.
__device__ __forceinline__ int upsampled(const Comp& c, const uint8_t* p, int y, int x) {
  if (c.hx == 1 && c.vx == 1) return p[(long long)y * c.pw + x];
  if (c.hx == 4 || (c.hx == 2 && c.dw <= 2)) return p[(long long)(y / c.vx) * c.pw + x / c.hx];
  const int r = c.vx == 2 ? y >> 1 : y;
  const uint8_t* row = p + (long long)r * c.pw;
  if (c.vx == 2) {
    const int nb = (y & 1) ? min(r + 1, c.dh - 1) : max(r - 1, 0);
    const uint8_t* row2 = p + (long long)nb * c.pw;
    if (c.hx == 1) return (3 * row[x] + row2[x] + ((y & 1) ? 2 : 1)) >> 2;
    const int i = x >> 1, o = (x & 1) ? min(i + 1, c.dw - 1) : max(i - 1, 0);
    const int ci = 3 * row[i] + row2[i], co = 3 * row[o] + row2[o];
    return (3 * ci + co + ((x & 1) ? 7 : 8)) >> 4;
  }
  const int i = x >> 1, o = (x & 1) ? min(i + 1, c.dw - 1) : max(i - 1, 0);
  return (3 * row[i] + row[o] + ((x & 1) ? 2 : 1)) >> 2;
}

__global__ void __launch_bounds__(256) jpeg_color_kernel(const Img* __restrict__ imgs, const uint8_t* __restrict__ planes,
                                                         const int32_t* __restrict__ status,
                                                         const int64_t* __restrict__ out_offsets, uint8_t* __restrict__ out) {
  const Img& d = imgs[blockIdx.y];
  const int st = status[blockIdx.y];
  if (st == JS_SLOT) return;
  const long long npix = (long long)d.width * d.height;
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  uint8_t* o = out + out_offsets[blockIdx.y] + 3 * p;
  if (st != JS_OK) {
    o[0] = o[1] = o[2] = 0;
    return;
  }
  const int y = (int)(p / d.width), x = (int)(p % d.width);
  const int Y = upsampled(d.comp[0], planes + d.comp[0].plane_off, y, x);
  if (d.ncomp == 1) {
    o[0] = o[1] = o[2] = (uint8_t)Y;
    return;
  }
  const int cb = upsampled(d.comp[1], planes + d.comp[1].plane_off, y, x) - 128;
  const int cr = upsampled(d.comp[2], planes + d.comp[2].plane_off, y, x) - 128;
  // jdcolor.c build_ycc_rgb_table / ycc_rgb_convert (SCALEBITS 16)
  const int r = Y + ((91881 * cr + 32768) >> 16);
  const int g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
  const int b = Y + ((116130 * cb + 32768) >> 16);
  o[0] = (uint8_t)min(max(b, 0), 255);
  o[1] = (uint8_t)min(max(g, 0), 255);
  o[2] = (uint8_t)min(max(r, 0), 255);
}

}  // namespace

int jpeg_inspect(const uint8_t* file, long long n, int32_t* hw) {
  Parsed P;
  const int rc = parse_header(file, n, &P);
  if (rc == FRCNN_OK && hw) {
    hw[0] = P.height;
    hw[1] = P.width;
  }
  return rc;
}

int launch_jpeg_decode(frcnn_handle* h, cudaStream_t stream, const uint8_t* files_host, const uint8_t* files,
                       const int64_t* file_offsets_host, const int64_t* file_bytes_host, int batch, uint8_t* out,
                       const int64_t* out_offsets, long long out_bytes, int32_t* status) {
  std::vector<Img> imgs(batch);
  std::vector<HuffTab> tabs;
  std::vector<int2> chunks;
  long long total_blocks = 0, plane_bytes = 0, total_file_end = 0;
  int total_iv = 0, total_sub = 0;
  int max_blocks = 0;
  long long max_pix = 0;
  for (int b = 0; b < batch; ++b) {
    Parsed P;
    const long long off = file_offsets_host[b], nb = file_bytes_host[b];
    if (off < 0 || nb <= 0) return fail(h, FRCNN_ERR_INVALID, "jpeg_decode: a file has no bytes%s%s");
    const int rc = parse_header(files_host + off, nb, &P);
    if (rc) return fail(h, rc, rc == FRCNN_ERR_UNSUPPORTED ? "jpeg_decode: unsupported file%s%s" : "jpeg_decode: invalid header%s%s");
    Img& d = imgs[b];
    memset(&d, 0, sizeof(d));
    d.width = P.width;
    d.height = P.height;
    d.ncomp = P.ncomp;
    int hm = 1, vm = 1;
    for (int c = 0; c < P.ncomp; ++c) {
      hm = std::max(hm, P.h[c]);
      vm = std::max(vm, P.v[c]);
    }
    // tables: DC and AC per component, shared within the image when the ids repeat
    int tab_of[8];
    for (int i = 0; i < 8; ++i) tab_of[i] = -1;
    for (int c = 0; c < P.ncomp; ++c) {
      const int ids[2] = {P.td[c], 4 + P.ta[c]};
      for (int cls = 0; cls < 2; ++cls) {
        int& t = tab_of[ids[cls]];
        if (t < 0) {
          t = (int)tabs.size();
          tabs.emplace_back();
          derive_table(P.ht[ids[cls]], &tabs.back());
        }
        (cls ? d.ac_tab : d.dc_tab)[c] = t;
      }
      memcpy(d.quant[c], P.qt[P.tq[c]], sizeof(d.quant[c]));
    }
    if (P.ncomp == 1) {
      Comp& c = d.comp[0];
      c.h = c.v = c.hx = c.vx = 1;
      const int wb = (int)((P.width * (long long)P.h[0] + hm * 8 - 1) / (hm * 8));
      const int hb = (int)((P.height * (long long)P.v[0] + vm * 8 - 1) / (vm * 8));
      d.mcux = wb;
      d.mcuy = hb;
      d.bpm = 1;
      d.blk_comp[0] = 0;
      c.dw = P.width;
      c.dh = P.height;
      c.pw = wb * 8;
      c.plane_off = plane_bytes;
      plane_bytes += align_up((size_t)c.pw * hb * 8, 256);
    } else {
      d.mcux = (P.width + 8 * hm - 1) / (8 * hm);
      d.mcuy = (P.height + 8 * vm - 1) / (8 * vm);
      int i = 0;
      for (int ci = 0; ci < 3; ++ci) {
        Comp& c = d.comp[ci];
        c.h = P.h[ci];
        c.v = P.v[ci];
        c.hx = hm / c.h;
        c.vx = vm / c.v;
        c.dw = (int)((P.width * (long long)c.h + hm - 1) / hm);
        c.dh = (int)((P.height * (long long)c.v + vm - 1) / vm);
        c.pw = d.mcux * c.h * 8;
        c.plane_off = plane_bytes;
        plane_bytes += align_up((size_t)c.pw * d.mcuy * c.v * 8, 256);
        for (int y = 0; y < c.v; ++y)
          for (int x = 0; x < c.h; ++x, ++i) {
            d.blk_comp[i] = (int8_t)ci;
            d.blk_dy[i] = (int8_t)y;
            d.blk_dx[i] = (int8_t)x;
          }
      }
      d.bpm = i;
    }
    const int n_mcu = d.mcux * d.mcuy;
    d.ri = P.dri ? std::min(P.dri, n_mcu) : n_mcu;
    d.n_iv = (n_mcu + d.ri - 1) / d.ri;
    d.iv_base = total_iv;
    total_iv += d.n_iv;
    d.coef_base = total_blocks;
    total_blocks += (long long)n_mcu * d.bpm;
    max_blocks = std::max(max_blocks, n_mcu * d.bpm);
    max_pix = std::max(max_pix, (long long)d.width * d.height);
    d.scan_off = off + P.scan;
    d.file_end = off + nb;
    total_file_end = std::max(total_file_end, d.file_end);
    const long long scan_bytes = d.file_end - d.scan_off;
    const long long cap = (scan_bytes * 8 + SUB_BITS - 1) / SUB_BITS + d.n_iv;
    if (cap + total_sub > (1LL << 30)) return fail(h, FRCNN_ERR_UNSUPPORTED, "jpeg_decode: batch too large%s%s");
    d.sub_base = total_sub;
    d.sub_cap = (int)cap;
    total_sub += (int)cap;
    d.chunk_base = (int)chunks.size();
    d.n_chunks = (int)((scan_bytes + CHUNK - 1) / CHUNK);
    for (int c = 0; c < d.n_chunks; ++c) chunks.push_back(make_int2(b, c));
    d.end_pos = d.file_end;
  }
  if (chunks.empty()) chunks.push_back(make_int2(0, 0));
  // one upload: descriptors, tables, chunk list
  const size_t o_img = 0, o_tab = align_up(sizeof(Img) * batch, 256),
               o_chunk = o_tab + align_up(sizeof(HuffTab) * tabs.size(), 256),
               blob = o_chunk + align_up(sizeof(int2) * chunks.size(), 256);
  int rc;
  if ((rc = host_staging(h, stream, blob))) return rc;
  uint8_t* pin = static_cast<uint8_t*>(h->pinned);
  memcpy(pin + o_img, imgs.data(), sizeof(Img) * batch);
  memcpy(pin + o_tab, tabs.data(), sizeof(HuffTab) * tabs.size());
  memcpy(pin + o_chunk, chunks.data(), sizeof(int2) * chunks.size());
  void *dev_blob, *clean, *chunk_sum, *chunk_pre, *iv_start, *sub_off, *sub_iv, *rec_a, *rec_b, *chg_a, *chg_b, *pre, *coef,
      *planes;
  if ((rc = arena_get(h, stream, blob, &dev_blob)) || (rc = arena_get(h, stream, total_file_end + 16, &clean)) ||
      (rc = arena_get(h, stream, 4 * chunks.size(), &chunk_sum)) || (rc = arena_get(h, stream, 8 * chunks.size(), &chunk_pre)) ||
      (rc = arena_get(h, stream, 4 * (size_t)total_iv, &iv_start)) || (rc = arena_get(h, stream, 4 * (size_t)total_iv, &sub_off)) ||
      (rc = arena_get(h, stream, 4 * (size_t)total_sub, &sub_iv)) ||
      (rc = arena_get(h, stream, sizeof(SubRec) * (size_t)total_sub, &rec_a)) ||
      (rc = arena_get(h, stream, sizeof(SubRec) * (size_t)total_sub, &rec_b)) ||
      (rc = arena_get(h, stream, (size_t)total_sub, &chg_a)) || (rc = arena_get(h, stream, (size_t)total_sub, &chg_b)) ||
      (rc = arena_get(h, stream, sizeof(SubPre) * (size_t)total_sub, &pre)) ||
      (rc = arena_get(h, stream, 128 * (size_t)total_blocks, &coef)) || (rc = arena_get(h, stream, plane_bytes, &planes)))
    return rc;
  FRCNN_CUDA(h, cudaMemcpyAsync(dev_blob, pin, blob, cudaMemcpyHostToDevice, stream));
  FRCNN_CUDA(h, cudaEventRecord(h->pinned_done, stream));
  FRCNN_CUDA(h, cudaMemsetAsync(iv_start, 0, 4 * (size_t)total_iv, stream));   // interval 0 starts at byte 0
  Img* dimg = reinterpret_cast<Img*>(static_cast<uint8_t*>(dev_blob) + o_img);
  const HuffTab* dtab = reinterpret_cast<const HuffTab*>(static_cast<uint8_t*>(dev_blob) + o_tab);
  const int2* dchunk = reinterpret_cast<const int2*>(static_cast<uint8_t*>(dev_blob) + o_chunk);
  const int n_chunks = (int)chunks.size();
  jpeg_unstuff_count_kernel<<<n_chunks, 256, 0, stream>>>(files, dimg, dchunk, static_cast<uint32_t*>(chunk_sum));
  FRCNN_LAUNCH_CHECK(h, "jpeg_unstuff_count_kernel");
  jpeg_unstuff_scan_kernel<<<batch, 256, 0, stream>>>(dimg, static_cast<uint32_t*>(chunk_sum), static_cast<uint2*>(chunk_pre));
  FRCNN_LAUNCH_CHECK(h, "jpeg_unstuff_scan_kernel");
  jpeg_unstuff_write_kernel<<<n_chunks, 256, 0, stream>>>(files, dimg, dchunk, static_cast<uint2*>(chunk_pre),
                                                          static_cast<uint8_t*>(clean), static_cast<uint32_t*>(iv_start));
  FRCNN_LAUNCH_CHECK(h, "jpeg_unstuff_write_kernel");
  jpeg_huffman_kernel<<<batch, HUFF_THREADS, 0, stream>>>(
      dimg, dtab, static_cast<uint8_t*>(clean), static_cast<uint32_t*>(iv_start), static_cast<uint32_t*>(sub_off),
      static_cast<uint32_t*>(sub_iv), static_cast<SubRec*>(rec_a), static_cast<SubRec*>(rec_b), static_cast<uint8_t*>(chg_a),
      static_cast<uint8_t*>(chg_b), static_cast<SubPre*>(pre), static_cast<int16_t*>(coef), out_offsets, out_bytes, status);
  FRCNN_LAUNCH_CHECK(h, "jpeg_huffman_kernel");
  jpeg_idct_kernel<<<dim3((max_blocks + 127) / 128, batch), 128, 0, stream>>>(dimg, static_cast<int16_t*>(coef), status,
                                                                              static_cast<uint8_t*>(planes));
  FRCNN_LAUNCH_CHECK(h, "jpeg_idct_kernel");
  jpeg_color_kernel<<<dim3((unsigned)((max_pix + 255) / 256), batch), 256, 0, stream>>>(dimg, static_cast<uint8_t*>(planes),
                                                                                       status, out_offsets, out);
  FRCNN_LAUNCH_CHECK(h, "jpeg_color_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
