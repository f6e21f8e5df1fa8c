// SURVEY 8f-4, host-side input pipeline on the device: the pixels of shapes.Image.data (shapes.py:19-29:
// cv2.resize(INTER_CUBIC) + cv2.flip) with the mean subtraction of resnet.preprocess (resnet.py:64-75) fused in, and
// the GT-box scale / mirror of shapes.py:93-132, 292-300.
//
// The resize is OpenCV's uint8 bicubic in its generic fixed-point form (modules/imgproc/src/resize.cpp): per axis
// f = (float)((d + 0.5) * scale - 0.5), s = floor(f), four float32 coefficients (A = -0.75) stored as
// cvRound(c * 2048) shorts, taps s-1 .. s+2 clamped to the image, horizontal pass in int32, vertical pass in int32,
// (sum + 2^21) >> 22, saturate.  Integer arithmetic, so the device result equals oracle/image_oracle.py bit for bit;
// against cv2.resize the tolerance is one grey level (cv2's own SIMD and generic paths differ from each other by that).
#include "common.cuh"

namespace frcnn {

// one record per output column / row: first tap (unclamped) and the four x2048 coefficients
struct CubicTap { int s; short c[4]; int pad; };

// output position d of an axis resized from src to dst
__device__ __forceinline__ CubicTap cubic_tap(int src, int dst, int d) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn((double)dst, (double)src));
  float f = (float)__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5);
  const int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  const float A = -0.75f, x = f, x1 = __fadd_rn(x, 1.0f), xm = __fsub_rn(1.0f, x);
  float c[4];
  c[0] = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, x1), __fmul_rn(5.0f, A)), x1), __fmul_rn(8.0f, A)), x1), __fmul_rn(4.0f, A));
  c[1] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.0f), x), __fadd_rn(A, 3.0f)), x), x), 1.0f);
  c[2] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.0f), xm), __fadd_rn(A, 3.0f)), xm), xm), 1.0f);
  c[3] = __fsub_rn(__fsub_rn(__fsub_rn(1.0f, c[0]), c[1]), c[2]);
  CubicTap t;
  t.s = s - 1;
  t.pad = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) t.c[k] = (short)max(-32768, min(32767, __float2int_rn(__fmul_rn(c[k], 2048.0f))));
  return t;
}

__global__ void __launch_bounds__(256)
cubic_table_kernel(int src_w, int dst_w, int src_h, int dst_h, CubicTap* __restrict__ xt, CubicTap* __restrict__ yt) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= dst_w + dst_h) return;
  const bool is_x = i < dst_w;
  const int d = is_x ? i : i - dst_w;
  (is_x ? xt : yt)[d] = cubic_tap(is_x ? src_w : src_h, is_x ? dst_w : dst_h, d);
}

// one thread per output pixel (all channels); out_u8 and / or out_f32 (pixel - mean[c], float64 subtraction stored as
// float32) may be requested; flip mirrors the OUTPUT columns (cv2.flip(img, 1) after the resize)
__global__ void __launch_bounds__(256)
resize_cubic_kernel(const unsigned char* __restrict__ src, int src_h, int src_w, int cn, int dst_h, int dst_w,
                    const CubicTap* __restrict__ xt, const CubicTap* __restrict__ yt, int flip,
                    unsigned char* __restrict__ out_u8, float* __restrict__ out_f32, double m0, double m1, double m2,
                    double m3) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31), dy = blockIdx.y * 8 + (threadIdx.x >> 5), img = blockIdx.z;
  if (dx >= dst_w || dy >= dst_h) return;
  const CubicTap tx = xt[dx], ty = yt[dy];
  const unsigned char* s_img = src + (size_t)img * src_h * src_w * cn;
  int xo[4], yo[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    xo[k] = min(max(tx.s + k, 0), src_w - 1) * cn;
    yo[k] = min(max(ty.s + k, 0), src_h - 1);
  }
  const int ox = flip ? dst_w - 1 - dx : dx;
  const size_t o = (((size_t)img * dst_h + dy) * dst_w + ox) * cn;
  const double mean[4] = {m0, m1, m2, m3};
  for (int c = 0; c < cn; ++c) {
    int acc = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned char* row = s_img + (size_t)yo[j] * src_w * cn + c;
      const int h = (int)row[xo[0]] * tx.c[0] + (int)row[xo[1]] * tx.c[1] + (int)row[xo[2]] * tx.c[2] + (int)row[xo[3]] * tx.c[3];
      acc += h * ty.c[j];
    }
    const int v = min(255, max(0, (acc + (1 << 21)) >> 22));
    if (out_u8) out_u8[o + c] = (unsigned char)v;
    if (out_f32) out_f32[o + c] = (float)__dsub_rn((double)v, mean[c & 3]);
  }
}

// Tiled form of the same arithmetic, channel count known at compile time: a CTA produces 32 x 8 output pixels.  The
// horizontal pass of every source row the tile's eight output rows touch is computed ONCE into shared memory (int32,
// exactly the per-pixel kernel's `h`; a thread keeps its column's four clamped tap offsets and coefficients in
// registers and walks down the rows), the vertical pass reads it back.  The float64 mean subtraction becomes a look-up
// in a 256-entry table per channel (cubic_table_kernel fills it with (float)((double)v - mean[c]), the same two
// roundings).  The first version of this file spent 214 instructions per output value (runtime channel loops, two
// integer divisions per horizontal sum, three float64-pipe operations per value); this one about 30.
// Used while eight output rows span at most TILE_ROWS source rows (any enlargement, reductions down to about 1/4) and
// the image has 1, 3 or 4 channels; the per-pixel kernel takes the rest.
// Two tile heights: 32 output rows per CTA (four per thread: the column's taps, the mean table and the tile set-up
// are paid once for four pixels, and neighbouring output rows share more source rows) while they span at most 72 source
// rows (scale <= 2.1), else 8 rows / 40 source rows.
constexpr int TILE_W = 32;

template <int CN, int TILE_H, int TILE_ROWS>
__global__ void __launch_bounds__(256)
resize_cubic_tile_kernel(const unsigned char* __restrict__ src, int src_h, int src_w, int dst_h, int dst_w,
                         const CubicTap* __restrict__ xt, const CubicTap* __restrict__ yt, const float* __restrict__ lut,
                         int flip, unsigned char* __restrict__ out_u8, float* __restrict__ out_f32) {
  __shared__ int hs[TILE_ROWS][TILE_W * CN];
  __shared__ float s_lut[CN][256];
  const int dx0 = blockIdx.x * TILE_W, dy0 = blockIdx.y * TILE_H, img = blockIdx.z;
  const int tid = threadIdx.x, x = tid & 31, wy = tid >> 5;
  for (int i = tid; i < CN * 256; i += 256) s_lut[i >> 8][i & 255] = lut[i];
  const int r0 = yt[dy0].s;                                          // first source row of the tile (unclamped)
  const int n_rows = yt[min(dy0 + TILE_H, dst_h) - 1].s + 4 - r0;   // <= TILE_ROWS (the launcher checked the span)
  const int dx = min(dx0 + x, dst_w - 1);                           // columns past the edge repeat the last one, never stored
  const CubicTap tx = xt[dx];
  int xo[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) xo[k] = min(max(tx.s + k, 0), src_w - 1) * CN;
  const unsigned char* s_img = src + (size_t)img * src_h * src_w * CN;
  for (int row = wy; row < n_rows; row += 8) {
    const unsigned char* rp = s_img + (size_t)min(max(r0 + row, 0), src_h - 1) * src_w * CN;
#pragma unroll
    for (int c = 0; c < CN; ++c)
      hs[row][c * TILE_W + x] = (int)rp[xo[0] + c] * tx.c[0] + (int)rp[xo[1] + c] * tx.c[1] + (int)rp[xo[2] + c] * tx.c[2] +
                            (int)rp[xo[3] + c] * tx.c[3];
  }
  __syncthreads();
  if (dx0 + x >= dst_w) return;
  const int ox = flip ? dst_w - 1 - dx : dx;
#pragma unroll 1
  for (int dy = dy0 + wy; dy < min(dy0 + TILE_H, dst_h); dy += 8) {
    const CubicTap ty = yt[dy];
    const int rr = ty.s - r0;
    const size_t o = (((size_t)img * dst_h + dy) * dst_w + ox) * CN;
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const int acc = hs[rr][c * TILE_W + x] * ty.c[0] + hs[rr + 1][c * TILE_W + x] * ty.c[1] + hs[rr + 2][c * TILE_W + x] * ty.c[2] +
                      hs[rr + 3][c * TILE_W + x] * ty.c[3];
      const int v = min(255, max(0, (acc + (1 << 21)) >> 22));
      if (out_u8) out_u8[o + c] = (unsigned char)v;
      if (out_f32) out_f32[o + c] = s_lut[c][v];
    }
  }
}

// (float)((double)v - mean[c]) for v = 0..255 and up to four channels
__global__ void mean_lut_kernel(float* __restrict__ lut, double m0, double m1, double m2, double m3) {
  const int v = threadIdx.x;
  lut[v] = (float)__dsub_rn((double)v, m0);
  lut[256 + v] = (float)__dsub_rn((double)v, m1);
  lut[512 + v] = (float)__dsub_rn((double)v, m2);
  lut[768 + v] = (float)__dsub_rn((double)v, m3);
}

// ---- ragged batch: differently sized sources, each resized to its own size inside one padded output ----------------
// Every geometry lives on the device, so the launch configuration depends on the padded shape only and one captured
// graph serves every mix of sizes.  Per image: tap tables at a fixed stride of dst_width + dst_height entries, then one
// CTA per 32 x 32 output tile of the padded image.  A tile outside the image's extent writes zeros.  A tile whose 32
// rows span at most 72 source rows (scale <= 2.1, as the uniform launcher's tall tiles) takes the shared-memory
// horizontal pass; any other computes each pixel straight from the source, the per-pixel kernel's integer sums, which
// give the same values.  The mirror works within the image's own width.
struct RaggedImage { long long off; int src_h, src_w, dst_h, dst_w; };

// geom[img] = (src_h, src_w, dst_h, dst_w); the output extent is clamped to the padded image, and a source with a
// non-positive size or bytes outside [0, src_bytes) gets an empty extent (an all-zero image, nothing read)
__device__ __forceinline__ RaggedImage ragged_image(const long long* offsets, long long src_bytes, const int* geom, int cn,
                                                    int dst_height, int dst_width, int img) {
  RaggedImage r;
  r.src_h = geom[4 * img];
  r.src_w = geom[4 * img + 1];
  r.dst_h = min(max(geom[4 * img + 2], 0), dst_height);
  r.dst_w = min(max(geom[4 * img + 3], 0), dst_width);
  r.off = offsets[img];
  const long long px = (long long)max(r.src_h, 0) * max(r.src_w, 0);
  if (px == 0 || px > src_bytes || r.off < 0 || r.off > src_bytes || px * cn > src_bytes - r.off) r.dst_h = r.dst_w = 0;
  return r;
}

__global__ void __launch_bounds__(256)
cubic_table_ragged_kernel(const long long* __restrict__ offsets, long long src_bytes, const int* __restrict__ geom, int cn,
                          int dst_height, int dst_width, CubicTap* __restrict__ tab) {
  const int i = blockIdx.x * 256 + threadIdx.x, img = blockIdx.y;
  const RaggedImage r = ragged_image(offsets, src_bytes, geom, cn, dst_height, dst_width, img);
  CubicTap* xt = tab + (size_t)img * (dst_width + dst_height);
  if (i < r.dst_w) xt[i] = cubic_tap(r.src_w, r.dst_w, i);
  else if (i >= dst_width && i - dst_width < r.dst_h) xt[i] = cubic_tap(r.src_h, r.dst_h, i - dst_width);
}

template <int CN>
__global__ void __launch_bounds__(256, CN == 4 ? 5 : 6)   // as many CTAs per SM as the shared memory (up to 30 KB, 40 KB at CN 4) allows
resize_cubic_ragged_kernel(const unsigned char* __restrict__ src, const long long* __restrict__ offsets, long long src_bytes,
                           const int* __restrict__ geom, const unsigned char* __restrict__ flip, int dst_height, int dst_width,
                           const CubicTap* __restrict__ tab, const float* __restrict__ lut, unsigned char* __restrict__ out_u8,
                           float* __restrict__ out_f32) {
  constexpr int TILE_H = 32, TILE_ROWS = 72;
  __shared__ int hs[TILE_ROWS][TILE_W * CN];
  __shared__ float s_lut[CN][256];
  const int dx0 = blockIdx.x * TILE_W, dy0 = blockIdx.y * TILE_H, img = blockIdx.z;
  const int tid = threadIdx.x, x = tid & 31, wy = tid >> 5;
  const int px = dx0 + x, y_end = min(dy0 + TILE_H, dst_height);
  const RaggedImage r = ragged_image(offsets, src_bytes, geom, CN, dst_height, dst_width, img);
  const size_t img_base = (size_t)img * dst_height * dst_width * CN;
  // rows [dy0, y_valid) of column px lie inside the image; the rest of the tile is padding
  const int y_valid = px < r.dst_w ? min(y_end, r.dst_h) : dy0;
  if (dx0 < r.dst_w && dy0 < r.dst_h) {
    for (int i = tid; i < CN * 256; i += 256) s_lut[i >> 8][i & 255] = lut[i];
    const unsigned char* s_img = src + r.off;
    const CubicTap* xt = tab + (size_t)img * (dst_width + dst_height);
    const CubicTap* yt = xt + dst_width;
    // source-side column of output column px; columns past the extent repeat an edge column and are never stored
    const int dx = (flip && flip[img]) ? max(r.dst_w - 1 - px, 0) : min(px, r.dst_w - 1);
    const CubicTap tx = xt[dx];
    int xo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) xo[k] = min(max(tx.s + k, 0), r.src_w - 1) * CN;
    const int r0 = yt[dy0].s;
    const int n_rows = yt[min(dy0 + TILE_H, r.dst_h) - 1].s + 4 - r0;
    if (n_rows <= TILE_ROWS) {                                      // the same for the whole CTA
      for (int row = wy; row < n_rows; row += 8) {
        const unsigned char* rp = s_img + (size_t)min(max(r0 + row, 0), r.src_h - 1) * r.src_w * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c)
          hs[row][c * TILE_W + x] = (int)rp[xo[0] + c] * tx.c[0] + (int)rp[xo[1] + c] * tx.c[1] +
                                    (int)rp[xo[2] + c] * tx.c[2] + (int)rp[xo[3] + c] * tx.c[3];
      }
      __syncthreads();
#pragma unroll 1
      for (int dy = dy0 + wy; dy < y_valid; dy += 8) {
        const CubicTap ty = yt[dy];
        const int rr = ty.s - r0;
        const size_t o = img_base + ((size_t)dy * dst_width + px) * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c) {
          const int acc = hs[rr][c * TILE_W + x] * ty.c[0] + hs[rr + 1][c * TILE_W + x] * ty.c[1] +
                          hs[rr + 2][c * TILE_W + x] * ty.c[2] + hs[rr + 3][c * TILE_W + x] * ty.c[3];
          const int v = min(255, max(0, (acc + (1 << 21)) >> 22));
          if (out_u8) out_u8[o + c] = (unsigned char)v;
          if (out_f32) out_f32[o + c] = s_lut[c][v];
        }
      }
    } else {
      __syncthreads();
#pragma unroll 1
      for (int dy = dy0 + wy; dy < y_valid; dy += 8) {
        const CubicTap ty = yt[dy];
        const size_t o = img_base + ((size_t)dy * dst_width + px) * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c) {
          int acc = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const unsigned char* rp = s_img + (size_t)min(max(ty.s + j, 0), r.src_h - 1) * r.src_w * CN + c;
            acc += ((int)rp[xo[0]] * tx.c[0] + (int)rp[xo[1]] * tx.c[1] + (int)rp[xo[2]] * tx.c[2] +
                    (int)rp[xo[3]] * tx.c[3]) * ty.c[j];
          }
          const int v = min(255, max(0, (acc + (1 << 21)) >> 22));
          if (out_u8) out_u8[o + c] = (unsigned char)v;
          if (out_f32) out_f32[o + c] = s_lut[c][v];
        }
      }
    }
  }
  if (px >= dst_width) return;
  for (int dy = dy0 + wy; dy < y_end; dy += 8) {
    if (dy < y_valid) continue;
    const size_t o = img_base + ((size_t)dy * dst_width + px) * CN;
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      if (out_u8) out_u8[o + c] = 0;
      if (out_f32) out_f32[o + c] = 0.0f;
    }
  }
}

// boxes [n,4] f64 -> corners * ratio, then mirrored about flip_width when flip_width >= 0 (per image: ratio[b], width[b])
__global__ void gt_transform_kernel(const double* __restrict__ boxes, const int* __restrict__ n_box, int n_max,
                                    const double* __restrict__ ratio, const double* __restrict__ flip_width,
                                    double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, img = blockIdx.y;
  if (i >= n_max) return;
  const size_t o = ((size_t)img * n_max + i) * 4;
  if (n_box && i >= n_box[img]) {
    out[o] = out[o + 1] = out[o + 2] = out[o + 3] = 0.0;
    return;
  }
  const double r = ratio[img];
  const double x1 = __dmul_rn(boxes[o], r), y1 = __dmul_rn(boxes[o + 1], r), x2 = __dmul_rn(boxes[o + 2], r), y2 = __dmul_rn(boxes[o + 3], r);
  const double w = flip_width ? flip_width[img] : -1.0;
  if (w >= 0.0) {
    out[o] = __dsub_rn(w, x2); out[o + 1] = y1; out[o + 2] = __dsub_rn(w, x1); out[o + 3] = y2;
  } else {
    out[o] = x1; out[o + 1] = y1; out[o + 2] = x2; out[o + 3] = y2;
  }
}

int launch_image_resize(frcnn_handle* h, cudaStream_t stream, const uint8_t* src, int src_h, int src_w, int cn, int dst_h,
                        int dst_w, int flip, int batch, const double* mean_host, uint8_t* out_u8, float* out_f32) {
  void* tab = nullptr;
  int rc = arena_get(h, stream, (size_t)(dst_w + dst_h) * sizeof(CubicTap), &tab);
  if (rc) return rc;
  CubicTap* xt = static_cast<CubicTap*>(tab);
  CubicTap* yt = xt + dst_w;
  cubic_table_kernel<<<(dst_w + dst_h + 255) / 256, 256, 0, stream>>>(src_w, dst_w, src_h, dst_h, xt, yt);
  FRCNN_LAUNCH_CHECK(h, "cubic_table_kernel");
  double m[4] = {0.0, 0.0, 0.0, 0.0};
  if (mean_host)
    for (int c = 0; c < cn && c < 4; ++c) m[c] = mean_host[c];
  dim3 grid((dst_w + 31) / 32, (dst_h + 7) / 8, batch);
  // source rows touched by T consecutive output rows: at most ceil((T - 1) * src_h / dst_h) + 5 (first taps of rows
  // that are T - 1 apart differ by at most ceil((T - 1) * scale) + 1, plus the four taps)
  const long long span8 = (7LL * src_h + dst_h - 1) / dst_h + 5, span32 = (31LL * src_h + dst_h - 1) / dst_h + 5;
  if ((cn == 1 || cn == 3 || cn == 4) && span8 <= 40) {
    void* lut = nullptr;
    if ((rc = arena_get(h, stream, 4 * 256 * sizeof(float), &lut))) return rc;
    float* lutf = static_cast<float*>(lut);
    mean_lut_kernel<<<1, 256, 0, stream>>>(lutf, m[0], m[1], m[2], m[3]);
    FRCNN_LAUNCH_CHECK(h, "mean_lut_kernel");
    const bool tall = span32 <= 72;
    const dim3 tgrid((dst_w + 31) / 32, tall ? (dst_h + 31) / 32 : (dst_h + 7) / 8, batch);
#define FRCNN_TILE(CN)                                                                                                  \
  if (tall) resize_cubic_tile_kernel<CN, 32, 72><<<tgrid, 256, 0, stream>>>(src, src_h, src_w, dst_h, dst_w, xt, yt, lutf, flip, out_u8, out_f32); \
  else resize_cubic_tile_kernel<CN, 8, 40><<<tgrid, 256, 0, stream>>>(src, src_h, src_w, dst_h, dst_w, xt, yt, lutf, flip, out_u8, out_f32)
    if (cn == 1) { FRCNN_TILE(1); } else if (cn == 3) { FRCNN_TILE(3); } else { FRCNN_TILE(4); }
#undef FRCNN_TILE
    FRCNN_LAUNCH_CHECK(h, "resize_cubic_tile_kernel");
    return FRCNN_OK;
  }
  resize_cubic_kernel<<<grid, 256, 0, stream>>>(src, src_h, src_w, cn, dst_h, dst_w, xt, yt, flip, out_u8, out_f32, m[0], m[1],
                                                m[2], m[3]);
  FRCNN_LAUNCH_CHECK(h, "resize_cubic_kernel");
  return FRCNN_OK;
}

int launch_image_resize_ragged(frcnn_handle* h, cudaStream_t stream, const uint8_t* src, const int64_t* src_offsets,
                               long long src_bytes, const int32_t* geom, const uint8_t* flip, int cn, int dst_height,
                               int dst_width, int batch, const double* mean_host, uint8_t* out_u8, float* out_f32) {
  void *tab = nullptr, *lut = nullptr;
  int rc = arena_get(h, stream, (size_t)batch * (dst_width + dst_height) * sizeof(CubicTap), &tab);
  if (rc || (rc = arena_get(h, stream, 4 * 256 * sizeof(float), &lut))) return rc;
  CubicTap* tabc = static_cast<CubicTap*>(tab);
  float* lutf = static_cast<float*>(lut);
  const long long* offs = reinterpret_cast<const long long*>(src_offsets);
  cubic_table_ragged_kernel<<<dim3((dst_width + dst_height + 255) / 256, batch), 256, 0, stream>>>(
      offs, src_bytes, geom, cn, dst_height, dst_width, tabc);
  FRCNN_LAUNCH_CHECK(h, "cubic_table_ragged_kernel");
  double m[4] = {0.0, 0.0, 0.0, 0.0};
  if (mean_host)
    for (int c = 0; c < cn && c < 4; ++c) m[c] = mean_host[c];
  mean_lut_kernel<<<1, 256, 0, stream>>>(lutf, m[0], m[1], m[2], m[3]);
  FRCNN_LAUNCH_CHECK(h, "mean_lut_kernel");
  const dim3 grid((dst_width + TILE_W - 1) / TILE_W, (dst_height + 31) / 32, batch);
#define FRCNN_RAGGED(CN) \
  resize_cubic_ragged_kernel<CN><<<grid, 256, 0, stream>>>(src, offs, src_bytes, geom, flip, dst_height, dst_width, tabc, lutf, out_u8, out_f32)
  switch (cn) {
    case 1: FRCNN_RAGGED(1); break;
    case 2: FRCNN_RAGGED(2); break;
    case 3: FRCNN_RAGGED(3); break;
    default: FRCNN_RAGGED(4); break;
  }
#undef FRCNN_RAGGED
  FRCNN_LAUNCH_CHECK(h, "resize_cubic_ragged_kernel");
  return FRCNN_OK;
}

int launch_gt_transform(frcnn_handle* h, cudaStream_t stream, const double* boxes, const int32_t* n_box, int n_max, int batch,
                        const double* ratio, const double* flip_width, double* out) {
  dim3 grid((n_max + 127) / 128, batch);
  gt_transform_kernel<<<grid, 128, 0, stream>>>(boxes, n_box, n_max, ratio, flip_width, out);
  FRCNN_LAUNCH_CHECK(h, "gt_transform_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
