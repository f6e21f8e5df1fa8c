// K-e: detector post-processing, one CTA per image (voc_dets.py:51-86).
//
//   per row: class = argmax(out_cls[row]) (first maximum), skip 'bg' / below threshold / class K-1 when 'bg' is not
//            last (no regression columns);
//            deltas = out_reg[row, 4c:4c+4] / [10,10,5,5] (float32);
//            box = util.transform(roi, deltas) (util.py:55-74: tx*wa in float32, rest float64,
//            no rounding, no clipping) * stride;
//   per class (order of first appearance): greedy NMS in float64 (+1 areas, 0.5, max_boxes),
//            visit order (prob desc, position desc);
//   per kept row: int(round(v / resize_ratio)) -- Python round == half-to-even == rint.
#include "common.cuh"

namespace frcnn {

constexpr int PP_THREADS = 1024;     // one CTA per image: 32 warps so that every class has a warp in the NMS phase
constexpr int PP_MAX_ROWS = 1024;
constexpr int PP_MAX_CLASSES = 128;

struct __align__(8) BoxI16 { short x1, y1, x2, y2; };

__global__ void __launch_bounds__(PP_THREADS)
det_postprocess_kernel(const BoxI16* __restrict__ rois_all, const float* __restrict__ cls_all,
                       const float* __restrict__ reg_all, const double* __restrict__ ratio_all,
                       const int* __restrict__ n_rows_all, int M, int K,
                       int bg, int stride, float det_thr, double nms_thr, int max_boxes,
                       int* __restrict__ det_boxes, float* __restrict__ det_probs, int* __restrict__ det_cls,
                       int* __restrict__ det_count) {
  // dynamic smem, sized by M: double4 box[M] | double area[M] | u64 key[M] | float prob[M] | short cls[M] |
  // short sorted[M] | short keep[M] | uchar dead[M]
  extern __shared__ __align__(32) unsigned char pp_smem[];
  double4* s_box = reinterpret_cast<double4*>(pp_smem);      // decoded boxes (by row)
  double* s_area = reinterpret_cast<double*>(s_box + M);     // areas in per-class visit order
  unsigned long long* s_key = reinterpret_cast<unsigned long long*>(s_area + M);   // class << 48 | mono(prob) << 16 | row
  float* s_prob = reinterpret_cast<float*>(s_key + M);
  short* s_cls = reinterpret_cast<short*>(s_prob + M);       // class of the row, -1 = dropped
  short* s_sorted = s_cls + M;                               // row ids in (class order, visit order)
  short* s_keep = s_sorted + M;                              // per-class pick lists (positions in the class)
  unsigned char* s_dead = reinterpret_cast<unsigned char*>(s_keep + M);
  __shared__ int s_first[PP_MAX_CLASSES], s_cnt[PP_MAX_CLASSES], s_off[PP_MAX_CLASSES + 1];
  __shared__ int s_order[PP_MAX_CLASSES], s_nkeep[PP_MAX_CLASSES], s_koff[PP_MAX_CLASSES + 1];
  __shared__ int s_ncls;

  const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const BoxI16* rois = rois_all + (size_t)img * M;
  const float* ocls = cls_all + (size_t)img * M * K;
  const float* oreg = reg_all + (size_t)img * M * 4 * (K - 1);
  const double ratio = ratio_all[img];
  const int m_live = n_rows_all ? min(max(n_rows_all[img], 0), M) : M;      // rows the detector really saw

  for (int c = tid; c < K; c += PP_THREADS) { s_first[c] = 0x7fffffff; s_cnt[c] = 0; }
  __syncthreads();

  // 1+2: class choice and float64 decode
  for (int r = tid; r < M; r += PP_THREADS) {
    if (r >= m_live) { s_cls[r] = -1; s_key[r] = ~0ull; continue; }
    const float* p = ocls + (size_t)r * K;
    int c = 0;
    float conf = p[0];
    for (int q = 1; q < K; ++q) { const float v = p[q]; if (v > conf) { conf = v; c = q; } }
    // out_reg holds 4(K-1) columns indexed by class: with 'bg' not last, class K-1 has none and its rows are dropped
    // (the reference's slice out_reg[4c:4c+4] is empty there)
    if (c == bg || c == K - 1 || conf < det_thr) { s_cls[r] = -1; s_key[r] = ~0ull; continue; }
    const float* t = oreg + (size_t)r * 4 * (K - 1) + 4 * c;
    const float tx = __fdiv_rn(t[0], 10.f), ty = __fdiv_rn(t[1], 10.f), tw = __fdiv_rn(t[2], 5.f), th = __fdiv_rn(t[3], 5.f);
    const BoxI16 b = rois[r];
    const double cxa = (double)(short)(b.x1 + b.x2) / 2.0, cya = (double)(short)(b.y1 + b.y2) / 2.0;
    const short wa = (short)(b.x2 - b.x1), ha = (short)(b.y2 - b.y1);
    const double cx = __dadd_rn((double)__fmul_rn(tx, (float)wa), cxa);
    const double cy = __dadd_rn((double)__fmul_rn(ty, (float)ha), cya);
    const double w = __dmul_rn(exp((double)tw), (double)wa), hh = __dmul_rn(exp((double)th), (double)ha);
    const double x = __dsub_rn(cx, w / 2.0), y = __dsub_rn(cy, hh / 2.0);
    const double s = (double)stride;
    const double4 o = make_double4(__dmul_rn(s, x), __dmul_rn(s, y), __dmul_rn(s, __dadd_rn(x, w)), __dmul_rn(s, __dadd_rn(y, hh)));
    s_box[r] = o;
    s_prob[r] = conf;
    s_cls[r] = (short)c;
    s_key[r] = ((unsigned long long)c << 48) | ((unsigned long long)mono_key(conf) << 16) | (unsigned)r;
    atomicMin(&s_first[c], r);
    atomicAdd(&s_cnt[c], 1);
  }
  __syncthreads();

  // 3: classes in order of first appearance, segment offsets (warp 0: a class's place = the number of present classes
  // that appear earlier; offsets by a running warp scan over the places)
  if (warp == 0) {
    int nc = 0;
    for (int c0 = 0; c0 < K; c0 += 32) nc += __popc(__ballot_sync(0xffffffffu, c0 + lane < K && s_cnt[c0 + lane] > 0));
    for (int c = lane; c < K; c += 32) {
      if (s_cnt[c] == 0) continue;
      const int f = s_first[c];
      int place = 0;
      for (int q = 0; q < K; ++q) place += (s_cnt[q] > 0 && s_first[q] < f) ? 1 : 0;     // first rows are distinct
      s_order[place] = c;
    }
    __syncwarp();
    int run = 0;
    for (int i0 = 0; i0 < nc; i0 += 32) {
      const int i = i0 + lane;
      const int cnt = i < nc ? s_cnt[s_order[i]] : 0;
      int incl = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
      }
      if (i < nc) s_off[s_order[i]] = run + incl - cnt;
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_ncls = nc;
  }
  __syncthreads();

  // 4a: visit rank inside the class: (prob desc, position-in-class desc) = the number of rows of the class with a larger
  // packed key.  Rows are spread over the lanes of a warp (eight partial counts per row, reduced by shuffles): the
  // first version walked all M rows per thread with two dependent shared loads and a branch per step (74 k cycles).
  {
    constexpr int PARTS = 8;                           // lanes per row
    const int part = lane & (PARTS - 1);
    for (int base = warp * (32 / PARTS); base < M; base += PP_THREADS / PARTS) {    // warp-uniform: shuffles inside
      const int r = base + lane / PARTS;
      const unsigned long long kr = r < M ? s_key[r] : ~0ull;
      const bool row_live = kr != ~0ull;
      int rank = 0;
      for (int q = part; q < M; q += PARTS) {
        const unsigned long long kq = s_key[q];
        rank += (((kq ^ kr) >> 48) == 0ull && kq > kr) ? 1 : 0;        // dropped rows (~0) never share a live row's class
      }
#pragma unroll
      for (int d = 1; d < PARTS; d <<= 1) rank += __shfl_xor_sync(0xffffffffu, rank, d);
      if (row_live && part == 0) s_sorted[s_off[(int)(kr >> 48)] + rank] = (short)r;
    }
  }
  __syncthreads();
  const int total_rows = (s_ncls > 0) ? s_off[s_order[s_ncls - 1]] + s_cnt[s_order[s_ncls - 1]] : 0;
  for (int i = tid; i < total_rows; i += PP_THREADS) {
    const double4 b = s_box[s_sorted[i]];
    s_area[i] = __dmul_rn(__dadd_rn(__dsub_rn(b.z, b.x), 1.0), __dadd_rn(__dsub_rn(b.w, b.y), 1.0));
    s_dead[i] = 0;
  }
  __syncthreads();

  // 4b: greedy NMS, one warp per class
  for (int ci = warp; ci < s_ncls; ci += PP_THREADS / 32) {
    const int c = s_order[ci];
    const int off = s_off[c], n = s_cnt[c];
    int kept = 0;
    for (int cur = 0; cur < n && kept < max_boxes; ++cur) {
      if (s_dead[off + cur]) continue;              // warp-uniform (flags synchronised below)
      if (lane == 0) s_keep[off + kept] = (short)cur;
      ++kept;
      const double4 a = s_box[s_sorted[off + cur]];
      const double a_area = s_area[off + cur];
      for (int j = cur + 1 + lane; j < n; j += 32) {
        if (s_dead[off + j]) continue;
        const double4 b = s_box[s_sorted[off + j]];
        const double iw = fmax(0.0, __dadd_rn(__dsub_rn(fmin(a.z, b.z), fmax(a.x, b.x)), 1.0));
        const double ih = fmax(0.0, __dadd_rn(__dsub_rn(fmin(a.w, b.w), fmax(a.y, b.y)), 1.0));
        const double inter = __dmul_rn(iw, ih);
        const double uni = __dsub_rn(__dadd_rn(a_area, s_area[off + j]), inter);
        if (!(__ddiv_rn(inter, uni) <= nms_thr)) s_dead[off + j] = 1;
      }
      __syncwarp();
    }
    if (lane == 0) s_nkeep[c] = kept;
  }
  __syncthreads();

  // 5: outputs
  if (tid == 0) {
    int off = 0;
    for (int i = 0; i < s_ncls; ++i) { s_koff[i] = off; off += s_nkeep[s_order[i]]; }
    s_koff[s_ncls] = off;
    det_count[img] = off;
  }
  __syncthreads();
  for (int o_row = tid; o_row < s_koff[s_ncls]; o_row += PP_THREADS) {
    int ci = 0;
    while (s_koff[ci + 1] <= o_row) ++ci;                 // class segment of this output row (at most K steps)
    const int c = s_order[ci];
    const int off = s_off[c], q = o_row - s_koff[ci];
    const int row = s_sorted[off + s_keep[off + q]];
    const double4 b = s_box[row];
    const size_t o = (size_t)img * M + o_row;
    det_boxes[4 * o + 0] = (int)rint(__ddiv_rn(b.x, ratio));
    det_boxes[4 * o + 1] = (int)rint(__ddiv_rn(b.y, ratio));
    det_boxes[4 * o + 2] = (int)rint(__ddiv_rn(b.z, ratio));
    det_boxes[4 * o + 3] = (int)rint(__ddiv_rn(b.w, ratio));
    det_probs[o] = s_prob[row];
    det_cls[o] = c;
  }
  for (int q = s_koff[s_ncls] + tid; q < M; q += PP_THREADS) {
    const size_t o = (size_t)img * M + q;
    det_boxes[4 * o] = det_boxes[4 * o + 1] = det_boxes[4 * o + 2] = det_boxes[4 * o + 3] = 0;
    det_probs[o] = 0.f;
    det_cls[o] = -1;
  }
}

int launch_det_postprocess(frcnn_handle* h, cudaStream_t stream, const int16_t* rois, const float* out_cls,
                           const float* out_reg, const double* ratio, const int32_t* n_rows, int M, int K, int bg, int stride,
                           double det_thr, double nms_thr, int max_boxes, int batch, int32_t* det_boxes,
                           float* det_probs, int32_t* det_cls, int32_t* det_count) {
  if (M > PP_MAX_ROWS || K > PP_MAX_CLASSES)
    return fail(h, FRCNN_ERR_UNSUPPORTED, "det_postprocess: more than 1024 rows or 128 classes per image%s%s");
  const size_t smem = (size_t)M * (32 + 8 + 8 + 4 + 2 + 2 + 2 + 1) + 64;
  FRCNN_CUDA(h, cudaFuncSetAttribute(det_postprocess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  det_postprocess_kernel<<<batch, PP_THREADS, smem, stream>>>(reinterpret_cast<const BoxI16*>(rois), out_cls, out_reg,
                                                           ratio, n_rows, M, K, bg, stride, (float)det_thr, nms_thr,
                                                           max_boxes, det_boxes, det_probs, det_cls, det_count);
  FRCNN_LAUNCH_CHECK(h, "det_postprocess_kernel");
  return FRCNN_OK;
}

}  // namespace frcnn
