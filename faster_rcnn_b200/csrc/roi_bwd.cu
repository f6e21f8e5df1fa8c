// K-d backward (custom_layers.py:35-56 under TF autodiff: ResizeBilinearGrad + slice-grad + AddN), both modes:
// block-stationary gather over precomputed work lists.
//
// dX is cut into 2x2-cell blocks.  A plan step (two small kernels) writes, for every block, the ordered list of dY rows
// (roi, ph, pw) that contribute to it -- resize mode: the bins with a bilinear tap inside the block, together
// with the four tap weights wy*wx; max mode: the bins that cover a cell of the block -- in ascending
// (roi, ph, pw) order.  One CTA of the plan kernel owns one block: RoIs are tested 256 at a time, the entry
// counts are prefix-summed across the CTA, the block's list is carved from a global bump counter (only its
// LOCATION depends on scheduling, its content and order never do) and filled in order.
//
// The streaming kernel is then a sparse x dense product with no bookkeeping on the critical path: a warp owns
// (block, 128*CPB channels, contiguous slice of the block's list) and keeps the four cells' accumulators in
// registers (static indexing: every entry carries the weights of all four cells, absent cells are masked).
// dY rows travel global -> shared with cp.async into a per-LANE ring (a lane only ever reads what it copied
// itself, so the ring needs no barrier): D rows of 512*CPB bytes per warp are in flight while the FMAs of the
// oldest one issue, and the list entries are staged the same way 32 at a time.  Slices of one block are added
// in slice order through shared memory: no atomics, one fixed summation order, bit-reproducible run to run.
//
// Against the cell-stationary gather of round 1 a dY row is fetched by 2.06 blocks instead of 3.48 cells in resize
// mode (2.64 instead of 5.02 bin covers in max mode, C5 RoIs), the crop / tap-table round trips that serialised every
// RoI chunk are gone, and twice the bytes are in flight per SM.
//
// This path takes every pool size up to ROI_MAX_TABLE_P and any RoI count whose work list fits its index formats
// (roi_bwd_blk_eligible); the plan step has a narrow instance (one-byte masks, P <= 8 and N < 65536: the tuned shapes)
// and a wide one (32-bit masks).  Everything else -- C % 4 != 0, unaligned buffers, larger pools or maps -- takes the
// scalar-channel kernel at the end of this file.
#include <type_traits>

#include "roi_common.cuh"

namespace frcnn {

constexpr int BLK = 2;                       // block edge in cells
constexpr unsigned ENT_MASK_SHIFT = 28;      // entry word = dY row index | cell mask << 28
constexpr unsigned ENT_IDX_MASK = (1u << ENT_MASK_SHIFT) - 1u;
constexpr int ROI_MAX_COMPACT = 2;           // internal mode: max pooling with the one-byte (dy << 4 | dx) arg-max of roi.cu

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16_if(void* smem_dst, const void* gsrc, bool pred) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("{ .reg .pred p; setp.ne.b32 p, %2, 0; @p cp.async.cg.shared.global [%0], [%1], 16; }"
               ::"r"(s), "l"(gsrc), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void cp_async4_if(void* smem_dst, const void* gsrc, bool pred) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("{ .reg .pred p; setp.ne.b32 p, %2, 0; @p cp.async.ca.shared.global [%0], [%1], 4; }"
               ::"r"(s), "l"(gsrc), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------------------------------------------------------------------------------
// plan: per-block work lists
// ---------------------------------------------------------------------------------------
// Which outputs of a RoI touch a block separates per axis: bin (ph, pw) touches block (by, bx) iff output row ph
// touches block row by and output column pw touches block column bx.  roi_bwd_mask_kernel writes those two
// relations once per (RoI, block row) and (RoI, block column) as P-bit masks M (uint8_t for P <= 8, else uint32_t),
// laid out [axis block][RoI] so that the plan kernel's RoI sweep is a coalesced stream: the sweep then costs a few
// instructions per 32 RoIs instead of re-deriving the taps of every RoI in every block (the first version of this
// file did that and spent 270 us on the C5 x 8 plan against 630 us for the streaming kernel).
template <int MODE, typename M>
__global__ void __launch_bounds__(256)
roi_bwd_mask_kernel(const void* __restrict__ rois, int dtype, int N, int n_pad, int H, int W, int P, int blocks_y,
                    int blocks_x, M* __restrict__ ymask, M* __restrict__ xmask, unsigned* __restrict__ counter) {
  const int r = blockIdx.x * 256 + threadIdx.x, ab = blockIdx.y, img = blockIdx.z;   // ab: block rows, then block columns
  if (r == 0 && ab == 0) counter[img] = 0u;              // the plan kernel's bump allocators (saves a memset node per call)
  if (r >= n_pad) return;
  const bool is_y = ab < blocks_y;
  M* dst = is_y ? ymask + ((size_t)img * blocks_y + ab) * n_pad : xmask + ((size_t)img * blocks_x + (ab - blocks_y)) * n_pad;
  if (r >= N) {                                        // padding reads as "touches nothing"
    dst[r] = 0;
    return;
  }
  const Crop k = load_crop(rois, dtype, (size_t)img * N + r, W, H);
  const int origin = (is_y ? ab : ab - blocks_y) * BLK;
  const int lo0 = is_y ? k.y1 : k.x1, len = is_y ? k.h : k.w;
  unsigned m = 0u;
  if (k.w > 0 && k.h > 0 && lo0 < origin + BLK && lo0 + len > origin) {
    if (MODE == FRCNN_ROI_RESIZE) {
      const float scale = (float)len / (float)P;
      for (int p = 0; p < P; ++p) {
        const Tap t = axis_tap(p, scale, len);
        if ((unsigned)(lo0 + t.lo - origin) < (unsigned)BLK || (unsigned)(lo0 + t.hi - origin) < (unsigned)BLK) m |= 1u << p;
      }
    } else {
      for (int p = 0; p < P; ++p) {
        const int a = lo0 + (p * len) / P, b = lo0 + ((p + 1) * len + P - 1) / P;
        if (a < origin + BLK && b > origin) m |= 1u << p;
      }
    }
  }
  dst[r] = (M)m;
}

// weights of the block's two rows (columns) for output index p of one axis, and which of them a tap lands on
__device__ __forceinline__ unsigned axis_weights(int p, float scale, int in_size, int origin, float& w0, float& w1) {
  const Tap t = axis_tap(p, scale, in_size);
  const int lo = origin + t.lo, hi = origin + t.hi;      // relative to the block
  const float a = 1.0f - t.lerp, b = t.lerp;
  w0 = 0.f;
  w1 = 0.f;
  unsigned hit = 0u;
  if (lo == 0) { w0 = a; hit |= 1u; }
  if (lo == 1) { w1 = a; hit |= 2u; }
  if (hi == 0) { w0 = w0 + b; hit |= 1u; }               // lo == hi (last row of a crop): both taps add up
  if (hi == 1) { w1 = w1 + b; hit |= 2u; }
  return hit;
}

// k / n for k < 64, 1 <= n <= 8 (multiply-shift, exact on that range): the narrow plan's entry decode
__constant__ unsigned short c_div_magic[9] = {0, 512, 256, 171, 128, 103, 86, 74, 64};

// One CTA per block; warp w sweeps the w-th contiguous eighth of the RoIs (so the list order is warp-major = RoI
// order).  The sweep compacts the touching RoIs of up to PLAN_ROUND RoIs into a per-warp queue; the entries are
// then produced with one LANE PER ENTRY (binary search of the entry's RoI in the queue's offsets): producing them
// with one lane per RoI left ~5 of 32 lanes busy and was 4x slower.
constexpr int PLAN_ROUND = 256;              // RoIs per queue round and warp

// PER_WARP: every warp of the CTA plans a block of its own (short RoI lists, e.g. 320 RoIs x 64 images = 38912 blocks:
// with one CTA per block the launch is a queue of tiny CTAs whose barriers and allocation round trip are exposed 260
// times per SM; with independent warps four times as many chains are in flight).
// M: the mask word.  uint8_t (P <= 8, N < 65536) packs a queued RoI into one word and decodes an entry with a
// multiply-shift division and bit clearing; uint32_t keeps the full RoI index and both masks, whose rounds can hold
// 256 RoIs x 1024 entries.
template <int MODE, typename M, int WARPS, bool PER_WARP>
__global__ void __launch_bounds__(WARPS * 32)
roi_bwd_plan_kernel(const void* __restrict__ rois, int dtype, int N, int n_pad, int H, int W, int P, int blocks_y,
                    int blocks_x, unsigned capacity, const M* __restrict__ ymask,
                    const M* __restrict__ xmask, unsigned* __restrict__ counter, int2* __restrict__ blk_tab,
                    unsigned* __restrict__ ent_idx, float4* __restrict__ ent_w) {
  constexpr bool WIDE = sizeof(M) == 4;
  using M4 = std::conditional_t<WIDE, uint4, uchar4>;
  using Rec = std::conditional_t<WIDE, uint3, unsigned>;   // narrow: RoI index | my << 16 | mx << 24; wide: (r, my, mx)
  using Start = std::conditional_t<WIDE, int, unsigned short>;
  __shared__ int s_wtot[WARPS];
  __shared__ unsigned s_wbase[WARPS];
  __shared__ Rec s_qroi[WARPS][PLAN_ROUND];
  __shared__ Start s_qstart[WARPS][PLAN_ROUND];             // first entry of the RoI inside the round
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int VW = PER_WARP ? 1 : WARPS;                  // warps that share one block's RoIs
  const int vwarp = PER_WARP ? 0 : warp;
  const int b = PER_WARP ? blockIdx.x * WARPS + warp : blockIdx.x, img = blockIdx.y, n_blocks = blocks_y * blocks_x;
  if (PER_WARP && b >= n_blocks) return;
  const int by = b / blocks_x, bx = b - by * blocks_x;
  const int Y0 = by * BLK, X0 = bx * BLK;
  const M* ym = ymask + ((size_t)img * blocks_y + by) * n_pad;
  const M* xm = xmask + ((size_t)img * blocks_x + bx) * n_pad;
  const int per_warp = ((N + VW - 1) / VW + 31) / 32 * 32;
  const int r_lo = min(n_pad, vwarp * per_warp), r_hi = min(n_pad, r_lo + per_warp);   // padding masks are zero

  // pass 1: entries of this warp's RoI range (four RoIs per lane and step)
  int mine = 0;
  for (int r = r_lo + 4 * lane; r < r_hi; r += 128) {
    const M4 a = *reinterpret_cast<const M4*>(ym + r), c = *reinterpret_cast<const M4*>(xm + r);
    mine += __popc(a.x) * __popc(c.x) + __popc(a.y) * __popc(c.y) + __popc(a.z) * __popc(c.z) + __popc(a.w) * __popc(c.w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  unsigned pos_warp;
  if (PER_WARP) {
    unsigned base = 0u;
    int total = mine;
    if (lane == 0) {
      base = atomicAdd(counter + img, (unsigned)total);
      if (base + (unsigned)total > capacity) {          // cannot happen with the launcher's bound; never write out of range
        base = 0u;
        total = 0;
      }
      base += (unsigned)img * capacity;
      blk_tab[(size_t)img * n_blocks + b] = make_int2((int)base, total);
    }
    total = __shfl_sync(0xffffffffu, total, 0);
    pos_warp = __shfl_sync(0xffffffffu, base, 0);
    if (total == 0) return;
  } else {
    if (lane == 0) s_wtot[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
      int total = 0;
      for (int i = 0; i < WARPS; ++i) total += s_wtot[i];
      // one bump counter per image
      unsigned base = atomicAdd(counter + img, (unsigned)total);
      if (base + (unsigned)total > capacity) {          // cannot happen with the launcher's bound; never write out of range
        base = 0u;
        total = 0;
      }
      base += (unsigned)img * capacity;                 // every image owns `capacity` list entries
      blk_tab[(size_t)img * n_blocks + b] = make_int2((int)base, total);
      unsigned run = base;
      for (int i = 0; i < WARPS; ++i) {
        s_wbase[i] = run;
        run += (unsigned)s_wtot[i];
      }
      if (total == 0) s_wtot[0] = -1;                   // overflow / empty marker
    }
    __syncthreads();
    if (s_wtot[0] < 0 || mine == 0) return;             // warp-uniform (mine is the reduced warp total)
    pos_warp = s_wbase[warp];
  }

  // pass 2: the entries, RoIs in index order, (ph, pw) row-major inside a RoI
  Rec* qroi = s_qroi[warp];
  Start* qstart = s_qstart[warp];
  for (int round_lo = r_lo; round_lo < r_hi; round_lo += PLAN_ROUND) {
    const int round_hi = min(r_hi, round_lo + PLAN_ROUND);
    int nq = 0, ne = 0;                                  // queued RoIs / entries of this round (warp-uniform)
    // the round's mask bytes are fetched up front: eight dependent L2 round trips became one (4.4 k -> 1.2 k cycles)
    unsigned pre_y[PLAN_ROUND / 32], pre_x[PLAN_ROUND / 32];
#pragma unroll
    for (int it = 0; it < PLAN_ROUND / 32; ++it) {
      const int r = round_lo + it * 32 + lane;
      pre_y[it] = r < round_hi ? (unsigned)ym[r] : 0u;
      pre_x[it] = r < round_hi ? (unsigned)xm[r] : 0u;
    }
#pragma unroll
    for (int it = 0; it < PLAN_ROUND / 32; ++it) {
      const int r = round_lo + it * 32 + lane;
      const unsigned my = pre_y[it], mx = pre_x[it];
      const int cnt = __popc(my) * __popc(mx);
      const unsigned hits = __ballot_sync(0xffffffffu, cnt > 0);
      if (hits == 0u) continue;
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (cnt > 0) {
        const int q = nq + __popc(hits & ((1u << lane) - 1u));
        if constexpr (WIDE) qroi[q] = make_uint3((unsigned)r, my, mx);
        else qroi[q] = (unsigned)r | (my << 16) | (mx << 24);
        qstart[q] = (Start)(ne + incl - cnt);
      }
      nq += __popc(hits);
      ne += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    // Long lists: four entries per lane and step, their chains (queue search, crop load, tap weights) independent of
    // each other; short lists (most blocks: a few dozen entries per warp) one entry per lane, or three quarters of the
    // lanes would execute the four-wide step for nothing.
    auto generate = [&](auto eu_tag) {
    constexpr int EU = decltype(eu_tag)::value;
    for (int e0 = lane; e0 < ne; e0 += 32 * EU) {
      Rec rec[EU];
      int kk[EU];
#pragma unroll
      for (int u = 0; u < EU; ++u) {
        const int e = min(e0 + 32 * u, ne - 1);          // lanes past the end repeat the last entry and do not store
        int lo = 0;                                      // last queued RoI whose first entry is <= e
#pragma unroll
        for (int step = PLAN_ROUND / 2; step > 0; step >>= 1) {
          const int mid = lo + step;
          if (mid < nq && (int)qstart[mid] <= e) lo = mid;
        }
        rec[u] = qroi[lo];
        kk[u] = e - (int)qstart[lo];
      }
#pragma unroll
      for (int u = 0; u < EU; ++u) {
        const int e = e0 + 32 * u;
        int r, ph, pw;                                   // entry k of a RoI is bin (iy-th bit of my, ix-th bit of mx)
        if constexpr (WIDE) {
          r = (int)rec[u].x;
          const unsigned my = rec[u].y, mx = rec[u].z;
          const int k = kk[u], nx = __popc(mx);
          const int iy = k / nx, ix = k - iy * nx;
          ph = (int)__fns(my, 0, iy + 1);
          pw = (int)__fns(mx, 0, ix + 1);
        } else {
          r = (int)(rec[u] & 0xffffu);
          unsigned my = (rec[u] >> 16) & 0xffu, mx = rec[u] >> 24;
          const int k = kk[u], nx = __popc(mx);
          const int iy = (int)((unsigned)k * c_div_magic[nx]) >> 9, ix = k - iy * nx;
#pragma unroll
          for (int i = 0; i < 7; ++i) {                  // masks have at most 8 bits: drop the iy / ix lowest ones
            if (i < iy) my &= my - 1u;
            if (i < ix) mx &= mx - 1u;
          }
          ph = __ffs(my) - 1;
          pw = __ffs(mx) - 1;
        }
        const unsigned row = (unsigned)((r * P + ph) * P + pw);
        const unsigned pos = pos_warp + (unsigned)e;
        const bool live = e < ne;
        if (MODE == ROI_MAX_COMPACT) {
          // the block's four cells as arg-max codes of THIS bin ((dy << 4) | dx from the bin's first cell); a cell the
          // code cannot describe (outside [0,16) in either direction) gets 0xffff, which no stored byte equals
          const Crop c = load_crop(rois, dtype, (size_t)img * N + r, W, H);
          const int ya = c.y1 + (ph * c.h) / P, xa = c.x1 + (pw * c.w) / P;
          unsigned code[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int dy = Y0 + (q >> 1) - ya, dx = X0 + (q & 1) - xa;
            code[q] = ((unsigned)dy < 16u && (unsigned)dx < 16u) ? (unsigned)((dy << 4) | dx) : 0xffffu;
          }
          if (live) {
            ent_idx[pos] = row;
            reinterpret_cast<uint4*>(ent_w)[pos] = make_uint4(code[0], code[1], code[2], code[3]);
          }
        } else if (MODE == FRCNN_ROI_RESIZE) {
          const Crop c = load_crop(rois, dtype, (size_t)img * N + r, W, H);
          float wy0, wy1, wx0, wx1;
          const unsigned hy = axis_weights(ph, (float)c.h / (float)P, c.h, c.y1 - Y0, wy0, wy1);
          const unsigned hx = axis_weights(pw, (float)c.w / (float)P, c.w, c.x1 - X0, wx0, wx1);
          const unsigned mask = ((hy & 1u) ? hx : 0u) | ((hy & 2u) ? hx << 2 : 0u);
          if (live) {
            ent_idx[pos] = row | (mask << ENT_MASK_SHIFT);
            ent_w[pos] = make_float4(__fmul_rn(wy0, wx0), __fmul_rn(wy0, wx1), __fmul_rn(wy1, wx0), __fmul_rn(wy1, wx1));
          }
        } else {
          if (live) ent_idx[pos] = row;
        }
      }
    }
    };
    if (ne > 64) generate(std::integral_constant<int, 4>());
    else generate(std::integral_constant<int, 1>());
    __syncwarp();                                        // the queue is rewritten by the next round
    pos_warp += (unsigned)ne;
  }
}

// ---------------------------------------------------------------------------------------
// streaming kernel
// ---------------------------------------------------------------------------------------
constexpr int BLK_WARPS = 8;

template <int MODE, int CPB, int D>
struct BlkSmem {
  // one ring slot: dY row (+ arg-max row: int32 = as large again, one byte per element = a quarter)
  static constexpr int ROW_F4 = CPB * 32 + (MODE == FRCNN_ROI_MAX ? CPB * 32 : (MODE == ROI_MAX_COMPACT ? CPB * 8 : 0));
  static constexpr int RING_F4 = D * ROW_F4;
  static constexpr int ENT_F4 = (MODE != FRCNN_ROI_MAX ? 64 : 0) + 16;        // 2 x 32 weights / cell codes + 2 x 32 index words
  static constexpr int WARP_F4 = RING_F4 + ENT_F4;
  static constexpr size_t BYTES = (size_t)BLK_WARPS * WARP_F4 * 16;
};

// PARTS warps share one block (each a contiguous slice of its list), 8 / PARTS blocks per CTA.
template <int MODE, int CPB, int D, int PARTS, bool FULL>
__global__ void __launch_bounds__(BLK_WARPS * 32)
roi_bwd_blk_kernel(const float* __restrict__ gout, const int* __restrict__ argmax, const int2* __restrict__ blk_tab,
                   const unsigned* __restrict__ ent_idx, const float4* __restrict__ ent_w, int H, int W, int C, int N,
                   int P, int blocks_x, int n_blocks, float* __restrict__ gfeat) {
  using S = BlkSmem<MODE, CPB, D>;
  constexpr int UNITS = BLK_WARPS / PARTS;
  static_assert(D >= 4 && D <= 16 && (D & (D - 1)) == 0, "ring depth");
  extern __shared__ float4 smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4* ring = smem + warp * S::WARP_F4;
  float4* entw = ring + S::RING_F4;                                           // resize: tap weights; compact max: cell codes
  unsigned* enti = reinterpret_cast<unsigned*>(ring + S::RING_F4 + (MODE != FRCNN_ROI_MAX ? 64 : 0));
  const int unit = blockIdx.x * UNITS + warp / PARTS, part = warp % PARTS;
  const int img = blockIdx.z;
  const bool live = unit < n_blocks;
  int begin = 0, n = 0;
  if (live) {
    const int2 tab = __ldg(blk_tab + (size_t)img * n_blocks + unit);
    const int b0 = (int)((long long)tab.y * part / PARTS), b1 = (int)((long long)tab.y * (part + 1) / PARTS);
    begin = tab.x + b0;
    n = b1 - b0;
  }
  const int Y0 = (unit / blocks_x) * BLK, X0 = (unit % blocks_x) * BLK;
  const int cbase = blockIdx.y * (CPB * 128) + 4 * lane;
  int coff[CPB];                                     // lanes beyond C read channel 0 and are never stored
#pragma unroll
  for (int j = 0; j < CPB; ++j) coff[j] = (FULL || cbase + j * 128 < C) ? cbase + j * 128 : 0;
  const size_t img_off = (size_t)img * N * P * P * C;
  const float* g_img = gout + img_off;
  const int* a_img = (MODE == FRCNN_ROI_MAX) ? argmax + img_off : nullptr;
  const unsigned char* a8_img = (MODE == ROI_MAX_COMPACT) ? reinterpret_cast<const unsigned char*>(argmax) + img_off : nullptr;
  const unsigned* ei = ent_idx + begin;
  const float4* ew = (MODE != FRCNN_ROI_MAX) ? ent_w + begin : nullptr;

  float4 acc[4][CPB];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int j = 0; j < CPB; ++j) acc[q][j] = make_float4(0.f, 0.f, 0.f, 0.f);
  int cellid[4];                                     // max mode: flat index of the block's cells (-1 outside the map)
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int y = Y0 + (q >> 1), x = X0 + (q & 1);
    cellid[q] = (y < H && x < W) ? y * W + x : -1;
  }

  auto fetch_batch = [&](int b) {
    const int e = 32 * b + lane;
    if (e < n) {
      if (MODE != FRCNN_ROI_MAX) cp_async16(entw + (b & 1) * 32 + lane, ew + e);
      cp_async4(enti + (b & 1) * 32 + lane, ei + e);
    }
  };
  // request the dY (and arg-max) row of list entry i into ring slot `s`; predicated, not branched: entries past the
  // end of the list are simply not loaded (the stale index word they would use is never dereferenced)
  auto issue_row = [&](int i, int s) {
    const unsigned row = enti[i & 63] & ENT_IDX_MASK;  // entry buffers: 2 x 32 entries back to back
    const size_t off = (size_t)row * C;
    const bool p = i < n;
    float4* slot = ring + s * S::ROW_F4 + lane;
#pragma unroll
    for (int j = 0; j < CPB; ++j) {
      cp_async16_if(slot + j * 32, g_img + off + coff[j], p);
      if (MODE == FRCNN_ROI_MAX) cp_async16_if(slot + (CPB + j) * 32, a_img + off + coff[j], p);
      if (MODE == ROI_MAX_COMPACT)
        cp_async4_if(reinterpret_cast<unsigned*>(ring + s * S::ROW_F4 + CPB * 32) + j * 32 + lane, a8_img + off + coff[j], p);
    }
  };
  // add list entry i (its rows sit in ring slot `s`) into the four cells
  auto consume = [&](int i, int s) {
    const float4* slot = ring + s * S::ROW_F4 + lane;
    if (MODE == FRCNN_ROI_RESIZE) {
      const float4 w = entw[i & 63];
      const unsigned mask = enti[i & 63] >> ENT_MASK_SHIFT;
      unsigned long long g2[CPB][2];
#pragma unroll
      for (int j = 0; j < CPB; ++j) {
        const float4 g = slot[j * 32];
        g2[j][0] = pack2(g.x, g.y);
        g2[j][1] = pack2(g.z, g.w);
      }
      // the tap weight wy*wx was formed by the plan kernel; one packed FMA per element pair and cell
#define FRCNN_BLK_ACCUM(Q, WV)                                                                  \
  if (mask & (1u << (Q))) {                                                                      \
    const unsigned long long ww = pack2(WV, WV);                                                 \
    _Pragma("unroll") for (int j = 0; j < CPB; ++j) {                                            \
      unpack2(fma2(g2[j][0], ww, pack2(acc[Q][j].x, acc[Q][j].y)), acc[Q][j].x, acc[Q][j].y);     \
      unpack2(fma2(g2[j][1], ww, pack2(acc[Q][j].z, acc[Q][j].w)), acc[Q][j].z, acc[Q][j].w);     \
    }                                                                                            \
  }
      FRCNN_BLK_ACCUM(0, w.x)
      FRCNN_BLK_ACCUM(1, w.y)
      FRCNN_BLK_ACCUM(2, w.z)
      FRCNN_BLK_ACCUM(3, w.w)
#undef FRCNN_BLK_ACCUM
    } else if (MODE == ROI_MAX_COMPACT) {
      const uint4 code = *reinterpret_cast<const uint4*>(entw + (i & 63));
      const unsigned cq[4] = {code.x, code.y, code.z, code.w};
#pragma unroll
      for (int j = 0; j < CPB; ++j) {
        const float4 g = slot[j * 32];
        const unsigned a = (reinterpret_cast<const unsigned*>(ring + s * S::ROW_F4 + CPB * 32) + j * 32)[lane];
        const unsigned ax = a & 0xffu, ay = (a >> 8) & 0xffu, az = (a >> 16) & 0xffu, aw = a >> 24;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (ax == cq[q]) acc[q][j].x += g.x;
          if (ay == cq[q]) acc[q][j].y += g.y;
          if (az == cq[q]) acc[q][j].z += g.z;
          if (aw == cq[q]) acc[q][j].w += g.w;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < CPB; ++j) {
        const float4 g = slot[j * 32];
        const int4 a = *reinterpret_cast<const int4*>(slot + (CPB + j) * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (a.x == cellid[q]) acc[q][j].x += g.x;
          if (a.y == cellid[q]) acc[q][j].y += g.y;
          if (a.z == cellid[q]) acc[q][j].z += g.z;
          if (a.w == cellid[q]) acc[q][j].w += g.w;
        }
      }
    }
  };

  if (n > 0) {                                       // warp-uniform
    fetch_batch(0);
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
    fetch_batch(1);
    cp_async_commit();
#pragma unroll
    for (int s = 0; s < D; ++s) {
      issue_row(s, s);
      cp_async_commit();
    }
    // groups of D entries: ring slots and the batch hand-over points are compile-time positions inside a group.
    // Entry batch i/32 + 1 was committed >= D groups before the first issue_row that reads it (D <= 16), so it
    // has landed for the copying lane; the __syncwarp makes it visible to the other lanes.
    int i0 = 0;
    for (; i0 + D <= n; i0 += D) {
      const bool handover = (i0 & 31) == 32 - D;      // this group ends a batch of 32 entries
      if (handover) __syncwarp();
#pragma unroll
      for (int u = 0; u < D; ++u) {
        cp_async_wait<D - 1>();                       // row i0 + u has landed
        consume(i0 + u, u);
        if (u == D - 1 && handover) {                 // batch i0/32 is consumed: its buffer takes batch i0/32 + 2
          __syncwarp();
          fetch_batch((i0 >> 5) + 2);
        }
        issue_row(i0 + u + D, u);
        cp_async_commit();
      }
    }
    if (i0 < n) {                                     // ragged tail: fewer than D entries, everything already requested
      cp_async_wait<0>();
      if ((i0 & 31) == 32 - D) __syncwarp();
      for (int i = i0; i < n; ++i) consume(i, i & (D - 1));
    }
    cp_async_wait<0>();
  }

  if (PARTS == 1) {
    if (!live) return;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (cellid[q] < 0) continue;
      float* dst = gfeat + ((size_t)img * H * W + cellid[q]) * C + cbase;
#pragma unroll
      for (int j = 0; j < CPB; ++j)
        if (FULL || cbase + j * 128 < C) *reinterpret_cast<float4*>(dst + j * 128) = acc[q][j];
    }
    return;
  }
  // slices of one block are added in slice order through shared memory (the rings are drained and reused)
  __syncthreads();
  float4* red = smem;                                // [warp][4 * CPB][32]
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int j = 0; j < CPB; ++j) red[(warp * (4 * CPB) + q * CPB + j) * 32 + lane] = acc[q][j];
  __syncthreads();
  if (!live) return;
  for (int item = part; item < 4 * CPB; item += PARTS) {
    const int q = item / CPB, j = item - q * CPB;
    const int y = Y0 + (q >> 1), x = X0 + (q & 1);
    if (y >= H || x >= W || !(FULL || cbase + j * 128 < C)) continue;
    float4 s = red[((warp - part) * (4 * CPB) + item) * 32 + lane];
    for (int p2 = 1; p2 < PARTS; ++p2) {
      const float4 v = red[((warp - part + p2) * (4 * CPB) + item) * 32 + lane];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    *reinterpret_cast<float4*>(gfeat + ((size_t)img * H * W + (size_t)y * W + x) * C + cbase + j * 128) = s;
  }
}

template <int MODE, int CPB, int D, int PARTS, bool FULL>
static int launch_blk_one(frcnn_handle* h, cudaStream_t stream, dim3 grid, const float* gout, const int* argmax,
                          const int2* tab, const unsigned* ent_idx, const float4* ent_w, int H, int W, int C, int N,
                          int P, int blocks_x, int n_blocks, float* gfeat) {
  using S = BlkSmem<MODE, CPB, D>;
  auto kern = roi_bwd_blk_kernel<MODE, CPB, D, PARTS, FULL>;
  FRCNN_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::BYTES));
  kern<<<grid, BLK_WARPS * 32, S::BYTES, stream>>>(gout, argmax, tab, ent_idx, ent_w, H, W, C, N, P, blocks_x, n_blocks,
                                                   gfeat);
  FRCNN_LAUNCH_CHECK(h, "roi_bwd_blk_kernel");
  return FRCNN_OK;
}

template <int MODE, int CPB, int D, bool FULL>
static int launch_blk_parts(frcnn_handle* h, cudaStream_t stream, int parts, int slabs, int batch, const float* gout,
                            const int* argmax, const int2* tab, const unsigned* ent_idx, const float4* ent_w, int H,
                            int W, int C, int N, int P, int blocks_x, int n_blocks, float* gfeat) {
#define FRCNN_BLK_CASE(PARTS)                                                                                       \
  case PARTS:                                                                                                       \
    return launch_blk_one<MODE, CPB, D, PARTS, FULL>(                                                               \
        h, stream, dim3((n_blocks + BLK_WARPS / PARTS - 1) / (BLK_WARPS / PARTS), slabs, batch), gout, argmax, tab,  \
        ent_idx, ent_w, H, W, C, N, P, blocks_x, n_blocks, gfeat);
  switch (parts) {
    FRCNN_BLK_CASE(1)
    FRCNN_BLK_CASE(2)
    FRCNN_BLK_CASE(4)
    default:
    FRCNN_BLK_CASE(8)
  }
#undef FRCNN_BLK_CASE
}

// upper bound of the work-list entries of a launch: a resize bin has taps in <= 2 x 2 blocks; a max bin spans
// <= ceil(H/P)+1 rows and columns
static long long work_list_entries(int mode, int H, int W, int N, int P, int batch) {
  long long per_bin = 4;
  if (mode == FRCNN_ROI_MAX) {
    const long long ly = (H + P - 1) / P + 1, lx = (W + P - 1) / P + 1;
    per_bin = (ly / BLK + 1) * (lx / BLK + 1);
  }
  return (long long)batch * N * P * P * per_bin;
}

// true when the work-list path takes this problem: float4 channels, masks of at most 32 bits, dY row indices that fit
// the entry word and list positions that fit an int
static bool roi_bwd_blk_eligible(int mode, int H, int W, int C, int N, int P, int batch) {
  return C % 4 == 0 && P <= ROI_MAX_TABLE_P && H < 32768 && W < 32768 && (long long)N * P * P < (1LL << ENT_MASK_SHIFT) &&
         work_list_entries(mode, H, W, N, P, batch) < (1LL << 31);
}

// mask + plan kernels; plan CTAs: 8 warps sweep 2000 RoIs in one queue round each, short RoI lists take smaller CTAs
// (38912 of them at C1 x 64)
template <int MODE, typename M>
static void launch_plan(cudaStream_t stream, const void* rois, int dtype, int N, int n_pad, int H, int W, int P,
                        int blocks_y, int blocks_x, int batch, unsigned capacity, void* ym, void* xm, unsigned* counter,
                        int2* tab, unsigned* ent_idx, float4* ent_w) {
  constexpr int MASK_MODE = MODE == FRCNN_ROI_RESIZE ? FRCNN_ROI_RESIZE : FRCNN_ROI_MAX;
  M *y = static_cast<M*>(ym), *x = static_cast<M*>(xm);
  const int n_blocks = blocks_y * blocks_x;
  roi_bwd_mask_kernel<MASK_MODE, M><<<dim3((n_pad + 255) / 256, blocks_y + blocks_x, batch), 256, 0, stream>>>(
      rois, dtype, N, n_pad, H, W, P, blocks_y, blocks_x, y, x, counter);
  if (N > 1024)
    roi_bwd_plan_kernel<MODE, M, 8, false><<<dim3(n_blocks, batch), 256, 0, stream>>>(
        rois, dtype, N, n_pad, H, W, P, blocks_y, blocks_x, capacity, y, x, counter, tab, ent_idx, ent_w);
  else if (N > 512)
    roi_bwd_plan_kernel<MODE, M, 4, false><<<dim3(n_blocks, batch), 128, 0, stream>>>(
        rois, dtype, N, n_pad, H, W, P, blocks_y, blocks_x, capacity, y, x, counter, tab, ent_idx, ent_w);
  else
    roi_bwd_plan_kernel<MODE, M, 8, true><<<dim3((n_blocks + 7) / 8, batch), 256, 0, stream>>>(
        rois, dtype, N, n_pad, H, W, P, blocks_y, blocks_x, capacity, y, x, counter, tab, ent_idx, ent_w);
}

static int launch_roi_bwd_blk(frcnn_handle* h, cudaStream_t stream, int mode, const float* gout, const void* rois,
                              int dtype, const int32_t* argmax, int H, int W, int C, int N, int P, int batch, float* gfeat,
                              int compact) {
  const int blocks_x = (W + BLK - 1) / BLK, blocks_y = (H + BLK - 1) / BLK, n_blocks = blocks_x * blocks_y;
  const long long cap = work_list_entries(mode, H, W, N, P, batch);
  const bool wide = P > 8 || N >= 65536;               // the narrow plan's masks are bytes, its queue keeps 16-bit RoIs
  const size_t mask_bytes = wide ? sizeof(uint32_t) : sizeof(uint8_t);
  const int n_pad = (N + 15) / 16 * 16;
  void *p_cnt = nullptr, *p_tab = nullptr, *p_idx = nullptr, *p_w = nullptr, *p_ym = nullptr, *p_xm = nullptr;
  int rc;
  if ((rc = arena_get(h, stream, align_up((size_t)batch * sizeof(unsigned), 256), &p_cnt))) return rc;
  if ((rc = arena_get(h, stream, (size_t)batch * n_blocks * sizeof(int2), &p_tab))) return rc;
  if ((rc = arena_get(h, stream, (size_t)batch * blocks_y * n_pad * mask_bytes, &p_ym))) return rc;
  if ((rc = arena_get(h, stream, (size_t)batch * blocks_x * n_pad * mask_bytes, &p_xm))) return rc;
  if ((rc = arena_get(h, stream, (size_t)cap * sizeof(unsigned), &p_idx))) return rc;
  if ((mode == FRCNN_ROI_RESIZE || compact) && (rc = arena_get(h, stream, (size_t)cap * sizeof(float4), &p_w))) return rc;
  int2* tab = static_cast<int2*>(p_tab);
  unsigned* eidx = static_cast<unsigned*>(p_idx);
  float4* ew = static_cast<float4*>(p_w);
#define FRCNN_PLAN(MODE, M)                                                                                        \
  launch_plan<MODE, M>(stream, rois, dtype, N, n_pad, H, W, P, blocks_y, blocks_x, batch, (unsigned)(cap / batch), \
                       p_ym, p_xm, static_cast<unsigned*>(p_cnt), tab, eidx, ew)
  if (compact) FRCNN_PLAN(ROI_MAX_COMPACT, uint8_t);   // launch_roi_bwd: the one-byte arg-max has P <= 8, N < 65536
  else if (mode == FRCNN_ROI_RESIZE) { if (wide) FRCNN_PLAN(FRCNN_ROI_RESIZE, uint32_t); else FRCNN_PLAN(FRCNN_ROI_RESIZE, uint8_t); }
  else if (wide) FRCNN_PLAN(FRCNN_ROI_MAX, uint32_t);
  else FRCNN_PLAN(FRCNN_ROI_MAX, uint8_t);
#undef FRCNN_PLAN
  FRCNN_LAUNCH_CHECK(h, "roi_bwd_mask_kernel");
  FRCNN_LAUNCH_CHECK(h, "roi_bwd_plan_kernel");

  // (channels per lane, ring depth): 2 x 8 = 8 KB of dY in flight per warp where 256 channels exist; the int32 max mode
  // carries an arg-max row as large as the dY row and keeps 1 x 8 (same-box A/B on a B200, C5 x 8: resize 0.66 ms
  // against 0.68 (2 x 4) / 0.75 (1 x 8) / 0.80 (1 x 16); max 1.32 against 1.30 (2 x 4) / 1.56 (1 x 4); one-byte
  // arg-max 1.15 (2 x 8) against 1.25 (2 x 4) / 1.40 (1 x 8)).
  int cpb = C >= 256 ? 2 : 1;
  if (mode == FRCNN_ROI_MAX && !compact) cpb = 1;
  const int slabs = (C + cpb * 128 - 1) / (cpb * 128);
  const bool full = C % (cpb * 128) == 0;
  // slices per block: enough warps for ~4 waves of 24 resident warps per SM, at most 8
  const long long units = (long long)n_blocks * batch * slabs;
  const long long want = 4LL * 24 * h->sm_count;
  int parts = units >= want ? 1 : (units * 2 >= want ? 2 : (units * 4 >= want ? 4 : 8));
  // long lists are also sliced in large launches: the eight warps of a CTA then work on 8 / parts blocks in equal
  // shares instead of on eight blocks of unequal length (C5 x 8: 0.77 -> 0.63 ms with four slices)
  const long long avg_list = (long long)N * P * P * (mode == FRCNN_ROI_MAX ? 3 : 2) / n_blocks;
  if (parts < 4 && avg_list >= 256) parts = 4;
  else if (parts < 2 && avg_list >= 128) parts = 2;
  if (N < 256) parts = 1;                              // short lists: one warp walks the whole list (reference order)
#define FRCNN_BLK_GO(MODE, CPB, D)                                                                                   \
  return full ? launch_blk_parts<MODE, CPB, D, true>(h, stream, parts, slabs, batch, gout, argmax, tab, eidx, ew, H, \
                                                     W, C, N, P, blocks_x, n_blocks, gfeat)                         \
              : launch_blk_parts<MODE, CPB, D, false>(h, stream, parts, slabs, batch, gout, argmax, tab, eidx, ew,  \
                                                      H, W, C, N, P, blocks_x, n_blocks, gfeat);
  if (mode == FRCNN_ROI_RESIZE) {
    if (cpb == 2) { FRCNN_BLK_GO(FRCNN_ROI_RESIZE, 2, 8) }
    FRCNN_BLK_GO(FRCNN_ROI_RESIZE, 1, 8)
  }
  if (compact) {
    if (cpb == 2) { FRCNN_BLK_GO(ROI_MAX_COMPACT, 2, 8) }
    FRCNN_BLK_GO(ROI_MAX_COMPACT, 1, 8)
  }
  FRCNN_BLK_GO(FRCNN_ROI_MAX, 1, 8)
#undef FRCNN_BLK_GO
}

// ---------------------------------------------------------------------------------------
// scalar-channel fallback for the problems roi_bwd_blk_eligible rejects (C % 4 != 0, pool sizes above
// ROI_MAX_TABLE_P, ...) and unaligned buffers: 8x8 tile, one channel per thread, every CTA scans all RoIs.
// Not a performance path.
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

int launch_roi_bwd(frcnn_handle* h, cudaStream_t stream, int mode, const float* gout, const void* rois, int dtype,
                   const int32_t* argmax, int H, int W, int C, int N, int P, int batch, float* gfeat, int compact) {
  if (compact) {
    const bool ok = mode == FRCNN_ROI_MAX && P <= 8 && N < 65536 && roi_compact_supported(H, W, C, P) &&
                    roi_bwd_blk_eligible(mode, H, W, C, N, P, batch) &&
                    (reinterpret_cast<uintptr_t>(gout) % 16 == 0) && (reinterpret_cast<uintptr_t>(gfeat) % 16 == 0) &&
                    (reinterpret_cast<uintptr_t>(argmax) % 4 == 0);
    if (!ok) return fail(h, FRCNN_ERR_UNSUPPORTED, "roi_bwd: compact arg-max needs max mode, C %% 4 == 0, pool <= 8, fewer than 65536 RoIs, bins of at most 16 x 16 cells and a work list below 2^31 entries%s%s");
    return launch_roi_bwd_blk(h, stream, mode, gout, rois, dtype, argmax, H, W, C, N, P, batch, gfeat, 1);
  }
  const bool aligned = (reinterpret_cast<uintptr_t>(gout) % 16 == 0) && (reinterpret_cast<uintptr_t>(gfeat) % 16 == 0) &&
                       (mode != FRCNN_ROI_MAX || reinterpret_cast<uintptr_t>(argmax) % 16 == 0);
  if (aligned && roi_bwd_blk_eligible(mode, H, W, C, N, P, batch))
    return launch_roi_bwd_blk(h, stream, mode, gout, rois, dtype, argmax, H, W, C, N, P, batch, gfeat, 0);
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
