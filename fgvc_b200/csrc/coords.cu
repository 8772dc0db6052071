// K3: bilinear up-sampling fused with img2coord (top-5 soft-argmax), the analytic
// frame-0 gaussian variant, and the VOS-style mask decode.  HBM-bound on the feature-res
// maps only: the full-resolution [T,P,h,w] tensor the reference ships to the host
// (vanilla_tracker.py:396-406) is never materialised.
#include "common.cuh"

namespace fgvc {

// F.interpolate(mode='bilinear', align_corners=False) source coordinates
struct Lerp {
  int i0, i1;
  float w1;
};
__device__ __forceinline__ Lerp lerp_coord(int dst, float scale, int in_size) {
  float s = fmaxf(((float)dst + 0.5f) * scale - 0.5f, 0.f);
  int i0 = min((int)s, in_size - 1);
  Lerp l;
  l.i0 = i0;
  l.i1 = min(i0 + 1, in_size - 1);
  l.w1 = s - (float)i0;
  return l;
}

struct BilinearSrc {
  const float* m;  // [H][W] (shared or global)
  int H, W;
  float sy, sx;
  __device__ __forceinline__ float at(int oy, int ox) const {
    Lerp ly = lerp_coord(oy, sy, H), lx = lerp_coord(ox, sx, W);
    float w0x = 1.f - lx.w1, w0y = 1.f - ly.w1;
    const float* r0 = m + ly.i0 * W;
    const float* r1 = m + ly.i1 * W;
    return w0y * (w0x * r0[lx.i0] + lx.w1 * r0[lx.i1]) + ly.w1 * (w0x * r1[lx.i0] + lx.w1 * r1[lx.i1]);
  }
};

struct GaussSrc {
  float cx, cy, denom;
  __device__ __forceinline__ float at(int oy, int ox) const {
    float dx = (float)ox - cx, dy = (float)oy - cy;
    return expf(__fdiv_rn(-(dx * dx + dy * dy), denom));
  }
};

constexpr int CK = 8;  // candidates kept per thread (>= img2coord topk)

// (value, index) ordering used by the soft-argmax: larger value first, exact ties -> higher index
// first (what a stable ascending argsort read from the back gives; np.argsort in img2coord)
__device__ __forceinline__ bool key_gt(float v, int i, float w, int j) { return v > w || (v == w && i > j); }

// sorted insert under that ordering; independent of the order in which pixels are visited
template <int K>
__device__ __forceinline__ void push_key(TopK<K>& t, float x, int i) {
  if (!key_gt(x, i, t.v[K - 1], t.id[K - 1])) return;
  bool c[K];
#pragma unroll
  for (int j = 0; j < K; ++j) c[j] = key_gt(x, i, t.v[j], t.id[j]);
#pragma unroll
  for (int j = K - 1; j > 0; --j) {
    t.v[j] = c[j - 1] ? t.v[j - 1] : (c[j] ? x : t.v[j]);
    t.id[j] = c[j - 1] ? t.id[j - 1] : (c[j] ? i : t.id[j]);
  }
  t.v[0] = c[0] ? x : t.v[0];
  t.id[0] = c[0] ? i : t.id[0];
}

// Block-wide selection of the `topk` best (value, index) pairs from the per-thread sorted lists:
// topk rounds of block arg-max over the list heads.  Results in win_v / win_i (shared).
__device__ void block_topk(const TopK<CK>& top, int topk, float* win_v, int* win_i) {
  __shared__ float red_v[8];
  __shared__ int red_i[8];
  __shared__ int red_t[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int head = 0;
  for (int r = 0; r < topk; ++r) {
    float v = -INFINITY;
    int i = -1;
#pragma unroll
    for (int j = 0; j < CK; ++j)
      if (j == head) { v = top.v[j]; i = top.id[j]; }
    int t = tid;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, v, o);
      int oi = __shfl_xor_sync(0xffffffffu, i, o);
      int ot = __shfl_xor_sync(0xffffffffu, t, o);
      if (key_gt(ov, oi, v, i)) { v = ov; i = oi; t = ot; }
    }
    __syncthreads();
    if (lane == 0) { red_v[warp] = v; red_i[warp] = i; red_t[warp] = t; }
    __syncthreads();
    float bv = red_v[0]; int bi = red_i[0], bt = red_t[0];
#pragma unroll
    for (int w = 1; w < 8; ++w)
      if (key_gt(red_v[w], red_i[w], bv, bi)) { bv = red_v[w]; bi = red_i[w]; bt = red_t[w]; }
    if (tid == bt) ++head;
    if (tid == 0) { win_v[r] = bv; win_i[r] = bi; }
  }
  __syncthreads();
}

// img2coord on the winners (vanilla_tracker.py:181-190): ascending order, fp32 sum + 1e-9, fp32
// weights, fp64 weighted mean of (idx % w, idx // w); an all-zero map gives -1
__device__ void write_coords(const float* win_v, const int* win_i, int topk, int out_w, bool nonzero, float* out_xy) {
  float x = -1.f, y = -1.f;
  if (nonzero) {
    float s = 0.f;
    for (int r = topk - 1; r >= 0; --r) s += win_v[r];
    s += 1e-9f;
    double ax = 0.0, ay = 0.0;
    for (int r = topk - 1; r >= 0; --r) {
      double w = (double)__fdiv_rn(win_v[r], s);
      ax += (double)(win_i[r] % out_w) * w;
      ay += (double)(win_i[r] / out_w) * w;
    }
    x = (float)ax; y = (float)ay;
  }
  out_xy[0] = x; out_xy[1] = y;
}

// brute-force soft-argmax over an implicit out_h x out_w map (used for the analytic gaussian)
template <class Src>
__device__ void soft_argmax_block(const Src& src, int out_h, int out_w, int topk, float* out_xy) {
  __shared__ double red_s[8];
  __shared__ float win_v[CK];
  __shared__ int win_i[CK];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  TopK<CK> top;
  top.init();
  double sum = 0.0;
  const int total = out_h * out_w;
  for (int o = tid; o < total; o += 256) {
    int oy = o / out_w, ox = o - oy * out_w;
    float v = src.at(oy, ox);
    sum += (double)v;
    push_key(top, v, o);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) red_s[warp] = sum;
  block_topk(top, topk, win_v, win_i);
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < 8; ++w) tot += red_s[w];
    write_coords(win_v, win_i, topk, out_w, tot != 0.0, out_xy);   // np.sum(map) == 0 -> -1
  }
}

// first / last output index whose source cell (floor of the clamped source coordinate) is i0
__device__ __forceinline__ void cell_range(int i0, int in_size, int out_size, float scale, int* lo, int* hi) {
  // lerp_coord(o).i0 is non-decreasing in o: locate the run of outputs that map to i0 by search
  // around the analytic estimate (scale = in/out, src = (o + 0.5) * scale - 0.5)
  int g = (int)floorf(((float)i0 + 0.5f) / scale - 0.5f);
  g = max(0, min(out_size - 1, g));
  while (g > 0 && lerp_coord(g - 1, scale, in_size).i0 >= i0) --g;
  while (g < out_size - 1 && lerp_coord(g, scale, in_size).i0 < i0) ++g;
  *lo = g;                       // first o with i0(o) >= i0
  // last o with i0(o) <= i0: analytic estimate (the last rows / columns all clamp to in_size - 1), then the same
  // exact correction by search
  int h = i0 >= in_size - 1 ? out_size - 1 : (int)ceilf(((float)i0 + 1.5f) / scale - 0.5f) - 1;
  h = max(g, min(out_size - 1, h));
  while (h > g && lerp_coord(h, scale, in_size).i0 > i0) --h;
  while (h < out_size - 1 && lerp_coord(h + 1, scale, in_size).i0 <= i0) ++h;
  *hi = h;
}

// Soft-argmax of the bilinearly up-sampled map WITHOUT evaluating every output pixel.  An up-sampled
// value is a convex combination of its 4 taps, so it cannot exceed their maximum:
//   1. seed: the largest SOURCE pixel (found while the map is streamed); the 5 x 5 output pixels nearest to it are
//      evaluated; tau = the topk-th best up-sampled value found there -- `topk` distinct outputs
//      reach it, so it is a lower bound of the final topk-th value, whatever set of outputs was looked at;
//   2. scan the source cells; only cells whose largest tap reaches tau (minus a rounding margin) can hold a
//      winner -- evaluate just those (each output belongs to exactly one cell, so none is seen twice).
// Peaked heat-maps touch a handful of cells; a flat map degrades to the full evaluation.  Exact.
// Zero test: labels are non-negative (convex combinations of gaussians / one-hots), for which
// "sum of the up-sampled map == 0" <=> "every source value is 0".
// ONE WARP PER MAP, no block barriers: the map is streamed from global memory once (16-byte loads: arg-max, zero
// test, and the maximum of each of a lane's <= 32 load slots, kept in shared memory); step 2 re-reads only the
// slots whose maximum reaches tau.  8 maps per CTA progress independently, so the serial part of one map (seed
// rectangle, selections) hides behind the others.
// (The first version -- one CTA per map staged in shared memory, 5 seeds, three block-wide selections, the seeds'
// output ranges searched by every thread, a division per cell -- took 11 k instructions per thread and 35 ms for
// the 255 k maps of a 250-frame, 1024-point clip; this one takes ~3 ms, the time to read the maps.)

// warp-wide selection of the `topk` best pairs from the lanes' sorted lists -> win_v / win_i (lane 0 writes)
__device__ __forceinline__ void warp_topk(const TopK<CK>& top, int topk, float* win_v, int* win_i) {
  const int lane = threadIdx.x & 31;
  int head = 0;
  for (int r = 0; r < topk; ++r) {
    float v = -INFINITY;
    int i = -1;
#pragma unroll
    for (int j = 0; j < CK; ++j)
      if (j == head) { v = top.v[j]; i = top.id[j]; }
    int t = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, v, o);
      const int oi = __shfl_xor_sync(0xffffffffu, i, o);
      const int ot = __shfl_xor_sync(0xffffffffu, t, o);
      if (key_gt(ov, oi, v, i)) { v = ov; i = oi; t = ot; }
    }
    if (lane == t) ++head;
    if (lane == 0) { win_v[r] = v; win_i[r] = i; }
  }
  __syncwarp();
}

// step 2 for one hot pixel: list the cells it is a tap of (each cell from its first hot tap only) with their output
// ranges in the warp's shared list; a cell that does not fit is evaluated on the spot
constexpr int CELL_CAP = 128;
// (only outputs that reach tau can be winners: the lists then see a handful of insertions instead of filling up)
__device__ __forceinline__ void eval_cell(const BilinearSrc& src, int y0, int y1, int x0, int x1, int out_w,
                                          float tau_safe, TopK<CK>& top) {
  for (int oy = y0; oy <= y1; ++oy)
    for (int ox = x0; ox <= x1; ++ox) {
      const float v = src.at(oy, ox);
      if (v >= tau_safe) push_key(top, v, oy * out_w + ox);
    }
}
__device__ __forceinline__ void list_hot_cells(const BilinearSrc& src, int i, float tau_safe, int out_h, int out_w,
                                               uint2* cells, int* n_cells, TopK<CK>& top) {
  const float* m = src.m;
  const int H = src.H, W = src.W;
  const int pi = i / W, pj = i - pi * W;
  for (int d = 0; d < 4; ++d) {
    const int di = d >> 1, dj = d & 1;
    const int i0 = pi - di, j0 = pj - dj;
    if (i0 < 0 || j0 < 0) continue;
    bool earlier = false;                      // an earlier tap (i0 + ei, j0 + ej), (ei, ej) < (di, dj), is hot too
    for (int e = 0; e < d; ++e) earlier |= __ldg(m + (i0 + (e >> 1)) * W + min(j0 + (e & 1), W - 1)) >= tau_safe;
    if (earlier) continue;
    int y0, y1, x0, x1;
    cell_range(i0, H, out_h, src.sy, &y0, &y1);
    cell_range(j0, W, out_w, src.sx, &x0, &x1);
    if (lerp_coord(y0, src.sy, H).i0 != i0 || lerp_coord(x0, src.sx, W).i0 != j0) continue;   // cell without outputs
    const int slot = (out_h <= 65535 && out_w <= 65535) ? atomicAdd(n_cells, 1) : CELL_CAP;
    if (slot < CELL_CAP) cells[slot] = make_uint2((uint32_t)y0 | ((uint32_t)y1 << 16), (uint32_t)x0 | ((uint32_t)x1 << 16));
    else eval_cell(src, y0, y1, x0, x1, out_w, tau_safe, top);
  }
}

constexpr int MAPS_PER_CTA = 8;
constexpr int SLOTS = 32;          // per-lane slot maxima kept in shared memory (4 KB per map)

// blockDim.x / 32 maps per CTA (<= MAPS_PER_CTA)
__global__ void __launch_bounds__(32 * MAPS_PER_CTA, 4)
heatmap_coords_kernel(const float* __restrict__ maps, int n_maps, int H, int W, int out_h, int out_w, int topk,
                      float* __restrict__ out_xy) {
  __shared__ float win_v_s[MAPS_PER_CTA][CK];
  __shared__ int win_i_s[MAPS_PER_CTA][CK];
  __shared__ float slot_max_s[MAPS_PER_CTA][SLOTS * 32];
  __shared__ uint2 cells_s[MAPS_PER_CTA][CELL_CAP];
  __shared__ int n_cells_s[MAPS_PER_CTA];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int map = blockIdx.x * (blockDim.x >> 5) + warp;
  if (map >= n_maps) return;
  float* win_v = win_v_s[warp];
  int* win_i = win_i_s[warp];
  const float* m = maps + (int64_t)map * H * W;
  out_xy += 2 * (int64_t)map;
  const int n = H * W;
  // ---- 0. stream the map once: arg-max, zero test, and the maximum of every SLOT (a lane's pixels are cut into
  // <= 32 slots of consecutive loads) kept in shared memory, so that step 2 re-reads only the slots that can
  // hold a hot pixel
  float* slot_max = slot_max_s[warp];
  const bool vec = (n & 3) == 0 && (reinterpret_cast<uintptr_t>(m) & 15) == 0;
  const int n_it = vec ? ((n >> 2) + 127) / 128 : (n + 127) / 128;    // iterations of 4 loads per lane
  const int per_slot = (n_it + SLOTS - 1) / SLOTS;
  float bv = -INFINITY, mn = INFINITY;
  int bi = 0;
  for (int s0 = 0, slot = 0; s0 < n_it; s0 += per_slot, ++slot) {
    float smx = -INFINITY;
    for (int it = s0; it < min(s0 + per_slot, n_it); ++it) {
      if (vec) {
        const float4* m4 = reinterpret_cast<const float4*>(m);
        const int n4 = n >> 2;
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldg(m4 + min(it * 128 + 32 * u + lane, n4 - 1));   // clamped: a repeat
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float mx = fmaxf(fmaxf(v[u].x, v[u].y), fmaxf(v[u].z, v[u].w));
          mn = fminf(mn, fminf(fminf(v[u].x, v[u].y), fminf(v[u].z, v[u].w)));
          smx = fmaxf(smx, mx);
          if (mx > bv) { bv = mx; bi = min(it * 128 + 32 * u + lane, n4 - 1); }
        }
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = min(it * 128 + 32 * u + lane, n - 1);
          const float v = __ldg(m + i);
          mn = fminf(mn, v);
          smx = fmaxf(smx, v);
          if (v > bv) { bv = v; bi = i; }
        }
      }
    }
    slot_max[slot * 32 + lane] = smx;
  }
  if (vec) {                                     // which of the 4 pixels of the best load
    const float4 v = __ldg(reinterpret_cast<const float4*>(m) + bi);
    bi = 4 * bi + (v.x == bv ? 0 : (v.y == bv ? 1 : (v.z == bv ? 2 : 3)));
  }
  // every value is 0 <=> min == 0 and max == 0
  if (!__any_sync(0xffffffffu, !(mn == 0.f && bv == 0.f))) {   // np.sum(map) == 0 -> (-1, -1)
    if (lane == 0) { out_xy[0] = -1.f; out_xy[1] = -1.f; }
    return;
  }
  // the largest source pixel
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv) { bv = ov; bi = oi; }
  }
  const BilinearSrc src{m, H, W, (float)H / (float)out_h, (float)W / (float)out_w};
  // ---- 1. tau from the output pixels around the seed (any distinct outputs give a valid lower bound)
  TopK<CK> top;
  top.init();
  {
    const int sy = bi / W, sx = bi - sy * W;
    // (the 5 x 5 outputs nearest to the seed pixel's centre: one per lane)
    const int ry = 2, rx = 2;
    const int cy = (int)(((float)sy + 0.5f) / src.sy), cx = (int)(((float)sx + 0.5f) / src.sx);
    const int y0 = max(cy - ry, 0), y1 = min(cy + ry, out_h - 1), x0 = max(cx - rx, 0), x1 = min(cx + rx, out_w - 1);
    const int nx = x1 - x0 + 1, cnt = (y1 - y0 + 1) * nx;
    for (int i = lane; i < cnt; i += 32) {
      const int oy = y0 + i / nx, ox = x0 + i % nx;
      push_key(top, src.at(oy, ox), oy * out_w + ox);
    }
  }
  warp_topk(top, topk, win_v, win_i);
  const float tau = (win_i[topk - 1] >= 0) ? win_v[topk - 1] : -INFINITY;
  const float tau_safe = tau == -INFINITY ? -INFINITY : tau - fabsf(tau) * 4e-6f - 1e-30f;
  __syncwarp();
  // ---- 2. cells that can hold a winner: a cell needs a tap >= tau, i.e. a hot PIXEL; visit the <= 4 cells each
  // hot pixel is a tap of
  top.init();
  uint2* cells = cells_s[warp];
  int* n_cells = n_cells_s + warp;
  if (lane == 0) *n_cells = 0;
  __syncwarp();
  for (int s0 = 0, slot = 0; s0 < n_it; s0 += per_slot, ++slot) {
    if (!(slot_max[slot * 32 + lane] >= tau_safe)) continue;
    for (int it = s0; it < min(s0 + per_slot, n_it); ++it)
      for (int u = 0; u < 4; ++u) {
        if (vec) {
          const int i4 = it * 128 + 32 * u + lane;
          if (i4 >= (n >> 2)) continue;
          const float4 v = __ldg(reinterpret_cast<const float4*>(m) + i4);
          if (v.x >= tau_safe) list_hot_cells(src, 4 * i4, tau_safe, out_h, out_w, cells, n_cells, top);
          if (v.y >= tau_safe) list_hot_cells(src, 4 * i4 + 1, tau_safe, out_h, out_w, cells, n_cells, top);
          if (v.z >= tau_safe) list_hot_cells(src, 4 * i4 + 2, tau_safe, out_h, out_w, cells, n_cells, top);
          if (v.w >= tau_safe) list_hot_cells(src, 4 * i4 + 3, tau_safe, out_h, out_w, cells, n_cells, top);
        } else {
          const int i = it * 128 + 32 * u + lane;
          if (i < n && __ldg(m + i) >= tau_safe) list_hot_cells(src, i, tau_safe, out_h, out_w, cells, n_cells, top);
        }
      }
  }
  __syncwarp();
  // the listed cells, spread over the warp: large cells (strong up-sampling) output by output, small ones cell by cell
  const int nc = min(*n_cells, CELL_CAP);
  if (src.sy * src.sx < 1.f / 12.f) {
    for (int c = 0; c < nc; ++c) {
      const uint2 r = cells[c];
      const int y0 = r.x & 0xffff, y1 = r.x >> 16, x0 = r.y & 0xffff, x1 = r.y >> 16;
      const int nx = x1 - x0 + 1, cnt = (y1 - y0 + 1) * nx;
      for (int k = lane; k < cnt; k += 32) {
        const int oy = y0 + k / nx, ox = x0 + k % nx;
        const float v = src.at(oy, ox);
        if (v >= tau_safe) push_key(top, v, oy * out_w + ox);
      }
    }
  } else {
    for (int c = lane; c < nc; c += 32) {
      const uint2 r = cells[c];
      eval_cell(src, r.x & 0xffff, r.x >> 16, r.y & 0xffff, r.y >> 16, out_w, tau_safe, top);
    }
  }
  warp_topk(top, topk, win_v, win_i);
  if (lane == 0) write_coords(win_v, win_i, topk, out_w, true, out_xy);
}

__global__ void __launch_bounds__(256)
gaussian_coords_kernel(const float* __restrict__ pts, int out_h, int out_w, float denom, int topk,
                       float* __restrict__ out_xy) {
  GaussSrc src{__ldg(pts + 2 * blockIdx.x), __ldg(pts + 2 * blockIdx.x + 1), denom};
  soft_argmax_block(src, out_h, out_w, topk, out_xy + 2 * blockIdx.x);
}

// ---- VOS decode ----------------------------------------------------------------------
// Label maps are read either channel-major (NCHW: maps[l][pix]) or straight from the
// pixel-major label bank (lab[pix][Lp]).  Two passes over the OUTPUT pixels, one thread per
// pixel: (1) per-channel min/max of the up-sampled map (warp shuffle -> shared -> one global
// atomic per channel and block, on order-preserving uint keys), (2) normalise + argmax.
__device__ __forceinline__ uint32_t f2key(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct Tap {   // bilinear taps of one output pixel
  int p00, p01, p10, p11;
  float w00, w01, w10, w11;
};
__device__ __forceinline__ Tap make_tap(int oy, int ox, int H, int W, float sy, float sx) {
  Lerp ly = lerp_coord(oy, sy, H), lx = lerp_coord(ox, sx, W);
  Tap t;
  t.p00 = ly.i0 * W + lx.i0; t.p01 = ly.i0 * W + lx.i1; t.p10 = ly.i1 * W + lx.i0; t.p11 = ly.i1 * W + lx.i1;
  float w0x = 1.f - lx.w1, w0y = 1.f - ly.w1;
  t.w00 = w0x; t.w01 = lx.w1; t.w10 = w0y; t.w11 = ly.w1;   // (x weights, y weights) kept separate
  return t;
}
// same association as BilinearSrc::at: wy0*(wx0*a + wx1*b) + wy1*(wx0*c + wx1*d)
__device__ __forceinline__ float tap_val(const Tap& t, float a, float b, float c, float d) {
  return t.w10 * (t.w00 * a + t.w01 * b) + t.w11 * (t.w00 * c + t.w01 * d);
}

template <bool PM>
__device__ __forceinline__ float label_at(const float* __restrict__ src, int l, int pix, int stride_l, int stride_p) {
  return __ldg(src + (int64_t)l * stride_l + (int64_t)pix * stride_p);
}

template <bool PM>
__global__ void __launch_bounds__(256)
decode_minmax_kernel(const float* __restrict__ src, int L, int H, int W, int stride_l, int stride_p, int out_h,
                     int out_w, uint32_t* __restrict__ minmax /*[L] min keys, [L] max keys*/) {
  extern __shared__ uint32_t skey[];   // [2L]
  for (int i = threadIdx.x; i < 2 * L; i += 256) skey[i] = i < L ? 0xffffffffu : 0u;
  __syncthreads();
  const int o = blockIdx.x * 256 + threadIdx.x;
  const bool valid = o < out_h * out_w;
  const int oy = valid ? o / out_w : 0, ox = valid ? o - oy * out_w : 0;
  const Tap t = make_tap(oy, ox, H, W, (float)H / (float)out_h, (float)W / (float)out_w);
  for (int l = 0; l < L; ++l) {
    float v = tap_val(t, label_at<PM>(src, l, t.p00, stride_l, stride_p), label_at<PM>(src, l, t.p01, stride_l, stride_p),
                      label_at<PM>(src, l, t.p10, stride_l, stride_p), label_at<PM>(src, l, t.p11, stride_l, stride_p));
    float mn = valid ? v : INFINITY, mx = valid ? v : -INFINITY;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, s));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&skey[l], f2key(mn));
      atomicMax(&skey[L + l], f2key(mx));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * L; i += 256) {
    if (i < L) atomicMin(minmax + i, skey[i]);
    else atomicMax(minmax + i, skey[i]);
  }
}

template <bool PM>
__global__ void __launch_bounds__(256)
decode_argmax_kernel(const float* __restrict__ src, int L, int H, int W, int stride_l, int stride_p, int out_h,
                     int out_w, const uint32_t* __restrict__ minmax, uint8_t* __restrict__ out) {
  int o = blockIdx.x * 256 + threadIdx.x;
  if (o >= out_h * out_w) return;
  int oy = o / out_w, ox = o - oy * out_w;
  const Tap t = make_tap(oy, ox, H, W, (float)H / (float)out_h, (float)W / (float)out_w);
  float best = -INFINITY;
  int arg = 0;
  for (int l = 0; l < L; ++l) {
    float v = tap_val(t, label_at<PM>(src, l, t.p00, stride_l, stride_p), label_at<PM>(src, l, t.p01, stride_l, stride_p),
                      label_at<PM>(src, l, t.p10, stride_l, stride_p), label_at<PM>(src, l, t.p11, stride_l, stride_p));
    float mn = key2f(__ldg(minmax + l)), mx = key2f(__ldg(minmax + L + l));
    if (mx > 0.f) v = __fdiv_rn(v - mn, (mx - mn) + 1e-12f);
    if (v > best) { best = v; arg = l; }
  }
  out[o] = (uint8_t)arg;
}

// batched form for a clip: blockIdx.y walks a list of jobs (a job range of one bank, or every job of several lanes);
// each decodes the label-bank slot of its out_slot into masks[slot] using its own min-max keys
// Per-channel min / max of the up-sampled map.  Within one source cell the bilinear value is
// monotone along each axis, so its extremes over the output pixels of that cell sit on the four
// corner-most output pixels: 4 evaluations per cell instead of (out/in)^2.  One thread per source
// cell; the values are produced by the same tap arithmetic as the arg-max pass.
// Jobs: RangeJobs or LaneJobs (common.cuh), blockIdx.y = job.
template <class Jobs>
__global__ void __launch_bounds__(256)
decode_minmax_jobs_kernel(const Jobs jobs, int H, int W, int out_h, int out_w) {
  extern __shared__ uint32_t skey[];   // [2L]
  const JobRef jr = jobs.at(blockIdx.y);
  const int L = jr.L, Lp = jr.Lp;
  const float* src = jr.lab + (int64_t)jr.slot * H * W * Lp;
  for (int i = threadIdx.x; i < 2 * L; i += 256) skey[i] = i < L ? 0xffffffffu : 0u;
  __syncthreads();
  const int cell = blockIdx.x * 256 + threadIdx.x;
  const bool valid = cell < H * W;
  const float sy = (float)H / (float)out_h, sx = (float)W / (float)out_w;
  int oy[2] = {0, 0}, ox[2] = {0, 0};
  bool any = false;
  if (valid) {
    cell_range(cell / W, H, out_h, sy, &oy[0], &oy[1]);
    cell_range(cell % W, W, out_w, sx, &ox[0], &ox[1]);
    any = lerp_coord(oy[0], sy, H).i0 == cell / W && lerp_coord(ox[0], sx, W).i0 == cell % W;   // cell has outputs
  }
  Tap t[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) t[c] = make_tap(oy[c >> 1], ox[c & 1], H, W, sy, sx);
  for (int l = 0; l < L; ++l) {
    float mn = INFINITY, mx = -INFINITY;
    if (any) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float v = tap_val(t[c], label_at<true>(src, l, t[c].p00, 1, Lp), label_at<true>(src, l, t[c].p01, 1, Lp),
                          label_at<true>(src, l, t[c].p10, 1, Lp), label_at<true>(src, l, t[c].p11, 1, Lp));
        mn = fminf(mn, v); mx = fmaxf(mx, v);
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, s));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&skey[l], f2key(mn));
      atomicMax(&skey[L + l], f2key(mx));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * L; i += 256) {
    if (i < L) atomicMin(jr.mn + i, skey[i]);
    else atomicMax(jr.mx + (i - L), skey[i]);
  }
}

// One CTA = a 64 x 4 tile of output pixels of one frame (blockIdx.z): no index division, neighbouring threads share
// their source taps.  Per-channel constants in shared memory as (min, max, reciprocal of the range, -).
template <class Jobs>
__global__ void __launch_bounds__(256)
decode_argmax_jobs_kernel(const Jobs jobs, int H, int W, int out_h, int out_w, uint8_t* __restrict__ masks) {
  // [Lp] (min, divisor, reciprocal of the divisor, -) with divisor = (max - min) + 1e-12.  Channels that are not
  // normalised (max <= 0: the map stays as it is) get (0, 1, 1): (v - 0) / 1 = v exactly; the pad channels get
  // min = +inf: their value becomes -inf and can never win.  The inner loop then has no per-channel case split.
  extern __shared__ float4 scst[];
  const JobRef jr = jobs.at(blockIdx.z);
  const int L = jr.L, Lp = jr.Lp;
  for (int i = threadIdx.x; i < Lp; i += 256) {
    float4 cs = make_float4(INFINITY, 1.f, 1.f, 0.f);
    if (i < L) {
      const float mn = key2f(__ldg(jr.mn + i)), mx = key2f(__ldg(jr.mx + i));
      const float dv = (mx - mn) + 1e-12f;
      cs = mx > 0.f ? make_float4(mn, dv, __frcp_rn(dv), 0.f) : make_float4(0.f, 1.f, 1.f, 0.f);
    }
    scst[i] = cs;
  }
  __syncthreads();
  const int ox = blockIdx.x * 64 + (threadIdx.x & 63), oy = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (ox >= out_w || oy >= out_h) return;
  const int slot = jr.slot;
  const float4* src = reinterpret_cast<const float4*>(jr.lab + (int64_t)slot * H * W * Lp);
  const int l4n = Lp / 4;
  const Tap t = make_tap(oy, ox, H, W, (float)H / (float)out_h, (float)W / (float)out_w);
  const float4* s00 = src + (int64_t)t.p00 * l4n;
  const float4* s01 = src + (int64_t)t.p01 * l4n;
  const float4* s10 = src + (int64_t)t.p10 * l4n;
  const float4* s11 = src + (int64_t)t.p11 * l4n;
  float best = -INFINITY, bar = -INFINITY;             // bar = best - 1e-6
  int arg = 0;
  for (int l4 = 0; l4 < l4n; ++l4) {
    const float4 a = __ldg(s00 + l4), b = __ldg(s01 + l4), c = __ldg(s10 + l4), d = __ldg(s11 + l4);
    const float v4[4] = {tap_val(t, a.x, b.x, c.x, d.x), tap_val(t, a.y, b.y, c.y, d.y),
                         tap_val(t, a.z, b.z, c.z, d.z), tap_val(t, a.w, b.w, c.w, d.w)};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int l = 4 * l4 + k;
      const float4 cs = scst[l];
      // The exact (correctly rounded) division is only needed for channels that can still win: the product
      // with the rounded reciprocal is within 2 ulp of the quotient (which lies in [0, 1]), so a channel whose
      // product is more than 1e-6 below the best exact quotient so far cannot reach it.  Same arg-max, bit for bit.
      const float num = v4[k] - cs.x;
      if (num * cs.z < bar) continue;
      const float v = __fdiv_rn(num, cs.y);
      if (v > best) { best = v; bar = v - 1e-6f; arg = l; }
    }
  }
  masks[((int64_t)slot * out_h + oy) * out_w + ox] = (uint8_t)arg;
}

// min keys are initialised to 0xffffffff and max keys to 0 by init_minmax_kernel
__global__ void init_minmax_kernel(uint32_t* mm, int n_frames, int L) {
  int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n_frames * 2 * L) mm[i] = (i % (2 * L)) < L ? 0xffffffffu : 0u;
}

int launch_decode_jobs(const float* lab, const fgvc_job* jobs_dev, int job_begin, int job_end, int L, int Lp, int H,
                       int W, int out_h, int out_w, uint32_t* minmax, uint8_t* masks, cudaStream_t st) {
  const int n = job_end - job_begin;
  if (n <= 0) return FGVC_OK;
  init_minmax_kernel<<<cdiv(n * 2 * L, 256), 256, 0, st>>>(minmax, n, L);
  FGVC_LAUNCH_CHECK();
  dim3 grid(cdiv(out_w, 64), cdiv(out_h, 4), n), grid_cells(cdiv(H * W, 256), n);
  const RangeJobs jobs{lab, jobs_dev, job_begin, L, Lp, minmax};
  decode_minmax_jobs_kernel<<<grid_cells, 256, 2 * L * 4, st>>>(jobs, H, W, out_h, out_w);
  FGVC_LAUNCH_CHECK();
  decode_argmax_jobs_kernel<<<grid, 256, Lp * 16, st>>>(jobs, H, W, out_h, out_w, masks);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

// The decode of every job of every lane (LaneJobs) in the two launches above; the min-max keys are initialised by two
// memsets (min keys first, then max keys), so the decode is two kernel launches whatever the number of lanes.
int launch_decode_lanes(const float* lab, const fgvc_job* jobs_dev, const fgvc_lane* lanes_dev,
                        const fgvc_lane* lanes_host, int n_lanes, int H, int W, int out_h, int out_w, uint32_t* minmax,
                        uint8_t* masks, cudaStream_t st) {
  int n = 0, max_L = 1, max_Lp = 4;
  int64_t n_keys = 0;
  for (int i = 0; i < n_lanes; ++i) {
    const int len = lanes_host[i].job_end - lanes_host[i].job_begin;
    n += len;
    n_keys += (int64_t)len * lanes_host[i].L;
    max_L = max(max_L, lanes_host[i].L);
    max_Lp = max(max_Lp, lanes_host[i].Lp);
  }
  if (n <= 0) return FGVC_OK;
  FGVC_CUDA(cudaMemsetAsync(minmax, 0xff, (size_t)n_keys * 4, st));
  FGVC_CUDA(cudaMemsetAsync(minmax + n_keys, 0x00, (size_t)n_keys * 4, st));
  dim3 grid(cdiv(out_w, 64), cdiv(out_h, 4), n), grid_cells(cdiv(H * W, 256), n);
  const LaneJobs jobs{lab, jobs_dev, lanes_dev, n_lanes, minmax, n_keys};
  decode_minmax_jobs_kernel<<<grid_cells, 256, 2 * max_L * 4, st>>>(jobs, H, W, out_h, out_w);
  FGVC_LAUNCH_CHECK();
  decode_argmax_jobs_kernel<<<grid, 256, max_Lp * 16, st>>>(jobs, H, W, out_h, out_w, masks);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

int launch_decode(const float* src, bool pixmajor, int L, int Lp, int H, int W, int out_h, int out_w,
                  uint32_t* minmax, uint8_t* out, cudaStream_t st) {
  FGVC_CUDA(cudaMemsetAsync(minmax, 0xff, (size_t)L * 4, st));
  FGVC_CUDA(cudaMemsetAsync(minmax + L, 0x00, (size_t)L * 4, st));
  const int blocks = cdiv(out_h * out_w, 256);
  const int sl = pixmajor ? 1 : H * W, sp = pixmajor ? Lp : 1;
  if (pixmajor) decode_minmax_kernel<true><<<blocks, 256, 2 * L * 4, st>>>(src, L, H, W, sl, sp, out_h, out_w, minmax);
  else decode_minmax_kernel<false><<<blocks, 256, 2 * L * 4, st>>>(src, L, H, W, sl, sp, out_h, out_w, minmax);
  FGVC_LAUNCH_CHECK();
  if (pixmajor) decode_argmax_kernel<true><<<blocks, 256, 0, st>>>(src, L, H, W, sl, sp, out_h, out_w, minmax, out);
  else decode_argmax_kernel<false><<<blocks, 256, 0, st>>>(src, L, H, W, sl, sp, out_h, out_w, minmax, out);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

}  // namespace fgvc

using namespace fgvc;

extern "C" int fgvc_heatmap_coords(const float* maps, int32_t n_maps, int32_t H, int32_t W, int32_t out_h,
                                   int32_t out_w, int32_t topk, float* out_xy, void* stream) {
  FGVC_CHECK_ARG(maps && out_xy && n_maps > 0 && H > 0 && W > 0 && out_h > 0 && out_w > 0,
                 "fgvc_heatmap_coords: bad arguments");
  FGVC_CHECK_ARG(topk >= 1 && topk <= CK, "fgvc_heatmap_coords: topk=%d not in [1,%d]", topk, CK);
  // few maps: spread them over the SMs (a map's critical path is one warp's)
  int mpc = MAPS_PER_CTA;
  while (mpc > 1 && cdiv(n_maps, mpc) < 2 * 148) mpc >>= 1;
  heatmap_coords_kernel<<<cdiv(n_maps, mpc), 32 * mpc, 0, (cudaStream_t)stream>>>(maps, n_maps, H, W, out_h, out_w, topk,
                                                                                  out_xy);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_gaussian_coords(const float* points_xy, int32_t P, int32_t out_h, int32_t out_w, float sigma,
                                    int32_t topk, float* out_xy, void* stream) {
  FGVC_CHECK_ARG(points_xy && out_xy && P > 0 && out_h > 0 && out_w > 0 && sigma > 0,
                 "fgvc_gaussian_coords: bad arguments");
  FGVC_CHECK_ARG(topk >= 1 && topk <= CK, "fgvc_gaussian_coords: topk=%d not in [1,%d]", topk, CK);
  gaussian_coords_kernel<<<P, 256, 0, (cudaStream_t)stream>>>(points_xy, out_h, out_w, 2.f * sigma * sigma, topk,
                                                              out_xy);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_decode_masks(const float* maps, int32_t L, int32_t H, int32_t W, int32_t out_h, int32_t out_w,
                                 float* scratch_minmax, uint8_t* out_mask, void* stream) {
  FGVC_CHECK_ARG(maps && scratch_minmax && out_mask && L > 0 && L <= 255 && H > 0 && W > 0 && out_h > 0 && out_w > 0,
                 "fgvc_decode_masks: bad arguments");
  return launch_decode(maps, false, L, L, H, W, out_h, out_w, reinterpret_cast<uint32_t*>(scratch_minmax), out_mask,
                       (cudaStream_t)stream);
}

extern "C" int fgvc_decode_masks_pixmajor(const float* lab_bank, int32_t slot, int32_t Lp, int32_t L, int32_t H,
                                          int32_t W, int32_t out_h, int32_t out_w, float* scratch_minmax,
                                          uint8_t* out_mask, void* stream) {
  FGVC_CHECK_ARG(lab_bank && scratch_minmax && out_mask && L > 0 && L <= 255 && Lp >= L && H > 0 && W > 0 &&
                     out_h > 0 && out_w > 0, "fgvc_decode_masks_pixmajor: bad arguments");
  return launch_decode(lab_bank + (int64_t)slot * H * W * Lp, true, L, Lp, H, W, out_h, out_w,
                       reinterpret_cast<uint32_t*>(scratch_minmax), out_mask, (cudaStream_t)stream);
}
