// Shared helpers for the fgvc_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <math.h>
#include <stdio.h>
#include <atomic>

#include "../../include/fgvc_b200.h"

namespace fgvc {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define FGVC_CHECK_ARG(cond, ...)                   \
  do {                                              \
    if (!(cond)) {                                  \
      fgvc::set_error(__VA_ARGS__);                 \
      return FGVC_ERR_INVALID;                      \
    }                                               \
  } while (0)

#define FGVC_CUDA(call)                                                                   \
  do {                                                                                    \
    cudaError_t e__ = (call);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      fgvc::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__,  \
                      __LINE__);                                                          \
      return FGVC_ERR_CUDA;                                                               \
    }                                                                                     \
  } while (0)

#define FGVC_LAUNCH_CHECK()                 \
  do {                                      \
    fgvc::g_launches.fetch_add(1);          \
    FGVC_CUDA(cudaGetLastError());          \
  } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// size in elements of one feature-bank slot: [2][n_pix][C]
__host__ __device__ inline int64_t feat_slot_floats(int n_pix, int C) { return 2ll * n_pix * C; }

// fp16 split of the F16 bank: X = 16 x, hi = fp16(X), lo = fp16(X - hi); x = (hi + lo) / 16 (exact in fp32).
// The 2^4 scale keeps `lo` (<= 2^-11 |X|) a normal fp16 number for every element that matters (|x| >= 2^-7 of a
// unit row), so all three products of the split can share ONE fp32 accumulator (= 256 x affinity).
#define FGVC_F16_SCALE 16.0f
#define FGVC_F16_INV (1.0f / 16.0f)
#define FGVC_F16_ACC_INV (1.0f / 256.0f)

// 4 consecutive channels of pixel `pix` of slot `slot`, reconstructed to fp32, for either bank format
template <int FMT>
__device__ __forceinline__ float4 bank_load4(const void* __restrict__ bank, int slot, int n_pix, int C, int pix, int c4) {
  if (FMT == FGVC_BANK_TF32) {
    const float4* hi = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(bank) +
                                                       (int64_t)slot * feat_slot_floats(n_pix, C));
    const float4* lo = hi + ((int64_t)n_pix * C) / 4;
    const int64_t o = ((int64_t)pix * C) / 4 + c4;
    float4 a = __ldg(hi + o), b = __ldg(lo + o);
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  } else {
    const uint2* hi = reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(bank) +
                                                     (int64_t)slot * feat_slot_floats(n_pix, C));
    const uint2* lo = hi + ((int64_t)n_pix * C) / 4;
    const int64_t o = ((int64_t)pix * C) / 4 + c4;
    uint2 a = __ldg(hi + o), b = __ldg(lo + o);
    float2 a0 = __half22float2(*reinterpret_cast<__half2*>(&a.x)), a1 = __half22float2(*reinterpret_cast<__half2*>(&a.y));
    float2 b0 = __half22float2(*reinterpret_cast<__half2*>(&b.x)), b1 = __half22float2(*reinterpret_cast<__half2*>(&b.y));
    return make_float4((a0.x + b0.x) * FGVC_F16_INV, (a0.y + b0.y) * FGVC_F16_INV, (a1.x + b1.x) * FGVC_F16_INV,
                       (a1.y + b1.y) * FGVC_F16_INV);
  }
}

__device__ __forceinline__ float tf32_round(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// ---- sorted (descending) top-K list held in registers -------------------------------
template <int K>
struct TopK {
  float v[K];
  int id[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int i = 0; i < K; ++i) {
      v[i] = -INFINITY;
      id[i] = -1;
    }
  }
  __device__ __forceinline__ float thr() const { return v[K - 1]; }
  // variant for exact ties: a later (higher-index) equal value goes ahead of earlier ones,
  // like a stable ascending argsort read from the back (np.argsort in img2coord)
  __device__ __forceinline__ void push_ge(float x, int i) {
    v[K - 1] = x;
    id[K - 1] = i;
#pragma unroll
    for (int j = K - 1; j > 0; --j) {
      if (v[j] >= v[j - 1]) {
        float tv = v[j]; v[j] = v[j - 1]; v[j - 1] = tv;
        int ti = id[j]; id[j] = id[j - 1]; id[j - 1] = ti;
      }
    }
  }
  // caller guarantees x > thr().  Select form of the sorted insert: K compares, then every slot
  // takes its left neighbour, the new element or itself (equal values keep arrival order).
  // The last slot is written without its compare (x > v[K-1] holds): with the compare in the
  // expression, nvcc 12.9 compiled TopK<4> in gather_labels_kernel to take the new index but keep
  // the old value there, which dropped the K-th winner (tests/test_gpu_label_kernels.py, K = 4).
  __device__ __forceinline__ void push(float x, int i) {
    bool c[K];
#pragma unroll
    for (int j = 0; j < K; ++j) c[j] = x > v[j];
    if (K > 1) {
      v[K - 1] = c[K - 2] ? v[K - 2] : x;
      id[K - 1] = c[K - 2] ? id[K - 2] : i;
    }
#pragma unroll
    for (int j = K - 2; j > 0; --j) {
      v[j] = c[j - 1] ? v[j - 1] : (c[j] ? x : v[j]);
      id[j] = c[j - 1] ? id[j - 1] : (c[j] ? i : id[j]);
    }
    v[0] = c[0] ? x : v[0];
    id[0] = c[0] ? i : id[0];
  }
};

// v[j] for a run-time j in [0,16): 4-level select tree (registers cannot be indexed dynamically)
__device__ __forceinline__ float select16(const float* v, int j) {
  float a[8], b[4];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = (j & 1) ? v[2 * i + 1] : v[2 * i];
#pragma unroll
  for (int i = 0; i < 4; ++i) b[i] = (j & 2) ? a[2 * i + 1] : a[2 * i];
  const float c0 = (j & 4) ? b[1] : b[0], c1 = (j & 4) ? b[3] : b[2];
  return (j & 8) ? c1 : c0;
}

// in-mask test shared by every kernel (affinity_utils.py:85-112):
// circle: dy^2 + dx^2 < r^2 (strict); square: |dy| <= r and |dx| <= r
__device__ __forceinline__ bool in_mask(int dy, int dx, int r, int mode) {
  if (mode == FGVC_MASK_CIRCLE) return dy * dy + dx * dx < r * r;
  return (dy <= r) && (dy >= -r) && (dx <= r) && (dx >= -r);
}
// largest |d| that can be in-mask
__host__ __device__ inline int mask_reach(int r, int mode) { return mode == FGVC_MASK_CIRCLE ? r - 1 : r; }

// grid barrier of a cooperative launch over a counter zeroed before the launch: the n-th barrier of every CTA
// (n = 1, 2, ...) returns once all CTAs reached their n-th.  The caller's stores before it are visible after it to
// ld.global.cg loads (the stores are fenced before the arrival).
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int n) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    const unsigned int want = n * gridDim.x;
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    } while (seen < want);
  }
  __syncthreads();
}

// F.interpolate(mode='bilinear', align_corners=False) taps of destination pixel (y, x) of an Hd x Wd map from an
// Hs x Ws one: src = max((dst + 0.5) * in / out - 0.5, 0), second tap clamped to the last row / column
struct BilinearTaps {
  int p00, p01, p10, p11;     // source pixels (y0, x0), (y0, x1), (y1, x0), (y1, x1)
  float ly, lx;
};
__device__ __forceinline__ BilinearTaps bilinear_taps(int y, int x, int Hs, int Ws, int Hd, int Wd) {
  const float fy = fmaxf(((float)y + 0.5f) * ((float)Hs / (float)Hd) - 0.5f, 0.f);
  const float fx = fmaxf(((float)x + 0.5f) * ((float)Ws / (float)Wd) - 0.5f, 0.f);
  const int y0 = min((int)fy, Hs - 1), x0 = min((int)fx, Ws - 1);
  const int y1 = min(y0 + 1, Hs - 1), x1 = min(x0 + 1, Ws - 1);
  BilinearTaps t;
  t.p00 = y0 * Ws + x0; t.p01 = y0 * Ws + x1; t.p10 = y1 * Ws + x0; t.p11 = y1 * Ws + x1;
  t.ly = fy - (float)y0; t.lx = fx - (float)x0;
  return t;
}
// same association as ATen's upsample_bilinear2d: (1-ly) * ((1-lx) * a + lx * b) + ly * ((1-lx) * c + lx * d)
__device__ __forceinline__ float4 bilinear_mix(const BilinearTaps& t, const float4& a, const float4& b, const float4& c,
                                               const float4& d) {
  const float ly = t.ly, lx = t.lx, hy = 1.f - ly, hx = 1.f - lx;
  float4 o;
  o.x = hy * (hx * a.x + lx * b.x) + ly * (hx * c.x + lx * d.x);
  o.y = hy * (hx * a.y + lx * b.y) + ly * (hx * c.y + lx * d.y);
  o.z = hy * (hx * a.z + lx * b.z) + ly * (hx * c.z + lx * d.z);
  o.w = hy * (hx * a.w + lx * b.w) + ly * (hx * c.w + lx * d.w);
  return o;
}

// One job of a clip-level c2f fine stage (fgvc_c2f_clip_weights): where its coarse arg-max table, its floors and its
// fine top-K lists live in the workspace, and which CTAs of the window-mode K1 launch are its (grid.y indices
// [y_begin, y_begin + n_mem * chunks), entry-major).
struct c2f_wjob {
  fgvc_job job;
  int32_t chunks;       // CTAs per (coarse tile, memory entry): c2f_window_chunks(Hc, Wc, n_mem)
  int32_t y_begin;
  int64_t best_off;     // elements: arg-max table [n_mem][Hc * Wc]
  int64_t floor_off;    // elements: floors [Hc * Wc]
  int64_t list_off;     // elements: lists [Hc * Wc][n_mem * chunks][K]
};

// host launchers implemented in the .cu files -------------------------------------------
int launch_affinity_topk_simt(const void* bank, int fmt, int H, int W, int C, const fgvc_job* jobs, int n_jobs,
                              const int32_t* mem_feat, int radius, int mode, int K, int groups,
                              float* tv, int32_t* ti, cudaStream_t st);
int launch_affinity_topk_tc(const float* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs, int n_jobs,
                            const int32_t* mem_feat, int radius, int mode, int K, int groups,
                            float* tv, int32_t* ti, float* dbg, int32_t* dbg_meta, int dbg_max_boxes,
                            cudaStream_t st);
bool tc_supported(int H, int W, int C, int K);
bool tc16_supported(int H, int W, int C, int K);
int launch_affinity_topk_tc16(const void* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs, int n_jobs,
                              const int32_t* mem_feat, int radius, int mode, int K, int groups, float* tv, int32_t* ti,
                              float* dbg, int32_t* dbg_meta, int dbg_max_boxes, cudaStream_t st, const float* floor = nullptr);
int launch_topk_floor16(const void* bank, int H, int W, int C, const fgvc_job* jobs, int n_jobs, const int32_t* seed_slot,
                        int radius, int mode, int K, float* floor_out, cudaStream_t st);
int64_t chain_workspace_bytes(int n_jobs, int n_pix, int K);
int launch_gather_chain(const float* tv, const int32_t* ti, int K, int groups, const fgvc_job* jobs, int job_begin,
                        int job_end, const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature,
                        int flags, float* lab, int Lp, void* ws, int64_t ws_bytes, cudaStream_t st);
int launch_gather_chain_lanes(const float* tv, const int32_t* ti, int K, int groups, const fgvc_job* jobs,
                              const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host, int n_lanes,
                              const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature, int flags,
                              float* lab, void* ws, int64_t ws_bytes, cudaStream_t st);
int launch_labels_to_nchw_jobs(const float* lab, const fgvc_job* jobs_dev, int job_begin, int job_end, int Lp, int L,
                               int n_pix, float* maps_nchw, cudaStream_t st);
void packed_tile_shape(int H, int W, int reach, int jobs_per_tile, int* QH, int* QW, int* BH, int* ncta);
int launch_affinity_topk_tc16_packed(const void* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs,
                                     const fgvc_tile_group* tgroups, int n_tgroups, const int32_t* uent,
                                     const int32_t* upos, int jobs_per_tile, int radius, int mode, int K, int groups,
                                     int split, float* tv, int32_t* ti, cudaStream_t st);
bool c2f_window_supported(int Hf, int Wf, int Cf, int K, int n_mem);
int launch_c2f_window_tc16(const void* fine_bank, int n_slots, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                           const fgvc_job& job, const int32_t* mem_feat, const int32_t* best, int rf, int K, int chunks,
                           float* floor_ws, float* tv, int32_t* ti, cudaStream_t st);
int launch_c2f_window_tc16_jobs(const void* fine_bank, int n_slots, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                                const c2f_wjob* wjobs_dev, int n_wjobs, int n_y, const int32_t* mem_feat,
                                const int32_t* best, int rf, int K, float* floor_ws, float* tv, int32_t* ti,
                                cudaStream_t st);
int c2f_window_chunks(int Hc, int Wc, int n_mem);
bool c2f_use_window(int engine, int bank_format, int Hf, int Wf, int Cf, int K, int n_mem);
int resident_ctas(const void* kernel, std::atomic<int>* cached, int* max_ctas);
int launch_c2f_chain_lanes(const float* cw, const int32_t* crow, int K, int job_base, const fgvc_job* jobs_dev,
                           const fgvc_c2f_lane* lanes_dev, const fgvc_c2f_lane* lanes_host, int n_lanes, int Hc, int Wc,
                           int Hf, int Wf, float* fine_lab, float* coarse_out, unsigned int* barrier, cudaStream_t st);
int launch_decode_jobs(const float* lab, const fgvc_job* jobs_dev, int job_begin, int job_end, int L, int Lp, int H,
                       int W, int out_h, int out_w, uint32_t* minmax, uint8_t* masks, cudaStream_t st);
int launch_labels_harden(float* lab_slot, int n_pix, int L, int Lp, cudaStream_t st);
int launch_decode(const float* src, bool pixmajor, int L, int Lp, int H, int W, int out_h, int out_w,
                  uint32_t* minmax, uint8_t* out, cudaStream_t st);

}  // namespace fgvc
