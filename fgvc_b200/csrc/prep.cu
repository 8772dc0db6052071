// K0: feature preparation and label layout kernels (HBM-bound, coalesced both ways).
#include "common.cuh"

namespace fgvc {

// One block = 32 consecutive pixels x all C channels of one frame.
// Read: for each channel a warp reads 32 consecutive pixels (128 B, coalesced).
// Write: for each pixel consecutive threads write consecutive channels (coalesced).
// smem tile[C][33] breaks the transpose bank conflicts.
template <int FMT>
__global__ void __launch_bounds__(256)
prep_features_kernel(const float* __restrict__ src, int64_t frame_stride, int64_t chan_stride, int C,
                     int n_pix, int normalize, void* __restrict__ bank_v, int first_slot) {
  extern __shared__ float tile[];  // [C][33] + norm[32]
  float* inv = tile + C * 33;
  const int frame = blockIdx.y;
  const int p0 = blockIdx.x * 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* s = src + frame * frame_stride;
  // HBM-bound: keep many bytes in flight per thread.  Full, 16-byte aligned tiles are read as float4 (4 pixels of
  // one channel per thread, 8 independent loads unrolled); ragged / misaligned ones element by element.
  const bool vec = p0 + 32 <= n_pix && (chan_stride & 3) == 0 && (frame_stride & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  if (vec) {
    const int quad = threadIdx.x & 7, c0 = threadIdx.x >> 3;       // 8 quads x 32 channels per pass
    for (int cb = 0; cb < C; cb += 256) {
      float4 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = cb + c0 + 32 * k;
        v[k] = c < C ? __ldg(reinterpret_cast<const float4*>(s + c * chan_stride + p0) + quad)
                     : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = cb + c0 + 32 * k;
        if (c < C) {
          float* t = tile + c * 33 + 4 * quad;
          t[0] = v[k].x; t[1] = v[k].y; t[2] = v[k].z; t[3] = v[k].w;
        }
      }
    }
  } else {
    for (int c = warp; c < C; c += 8) {
      int p = p0 + lane;
      tile[c * 33 + lane] = (p < n_pix) ? __ldg(s + c * chan_stride + p) : 0.f;
    }
  }
  __syncthreads();
  // per-pixel L2 norm over C: warp w handles pixels w, w+8, ...
  for (int pp = warp; pp < 32; pp += 8) {
    float acc = 0.f;
    for (int c = lane; c < C; c += 32) {
      float x = tile[c * 33 + pp];
      acc = fmaf(x, x, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    // one reciprocal per pixel (x * (1 / max(|x|, eps)) is within 1 ulp of F.normalize's x / max(|x|, eps))
    if (lane == 0) inv[pp] = normalize ? __frcp_rn(fmaxf(sqrtf(acc), 1e-12f)) : 1.f;
  }
  __syncthreads();
  const int64_t slot_off = (int64_t)(first_slot + frame) * feat_slot_floats(n_pix, C);
  // two consecutive channels per thread: 4-byte (fp16 pair) / 8-byte (fp32 pair) stores; a warp walks the channel
  // pairs of one pixel (no index division), 4 pixels per warp
  for (int pp = warp; pp < 32; pp += 8)
  for (int c = 2 * lane; c < C; c += 64) {
    const int p = p0 + pp;
    if (p < n_pix) {
      const float x0 = tile[c * 33 + pp] * inv[pp];
      const float x1 = tile[(c + 1) * 33 + pp] * inv[pp];
      if (FMT == FGVC_BANK_TF32) {
        float* hi = reinterpret_cast<float*>(bank_v) + slot_off;
        float* lo = hi + (int64_t)n_pix * C;
        const float h0 = tf32_round(x0), h1 = tf32_round(x1);
        *reinterpret_cast<float2*>(hi + (int64_t)p * C + c) = make_float2(h0, h1);
        *reinterpret_cast<float2*>(lo + (int64_t)p * C + c) = make_float2(x0 - h0, x1 - h1);
      } else {
        __half* hi = reinterpret_cast<__half*>(bank_v) + slot_off;
        __half* lo = hi + (int64_t)n_pix * C;
        const float X0 = x0 * FGVC_F16_SCALE, X1 = x1 * FGVC_F16_SCALE;        // exact (power of two)
        const __half h0 = __float2half_rn(X0), h1 = __float2half_rn(X1);
        *reinterpret_cast<__half2*>(hi + (int64_t)p * C + c) = __halves2half2(h0, h1);
        *reinterpret_cast<__half2*>(lo + (int64_t)p * C + c) =
            __halves2half2(__float2half_rn(X0 - __half2float(h0)), __float2half_rn(X1 - __half2float(h1)));
      }
    }
  }
}

// NCHW [L][n_pix] -> pixel-major [n_pix][Lp] (pad channels zero-filled); 32x32 tiles
__global__ void __launch_bounds__(256)
labels_to_pixmajor_kernel(const float* __restrict__ src, int64_t chan_stride, int L, int n_pix,
                          float* __restrict__ dst, int Lp) {
  __shared__ float t[32][33];
  const int p0 = blockIdx.x * 32, l0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    int l = l0 + j, p = p0 + tx;
    t[j][tx] = (l < L && p < n_pix) ? __ldg(src + l * chan_stride + p) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int p = p0 + j, l = l0 + tx;
    if (p < n_pix && l < Lp) dst[(int64_t)p * Lp + l] = t[tx][j];
  }
}

__global__ void __launch_bounds__(256)
labels_to_nchw_kernel(const float* __restrict__ src, int Lp, int L, int n_pix, float* __restrict__ dst) {
  __shared__ float t[32][33];
  const int p0 = blockIdx.x * 32, l0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    int p = p0 + j, l = l0 + tx;
    t[j][tx] = (p < n_pix && l < Lp) ? __ldg(src + (int64_t)p * Lp + l) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int l = l0 + j, p = p0 + tx;
    if (l < L && p < n_pix) dst[(int64_t)l * n_pix + p] = t[tx][j];
  }
}

// the same for the out_slots of jobs [job_begin, job_begin + gridDim.z): dst[slot][L][n_pix]
__global__ void __launch_bounds__(256)
labels_to_nchw_jobs_kernel(const float* __restrict__ lab, const fgvc_job* __restrict__ jobs, int job_begin, int Lp, int L,
                           int n_pix, float* __restrict__ maps) {
  __shared__ float t[32][33];
  const int slot = jobs[job_begin + blockIdx.z].out_slot;
  const float* src = lab + (int64_t)slot * n_pix * Lp;
  float* dst = maps + (int64_t)slot * L * n_pix;
  const int p0 = blockIdx.x * 32, l0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    int p = p0 + j, l = l0 + tx;
    t[j][tx] = (p < n_pix && l < Lp) ? __ldg(src + (int64_t)p * Lp + l) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int l = l0 + j, p = p0 + tx;
    if (l < L && p < n_pix) dst[(int64_t)l * n_pix + p] = t[tx][j];
  }
}

// wide variant (n_pix % 4 == 0): 64 pixels x 64 channels per CTA, 16-byte loads along the channels and 16-byte
// stores along the pixels
__global__ void __launch_bounds__(256)
labels_to_nchw_jobs_wide_kernel(const float* __restrict__ lab, const fgvc_job* __restrict__ jobs, int job_begin, int Lp,
                                int L, int n_pix, float* __restrict__ maps) {
  __shared__ float t[64][65];
  const int slot = jobs[job_begin + blockIdx.z].out_slot;
  const float* src = lab + (int64_t)slot * n_pix * Lp;
  float* dst = maps + (int64_t)slot * L * n_pix;
  const int p0 = blockIdx.x * 64, l0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int j = ty; j < 64; j += 16) {
    const int p = p0 + j, l = l0 + 4 * tx;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p < n_pix && l < Lp) v = __ldg(reinterpret_cast<const float4*>(src + (int64_t)p * Lp + l));
    t[j][4 * tx] = v.x; t[j][4 * tx + 1] = v.y; t[j][4 * tx + 2] = v.z; t[j][4 * tx + 3] = v.w;
  }
  __syncthreads();
#pragma unroll
  for (int j = ty; j < 64; j += 16) {
    const int l = l0 + j, p = p0 + 4 * tx;
    if (l < L && p < n_pix)
      *reinterpret_cast<float4*>(dst + (int64_t)l * n_pix + p) =
          make_float4(t[4 * tx][j], t[4 * tx + 1][j], t[4 * tx + 2][j], t[4 * tx + 3][j]);
  }
}

__global__ void __launch_bounds__(256)
gaussian_labels_kernel(const float* __restrict__ pts, int P, int H, int W, int stride, float denom,
                       float* __restrict__ dst, int Lp) {
  int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  int64_t total = (int64_t)H * W * Lp;
  if (i >= total) return;
  int p = (int)(i % Lp);
  int pix = (int)(i / Lp);
  float v = 0.f;
  if (p < P) {
    float x = (float)((pix % W) * stride), y = (float)((pix / W) * stride);
    float dx = x - __ldg(pts + 2 * p), dy = y - __ldg(pts + 2 * p + 1);
    // reference: exp(-((gx-cx)**2 + (gy-cy)**2) / (2*sigma**2))
    v = expf(__fdiv_rn(-(dx * dx + dy * dy), denom));
  }
  dst[i] = v;
}

// bilinear up-sampling of a pixel-major label map (F.interpolate(mode='bilinear', align_corners=False) semantics,
// bilinear_taps / bilinear_mix in common.cuh); one thread per
// (destination pixel, 4 channels): float4 loads and stores along the channel dimension are coalesced
__global__ void __launch_bounds__(256)
upsample_labels_kernel(const float* __restrict__ src, int Hs, int Ws, int Lp, float* __restrict__ dst, int Hd, int Wd) {
  const int l4n = Lp / 4;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= (int64_t)Hd * Wd * l4n) return;
  const int l4 = (int)(i % l4n);
  const int pix = (int)(i / l4n);
  const int y = pix / Wd, x = pix - y * Wd;
  const BilinearTaps t = bilinear_taps(y, x, Hs, Ws, Hd, Wd);
  const float4* s4 = reinterpret_cast<const float4*>(src);
  const float4 a = __ldg(s4 + (int64_t)t.p00 * l4n + l4), b = __ldg(s4 + (int64_t)t.p01 * l4n + l4);
  const float4 c = __ldg(s4 + (int64_t)t.p10 * l4n + l4), d = __ldg(s4 + (int64_t)t.p11 * l4n + l4);
  reinterpret_cast<float4*>(dst)[i] = bilinear_mix(t, a, b, c, d);
}

// hard propagation (vanilla_tracker.py:762-767): replace the soft labels of a slot by one_hot(argmax)
__global__ void __launch_bounds__(256)
labels_harden_kernel(float* __restrict__ lab, int n_pix, int L, int Lp) {
  int p = blockIdx.x * 256 + threadIdx.x;
  if (p >= n_pix) return;
  float* row = lab + (int64_t)p * Lp;
  float best = row[0];
  int arg = 0;
  for (int l = 1; l < L; ++l) {
    float v = row[l];
    if (v > best) { best = v; arg = l; }     // first maximum, like torch.argmax
  }
  for (int l = 0; l < Lp; ++l) row[l] = (l == arg) ? 1.f : 0.f;
}

int launch_labels_harden(float* lab_slot, int n_pix, int L, int Lp, cudaStream_t st) {
  labels_harden_kernel<<<cdiv(n_pix, 256), 256, 0, st>>>(lab_slot, n_pix, L, Lp);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

int launch_labels_to_nchw_jobs(const float* lab, const fgvc_job* jobs_dev, int job_begin, int job_end, int Lp, int L,
                               int n_pix, float* maps_nchw, cudaStream_t st) {
  const int n = job_end - job_begin;
  if (n <= 0) return FGVC_OK;
  const bool wide = n_pix % 4 == 0 && L >= 32 && (reinterpret_cast<uintptr_t>(maps_nchw) & 15) == 0;
  for (int z0 = 0; z0 < n; z0 += 65535) {
    if (wide) {
      dim3 grid(cdiv(n_pix, 64), cdiv(L, 64), min(65535, n - z0));
      labels_to_nchw_jobs_wide_kernel<<<grid, 256, 0, st>>>(lab, jobs_dev, job_begin + z0, Lp, L, n_pix, maps_nchw);
    } else {
      dim3 grid(cdiv(n_pix, 32), cdiv(L, 32), min(65535, n - z0));
      labels_to_nchw_jobs_kernel<<<grid, 256, 0, st>>>(lab, jobs_dev, job_begin + z0, Lp, L, n_pix, maps_nchw);
    }
    FGVC_LAUNCH_CHECK();
  }
  return FGVC_OK;
}

}  // namespace fgvc

using namespace fgvc;

extern "C" int fgvc_prep_features(const float* src, int64_t src_frame_stride, int64_t src_chan_stride,
                                  int32_t n_frames, int32_t C, int32_t H, int32_t W, int32_t normalize,
                                  void* feat_bank, int32_t bank_format, int32_t first_slot, void* stream) {
  FGVC_CHECK_ARG(src && feat_bank, "fgvc_prep_features: null pointer");
  FGVC_CHECK_ARG(n_frames > 0 && C > 0 && H > 0 && W > 0, "fgvc_prep_features: bad shape");
  FGVC_CHECK_ARG(C % 4 == 0 && C <= 1024, "fgvc_prep_features: C=%d must be a multiple of 4, <= 1024", C);
  int n_pix = H * W;
  size_t smem = (size_t)(C * 33 + 32) * sizeof(float);
  FGVC_CHECK_ARG(bank_format == FGVC_BANK_TF32 || bank_format == FGVC_BANK_F16, "fgvc_prep_features: bad bank format");
  if (smem > 48 * 1024) {      // per launch: the attribute is per device, and a process may use several
    if (bank_format == FGVC_BANK_TF32)
      FGVC_CUDA(cudaFuncSetAttribute(prep_features_kernel<FGVC_BANK_TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    else
      FGVC_CUDA(cudaFuncSetAttribute(prep_features_kernel<FGVC_BANK_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  }
  dim3 grid(cdiv(n_pix, 32), n_frames);
  if (bank_format == FGVC_BANK_TF32)
    prep_features_kernel<FGVC_BANK_TF32><<<grid, 256, smem, (cudaStream_t)stream>>>(
        src, src_frame_stride, src_chan_stride, C, n_pix, normalize, feat_bank, first_slot);
  else
    prep_features_kernel<FGVC_BANK_F16><<<grid, 256, smem, (cudaStream_t)stream>>>(
        src, src_frame_stride, src_chan_stride, C, n_pix, normalize, feat_bank, first_slot);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_labels_to_pixmajor(const float* src, int64_t src_chan_stride, int32_t L, int32_t n_pix,
                                       float* lab_bank, int32_t slot, int32_t Lp, void* stream) {
  FGVC_CHECK_ARG(src && lab_bank && L > 0 && n_pix > 0 && Lp >= L && Lp % 4 == 0,
                 "fgvc_labels_to_pixmajor: bad arguments (L=%d Lp=%d)", L, Lp);
  dim3 grid(cdiv(n_pix, 32), cdiv(Lp, 32));
  labels_to_pixmajor_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, src_chan_stride, L, n_pix,
                                                                    lab_bank + (int64_t)slot * n_pix * Lp, Lp);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_labels_to_nchw(const float* lab_bank, int32_t slot, int32_t Lp, int32_t L, int32_t n_pix,
                                   float* dst, void* stream) {
  FGVC_CHECK_ARG(dst && lab_bank && L > 0 && n_pix > 0 && Lp >= L, "fgvc_labels_to_nchw: bad arguments");
  dim3 grid(cdiv(n_pix, 32), cdiv(L, 32));
  labels_to_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(lab_bank + (int64_t)slot * n_pix * Lp, Lp, L,
                                                                n_pix, dst);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_upsample_labels(const float* src, int32_t Hs, int32_t Ws, int32_t Lp, float* lab_bank, int32_t slot,
                                    int32_t Hd, int32_t Wd, void* stream) {
  FGVC_CHECK_ARG(src && lab_bank && Hs > 0 && Ws > 0 && Hd > 0 && Wd > 0 && Lp > 0 && Lp % 4 == 0 && slot >= 0,
                 "fgvc_upsample_labels: bad arguments");
  const int64_t total = (int64_t)Hd * Wd * (Lp / 4);
  upsample_labels_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      src, Hs, Ws, Lp, lab_bank + (int64_t)slot * Hd * Wd * Lp, Hd, Wd);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

extern "C" int fgvc_gaussian_labels(const float* points_xy, int32_t P, int32_t H, int32_t W, int32_t stride,
                                    float sigma, float* lab_bank, int32_t slot, int32_t Lp, void* stream) {
  FGVC_CHECK_ARG(points_xy && lab_bank && P > 0 && Lp >= P && Lp % 4 == 0 && sigma > 0,
                 "fgvc_gaussian_labels: bad arguments");
  int64_t total = (int64_t)H * W * Lp;
  gaussian_labels_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      points_xy, P, H, W, stride, 2.f * sigma * sigma, lab_bank + (int64_t)slot * H * W * Lp, Lp);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}
