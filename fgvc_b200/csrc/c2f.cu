// K2: coarse-to-fine propagation (local_attention.py:721-880, SURVEY.md Appendix A.3).
//
// Coarse stage: K1 with K = 1 and one group per memory frame gives, for every coarse
// query and memory frame, the arg-max key inside the radius mask (:804-837).
// Fine stage (this file): one CTA per coarse query.  For every memory frame the
// (2*rf+1)^2 window of the fine key map centred at scale*(ky,kx) is read straight from
// the pixel-major fine bank -- the R^2-fold F.unfold blow-up of the reference (:790-793)
// never exists.  One warp per candidate: lanes stride the contiguous channel dimension
// (coalesced 128-bit loads), butterfly-reduce the dot product, and every lane keeps the
// same sorted top-K so there is no divergence.  Out-of-map candidates compete with
// affinity 0 and value 0 exactly as the zero padding of the reference does.
#include <stdlib.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "common.cuh"

namespace fgvc {

// WONLY: the weights-only form of fgvc_c2f_clip_weights -- job blockIdx.y of the table `wjobs` (its arg-max table at
// best_idx + best_off), and the (weight, row) pairs of the query go to w_out / row_out[job][q][k_out] instead of the
// gather.
template <int K, int FMT, bool WONLY = false>
__global__ void __launch_bounds__(256, WONLY ? 1 : 0)     // (weights-only: room for the job's entry without spills)
c2f_fine_kernel(const void* __restrict__ fine_bank, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                fgvc_job job, const int32_t* __restrict__ mem_feat, const int32_t* __restrict__ mem_label,
                const int32_t* __restrict__ best_idx, int rf, int k_out, float temperature,
                const float* __restrict__ fine_lab, int Lp, float* __restrict__ out,
                const c2f_wjob* __restrict__ wjobs = nullptr, float* __restrict__ w_out = nullptr,
                int32_t* __restrict__ row_out = nullptr) {
  if (WONLY) {
    job = wjobs[blockIdx.y].job;
    best_idx += wjobs[blockIdx.y].best_off;
  }
  extern __shared__ __align__(16) float qf[];  // [Cf]
  __shared__ float lv[8][K];
  __shared__ int li[8][K];
  __shared__ float sw[K];
  __shared__ int srow[K];
  const int q = blockIdx.x;
  const int qy = q / Wc, qx = q - qy * Wc;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nf = Hf * Wf, nc = Hc * Wc;
  for (int c4 = tid; c4 < Cf / 4; c4 += 256)
    *reinterpret_cast<float4*>(qf + 4 * c4) =
        bank_load4<FMT>(fine_bank, job.q_slot, nf, Cf, (qy * scale) * Wf + qx * scale, c4);
  __syncthreads();
  const int R = 2 * rf + 1;
  const int n_mem = job.mem_end - job.mem_begin;
  TopK<K> top;
  top.init();
  const int c4n = Cf / 4;
  for (int t = 0; t < n_mem; ++t) {
    const int slot = __ldg(mem_feat + job.mem_begin + t) & ~FGVC_MEM_UNMASKED;
    const int b = max(__ldg(best_idx + (int64_t)t * nc + q), 0) % nc;   // coarse arg-max key pixel
    const int cy = (b / Wc) * scale, cx = (b % Wc) * scale;
    for (int w = warp; w < R * R; w += 8) {
      int dy = w / R - rf, dx = w % R - rf;
      int y = cy + dy, x = cx + dx;
      float dot = 0.f;
      if (y >= 0 && y < Hf && x >= 0 && x < Wf) {
        for (int c = lane; c < c4n; c += 32) {
          float4 a = bank_load4<FMT>(fine_bank, slot, nf, Cf, y * Wf + x, c);
          float4 qq = *reinterpret_cast<const float4*>(qf + 4 * c);
          dot = fmaf(a.x, qq.x, dot); dot = fmaf(a.y, qq.y, dot);
          dot = fmaf(a.z, qq.z, dot); dot = fmaf(a.w, qq.w, dot);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      }
      // candidate id = t * R^2 + w; padded candidates carry affinity 0
      if (dot > top.thr()) top.push(dot, t * R * R + w);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < K; ++i) { lv[warp][i] = top.v[i]; li[warp][i] = top.id[i]; }
  }
  __syncthreads();
  if (tid == 0) {
    TopK<K> m;
    m.init();
    for (int w = 0; w < 8; ++w)
      for (int i = 0; i < K; ++i)
        if (li[w][i] >= 0 && lv[w][i] > m.thr()) m.push(lv[w][i], li[w][i]);
    float a[K];
#pragma unroll
    for (int i = 0; i < K; ++i) a[i] = __fdiv_rn(m.v[i], temperature);
    float mx = a[0], sum = 0.f;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      a[i] = (i < k_out && m.id[i] >= 0) ? expf(a[i] - mx) : 0.f;
      sum += a[i];
    }
    for (int i = 0; i < K; ++i) {
      bool ok = i < k_out && m.id[i] >= 0;
      float w = ok ? __fdiv_rn(a[i], sum) : 0.f;
      int row = -1;
      if (ok) {
        int t = m.id[i] / (R * R), wdx = m.id[i] - t * R * R;
        int b = max(__ldg(best_idx + (int64_t)t * nc + q), 0) % nc;
        int y = (b / Wc) * scale + wdx / R - rf, x = (b % Wc) * scale + wdx % R - rf;
        if (y >= 0 && y < Hf && x >= 0 && x < Wf)
          row = __ldg(mem_label + job.mem_begin + t) * nf + y * Wf + x;
      }
      sw[i] = w;
      srow[i] = row;   // row < 0: zero-padded candidate, contributes value 0
    }
  }
  __syncthreads();
  if (WONLY) {
    if (tid < k_out) {
      const int64_t o = ((int64_t)blockIdx.y * nc + q) * k_out + tid;
      w_out[o] = sw[tid];
      row_out[o] = srow[tid];
    }
    return;
  }
  const int l4n = Lp / 4;
  const float4* src = reinterpret_cast<const float4*>(fine_lab);
  float4* dst = reinterpret_cast<float4*>(out) + (int64_t)q * l4n;
  for (int c = tid; c < l4n; c += 256) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < K; ++j) {
      if (srow[j] >= 0 && sw[j] != 0.f) {
        float4 v = __ldg(src + (int64_t)srow[j] * l4n + c);
        acc.x = fmaf(sw[j], v.x, acc.x); acc.y = fmaf(sw[j], v.y, acc.y);
        acc.z = fmaf(sw[j], v.z, acc.z); acc.w = fmaf(sw[j], v.w, acc.w);
      }
    }
    dst[c] = acc;
  }
}

constexpr int C2F_TAIL_QB = 8;      // coarse queries per CTA: a coarse grid is small, keep the grid wide

// Tail of the tensor-core fine stage (topk_tc16.cu): per coarse query, the K best in-window fine keys are in
// tv / ti.  The reference's windows are zero padded (F.unfold(padding = rf), local_attention.py:790-793): every
// window position outside the fine map is a candidate too, with affinity 0 and value 0 -- their number is
// analytic, so they are inserted here; then soft-max over the K winners and the gather of fine label rows.
// The (weight, fine label row) pairs of the coarse queries [q0, q0 + QB) into sw / srow (shared): the first half of
// c2f_tail_kernel, shared with c2f_weights_kernel.  Called by all 256 threads of the CTA; the caller synchronises.
template <int K>
__device__ __forceinline__ void c2f_tail_pairs(const float* __restrict__ tv, const int32_t* __restrict__ ti, int k_in,
                                               int n_lists, int Hc, int Wc, int Hf, int Wf, int scale, const fgvc_job& job,
                                               const int32_t* __restrict__ mem_label,
                                               const int32_t* __restrict__ best_idx, int rf, float temperature, int q0,
                                               float (*sw)[K], int (*srow)[K]) {
  constexpr int QB = C2F_TAIL_QB;
  const int tid = threadIdx.x;
  const int nc = Hc * Wc, nf = Hf * Wf;
  const int n_mem = job.mem_end - job.mem_begin;
  __shared__ float sv[QB][K];
  __shared__ int sid[QB][K];
  if (n_lists <= 32) {
    // one warp per coarse query: lane l holds partial list l (sorted by K1; all its loads in flight together); K
    // rounds of a warp-wide arg-max over the list heads give the K best in the order the serial merge below finds
    // them (equal values: lower list first, then list order); the analytic number of zero-padded candidates is a
    // warp reduction; lane 0 finishes with the soft-max in the reference's summation order.
    const int warp = tid >> 5, lane = tid & 31;
    const int q = q0 + warp;                      // QB == 8 warps
    float lv[K];
    int li[K];
#pragma unroll
    for (int i = 0; i < K; ++i) { lv[i] = -INFINITY; li[i] = -1; }
    if (q < nc && lane < n_lists) {
      const int64_t o = ((int64_t)q * n_lists + lane) * k_in;
#pragma unroll
      for (int i = 0; i < K; ++i)
        if (i < k_in) { lv[i] = __ldg(tv + o + i); li[i] = __ldg(ti + o + i); }
    }
    int n_zero = 0;
    if (q < nc) {
      const int R = 2 * rf + 1;
      for (int t = lane; t < n_mem; t += 32) {
        const int bq = max(__ldg(best_idx + (int64_t)t * nc + q), 0) % nc;
        const int cy = (bq / Wc) * scale, cx = (bq % Wc) * scale;
        const int rows = min(cy + rf, Hf - 1) - max(cy - rf, 0) + 1, cols = min(cx + rf, Wf - 1) - max(cx - rf, 0) + 1;
        n_zero += R * R - rows * cols;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n_zero += __shfl_xor_sync(0xffffffffu, n_zero, o);
    const int nz = min(n_zero, K);
    int head = 0;
    float myv = -INFINITY;                        // lane r keeps the r-th best genuine candidate
    int myid = -1;
    for (int r = 0; r < K; ++r) {
      float v = -INFINITY;
      int id = -1;
#pragma unroll
      for (int j = 0; j < K; ++j)
        if (j == head) { v = lv[j]; id = li[j]; }
      if (id < 0) v = -INFINITY;                  // (a list ends at its first empty slot)
      int from = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, id, o);
        const int of = __shfl_xor_sync(0xffffffffu, from, o);
        if (ov > v || (ov == v && of < from)) { v = ov; id = oi; from = of; }
      }
      if (v == -INFINITY) id = -1;
      if (lane == from && id >= 0) ++head;
      if (lane == r) { myv = v; myid = id; }
    }
    // zero-padded candidates (affinity 0, value 0) go behind the genuine ones that are >= 0
    const int n_pos = __popc(__ballot_sync(0xffffffffu, lane < K && myid >= 0 && myv >= 0.f));
    const int src_lane = lane < n_pos ? lane : max(lane - nz, 0);
    float fv = __shfl_sync(0xffffffffu, myv, src_lane);
    int fid = __shfl_sync(0xffffffffu, myid, src_lane);
    if (lane >= n_pos && lane < n_pos + nz) { fv = 0.f; fid = -2; }      // id -2: padded candidate, value row of zeros
    if (lane < K) { sv[warp][lane] = fv; sid[warp][lane] = fid; }
    __syncwarp();
    if (lane == 0) {
      float a[K];
#pragma unroll
      for (int i = 0; i < K; ++i) a[i] = __fdiv_rn(sv[warp][i], temperature);
      const float mx = a[0];
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        a[i] = (i < k_in && sid[warp][i] != -1) ? expf(a[i] - mx) : 0.f;
        sum += a[i];
      }
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int id = sid[warp][i];
        const bool live = i < k_in && id != -1;
        sw[warp][i] = live ? __fdiv_rn(a[i], sum) : 0.f;
        int row = -1;
        if (live && id >= 0) {
          const int pos = id / nf;
          row = __ldg(mem_label + job.mem_begin + pos) * nf + (id - pos * nf);
        }
        srow[warp][i] = row;                      // row < 0: contributes value 0 (but its weight took soft-max mass)
      }
    }
  }
  if (n_lists > 32 && tid < QB) {
    const int q = q0 + tid;
    TopK<K> top;
    top.init();
    if (q < nc) {
      for (int l = 0; l < n_lists; ++l)                    // partial lists of the (entry, chunk) CTAs, each sorted
        for (int i = 0; i < k_in; ++i) {
          const float v = __ldg(tv + ((int64_t)q * n_lists + l) * k_in + i);
          const int id = __ldg(ti + ((int64_t)q * n_lists + l) * k_in + i);
          if (id < 0 || !(v > top.thr())) break;
          top.push(v, id);
        }
      // zero-padded window positions of all memory entries
      int n_zero = 0;
      const int R = 2 * rf + 1;
      for (int t = 0; t < n_mem && n_zero < K; ++t) {
        const int b = max(__ldg(best_idx + (int64_t)t * nc + q), 0) % nc;
        const int cy = (b / Wc) * scale, cx = (b % Wc) * scale;
        const int rows = min(cy + rf, Hf - 1) - max(cy - rf, 0) + 1, cols = min(cx + rf, Wf - 1) - max(cx - rf, 0) + 1;
        n_zero += R * R - rows * cols;
      }
      for (int z = 0; z < min(n_zero, K); ++z) {
        if (!(0.f > top.thr())) break;
        top.push(0.f, -2);                       // id -2: padded candidate, value row of zeros
      }
    }
    float a[K];
#pragma unroll
    for (int i = 0; i < K; ++i) a[i] = __fdiv_rn(top.v[i], temperature);
    const float mx = a[0];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      a[i] = (i < k_in && top.id[i] != -1) ? expf(a[i] - mx) : 0.f;
      sum += a[i];
    }
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const int id = top.id[i];
      const bool live = i < k_in && id != -1;
      sw[tid][i] = live ? __fdiv_rn(a[i], sum) : 0.f;
      int row = -1;
      if (live && id >= 0) {
        const int pos = id / nf;
        row = __ldg(mem_label + job.mem_begin + pos) * nf + (id - pos * nf);
      }
      srow[tid][i] = row;                        // row < 0: contributes value 0 (but its weight took soft-max mass)
    }
  }
}

template <int K>
__global__ void __launch_bounds__(256)
c2f_tail_kernel(const float* __restrict__ tv, const int32_t* __restrict__ ti, int k_in, int n_lists, int Hc, int Wc, int Hf, int Wf,
                int scale, fgvc_job job, const int32_t* __restrict__ mem_label, const int32_t* __restrict__ best_idx,
                int rf, float temperature, const float* __restrict__ fine_lab, int Lp, float* __restrict__ out) {
  constexpr int QB = C2F_TAIL_QB;
  __shared__ float sw[QB][K];
  __shared__ int srow[QB][K];
  const int q0 = blockIdx.x * QB;
  const int tid = threadIdx.x;
  const int nc = Hc * Wc;
  c2f_tail_pairs<K>(tv, ti, k_in, n_lists, Hc, Wc, Hf, Wf, scale, job, mem_label, best_idx, rf, temperature, q0, sw, srow);
  __syncthreads();
  const int l4n = Lp / 4;
  const float4* src = reinterpret_cast<const float4*>(fine_lab);
  float4* dst = reinterpret_cast<float4*>(out) + (int64_t)q0 * l4n;
  const int nq = min(QB, nc - q0);
  for (int i = tid; i < nq * l4n; i += 256) {
    const int q = i / l4n, c = i - q * l4n;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const float w = sw[q][j];
      if (w != 0.f && srow[q][j] >= 0) {
        const float4 v = __ldg(src + (int64_t)srow[q][j] * l4n + c);
        acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
        acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
      }
    }
    dst[i] = acc;
  }
}

template <int K>
static int launch_tail(const float* tv, const int32_t* ti, int k_in, int n_lists, int Hc, int Wc, int Hf, int Wf, int scale,
                       const fgvc_job& job, const int32_t* mem_label, const int32_t* best, int rf, float temperature,
                       const float* fine_lab, int Lp, float* out, cudaStream_t st) {
  c2f_tail_kernel<K><<<cdiv(Hc * Wc, C2F_TAIL_QB), 256, 0, st>>>(tv, ti, k_in, n_lists, Hc, Wc, Hf, Wf, scale, job, mem_label, best,
                                                       rf, temperature, fine_lab, Lp, out);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

template <int K, int FMT>
static int launch_fine(const void* fine_bank, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                       const fgvc_job& job, const int32_t* mem_feat, const int32_t* mem_label,
                       const int32_t* best, int rf, int k_out, float temperature, const float* fine_lab, int Lp,
                       float* out, cudaStream_t st) {
  c2f_fine_kernel<K, FMT><<<Hc * Wc, 256, Cf * sizeof(float), st>>>(fine_bank, Hc, Wc, Hf, Wf, Cf, scale, job,
                                                               mem_feat, mem_label, best, rf, k_out, temperature,
                                                               fine_lab, Lp, out);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

// The label-independent half of c2f_tail_kernel for the jobs of a c2f_wjob table: job blockIdx.y, its lists at
// tv / ti + list_off and its arg-max table at best_idx + best_off; the pairs go to w_out / row_out[job][q][k_in].
template <int K>
__global__ void __launch_bounds__(256)
c2f_weights_kernel(const float* __restrict__ tv, const int32_t* __restrict__ ti, int k_in, int Hc, int Wc, int Hf,
                   int Wf, int scale, const c2f_wjob* __restrict__ wjobs, const int32_t* __restrict__ mem_label,
                   const int32_t* __restrict__ best_idx, int rf, float temperature, float* __restrict__ w_out,
                   int32_t* __restrict__ row_out) {
  constexpr int QB = C2F_TAIL_QB;
  __shared__ float sw[QB][K];
  __shared__ int srow[QB][K];
  __shared__ c2f_wjob wj;                  // (shared: nothing of it has to stay in registers across the selection)
  if (threadIdx.x == 0) wj = wjobs[blockIdx.y];
  __syncthreads();
  const int q0 = blockIdx.x * QB;
  const int nc = Hc * Wc;
  c2f_tail_pairs<K>(tv + wj.list_off, ti + wj.list_off, k_in, (wj.job.mem_end - wj.job.mem_begin) * wj.chunks, Hc, Wc,
                    Hf, Wf, scale, wj.job, mem_label, best_idx + wj.best_off, rf, temperature, q0, sw, srow);
  __syncthreads();
  const int nq = min(QB, nc - q0);
  for (int i = threadIdx.x; i < nq * k_in; i += 256) {
    const int q = i / k_in, k = i - q * k_in;
    const int64_t o = ((int64_t)blockIdx.y * nc + q0) * k_in + i;
    w_out[o] = sw[q][k];
    row_out[o] = srow[q][k];
  }
}

// ------------------------------------------------------------------ the multi-lane c2f chain
// Every coarse-to-fine recurrence (lane) of a clip in ONE cooperative kernel.  Step s, for every lane still running:
// phase 1 gathers job s's coarse output out[q][c] = sum_k w * fine_lab[row][c] from the pairs of fgvc_c2f_clip_weights
// (per (query, 4 channels) the FMA sequence of the gathers of c2f_tail_kernel / c2f_fine_kernel: k ascending, pairs with
// weight 0 or row < 0 skipped) into the job's out_slot of the lane's coarse-output bank; grid barrier; phase 2
// up-samples it into the job's out_slot of the lane's fine bank (upsample_labels_kernel's taps and blend); grid
// barrier.  The items of all running lanes of a phase are dealt to the threads of the grid as one sequence, so a
// phase with many short lanes keeps every thread busy.  Loads of banks written in this kernel are ld.global.cg.
// (32-bit indices: a lane's phase has fewer than 2^31 items -- checked by the launcher -- and the grid fewer threads)
__device__ __forceinline__ int first_item(int me, int base_mod, int G) {
  // the first item i >= 0 of a lane with (base + i) % G == me, base_mod = base % G: the lane's items continue the
  // running sequence
  return me >= base_mod ? me - base_mod : me + G - base_mod;
}

template <int K>
__global__ void __launch_bounds__(256)
c2f_chain_lanes_kernel(const float* __restrict__ cw, const int32_t* __restrict__ crow, int k_in,
                       const fgvc_job* __restrict__ jobs, int job_base, const fgvc_c2f_lane* __restrict__ lanes,
                       int n_lanes, int n_steps, int Hc, int Wc, int Hf, int Wf, float* fine_lab, float* coarse_out,
                       unsigned int* barrier) {
  const int G = gridDim.x * 256, me = blockIdx.x * 256 + threadIdx.x;
  const int nc = Hc * Wc, nf = Hf * Wf;
  unsigned int n_bar = 0;
  for (int s = 0; s < n_steps; ++s) {
    int base = 0;                                  // items dealt so far in this phase, mod G
    for (int l = 0; l < n_lanes; ++l) {
      const fgvc_c2f_lane& ln = lanes[l];
      if (ln.job_end - ln.job_begin <= s) continue;
      const int l4n = ln.Lp / 4, j = ln.job_begin + s;
      const int slot = jobs[j].out_slot;
      const float4* src = reinterpret_cast<const float4*>(fine_lab + ln.lab_offset);
      float4* dst = reinterpret_cast<float4*>(coarse_out + ln.out_offset) + (int64_t)slot * nc * l4n;
      const int items = nc * l4n;
      const float* w = cw + (int64_t)(j - job_base) * nc * k_in;
      const int32_t* r = crow + (int64_t)(j - job_base) * nc * k_in;
      for (int i = first_item(me, base, G); i < items; i += G) {
        const int q = i / l4n, c = i - q * l4n;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
          if (k < k_in) {
            const float wk = __ldg(w + (int64_t)q * k_in + k);
            const int rk = __ldg(r + (int64_t)q * k_in + k);
            if (wk != 0.f && rk >= 0) {
              const float4 v = __ldcg(src + (int64_t)rk * l4n + c);     // written by the previous step's phase 2
              acc.x = fmaf(wk, v.x, acc.x); acc.y = fmaf(wk, v.y, acc.y);
              acc.z = fmaf(wk, v.z, acc.z); acc.w = fmaf(wk, v.w, acc.w);
            }
          }
        }
        dst[i] = acc;
      }
      base = (base + items % G) % G;
    }
    grid_barrier(barrier, ++n_bar);
    base = 0;
    for (int l = 0; l < n_lanes; ++l) {
      const fgvc_c2f_lane& ln = lanes[l];
      if (ln.job_end - ln.job_begin <= s) continue;
      const int l4n = ln.Lp / 4, j = ln.job_begin + s;
      const int slot = jobs[j].out_slot;
      const float4* src = reinterpret_cast<const float4*>(coarse_out + ln.out_offset) + (int64_t)slot * nc * l4n;
      float4* dst = reinterpret_cast<float4*>(fine_lab + ln.lab_offset) + (int64_t)slot * nf * l4n;
      const int items = nf * l4n;
      for (int i = first_item(me, base, G); i < items; i += G) {
        const int pix = i / l4n, l4 = i - pix * l4n;
        const int y = pix / Wf, x = pix - y * Wf;
        const BilinearTaps t = bilinear_taps(y, x, Hc, Wc, Hf, Wf);
        const float4 a = __ldcg(src + (int64_t)t.p00 * l4n + l4), b = __ldcg(src + (int64_t)t.p01 * l4n + l4);
        const float4 c = __ldcg(src + (int64_t)t.p10 * l4n + l4), d = __ldcg(src + (int64_t)t.p11 * l4n + l4);
        dst[i] = bilinear_mix(t, a, b, c, d);
      }
      base = (base + items % G) % G;
    }
    if (s + 1 < n_steps) grid_barrier(barrier, ++n_bar);
  }
}

template <int K>
static int launch_chain_t(const float* cw, const int32_t* crow, int k_in, int job_base, const fgvc_job* jobs_dev,
                          const fgvc_c2f_lane* lanes_dev, int n_lanes, int n_steps, int64_t max_items, int Hc, int Wc,
                          int Hf, int Wf, float* fine_lab, float* coarse_out, unsigned int* barrier, cudaStream_t st) {
  static std::atomic<int> cached[64];
  int max_ctas = 0;
  int rc = resident_ctas((const void*)c2f_chain_lanes_kernel<K>, cached, &max_ctas);
  if (rc) return rc;
  // every co-resident CTA: the phases are bandwidth work over up to (lanes x fine map x Lp / 4) items
  const int ctas = (int)min((int64_t)max_ctas, max((int64_t)1, (max_items + 255) / 256));
  int ki = k_in, jb = job_base, nl = n_lanes, ns = n_steps, hc = Hc, wc = Wc, hf = Hf, wf = Wf;
  void* args[] = {(void*)&cw, (void*)&crow, (void*)&ki, (void*)&jobs_dev, (void*)&jb, (void*)&lanes_dev, (void*)&nl,
                  (void*)&ns, (void*)&hc, (void*)&wc, (void*)&hf, (void*)&wf, (void*)&fine_lab, (void*)&coarse_out,
                  (void*)&barrier};
  FGVC_CUDA(cudaLaunchCooperativeKernel((const void*)c2f_chain_lanes_kernel<K>, dim3(ctas), dim3(256), args, 0, st));
  fgvc::g_launches.fetch_add(1);
  return FGVC_OK;
}

// the lanes are validated by the caller (fgvc_c2f_point_clip_tail_lanes); the barrier counter is zeroed here
int launch_c2f_chain_lanes(const float* cw, const int32_t* crow, int K, int job_base, const fgvc_job* jobs_dev,
                           const fgvc_c2f_lane* lanes_dev, const fgvc_c2f_lane* lanes_host, int n_lanes, int Hc, int Wc,
                           int Hf, int Wf, float* fine_lab, float* coarse_out, unsigned int* barrier, cudaStream_t st) {
  int n_steps = 0;
  int64_t items = 0;
  for (int i = 0; i < n_lanes; ++i) {
    n_steps = max(n_steps, lanes_host[i].job_end - lanes_host[i].job_begin);
    items += (int64_t)Hf * Wf * (lanes_host[i].Lp / 4);
    FGVC_CHECK_ARG((int64_t)Hf * Wf * (lanes_host[i].Lp / 4) < (1ll << 31),
                   "c2f chain: a %dx%d map of %d labels is too large", Hf, Wf, lanes_host[i].Lp);
  }
  FGVC_CUDA(cudaMemsetAsync(barrier, 0, 256, st));
  if (K <= 4) return launch_chain_t<4>(cw, crow, K, job_base, jobs_dev, lanes_dev, n_lanes, n_steps, items, Hc, Wc, Hf, Wf, fine_lab, coarse_out, barrier, st);
  if (K <= 10) return launch_chain_t<10>(cw, crow, K, job_base, jobs_dev, lanes_dev, n_lanes, n_steps, items, Hc, Wc, Hf, Wf, fine_lab, coarse_out, barrier, st);
  return launch_chain_t<16>(cw, crow, K, job_base, jobs_dev, lanes_dev, n_lanes, n_steps, items, Hc, Wc, Hf, Wf, fine_lab, coarse_out, barrier, st);
}

// the fine stage of fgvc_c2f_propagate runs as a window-mode K1 (+ tail) exactly when this holds (else c2f_fine_kernel)
bool c2f_use_window(int engine, int fine_format, int Hf, int Wf, int Cf, int K, int n_mem) {
  static const bool no_window = getenv("FGVC_C2F_SIMT") != nullptr;
  return !no_window && engine != FGVC_ENGINE_SIMT && fine_format == FGVC_BANK_F16 &&
         c2f_window_supported(Hf, Wf, Cf, K, n_mem);
}

}  // namespace fgvc

using namespace fgvc;

extern "C" int64_t fgvc_c2f_scratch_elems(int32_t n_mem, int32_t n_coarse) {
  // coarse per-frame arg-max table + one floor per coarse query + the fine top-K lists (K <= 16) of up to 4 chunk
  // CTAs per memory entry
  return ((int64_t)n_mem + 1 + (int64_t)n_mem * 4 * 16) * n_coarse;
}

extern "C" int fgvc_c2f_propagate(const void* coarse_bank, int32_t coarse_format, int32_t n_slots, int32_t Hc, int32_t Wc,
                                  int32_t C, const void* fine_bank, int32_t fine_format, int32_t Hf, int32_t Wf, int32_t Cf,
                                  const fgvc_job* job_dev, const fgvc_job* job_host, const int32_t* mem_feat_slot,
                                  const int32_t* mem_label_slot, int32_t radius, int32_t mask_mode,
                                  int32_t radius_fine, int32_t K, float temperature, const float* fine_lab_bank,
                                  int32_t Lp, float* out, float* scratch_val, int32_t* scratch_idx,
                                  int64_t scratch_elems, int32_t engine, void* stream) {
  FGVC_CHECK_ARG(coarse_bank && fine_bank && job_dev && job_host && mem_feat_slot && mem_label_slot &&
                     fine_lab_bank && out && scratch_val && scratch_idx, "fgvc_c2f_propagate: null pointer");
  FGVC_CHECK_ARG(Hc > 0 && Wc > 0 && Hf % Hc == 0 && Hf / Hc >= 1 && Wf >= Wc * (Hf / Hc) - (Hf / Hc) + 1,
                 "fgvc_c2f_propagate: fine map %dx%d is not a multiple of the coarse map %dx%d", Hf, Wf, Hc, Wc);
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_c2f_propagate: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(Cf % 4 == 0 && Lp % 4 == 0 && radius_fine >= 0 && temperature > 0, "fgvc_c2f_propagate: bad sizes");
  const int n_mem = job_host->mem_end - job_host->mem_begin;
  FGVC_CHECK_ARG(n_mem >= 1 && n_mem <= 64, "fgvc_c2f_propagate: memory length %d not in [1,64]", n_mem);
  FGVC_CHECK_ARG(scratch_elems >= fgvc_c2f_scratch_elems(n_mem, Hc * Wc),
                 "fgvc_c2f_propagate: scratch arrays need %lld elements each (fgvc_c2f_scratch_elems)",
                 (long long)fgvc_c2f_scratch_elems(n_mem, Hc * Wc));
  // coarse stage: top-1 per memory frame == groups = n_mem
  int rc = fgvc_affinity_topk(coarse_bank, coarse_format, n_slots, Hc, Wc, C, job_dev, 1, mem_feat_slot, radius, mask_mode, 1, n_mem,
                              scratch_val, scratch_idx, engine, stream);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int scale = Hf / Hc;
  // fine stage on the tensor cores (window-mode K1 + tail) whenever the fine bank allows; else one warp per candidate
  if (c2f_use_window(engine, fine_format, Hf, Wf, Cf, K, n_mem)) {
    float* floor_ws = scratch_val + (int64_t)n_mem * Hc * Wc;    // behind the coarse arg-max table: the floors,
    float* fv = floor_ws + (int64_t)Hc * Wc;                     // then the fine lists
    int32_t* fi = scratch_idx + (int64_t)(n_mem + 1) * Hc * Wc;
    const int chunks = c2f_window_chunks(Hc, Wc, n_mem);
    const int n_lists = n_mem * chunks;
    rc = launch_c2f_window_tc16(fine_bank, n_slots, Hc, Wc, Hf, Wf, Cf, scale, *job_host, mem_feat_slot, scratch_idx,
                                radius_fine, K, chunks, floor_ws, fv, fi, st);
    if (rc == FGVC_OK) {
      if (K <= 4) return launch_tail<4>(fv, fi, K, n_lists, Hc, Wc, Hf, Wf, scale, *job_host, mem_label_slot, scratch_idx, radius_fine, temperature, fine_lab_bank, Lp, out, st);
      if (K <= 10) return launch_tail<10>(fv, fi, K, n_lists, Hc, Wc, Hf, Wf, scale, *job_host, mem_label_slot, scratch_idx, radius_fine, temperature, fine_lab_bank, Lp, out, st);
      return launch_tail<16>(fv, fi, K, n_lists, Hc, Wc, Hf, Wf, scale, *job_host, mem_label_slot, scratch_idx, radius_fine, temperature, fine_lab_bank, Lp, out, st);
    }
    if (rc != FGVC_ERR_UNSUPPORTED) return rc;
  }
#define FGVC_FINE(KK)                                                                                              \
  return fine_format == FGVC_BANK_TF32                                                                             \
             ? launch_fine<KK, FGVC_BANK_TF32>(fine_bank, Hc, Wc, Hf, Wf, Cf, scale, *job_host, mem_feat_slot,      \
                                               mem_label_slot, scratch_idx, radius_fine, K, temperature,            \
                                               fine_lab_bank, Lp, out, st)                                          \
             : launch_fine<KK, FGVC_BANK_F16>(fine_bank, Hc, Wc, Hf, Wf, Cf, scale, *job_host, mem_feat_slot,       \
                                              mem_label_slot, scratch_idx, radius_fine, K, temperature,             \
                                              fine_lab_bank, Lp, out, st)
  if (K <= 4) { FGVC_FINE(4); }
  if (K <= 10) { FGVC_FINE(10); }
  FGVC_FINE(16);
#undef FGVC_FINE
}

// ------------------------------------------------------------------ clip level: the label-independent half
// workspace of fgvc_c2f_clip_weights (byte offsets, 256-aligned): the length-sorted coarse job table, the c2f_wjob
// table, the coarse arg-max tables (val + idx), the floors, the fine lists (val + idx)
namespace {
struct ClipLayout {
  int64_t cjobs, wjobs, best_val, best_idx, floor, list_val, list_idx, total;
};
int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }
ClipLayout clip_layout(const fgvc_job* jobs_host, int job_begin, int job_end, int Hc, int Wc, int K) {
  int64_t sum_mem = 0, sum_lists = 0;
  for (int j = job_begin; j < job_end; ++j) {
    const int m = jobs_host[j].mem_end - jobs_host[j].mem_begin;
    sum_mem += m;
    sum_lists += (int64_t)m * c2f_window_chunks(Hc, Wc, m);
  }
  const int64_t n = job_end - job_begin, nc = (int64_t)Hc * Wc;
  ClipLayout L;
  int64_t o = 0;
  L.cjobs = o; o += align256(n * (int64_t)sizeof(fgvc_job));
  L.wjobs = o; o += align256(n * (int64_t)sizeof(c2f_wjob));
  L.best_val = o; o += align256(sum_mem * nc * 4);
  L.best_idx = o; o += align256(sum_mem * nc * 4);
  L.floor = o; o += align256(n * nc * 4);
  L.list_val = o; o += align256(sum_lists * nc * K * 4);
  L.list_idx = o; o += align256(sum_lists * nc * K * 4);
  L.total = o;
  return L;
}
}  // namespace

extern "C" int64_t fgvc_c2f_clip_workspace_bytes(const fgvc_job* jobs_host, int32_t job_begin, int32_t job_end,
                                                 int32_t Hc, int32_t Wc, int32_t K) {
  if (jobs_host == nullptr || job_begin < 0 || job_end <= job_begin || Hc <= 0 || Wc <= 0 || K < 1 || K > 16) return -1;
  return clip_layout(jobs_host, job_begin, job_end, Hc, Wc, K).total;
}

extern "C" int fgvc_c2f_clip_weights(const void* coarse_bank, int32_t coarse_format, int32_t n_slots, int32_t Hc,
                                     int32_t Wc, int32_t C, const void* fine_bank, int32_t fine_format, int32_t Hf, int32_t Wf,
                                     int32_t Cf,
                                     const fgvc_job* jobs_host, int32_t job_begin, int32_t job_end,
                                     const int32_t* mem_feat_slot, const int32_t* mem_label_slot, int32_t radius,
                                     int32_t mask_mode, int32_t radius_fine, int32_t K, float temperature, float* weights,
                                     int32_t* rows, void* ws, int64_t ws_bytes, int32_t engine, void* stream) {
  FGVC_CHECK_ARG(coarse_bank && fine_bank && jobs_host && mem_feat_slot && mem_label_slot && weights && rows && ws,
                 "fgvc_c2f_clip_weights: null pointer");
  FGVC_CHECK_ARG(Hc > 0 && Wc > 0 && Hf % Hc == 0 && Hf / Hc >= 1 && Wf >= Wc * (Hf / Hc) - (Hf / Hc) + 1,
                 "fgvc_c2f_clip_weights: fine map %dx%d is not a multiple of the coarse map %dx%d", Hf, Wf, Hc, Wc);
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_c2f_clip_weights: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(Cf % 4 == 0 && radius_fine >= 0 && temperature > 0, "fgvc_c2f_clip_weights: bad sizes");
  FGVC_CHECK_ARG(job_begin >= 0 && job_end > job_begin && job_end - job_begin <= 65535,
                 "fgvc_c2f_clip_weights: job range [%d, %d) empty or longer than 65535", job_begin, job_end);
  const int n = job_end - job_begin, nc = Hc * Wc, scale = Hf / Hc;
  int max_mem = 0;
  for (int j = job_begin; j < job_end; ++j) {
    const int m = jobs_host[j].mem_end - jobs_host[j].mem_begin;
    FGVC_CHECK_ARG(m >= 1 && m <= 64, "fgvc_c2f_clip_weights: memory length %d of job %d not in [1,64]", m, j);
    max_mem = max(max_mem, m);
  }
  const ClipLayout L = clip_layout(jobs_host, job_begin, job_end, Hc, Wc, K);
  FGVC_CHECK_ARG(ws_bytes >= L.total, "fgvc_c2f_clip_weights: workspace of %lld bytes needed (fgvc_c2f_clip_workspace_bytes)",
                 (long long)L.total);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* base = reinterpret_cast<uint8_t*>(ws);
  fgvc_job* cjobs_dev = reinterpret_cast<fgvc_job*>(base + L.cjobs);
  c2f_wjob* wjobs_dev = reinterpret_cast<c2f_wjob*>(base + L.wjobs);
  float* best_val = reinterpret_cast<float*>(base + L.best_val);
  int32_t* best_idx = reinterpret_cast<int32_t*>(base + L.best_idx);
  float* floor_ws = reinterpret_cast<float*>(base + L.floor);
  float* lv = reinterpret_cast<float*>(base + L.list_val);
  int32_t* li = reinterpret_cast<int32_t*>(base + L.list_idx);

  // coarse stage: K1 with K = 1 and one group per memory entry gives one arg-max list per entry only when every job
  // of the launch has the same memory length -- one launch per length over a length-sorted copy of the jobs
  std::vector<int> order(n);
  std::iota(order.begin(), order.end(), 0);
  auto len = [&](int i) { return jobs_host[job_begin + i].mem_end - jobs_host[job_begin + i].mem_begin; };
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return len(a) < len(b); });
  std::vector<fgvc_job> cjobs(n);
  std::vector<c2f_wjob> wj(n);
  int64_t best_off = 0;
  for (int i = 0; i < n; ++i) {
    cjobs[i] = jobs_host[job_begin + order[i]];
    wj[order[i]].best_off = best_off;
    best_off += (int64_t)len(order[i]) * nc;
  }
  int n_y = 0;
  int64_t list_off = 0;
  for (int i = 0; i < n; ++i) {
    const int m = len(i);
    wj[i].job = jobs_host[job_begin + i];
    wj[i].chunks = c2f_window_chunks(Hc, Wc, m);
    wj[i].y_begin = n_y;
    wj[i].floor_off = (int64_t)i * nc;
    wj[i].list_off = list_off;
    n_y += m * wj[i].chunks;
    list_off += (int64_t)m * wj[i].chunks * K * nc;
  }
  // (pageable sources: the copies return once the tables are staged, so the vectors may go)
  FGVC_CUDA(cudaMemcpyAsync(cjobs_dev, cjobs.data(), n * sizeof(fgvc_job), cudaMemcpyHostToDevice, st));
  FGVC_CUDA(cudaMemcpyAsync(wjobs_dev, wj.data(), n * sizeof(c2f_wjob), cudaMemcpyHostToDevice, st));
  for (int a = 0; a < n;) {
    int b = a;
    while (b < n && len(order[b]) == len(order[a])) ++b;
    const int m = len(order[a]);
    const int64_t o = wj[order[a]].best_off;
    int rc = fgvc_affinity_topk(coarse_bank, coarse_format, n_slots, Hc, Wc, C, cjobs_dev + a, b - a, mem_feat_slot, radius,
                                mask_mode, 1, m, best_val + o, best_idx + o, engine, stream);
    if (rc) return rc;
    a = b;
  }

  // fine stage of every job: window-mode K1 + weights kernel on the tensor cores, else the one-warp-per-candidate
  // kernel in its weights-only form -- the choice fgvc_c2f_propagate makes for each job
  if (c2f_use_window(engine, fine_format, Hf, Wf, Cf, K, max_mem)) {
    int rc = launch_c2f_window_tc16_jobs(fine_bank, n_slots, Hc, Wc, Hf, Wf, Cf, scale, wjobs_dev, n, n_y, mem_feat_slot,
                                         best_idx, radius_fine, K, floor_ws, lv, li, st);
    if (rc == FGVC_OK) {
      dim3 grid(cdiv(nc, C2F_TAIL_QB), n);
#define FGVC_WEIGHTS(KK)                                                                                           \
  c2f_weights_kernel<KK><<<grid, 256, 0, st>>>(lv, li, K, Hc, Wc, Hf, Wf, scale, wjobs_dev, mem_label_slot, best_idx, \
                                               radius_fine, temperature, weights, rows)
      if (K <= 4) FGVC_WEIGHTS(4);
      else if (K <= 10) FGVC_WEIGHTS(10);
      else FGVC_WEIGHTS(16);
#undef FGVC_WEIGHTS
      FGVC_LAUNCH_CHECK();
      return FGVC_OK;
    }
    if (rc != FGVC_ERR_UNSUPPORTED) return rc;
  }
  const fgvc_job none = {0, 0, 1, 0};
  dim3 grid(nc, n);
#define FGVC_FINE_W(KK, FMT)                                                                                        \
  c2f_fine_kernel<KK, FMT, true><<<grid, 256, Cf * sizeof(float), st>>>(                                            \
      fine_bank, Hc, Wc, Hf, Wf, Cf, scale, none, mem_feat_slot, mem_label_slot, best_idx, radius_fine, K, temperature, \
      nullptr, 0, nullptr, wjobs_dev, weights, rows)
#define FGVC_FINE_K(KK)                                               \
  if (fine_format == FGVC_BANK_TF32) FGVC_FINE_W(KK, FGVC_BANK_TF32); \
  else FGVC_FINE_W(KK, FGVC_BANK_F16)
  if (K <= 4) { FGVC_FINE_K(4); }
  else if (K <= 10) { FGVC_FINE_K(10); }
  else { FGVC_FINE_K(16); }
#undef FGVC_FINE_K
#undef FGVC_FINE_W
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}
