// K1b: merge the per-group top-K lists, divide by the temperature, softmax over the K
// winners and gather + weighted-sum the label rows (local_attention.py:356-374).
// HBM/L2-bound: K label rows of Lp floats per query, read as float4, coalesced along L.
#include <stdlib.h>

#include "common.cuh"

namespace fgvc {

constexpr int QB = 64;  // queries per CTA

// Local-window ("HR") propagation (HRVanillaTracker.forward_test_main, vanilla_tracker.py:547-563): the candidates of
// a query are the (2r+1)^2 window positions of every memory frame, and the positions OUTSIDE the image are still
// candidates -- mmcv's Correlation and F.unfold(padding=r) give them affinity 0 and value 0.  K1 lists only the real
// keys; here the n_oob zero candidates of the query are merged analytically: they displace the negative real
// winners from the end of the (sorted) list.  Returns how many zeros enter the top-K.
template <int K>
__device__ __forceinline__ int zero_pad_count(const TopK<K>& top, int k_in, int flags, int q, int n_pix, int n_mem) {
  if (!(flags & FGVC_ZERO_PAD)) return 0;
  const int r = (flags >> 8) & 0xff, W = (flags >> 16) & 0xffff, H = n_pix / W;
  const int qy = q / W, qx = q - qy * W;
  const int cy = min(qy + r, H - 1) - max(qy - r, 0) + 1, cx = min(qx + r, W - 1) - max(qx - r, 0) + 1;
  const int n_oob = n_mem * ((2 * r + 1) * (2 * r + 1) - cy * cx);
  int nonneg = 0;
#pragma unroll
  for (int i = 0; i < K; ++i) nonneg += (i < k_in && top.id[i] >= 0 && top.v[i] >= 0.f) ? 1 : 0;
  return min(n_oob, k_in - nonneg);
}

template <int K>
__global__ void __launch_bounds__(256)
gather_labels_kernel(const float* __restrict__ tv, const int32_t* __restrict__ ti, int k_in, int groups,
                     const fgvc_job* __restrict__ jobs, int job_begin, const int32_t* __restrict__ mem_label,
                     int n_pix, float temperature, int flags, float* __restrict__ lab, int Lp) {
  __shared__ float sw[QB][K];
  __shared__ int srow[QB][K];
  const int jidx = job_begin + blockIdx.y;
  const fgvc_job job = jobs[jidx];
  const int q0 = blockIdx.x * QB;
  const int tid = threadIdx.x;
  if (tid < QB) {
    const int q = q0 + tid;
    TopK<K> top;
    top.init();
    if (q < n_pix) {
      for (int g = 0; g < groups; ++g) {
        int64_t o = (((int64_t)jidx * groups + g) * n_pix + q) * k_in;
        for (int i = 0; i < k_in; ++i) {
          float v = __ldg(tv + o + i);
          int id = __ldg(ti + o + i);
          if (id >= 0 && v > top.thr()) top.push(v, id);
        }
      }
    }
    // weights of the winners; empty entries (-inf) weigh 0.
    //   similarity  a = cos / temperature                      (dot_product, local_attention.py:321-323)
    //               a = (2 cos - 1) / sqrt(C) [= temperature]  (l2-distance on unit vectors, :324-327)
    //   weights     softmax(a) (:369)   or   clamp(a, 0)^2 ('cosine', :371)
    const int zt = q < n_pix ? zero_pad_count<K>(top, k_in, flags, q, n_pix, job.mem_end - job.mem_begin) : 0;
    float a[K];
#pragma unroll
    for (int i = 0; i < K; ++i)
      a[i] = (flags & FGVC_SIM_L2) ? __fdiv_rn(2.f * top.v[i] - 1.f, temperature) : __fdiv_rn(top.v[i], temperature);
    float m = zt > 0 ? fmaxf(a[0], 0.f) : a[0], sum = 0.f;
    if (flags & FGVC_WEIGHT_COSINE) {
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const float c = fmaxf(a[i], 0.f);
        a[i] = (i < k_in - zt && top.id[i] >= 0) ? c * c : 0.f;
      }
      sum = 1.f;
    } else {
#pragma unroll
      for (int i = 0; i < K; ++i) {
        a[i] = (i < k_in - zt && top.id[i] >= 0) ? expf(a[i] - m) : 0.f;
        sum += a[i];
      }
      sum += (float)zt * expf(0.f - m);          // the zero-padded winners: weight exp(0 / temperature), value 0
    }
#pragma unroll
    for (int i = 0; i < K; ++i) {
      int id = top.id[i];
      bool ok = i < k_in - zt && id >= 0;
      sw[tid][i] = ok ? ((flags & FGVC_WEIGHT_COSINE) ? a[i] : __fdiv_rn(a[i], sum)) : 0.f;
      int row = 0;
      if (ok) {
        int pos = id / n_pix;
        row = __ldg(mem_label + job.mem_begin + pos) * n_pix + (id - pos * n_pix);
      }
      srow[tid][i] = row;
    }
  }
  __syncthreads();
  const int l4n = Lp / 4;
  const float4* src = reinterpret_cast<const float4*>(lab);
  float4* dst = reinterpret_cast<float4*>(lab) + ((int64_t)job.out_slot * n_pix + q0) * l4n;
  const int nq = min(QB, n_pix - q0);
  for (int i = tid; i < nq * l4n; i += 256) {
    int q = i / l4n, c = i - q * l4n;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < K; ++j) {
      float w = sw[q][j];
      if (w != 0.f) {
        float4 v = __ldg(src + (int64_t)srow[q][j] * l4n + c);
        acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
        acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
      }
    }
    dst[i] = acc;
  }
}

template <int K>
static int launch_g(const float* tv, const int32_t* ti, int k_in, int groups, const fgvc_job* jobs,
                    int job_begin, int n, const int32_t* mem_label, int n_pix, float temperature, int flags,
                    float* lab, int Lp, cudaStream_t st) {
  dim3 grid(cdiv(n_pix, QB), n);
  gather_labels_kernel<K><<<grid, 256, 0, st>>>(tv, ti, k_in, groups, jobs, job_begin, mem_label, n_pix,
                                                temperature, flags, lab, Lp);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}


// ------------------------------------------------------------------ the gather CHAIN
// The recurrence of the reference loop (vanilla_tracker.py:345-394) lives only in the gather: frame t's
// labels are a sparse combination of the labels of its memory frames.  One launch per frame costs ~20 us of
// launch + drain latency for ~5 us of work, so a clip's chain is run by ONE persistent kernel:
//   gather_weights_kernel : label-independent part for ALL jobs at once (merge groups, temperature, soft-max):
//                           w[job][q][K], src_row[job][q][K] (label row = slot * n_pix + pixel);
//   gather_chain_kernel   : cooperative launch, every CTA owns a fixed slice of the queries; per job it
//                           gathers its slice, then all CTAs meet at a grid barrier (the next job reads rows
//                           other CTAs wrote: label loads are ld.global.cg, stores are fenced before the barrier).
template <int K>
__global__ void __launch_bounds__(256)
gather_weights_kernel(const float* __restrict__ tv, const int32_t* __restrict__ ti, int k_in, int groups,
                      const fgvc_job* __restrict__ jobs, int job_begin, const int32_t* __restrict__ mem_label,
                      const int32_t* __restrict__ pair_ref, int n_pix, float temperature, int flags,
                      float* __restrict__ cw, int32_t* __restrict__ crow) {
  const int jidx = job_begin + blockIdx.y;
  const int q = blockIdx.x * 256 + threadIdx.x;
  if (q >= n_pix) return;
  const fgvc_job job = jobs[jidx];
  TopK<K> top;
  top.init();
  if (pair_ref == nullptr) {
    for (int g = 0; g < groups; ++g) {
      const int64_t o = (((int64_t)jidx * groups + g) * n_pix + q) * k_in;
      // all loads of a list first (the kernel is latency-bound: ~11 stall cycles per instruction on dependent loads)
      float vb[K];
      int ib[K];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        vb[i] = i < k_in ? __ldg(tv + o + i) : -INFINITY;
        ib[i] = i < k_in ? __ldg(ti + o + i) : -1;
      }
#pragma unroll
      for (int i = 0; i < K; ++i)
        if (ib[i] >= 0 && vb[i] > top.thr()) top.push(vb[i], ib[i]);
    }
  } else {
    // shared per-(query frame, memory frame) lists: entry e of this job reads list pair_ref[e]; the key pixel
    // is kept, the position becomes the entry's position in THIS job's memory list
    for (int e = job.mem_begin; e < job.mem_end; ++e) {
      const int64_t o = ((int64_t)__ldg(pair_ref + e) * n_pix + q) * k_in;
      for (int i = 0; i < k_in; ++i) {
        const float v = __ldg(tv + o + i);
        const int id = __ldg(ti + o + i);
        if (id < 0 || !(v > top.thr())) break;            // the lists are sorted
        top.push(v, (e - job.mem_begin) * n_pix + id % n_pix);
      }
    }
  }
  const int zt = zero_pad_count<K>(top, k_in, flags, q, n_pix, job.mem_end - job.mem_begin);
  float a[K];
#pragma unroll
  for (int i = 0; i < K; ++i)
    a[i] = (flags & FGVC_SIM_L2) ? __fdiv_rn(2.f * top.v[i] - 1.f, temperature) : __fdiv_rn(top.v[i], temperature);
  const float m = zt > 0 ? fmaxf(a[0], 0.f) : a[0];
  float sum = 0.f;
  if (flags & FGVC_WEIGHT_COSINE) {
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const float c = fmaxf(a[i], 0.f);
      a[i] = (i < k_in - zt && top.id[i] >= 0) ? c * c : 0.f;
    }
    sum = 1.f;
  } else {
#pragma unroll
    for (int i = 0; i < K; ++i) {
      a[i] = (i < k_in - zt && top.id[i] >= 0) ? expf(a[i] - m) : 0.f;
      sum += a[i];
    }
    sum += (float)zt * expf(0.f - m);            // the zero-padded winners: weight exp(0 / temperature), value 0
  }
  const int64_t o = ((int64_t)blockIdx.y * n_pix + q) * K;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int id = top.id[i];
    const bool ok = i < k_in - zt && id >= 0;
    int row = 0;
    if (ok) {
      const int pos = id / n_pix;
      row = __ldg(mem_label + job.mem_begin + pos) * n_pix + (id - pos * n_pix);
    }
    cw[o + i] = ok ? ((flags & FGVC_WEIGHT_COSINE) ? a[i] : __fdiv_rn(a[i], sum)) : 0.f;
    crow[o + i] = row;
  }
}

constexpr int CH_Q = 32;      // queries staged per CTA pass

template <int K>
__global__ void __launch_bounds__(256)
gather_chain_kernel(const float* __restrict__ cw, const int32_t* __restrict__ crow, const fgvc_job* __restrict__ jobs,
                    int job_begin, int n_jobs, int n_pix, float* lab, int Lp, unsigned int* barrier) {
  __shared__ float sw[CH_Q][K];
  __shared__ int srow[CH_Q][K];
  const int tid = threadIdx.x;
  const int l4n = Lp / 4;
  const float4* src = reinterpret_cast<const float4*>(lab);
  // this CTA's queries: a contiguous slice (the same for every job)
  const int per = (n_pix + gridDim.x - 1) / gridDim.x;
  const int q_lo = blockIdx.x * per, q_hi = min(n_pix, q_lo + per);
  // single-pass slices (the usual case: the grid is sized for it): the label-independent (weight, row) pairs of job
  // j + 1 are fetched into registers while job j is gathered, so the only loads after a grid barrier are the label rows.
  // With L <= 4 (one float4 per label row) the launch sizes the grid at ceil(n_pix / 64) CTAs or fewer, so every map
  // of more than 32 pixels takes the multi-pass branch; so does any map of more than 32 x (resident CTAs) pixels.
  const bool one_pass = q_hi - q_lo <= CH_Q;
  constexpr int PRE = (CH_Q * K + 255) / 256;
  float pw[PRE];
  int pr[PRE];
  const int nq1 = max(q_hi - q_lo, 0);
  if (one_pass) {
#pragma unroll
    for (int u = 0; u < PRE; ++u) {
      const int i = tid + 256 * u;
      if (i < nq1 * K) {
        const int64_t o = ((int64_t)0 * n_pix + q_lo) * K + i;
        (&sw[0][0])[i] = __ldg(cw + o);
        (&srow[0][0])[i] = __ldg(crow + o);
      }
    }
    __syncthreads();
  }
  for (int j = 0; j < n_jobs; ++j) {
    const int out_slot = jobs[job_begin + j].out_slot;
    float4* dst = reinterpret_cast<float4*>(lab) + (int64_t)out_slot * n_pix * l4n;
    if (one_pass) {
      if (j + 1 < n_jobs) {
#pragma unroll
        for (int u = 0; u < PRE; ++u) {
          const int i = tid + 256 * u;
          if (i < nq1 * K) {
            const int64_t o = ((int64_t)(j + 1) * n_pix + q_lo) * K + i;
            pw[u] = __ldg(cw + o);
            pr[u] = __ldg(crow + o);
          }
        }
      }
      for (int i = tid; i < nq1 * l4n; i += 256) {
        const int q = i / l4n, c = i - q * l4n;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float w = sw[q][k];
          if (w != 0.f) {
            const float4 v = __ldcg(src + (int64_t)srow[q][k] * l4n + c);   // may have been written by another CTA
            acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
            acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
          }
        }
        dst[(int64_t)(q_lo + q) * l4n + c] = acc;
      }
      if (j + 1 < n_jobs) {
        __syncthreads();                               // everyone is done with this job's pairs
#pragma unroll
        for (int u = 0; u < PRE; ++u) {
          const int i = tid + 256 * u;
          if (i < nq1 * K) { (&sw[0][0])[i] = pw[u]; (&srow[0][0])[i] = pr[u]; }
        }
      }
    } else
    for (int q0 = q_lo; q0 < q_hi; q0 += CH_Q) {
      const int nq = min(CH_Q, q_hi - q0);
      __syncthreads();
      for (int i = tid; i < nq * K; i += 256) {
        const int64_t o = ((int64_t)j * n_pix + q0) * K + i;
        (&sw[0][0])[i] = __ldg(cw + o);
        (&srow[0][0])[i] = __ldg(crow + o);
      }
      __syncthreads();
      for (int i = tid; i < nq * l4n; i += 256) {
        const int q = i / l4n, c = i - q * l4n;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float w = sw[q][k];
          if (w != 0.f) {
            const float4 v = __ldcg(src + (int64_t)srow[q][k] * l4n + c);   // may have been written by another CTA
            acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
            acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
          }
        }
        dst[(int64_t)(q0 + q) * l4n + c] = acc;
      }
    }
    // grid barrier: every CTA's stores of job j are visible before anyone starts job j + 1
    if (j + 1 < n_jobs) grid_barrier(barrier, (unsigned int)(j + 1));
  }
}

// ------------------------------------------------------------------ the multi-lane gather chain
// Several independent recurrences of one clip (lanes: the forward and backward tracks of every point group) in ONE
// cooperative kernel.  Step s gathers job s of every lane that is still running, then all CTAs meet at the grid
// barrier, so a clip pays the longest lane's length in barriers instead of the sum over its lanes.  Each CTA owns the
// same fixed query slice in every lane; per (query, channel) the FMA sequence is gather_chain_kernel's, so every lane
// is bit for bit the single-lane chain over its jobs.  The (weight, row) pairs of all jobs come from ONE
// gather_weights_kernel launch over the job range [job_base, ...) holding every lane; rows are relative to the lane's
// bank.  In the one-pass branch the CTA walks its work items (step, lane) in order and copies the pairs of the next
// item into a second shared buffer (cp.async, no registers held) while it gathers the current one: they are
// label-independent, so this holds across barriers and lanes, and the shared memory does not grow with the lanes.

// first lane >= l that still runs at step s (n_lanes: none)
__device__ __forceinline__ int next_lane(const fgvc_lane* __restrict__ lanes, int n_lanes, int s, int l) {
  while (l < n_lanes && __ldg(&lanes[l].job_end) - __ldg(&lanes[l].job_begin) <= s) ++l;
  return l;
}

// index in the chain workspace of the (weight, row) pair of query q of job s of lane l
template <int K>
__device__ __forceinline__ int64_t lane_pairs(const fgvc_lane* __restrict__ lanes, int l, int s, int job_base, int n_pix,
                                              int q) {
  return ((int64_t)(__ldg(&lanes[l].job_begin) + s - job_base) * n_pix + q) * K;
}

// queries of a lane-chain CTA's one-pass slice.  The kernel is bounded to 2 resident CTAs per SM, where it needs no
// spill at any K (64 to 88 registers: the K label rows of a query are loaded at once); at 2 to 4 CTAs per SM a
// slice of 64 keeps 128 x 128 maps in the one-pass branch.
constexpr int CH_QL = 64;

// 4-byte global -> shared copy that holds no register until it lands (cp.async, sm_80+)
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  const unsigned int d = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem) : "memory");
}

template <int K>
__global__ void __launch_bounds__(256, 2)
gather_chain_lanes_kernel(const float* __restrict__ cw, const int32_t* __restrict__ crow,
                          const fgvc_job* __restrict__ jobs, int job_base, const fgvc_lane* __restrict__ lanes,
                          int n_lanes, int n_steps, int n_pix, float* lab, unsigned int* barrier) {
  // two buffers of (weight, row) pairs: the current work item's and the next one's, in flight
  __shared__ float sw[2][CH_QL][K];
  __shared__ int srow[2][CH_QL][K];
  const int tid = threadIdx.x;
  const int per = (n_pix + gridDim.x - 1) / gridDim.x;
  const int q_lo = blockIdx.x * per, q_hi = min(n_pix, q_lo + per);
  const bool one_pass = q_hi - q_lo <= CH_QL;
  const int nq1 = max(q_hi - q_lo, 0);
  int l = next_lane(lanes, n_lanes, 0, 0), b = 0;
  if (one_pass && l < n_lanes) {
    const int64_t o = lane_pairs<K>(lanes, l, 0, job_base, n_pix, q_lo);
    for (int i = tid; i < nq1 * K; i += 256) {
      (&sw[0][0][0])[i] = __ldg(cw + o + i);
      (&srow[0][0][0])[i] = __ldg(crow + o + i);
    }
    __syncthreads();
  }
  for (int s = 0; s < n_steps; ++s) {
    for (; l < n_lanes; l = next_lane(lanes, n_lanes, s, l + 1)) {
      const int l4n = __ldg(&lanes[l].Lp) / 4;
      float4* bank = reinterpret_cast<float4*>(lab + __ldg(&lanes[l].lab_offset));
      const int out_slot = jobs[__ldg(&lanes[l].job_begin) + s].out_slot;
      if (one_pass) {
        // the next work item: the next running lane of this step, else the first lane of the next step
        int ns = s, nl = next_lane(lanes, n_lanes, s, l + 1);
        if (nl == n_lanes) {
          ns = s + 1;
          nl = ns < n_steps ? next_lane(lanes, n_lanes, ns, 0) : n_lanes;
        }
        const bool more = nl < n_lanes;
        if (more) {
          const int64_t o = lane_pairs<K>(lanes, nl, ns, job_base, n_pix, q_lo);
          for (int i = tid; i < nq1 * K; i += 256) {
            cp_async4(&sw[b ^ 1][0][0] + i, cw + o + i);
            cp_async4(&srow[b ^ 1][0][0] + i, crow + o + i);
          }
          asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (int i = tid; i < nq1 * l4n; i += 256) {
          const int q = i / l4n, c = i - q * l4n;
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int k = 0; k < K; ++k) {
            const float w = sw[b][q][k];
            if (w != 0.f) {
              const float4 v = __ldcg(bank + (int64_t)srow[b][q][k] * l4n + c);   // may have been written by another CTA
              acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
              acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
            }
          }
          bank[((int64_t)out_slot * n_pix + q_lo + q) * l4n + c] = acc;
        }
        if (more) {
          asm volatile("cp.async.wait_all;" ::: "memory");
          __syncthreads();                             // the next item's pairs have landed, this item's are done
          b ^= 1;
        }
      } else {
        const int64_t o0 = lane_pairs<K>(lanes, l, s, job_base, n_pix, 0);
        for (int q0 = q_lo; q0 < q_hi; q0 += CH_QL) {
          const int nq = min(CH_QL, q_hi - q0);
          __syncthreads();
          for (int i = tid; i < nq * K; i += 256) {
            const int64_t o = o0 + (int64_t)q0 * K + i;
            (&sw[0][0][0])[i] = __ldg(cw + o);
            (&srow[0][0][0])[i] = __ldg(crow + o);
          }
          __syncthreads();
          for (int i = tid; i < nq * l4n; i += 256) {
            const int q = i / l4n, c = i - q * l4n;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < K; ++k) {
              const float w = sw[0][q][k];
              if (w != 0.f) {
                const float4 v = __ldcg(bank + (int64_t)srow[0][q][k] * l4n + c);   // may have been written by another CTA
                acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y);
                acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
              }
            }
            bank[((int64_t)out_slot * n_pix + q0 + q) * l4n + c] = acc;
          }
        }
      }
    }
    // grid barrier: every CTA's stores of step s are visible before anyone starts step s + 1
    if (s + 1 < n_steps) grid_barrier(barrier, (unsigned int)(s + 1));
    l = next_lane(lanes, n_lanes, s + 1, 0);
  }
}

int64_t chain_workspace_bytes(int n_jobs, int n_pix, int K) {
  const int Kt = K <= 4 ? 4 : (K <= 10 ? 10 : 16);
  return (int64_t)n_jobs * n_pix * Kt * 8 + 256;
}

// the label-independent (weight, row) pairs of jobs [job_begin, job_begin + n) into the chain workspace (cw, crow),
// and the grid barrier's counter reset; returns the counter
template <int K>
static int launch_weights_t(const float* tv, const int32_t* ti, int k_in, int groups, const fgvc_job* jobs, int job_begin,
                            int n, const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature,
                            int flags, void* ws, float** cw, int32_t** crow, unsigned int** barrier, cudaStream_t st) {
  const int64_t cells = (int64_t)n * n_pix * K;
  *cw = reinterpret_cast<float*>(ws);
  *crow = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(ws) + cells * 4);
  *barrier = reinterpret_cast<unsigned int*>(reinterpret_cast<uint8_t*>(ws) + cells * 8);
  FGVC_CUDA(cudaMemsetAsync(*barrier, 0, 256, st));
  dim3 gw(cdiv(n_pix, 256), n);
  gather_weights_kernel<K><<<gw, 256, 0, st>>>(tv, ti, k_in, groups, jobs, job_begin, mem_label, pair_ref, n_pix,
                                               temperature, flags, *cw, *crow);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}

// co-resident CTAs of a 256-thread chain kernel on the calling thread's device (they spin on the grid barrier:
// cooperative launch, sized from the occupancy; cached per device index, written once with the same value by any
// thread)
int resident_ctas(const void* kernel, std::atomic<int>* cached, int* max_ctas) {
  int dev = 0;
  FGVC_CUDA(cudaGetDevice(&dev));
  *max_ctas = (dev >= 0 && dev < 64) ? cached[dev].load(std::memory_order_relaxed) : 0;
  if (*max_ctas == 0) {
    int sms = 0, occ = 0;
    FGVC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    FGVC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 256, 0));
    *max_ctas = sms * (occ < 1 ? 1 : occ);
    if (dev >= 0 && dev < 64) cached[dev].store(*max_ctas, std::memory_order_relaxed);
  }
  return FGVC_OK;
}

template <int K>
static int launch_chain_t(const float* tv, const int32_t* ti, int k_in, int groups, const fgvc_job* jobs, int job_begin,
                          int n, const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature,
                          int flags, float* lab, int Lp, void* ws, cudaStream_t st) {
  float* cw;
  int32_t* crow;
  unsigned int* barrier;
  int rc = launch_weights_t<K>(tv, ti, k_in, groups, jobs, job_begin, n, mem_label, pair_ref, n_pix, temperature, flags,
                               ws, &cw, &crow, &barrier, st);
  if (rc) return rc;
  static std::atomic<int> cached[64];
  int max_ctas = 0;
  rc = resident_ctas((const void*)gather_chain_kernel<K>, cached, &max_ctas);
  if (rc) return rc;
  const int l4n = Lp / 4;
  // latency-bound (a few microseconds per frame): as many CTAs as can be co-resident, so that a CTA's slice is
  // one pass of <= CH_Q queries whenever possible
  // (short label rows: ~2 CTAs per SM; long rows want every resident thread for memory-level parallelism)
  // (measured on the bench clip, 6420 queries x 3 float4: 301 CTAs 337 us; 148 CTAs 558 us -- two passes per CTA;
  // 602 CTAs 379 us, 1184 CTAs 485 us -- the barrier grows)
  const int ctas = (int)min((int64_t)max_ctas, max((int64_t)1, ((int64_t)n_pix * l4n + 63) / 64));
  int n_jobs = n, jb = job_begin, npx = n_pix, lp = Lp;
  void* args[] = {(void*)&cw, (void*)&crow, (void*)&jobs, (void*)&jb, (void*)&n_jobs, (void*)&npx, (void*)&lab,
                  (void*)&lp, (void*)&barrier};
  FGVC_CUDA(cudaLaunchCooperativeKernel((const void*)gather_chain_kernel<K>, dim3(ctas), dim3(256), args, 0, st));
  fgvc::g_launches.fetch_add(1);
  return FGVC_OK;
}

// K1b for the consecutive jobs [job_begin, job_end) as one persistent chain (see above)
int launch_gather_chain(const float* tv, const int32_t* ti, int K, int groups, const fgvc_job* jobs, int job_begin,
                        int job_end, const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature,
                        int flags, float* lab, int Lp, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int n = job_end - job_begin;
  FGVC_CHECK_ARG(ws != nullptr && ws_bytes >= chain_workspace_bytes(n, n_pix, K),
                 "gather chain: workspace of %lld bytes needed (fgvc_chain_workspace_bytes)",
                 (long long)chain_workspace_bytes(n, n_pix, K));
  if (K <= 4) return launch_chain_t<4>(tv, ti, K, groups, jobs, job_begin, n, mem_label, pair_ref, n_pix, temperature, flags, lab, Lp, ws, st);
  if (K <= 10) return launch_chain_t<10>(tv, ti, K, groups, jobs, job_begin, n, mem_label, pair_ref, n_pix, temperature, flags, lab, Lp, ws, st);
  return launch_chain_t<16>(tv, ti, K, groups, jobs, job_begin, n, mem_label, pair_ref, n_pix, temperature, flags, lab, Lp, ws, st);
}

template <int K>
static int launch_chain_lanes_t(const float* tv, const int32_t* ti, int k_in, int groups, const fgvc_job* jobs,
                                int job_base, int n, const fgvc_lane* lanes_dev, int n_lanes, int n_steps, int max_l4n,
                                const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature,
                                int flags, float* lab, void* ws, cudaStream_t st) {
  float* cw;
  int32_t* crow;
  unsigned int* barrier;
  int rc = launch_weights_t<K>(tv, ti, k_in, groups, jobs, job_base, n, mem_label, pair_ref, n_pix, temperature, flags,
                               ws, &cw, &crow, &barrier, st);
  if (rc) return rc;
  static std::atomic<int> cached[64];
  int max_ctas = 0;
  rc = resident_ctas((const void*)gather_chain_lanes_kernel<K>, cached, &max_ctas);
  if (rc) return rc;
  // the grid rule of the single-lane chain, for the lane with the longest rows
  const int ctas = (int)min((int64_t)max_ctas, max((int64_t)1, ((int64_t)n_pix * max_l4n + 63) / 64));
  int jb = job_base, nl = n_lanes, ns = n_steps, npx = n_pix;
  void* args[] = {(void*)&cw, (void*)&crow, (void*)&jobs, (void*)&jb, (void*)&lanes_dev, (void*)&nl, (void*)&ns,
                  (void*)&npx, (void*)&lab, (void*)&barrier};
  FGVC_CUDA(cudaLaunchCooperativeKernel((const void*)gather_chain_lanes_kernel<K>, dim3(ctas), dim3(256), args, 0, st));
  fgvc::g_launches.fetch_add(1);
  return FGVC_OK;
}

// K1b for every lane of lanes_host[0, n_lanes) as one multi-lane chain (see gather_chain_lanes_kernel); the lanes are
// validated by the caller
int launch_gather_chain_lanes(const float* tv, const int32_t* ti, int K, int groups, const fgvc_job* jobs,
                              const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host, int n_lanes,
                              const int32_t* mem_label, const int32_t* pair_ref, int n_pix, float temperature, int flags,
                              float* lab, void* ws, int64_t ws_bytes, cudaStream_t st) {
  int jb = lanes_host[0].job_begin, je = lanes_host[0].job_end, n_steps = 0, max_l4n = 1;
  for (int i = 0; i < n_lanes; ++i) {
    jb = min(jb, lanes_host[i].job_begin);
    je = max(je, lanes_host[i].job_end);
    n_steps = max(n_steps, lanes_host[i].job_end - lanes_host[i].job_begin);
    max_l4n = max(max_l4n, lanes_host[i].Lp / 4);
  }
  const int n = je - jb;
  FGVC_CHECK_ARG(n <= 65535, "gather chain lanes: %d jobs in the lanes' range, at most 65535", n);
  FGVC_CHECK_ARG(ws != nullptr && ws_bytes >= chain_workspace_bytes(n, n_pix, K),
                 "gather chain lanes: workspace of %lld bytes needed (fgvc_chain_workspace_bytes)",
                 (long long)chain_workspace_bytes(n, n_pix, K));
  if (K <= 4) return launch_chain_lanes_t<4>(tv, ti, K, groups, jobs, jb, n, lanes_dev, n_lanes, n_steps, max_l4n, mem_label, pair_ref, n_pix, temperature, flags, lab, ws, st);
  if (K <= 10) return launch_chain_lanes_t<10>(tv, ti, K, groups, jobs, jb, n, lanes_dev, n_lanes, n_steps, max_l4n, mem_label, pair_ref, n_pix, temperature, flags, lab, ws, st);
  return launch_chain_lanes_t<16>(tv, ti, K, groups, jobs, jb, n, lanes_dev, n_lanes, n_steps, max_l4n, mem_label, pair_ref, n_pix, temperature, flags, lab, ws, st);
}

}  // namespace fgvc

using namespace fgvc;

extern "C" int64_t fgvc_chain_workspace_bytes(int32_t n_jobs, int32_t n_pix, int32_t K) {
  return chain_workspace_bytes(n_jobs, n_pix, K);
}

extern "C" int fgvc_gather_labels(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                  const fgvc_job* jobs, int32_t job_begin, int32_t job_end,
                                  const int32_t* mem_label_slot, int32_t n_pix, float temperature, int32_t flags,
                                  float* lab_bank, int32_t Lp, void* stream) {
  FGVC_CHECK_ARG(topk_val && topk_idx && jobs && mem_label_slot && lab_bank, "fgvc_gather_labels: null pointer");
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_gather_labels: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(groups >= 1 && job_end > job_begin && n_pix > 0, "fgvc_gather_labels: bad sizes");
  FGVC_CHECK_ARG(Lp > 0 && Lp % 4 == 0, "fgvc_gather_labels: Lp=%d must be a positive multiple of 4", Lp);
  FGVC_CHECK_ARG(temperature > 0.f, "fgvc_gather_labels: temperature must be > 0");
  cudaStream_t st = (cudaStream_t)stream;
  int n = job_end - job_begin;
  if (K <= 4) return launch_g<4>(topk_val, topk_idx, K, groups, jobs, job_begin, n, mem_label_slot, n_pix, temperature, flags, lab_bank, Lp, st);
  if (K <= 10) return launch_g<10>(topk_val, topk_idx, K, groups, jobs, job_begin, n, mem_label_slot, n_pix, temperature, flags, lab_bank, Lp, st);
  return launch_g<16>(topk_val, topk_idx, K, groups, jobs, job_begin, n, mem_label_slot, n_pix, temperature, flags, lab_bank, Lp, st);
}
