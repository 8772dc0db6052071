// Clip-level drivers: the sequential part of the reference loop
// (vanilla_tracker.py:345-412) enqueued by ONE C call, so that the host costs a few
// microseconds per frame instead of a Python round trip per kernel.
#include "common.cuh"

using namespace fgvc;

// Hard propagation over jobs [job_begin, job_end) of one label bank: the memory keeps one_hot(argmax) of every
// propagated frame, the prediction is decoded from the soft labels first (vanilla_tracker.py:762-798) -- so gather,
// NCHW copy, decode and hardening frame by frame.  scratch_minmax: 2L words.
static int hard_prop_tail(const float* topk_val, const int32_t* topk_idx, int K, int groups, const fgvc_job* jobs_dev,
                          const fgvc_job* jobs_host, int job_begin, int job_end, const int32_t* mem_label_slot, int H,
                          int W, float temperature, int flags, float* lab_bank, int Lp, int L, int out_h, int out_w,
                          float* scratch_minmax, uint8_t* masks, float* maps_nchw, void* stream) {
  const int n_pix = H * W;
  const int64_t mask_elems = (int64_t)out_h * out_w;
  cudaStream_t st = (cudaStream_t)stream;
  for (int j = job_begin; j < job_end; ++j) {
    int rc = fgvc_gather_labels(topk_val, topk_idx, K, groups, jobs_dev, j, j + 1, mem_label_slot, n_pix,
                                temperature, flags, lab_bank, Lp, stream);
    if (rc) return rc;
    const int slot = jobs_host[j].out_slot;
    float* lab_slot = lab_bank + (int64_t)slot * n_pix * Lp;
    if (maps_nchw) {
      rc = fgvc_labels_to_nchw(lab_bank, slot, Lp, L, n_pix, maps_nchw + (int64_t)slot * L * n_pix, stream);
      if (rc) return rc;
    }
    rc = launch_decode(lab_slot, true, L, Lp, H, W, out_h, out_w, reinterpret_cast<uint32_t*>(scratch_minmax),
                       masks + slot * mask_elems, st);
    if (rc) return rc;
    rc = launch_labels_harden(lab_slot, n_pix, L, Lp, st);
    if (rc) return rc;
  }
  return FGVC_OK;
}

// After K0 + K1 ran for the whole clip: for every job j (in order) gather the labels of its
// query frame (K1b) and decode them to a uint8 mask of the image size.
extern "C" int fgvc_mask_clip_tail(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                   const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                                   int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                                   float temperature, int32_t flags,
                                   float* lab_bank, int32_t Lp, int32_t L, int32_t out_h, int32_t out_w,
                                   float* scratch_minmax, uint8_t* masks, float* maps_nchw, void* chain_ws,
                                   int64_t chain_ws_bytes, void* stream) {
  FGVC_CHECK_ARG(jobs_dev && jobs_host && masks && scratch_minmax && lab_bank, "fgvc_mask_clip_tail: null pointer");
  FGVC_CHECK_ARG(L > 0 && L <= 255 && Lp >= L && Lp % 4 == 0, "fgvc_mask_clip_tail: bad label sizes");
  const int n_pix = H * W;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & FGVC_HARD_PROP)
    return hard_prop_tail(topk_val, topk_idx, K, groups, jobs_dev, jobs_host, job_begin, job_end, mem_label_slot, H, W,
                          temperature, flags, lab_bank, Lp, L, out_h, out_w, scratch_minmax, masks, maps_nchw, stream);
  // the recurrence lives only in the gather: run the chain first ...
  if (chain_ws != nullptr && job_end - job_begin > 1) {
    // ... as ONE persistent kernel with a grid barrier per frame (gather.cu)
    int rc = launch_gather_chain(topk_val, topk_idx, K, groups, jobs_dev, job_begin, job_end, mem_label_slot, nullptr,
                                 n_pix, temperature, flags, lab_bank, Lp, chain_ws, chain_ws_bytes, st);
    if (rc) return rc;
    if (maps_nchw) {
      rc = launch_labels_to_nchw_jobs(lab_bank, jobs_dev, job_begin, job_end, Lp, L, n_pix, maps_nchw, st);
      if (rc) return rc;
    }
  } else {
    for (int j = job_begin; j < job_end; ++j) {
      int rc = fgvc_gather_labels(topk_val, topk_idx, K, groups, jobs_dev, j, j + 1, mem_label_slot, n_pix,
                                  temperature, flags, lab_bank, Lp, stream);
      if (rc) return rc;
      if (maps_nchw) {
        const int slot = jobs_host[j].out_slot;
        rc = fgvc_labels_to_nchw(lab_bank, slot, Lp, L, n_pix, maps_nchw + (int64_t)slot * L * n_pix, stream);
        if (rc) return rc;
      }
    }
  }
  // ... then decode every frame of the range in two batched launches (scratch: [n_jobs][2L] words)
  return launch_decode_jobs(lab_bank, jobs_dev, job_begin, job_end, L, Lp, H, W, out_h, out_w,
                            reinterpret_cast<uint32_t*>(scratch_minmax), masks, st);
}

// The mask tails of the independent recurrences of a clip (the forward and the backward propagation from an annotated
// frame), each lane bit for bit fgvc_mask_clip_tail over its jobs and its bank with the chain workspace: ONE
// multi-lane gather chain, ONE NCHW copy over every job of every lane, ONE batched decode (min-max + arg-max) over
// every job of every lane.  With FGVC_HARD_PROP every lane runs the per-frame loop of fgvc_mask_clip_tail instead.
extern "C" int fgvc_mask_clip_tail_lanes(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                         const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                                         const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host, int32_t n_lanes,
                                         const int32_t* mem_label_slot, int32_t H, int32_t W, float temperature,
                                         int32_t flags, float* lab_bank, int32_t out_h, int32_t out_w,
                                         float* scratch_minmax, uint8_t* masks, float* maps_nchw, void* chain_ws,
                                         int64_t chain_ws_bytes, void* stream) {
  const bool hard = (flags & FGVC_HARD_PROP) != 0;
  FGVC_CHECK_ARG(topk_val && topk_idx && jobs_dev && jobs_host && lanes_dev && lanes_host && mem_label_slot &&
                     lab_bank && scratch_minmax && masks && (chain_ws || hard),
                 "fgvc_mask_clip_tail_lanes: null pointer");
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_mask_clip_tail_lanes: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(n_lanes >= 1 && H > 0 && W > 0 && out_h > 0 && out_w > 0 && groups >= 1,
                 "fgvc_mask_clip_tail_lanes: bad sizes");
  FGVC_CHECK_ARG(pair_ref == nullptr || groups == 1, "fgvc_mask_clip_tail_lanes: shared lists need groups == 1");
  FGVC_CHECK_ARG(pair_ref == nullptr || !hard, "fgvc_mask_clip_tail_lanes: hard propagation takes no shared lists");
  FGVC_CHECK_ARG(temperature > 0.f, "fgvc_mask_clip_tail_lanes: temperature must be > 0");
  int64_t n_jobs = 0;
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_lane& ln = lanes_host[i];
    FGVC_CHECK_ARG(ln.job_begin >= 0 && ln.job_end > ln.job_begin, "fgvc_mask_clip_tail_lanes: lane %d is empty", i);
    FGVC_CHECK_ARG(ln.L > 0 && ln.L <= 255 && ln.Lp >= ln.L && ln.Lp % 4 == 0 && ln.lab_offset >= 0 &&
                       ln.lab_offset % 4 == 0 && ln.coord_offset == 0,
                   "fgvc_mask_clip_tail_lanes: bad label sizes or offsets in lane %d", i);
    n_jobs += ln.job_end - ln.job_begin;
  }
  FGVC_CHECK_ARG(n_jobs <= 65535, "fgvc_mask_clip_tail_lanes: %lld jobs in all, at most 65535", (long long)n_jobs);
  if (hard) {
    for (int i = 0; i < n_lanes; ++i) {
      const fgvc_lane& ln = lanes_host[i];
      int rc = hard_prop_tail(topk_val, topk_idx, K, groups, jobs_dev, jobs_host, ln.job_begin, ln.job_end,
                              mem_label_slot, H, W, temperature, flags, lab_bank + ln.lab_offset, ln.Lp, ln.L, out_h,
                              out_w, scratch_minmax, masks, maps_nchw, stream);
      if (rc) return rc;
    }
    return FGVC_OK;
  }
  const int n_pix = H * W;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_gather_chain_lanes(topk_val, topk_idx, K, groups, jobs_dev, lanes_dev, lanes_host, n_lanes,
                                     mem_label_slot, pair_ref, n_pix, temperature, flags, lab_bank, chain_ws,
                                     chain_ws_bytes, st);
  if (rc) return rc;
  if (maps_nchw) {
    rc = launch_labels_to_nchw_lanes(lab_bank, jobs_dev, lanes_dev, lanes_host, n_lanes, n_pix, maps_nchw, st);
    if (rc) return rc;
  }
  return launch_decode_lanes(lab_bank, jobs_dev, lanes_dev, lanes_host, n_lanes, H, W, out_h, out_w,
                             reinterpret_cast<uint32_t*>(scratch_minmax), masks, st);
}

// Lowest out_slot of jobs [job_begin, job_end) when their out_slots run consecutively up (a forward track) or down (a
// track run backwards in time), else -1.  The K3 launch of a point tail covers the slots [lowest, lowest + n).
static int consecutive_slots(const fgvc_job* jobs_host, int job_begin, int job_end) {
  const int s0 = jobs_host[job_begin].out_slot, n = job_end - job_begin;
  const int dir = (n > 1 && jobs_host[job_begin + 1].out_slot < s0) ? -1 : 1;
  for (int j = job_begin; j < job_end; ++j)
    if (jobs_host[j].out_slot != s0 + dir * (j - job_begin)) return -1;
  return dir > 0 ? s0 : s0 - (n - 1);
}

// NCHW copies of jobs [job_begin, job_end) of a label bank into maps_nchw[slot][L][H*W], then ONE K3 launch (fused
// up-sample / soft-argmax) over all their (frame, point) maps into coords[slot][L][2].  The caller checked that the
// out_slots are consecutive.
static int nchw_and_coords(const float* bank, const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int job_begin,
                           int job_end, int Lp, int L, int H, int W, int out_h, int out_w, int coord_topk,
                           float* maps_nchw, float* coords, void* stream) {
  const int n_pix = H * W;
  int rc = launch_labels_to_nchw_jobs(bank, jobs_dev, job_begin, job_end, Lp, L, n_pix, maps_nchw, (cudaStream_t)stream);
  if (rc) return rc;
  const int slot0 = consecutive_slots(jobs_host, job_begin, job_end);
  return fgvc_heatmap_coords(maps_nchw + (int64_t)slot0 * L * n_pix, (job_end - job_begin) * L, H, W, out_h, out_w,
                             coord_topk, coords + (int64_t)slot0 * L * 2, stream);
}

// Point tracking tail: the gather chain over jobs [job_begin, job_end) with an NCHW copy of every
// propagated frame into maps_nchw[slot][L][H*W], then ONE K3 launch over all (frame, point) maps of the
// range: coords[slot][L][2].  The out_slots of the range must be consecutive (they are frame indices),
// ascending or descending.
extern "C" int fgvc_point_clip_tail(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                    const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                                    int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                                    float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L, int32_t out_h,
                                    int32_t out_w, int32_t coord_topk, float* maps_nchw, float* coords,
                                    void* chain_ws, int64_t chain_ws_bytes, void* stream) {
  FGVC_CHECK_ARG(jobs_dev && jobs_host && maps_nchw && coords && lab_bank, "fgvc_point_clip_tail: null pointer");
  FGVC_CHECK_ARG(job_end > job_begin, "fgvc_point_clip_tail: empty job range");
  const int n_pix = H * W;
  const int slot0 = consecutive_slots(jobs_host, job_begin, job_end);
  FGVC_CHECK_ARG(slot0 >= 0, "fgvc_point_clip_tail: out_slots must be consecutive");
  if (chain_ws != nullptr && job_end - job_begin > 1) {
    int rc = launch_gather_chain(topk_val, topk_idx, K, groups, jobs_dev, job_begin, job_end, mem_label_slot, nullptr,
                                 n_pix, temperature, flags, lab_bank, Lp, chain_ws, chain_ws_bytes, (cudaStream_t)stream);
    if (rc) return rc;
    return nchw_and_coords(lab_bank, jobs_dev, jobs_host, job_begin, job_end, Lp, L, H, W, out_h, out_w, coord_topk,
                           maps_nchw, coords, stream);
  }
  for (int j = job_begin; j < job_end; ++j) {
    const int slot = jobs_host[j].out_slot;
    int rc = fgvc_gather_labels(topk_val, topk_idx, K, groups, jobs_dev, j, j + 1, mem_label_slot, n_pix,
                                temperature, flags, lab_bank, Lp, stream);
    if (rc) return rc;
    rc = fgvc_labels_to_nchw(lab_bank, slot, Lp, L, n_pix, maps_nchw + (int64_t)slot * L * n_pix, stream);
    if (rc) return rc;
  }
  return fgvc_heatmap_coords(maps_nchw + (int64_t)slot0 * L * n_pix, (job_end - job_begin) * L, H, W, out_h, out_w,
                             coord_topk, coords + (int64_t)slot0 * L * 2, stream);
}

// The point tails of the independent recurrences of a clip (every forward and backward track of every point group),
// each lane bit for bit fgvc_point_clip_tail over its jobs with the chain workspace: one gather chain for all of them,
// then per lane the NCHW copies and one K3 launch -- bandwidth work, where one launch per lane costs nothing worth
// saving.  A single lane runs the multi-lane chain (gather.cu) too: with it a whole one-lane tail is not slower than
// with gather_chain_kernel on a B200 at 1000 W (128 x 128 map, 256 points x 49 frames: 1.60 against 1.76 ms; 1024
// points x 249 frames: 38.0 against 38.4 ms; 160 x 160, 15 points x 31 frames: 0.34 against 0.46 ms).  pair_ref names the shared per-(query frame, memory
// frame) lists of every memory entry, or is NULL.
extern "C" int fgvc_point_clip_tail_lanes(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                          const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                                          const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host, int32_t n_lanes,
                                          const int32_t* mem_label_slot, int32_t H, int32_t W, float temperature,
                                          int32_t flags, float* lab_bank, int32_t out_h, int32_t out_w,
                                          int32_t coord_topk, float* maps_nchw, float* coords, void* chain_ws,
                                          int64_t chain_ws_bytes, void* stream) {
  FGVC_CHECK_ARG(topk_val && topk_idx && jobs_dev && jobs_host && lanes_dev && lanes_host && mem_label_slot && lab_bank &&
                     maps_nchw && coords && chain_ws, "fgvc_point_clip_tail_lanes: null pointer");
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_point_clip_tail_lanes: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(n_lanes >= 1 && H > 0 && W > 0 && groups >= 1, "fgvc_point_clip_tail_lanes: bad sizes");
  FGVC_CHECK_ARG(pair_ref == nullptr || groups == 1, "fgvc_point_clip_tail_lanes: shared lists need groups == 1");
  FGVC_CHECK_ARG(temperature > 0.f, "fgvc_point_clip_tail_lanes: temperature must be > 0");
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_lane& ln = lanes_host[i];
    FGVC_CHECK_ARG(ln.job_begin >= 0 && ln.job_end > ln.job_begin, "fgvc_point_clip_tail_lanes: lane %d is empty", i);
    FGVC_CHECK_ARG(ln.L > 0 && ln.Lp >= ln.L && ln.Lp % 4 == 0 && ln.lab_offset >= 0 && ln.lab_offset % 4 == 0 &&
                       ln.coord_offset >= 0, "fgvc_point_clip_tail_lanes: bad label sizes or offsets in lane %d", i);
    FGVC_CHECK_ARG(consecutive_slots(jobs_host, ln.job_begin, ln.job_end) >= 0,
                   "fgvc_point_clip_tail_lanes: out_slots of lane %d must be consecutive", i);
  }
  const int n_pix = H * W;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_gather_chain_lanes(topk_val, topk_idx, K, groups, jobs_dev, lanes_dev, lanes_host, n_lanes,
                                     mem_label_slot, pair_ref, n_pix, temperature, flags, lab_bank, chain_ws,
                                     chain_ws_bytes, st);
  if (rc) return rc;
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_lane& ln = lanes_host[i];
    rc = nchw_and_coords(lab_bank + ln.lab_offset, jobs_dev, jobs_host, ln.job_begin, ln.job_end, ln.Lp, ln.L, H, W,
                         out_h, out_w, coord_topk, maps_nchw, coords + ln.coord_offset, stream);
    if (rc) return rc;
  }
  return FGVC_OK;
}

// The coarse-to-fine point tails of several recurrences of a clip (C2FPointTracker.track_queries): one multi-lane c2f
// chain (c2f.cu), then per lane the NCHW copies of its coarse outputs and one K3 launch.
extern "C" int fgvc_c2f_point_clip_tail_lanes(const float* weights, const int32_t* rows, int32_t K, int32_t job_base,
                                              const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                                              const fgvc_c2f_lane* lanes_dev, const fgvc_c2f_lane* lanes_host,
                                              int32_t n_lanes, int32_t Hc, int32_t Wc, int32_t Hf, int32_t Wf,
                                              float* fine_lab, float* coarse_out, int32_t out_h, int32_t out_w,
                                              int32_t coord_topk, float* maps_nchw, float* coords, void* barrier_ws,
                                              void* stream) {
  FGVC_CHECK_ARG(weights && rows && jobs_dev && jobs_host && lanes_dev && lanes_host && fine_lab && coarse_out &&
                     maps_nchw && coords && barrier_ws, "fgvc_c2f_point_clip_tail_lanes: null pointer");
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_c2f_point_clip_tail_lanes: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(n_lanes >= 1 && Hc > 0 && Wc > 0 && Hf > 0 && Wf > 0 && job_base >= 0,
                 "fgvc_c2f_point_clip_tail_lanes: bad sizes");
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_c2f_lane& ln = lanes_host[i];
    FGVC_CHECK_ARG(ln.job_begin >= job_base && ln.job_end > ln.job_begin,
                   "fgvc_c2f_point_clip_tail_lanes: lane %d is empty or starts before job_base", i);
    FGVC_CHECK_ARG(ln.L > 0 && ln.Lp >= ln.L && ln.Lp % 4 == 0 && ln.lab_offset >= 0 && ln.lab_offset % 4 == 0 &&
                       ln.out_offset >= 0 && ln.out_offset % 4 == 0 && ln.coord_offset >= 0,
                   "fgvc_c2f_point_clip_tail_lanes: bad label sizes or offsets in lane %d", i);
    FGVC_CHECK_ARG(consecutive_slots(jobs_host, ln.job_begin, ln.job_end) >= 0,
                   "fgvc_c2f_point_clip_tail_lanes: out_slots of lane %d must be consecutive", i);
  }
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_c2f_chain_lanes(weights, rows, K, job_base, jobs_dev, lanes_dev, lanes_host, n_lanes, Hc, Wc, Hf, Wf,
                                  fine_lab, coarse_out, reinterpret_cast<unsigned int*>(barrier_ws), st);
  if (rc) return rc;
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_c2f_lane& ln = lanes_host[i];
    rc = nchw_and_coords(coarse_out + ln.out_offset, jobs_dev, jobs_host, ln.job_begin, ln.job_end, ln.Lp, ln.L, Hc, Wc,
                         out_h, out_w, coord_topk, maps_nchw, coords + ln.coord_offset, stream);
    if (rc) return rc;
  }
  return FGVC_OK;
}
