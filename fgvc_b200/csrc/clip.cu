// Clip-level drivers: the sequential part of the reference loop
// (vanilla_tracker.py:345-412) enqueued by ONE C call, so that the host costs a few
// microseconds per frame instead of a Python round trip per kernel.
#include "common.cuh"

using namespace fgvc;

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
  const int64_t mask_elems = (int64_t)out_h * out_w;
  cudaStream_t st = (cudaStream_t)stream;
  if (flags & FGVC_HARD_PROP) {
    // hard propagation: the memory keeps one_hot(argmax) of every propagated frame, the prediction is
    // decoded from the soft labels first (vanilla_tracker.py:762-798) -- so decode per frame
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

// Lowest out_slot of jobs [job_begin, job_end) when their out_slots run consecutively up (a forward track) or down (a
// track run backwards in time), else -1.  The K3 launch of a point tail covers the slots [lowest, lowest + n).
static int consecutive_slots(const fgvc_job* jobs_host, int job_begin, int job_end) {
  const int s0 = jobs_host[job_begin].out_slot, n = job_end - job_begin;
  const int dir = (n > 1 && jobs_host[job_begin + 1].out_slot < s0) ? -1 : 1;
  for (int j = job_begin; j < job_end; ++j)
    if (jobs_host[j].out_slot != s0 + dir * (j - job_begin)) return -1;
  return dir > 0 ? s0 : s0 - (n - 1);
}

// Point tracking tail: the gather chain over jobs [job_begin, job_end) with an NCHW copy of every
// propagated frame into maps_nchw[slot][L][H*W], then ONE K3 launch (fused up-sample / soft-argmax)
// over all (frame, point) maps of the range: coords[slot][L][2].  The out_slots of the range must
// be consecutive (they are frame indices), ascending or descending.
static int point_clip_tail_impl(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                    const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                                    int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                                    float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L, int32_t out_h,
                                    int32_t out_w, int32_t coord_topk, float* maps_nchw, float* coords,
                                    void* chain_ws, int64_t chain_ws_bytes, const int32_t* pair_ref, void* stream) {
  FGVC_CHECK_ARG(jobs_dev && jobs_host && maps_nchw && coords && lab_bank, "fgvc_point_clip_tail: null pointer");
  FGVC_CHECK_ARG(job_end > job_begin, "fgvc_point_clip_tail: empty job range");
  const int n_pix = H * W;
  const int slot0 = consecutive_slots(jobs_host, job_begin, job_end);
  FGVC_CHECK_ARG(slot0 >= 0, "fgvc_point_clip_tail: out_slots must be consecutive");
  FGVC_CHECK_ARG(pair_ref == nullptr || chain_ws != nullptr, "fgvc_point_clip_tail_shared: needs the chain workspace");
  if (chain_ws != nullptr && (job_end - job_begin > 1 || pair_ref != nullptr)) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc = launch_gather_chain(topk_val, topk_idx, K, groups, jobs_dev, job_begin, job_end, mem_label_slot, pair_ref,
                                 n_pix, temperature, flags, lab_bank, Lp, chain_ws, chain_ws_bytes, st);
    if (rc) return rc;
    rc = launch_labels_to_nchw_jobs(lab_bank, jobs_dev, job_begin, job_end, Lp, L, n_pix, maps_nchw, st);
    if (rc) return rc;
  } else {
    for (int j = job_begin; j < job_end; ++j) {
      const int slot = jobs_host[j].out_slot;
      int rc = fgvc_gather_labels(topk_val, topk_idx, K, groups, jobs_dev, j, j + 1, mem_label_slot, n_pix,
                                  temperature, flags, lab_bank, Lp, stream);
      if (rc) return rc;
      rc = fgvc_labels_to_nchw(lab_bank, slot, Lp, L, n_pix, maps_nchw + (int64_t)slot * L * n_pix, stream);
      if (rc) return rc;
    }
  }
  return fgvc_heatmap_coords(maps_nchw + (int64_t)slot0 * L * n_pix, (job_end - job_begin) * L, H, W, out_h, out_w,
                             coord_topk, coords + (int64_t)slot0 * L * 2, stream);
}

extern "C" int fgvc_point_clip_tail(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                    const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                                    int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                                    float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L, int32_t out_h,
                                    int32_t out_w, int32_t coord_topk, float* maps_nchw, float* coords,
                                    void* chain_ws, int64_t chain_ws_bytes, void* stream) {
  return point_clip_tail_impl(topk_val, topk_idx, K, groups, jobs_dev, jobs_host, job_begin, job_end, mem_label_slot, H, W,
                              temperature, flags, lab_bank, Lp, L, out_h, out_w, coord_topk, maps_nchw, coords, chain_ws,
                              chain_ws_bytes, nullptr, stream);
}

// Same with SHARED top-k lists: the jobs of several with_first groups that have the same query frame look at the
// same memory frames except their first one, so K1 ran once per (query frame, memory frame) pair
// (one list per pair) and pair_ref[e] names the list of memory entry e of these jobs (indices into
// topk_val / topk_idx in units of H*W*K).  Needs the chain workspace.
extern "C" int fgvc_point_clip_tail_shared(const float* topk_val, const int32_t* topk_idx, int32_t K,
                                           const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                                           int32_t job_begin, int32_t job_end, const int32_t* mem_label_slot, int32_t H,
                                           int32_t W, float temperature, int32_t flags, float* lab_bank, int32_t Lp,
                                           int32_t L, int32_t out_h, int32_t out_w, int32_t coord_topk, float* maps_nchw,
                                           float* coords, void* chain_ws, int64_t chain_ws_bytes, void* stream) {
  FGVC_CHECK_ARG(pair_ref != nullptr, "fgvc_point_clip_tail_shared: null pair_ref");
  return point_clip_tail_impl(topk_val, topk_idx, K, 1, jobs_dev, jobs_host, job_begin, job_end, mem_label_slot, H, W,
                              temperature, flags, lab_bank, Lp, L, out_h, out_w, coord_topk, maps_nchw, coords, chain_ws,
                              chain_ws_bytes, pair_ref, stream);
}

// Several independent point tails of one clip (bidirectional tracking: the forward and the backward track of every
// point group), each lane bit for bit its own point_clip_tail_impl: one multi-lane gather chain for all of them
// (gather.cu), then per lane the NCHW copies and one K3 launch -- bandwidth work, where one launch per lane costs
// nothing worth saving.
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
    rc = launch_labels_to_nchw_jobs(lab_bank + ln.lab_offset, jobs_dev, ln.job_begin, ln.job_end, ln.Lp, ln.L, n_pix,
                                    maps_nchw, st);
    if (rc) return rc;
    const int slot0 = consecutive_slots(jobs_host, ln.job_begin, ln.job_end);
    rc = fgvc_heatmap_coords(maps_nchw + (int64_t)slot0 * ln.L * n_pix, (ln.job_end - ln.job_begin) * ln.L, H, W, out_h,
                             out_w, coord_topk, coords + ln.coord_offset + (int64_t)slot0 * ln.L * 2, stream);
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
  const int nc = Hc * Wc;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_c2f_chain_lanes(weights, rows, K, job_base, jobs_dev, lanes_dev, lanes_host, n_lanes, Hc, Wc, Hf, Wf,
                                  fine_lab, coarse_out, reinterpret_cast<unsigned int*>(barrier_ws), st);
  if (rc) return rc;
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_c2f_lane& ln = lanes_host[i];
    rc = launch_labels_to_nchw_jobs(coarse_out + ln.out_offset, jobs_dev, ln.job_begin, ln.job_end, ln.Lp, ln.L, nc,
                                    maps_nchw, st);
    if (rc) return rc;
    const int slot0 = consecutive_slots(jobs_host, ln.job_begin, ln.job_end);
    rc = fgvc_heatmap_coords(maps_nchw + (int64_t)slot0 * ln.L * nc, (ln.job_end - ln.job_begin) * ln.L, Hc, Wc, out_h,
                             out_w, coord_topk, coords + ln.coord_offset + (int64_t)slot0 * ln.L * 2, stream);
    if (rc) return rc;
  }
  return FGVC_OK;
}
