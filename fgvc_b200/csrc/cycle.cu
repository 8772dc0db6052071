// Forward-backward cycle consistency of point tracks (VanillaTracker, test_cfg.cycle_occlusion): every (group, frame t)
// prediction re-tracked toward the group's query frame as one lane of a multi-lane gather chain, then a visibility
// decision on the lane's last frame only.  A clip has up to (groups x frames) lanes, so everything around the chain is
// one launch over all lanes of a call: seeding, the NCHW copy of the last slots, K3, the decision.
#include "common.cuh"

namespace fgvc {

// slot 0 of every lane's bank = the gaussian labels of the group's track at frame t (gaussian_labels_kernel's
// arithmetic on coords[t]); blockIdx.y = lane
__global__ void __launch_bounds__(256)
cycle_seed_kernel(const fgvc_lane* __restrict__ lanes, const fgvc_cycle* __restrict__ cycles,
                  const float* __restrict__ coords, int H, int W, int stride, float denom, float* __restrict__ lab) {
  const fgvc_lane ln = lanes[blockIdx.y];
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= (int64_t)H * W * ln.Lp) return;
  const int p = (int)(i % ln.Lp);
  const int pix = (int)(i / ln.Lp);
  const float* pts = coords + ln.coord_offset + (int64_t)cycles[blockIdx.y].t * ln.L * 2;
  float v = 0.f;
  if (p < ln.L) {
    float x = (float)((pix % W) * stride), y = (float)((pix / W) * stride);
    float dx = x - __ldg(pts + 2 * p), dy = y - __ldg(pts + 2 * p + 1);
    v = expf(__fdiv_rn(-(dx * dx + dy * dy), denom));
  }
  lab[ln.lab_offset + i] = v;
}

// the last slot of every lane's bank -> maps_nchw + map_offset maps ([L][H*W], labels_to_nchw_kernel's tiles);
// blockIdx.z = lane
__global__ void __launch_bounds__(256)
cycle_last_nchw_kernel(const fgvc_lane* __restrict__ lanes, const fgvc_cycle* __restrict__ cycles,
                       const float* __restrict__ lab, int n_pix, float* __restrict__ maps) {
  __shared__ float t[32][33];
  const fgvc_lane ln = lanes[blockIdx.z];
  const int p0 = blockIdx.x * 32, l0 = blockIdx.y * 32;
  if (l0 >= ln.L) return;                                  // (whole block)
  const float* src = lab + ln.lab_offset + (int64_t)(ln.job_end - ln.job_begin) * n_pix * ln.Lp;
  float* dst = maps + cycles[blockIdx.z].map_offset * n_pix;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    int p = p0 + j, l = l0 + tx;
    t[j][tx] = (p < n_pix && l < ln.Lp) ? __ldg(src + (int64_t)p * ln.Lp + l) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int l = l0 + j, p = p0 + tx;
    if (l < ln.L && p < n_pix) dst[(int64_t)l * n_pix + p] = t[tx][j];
  }
}

// per (lane, point): c = the re-tracked position at s, visible iff |c - coords[s]| <= threshold (fp32 Euclidean
// distance); c goes to cycle_coords[t], the flag to vis[t]; blockIdx.y = lane
__global__ void __launch_bounds__(128)
cycle_decide_kernel(const fgvc_lane* __restrict__ lanes, const fgvc_cycle* __restrict__ cycles,
                    const float* __restrict__ xy, const float* __restrict__ coords, float threshold,
                    float* __restrict__ cycle_coords, uint8_t* __restrict__ vis) {
  const fgvc_lane ln = lanes[blockIdx.y];
  const fgvc_cycle cy = cycles[blockIdx.y];
  const int p = blockIdx.x * 128 + threadIdx.x;
  if (p >= ln.L) return;
  const float cx = __ldg(xy + (cy.map_offset + p) * 2), cyy = __ldg(xy + (cy.map_offset + p) * 2 + 1);
  const float* ps = coords + ln.coord_offset + ((int64_t)cy.s * ln.L + p) * 2;
  const float dx = __fsub_rn(cx, __ldg(ps)), dy = __fsub_rn(cyy, __ldg(ps + 1));
  const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
  const int64_t o = (int64_t)cy.t * ln.L + p;
  cycle_coords[ln.coord_offset + 2 * o] = cx;
  cycle_coords[ln.coord_offset + 2 * o + 1] = cyy;
  vis[ln.coord_offset / 2 + o] = d <= threshold ? 1 : 0;
}

}  // namespace fgvc

using namespace fgvc;

extern "C" int fgvc_point_cycle_lanes(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                                      const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                                      const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host,
                                      const fgvc_cycle* cycles_dev, const fgvc_cycle* cycles_host, int32_t n_lanes,
                                      const int32_t* mem_label_slot, int32_t H, int32_t W, int32_t stride, float sigma,
                                      float temperature, int32_t flags, float* lab_bank, int32_t out_h, int32_t out_w,
                                      int32_t coord_topk, float threshold, const float* coords, float* maps_nchw,
                                      float* xy_scratch, float* cycle_coords, uint8_t* vis, void* chain_ws,
                                      int64_t chain_ws_bytes, void* stream) {
  FGVC_CHECK_ARG(topk_val && topk_idx && jobs_dev && jobs_host && lanes_dev && lanes_host && cycles_dev && cycles_host &&
                     mem_label_slot && lab_bank && coords && maps_nchw && xy_scratch && cycle_coords && vis && chain_ws,
                 "fgvc_point_cycle_lanes: null pointer");
  FGVC_CHECK_ARG(K >= 1 && K <= 16, "fgvc_point_cycle_lanes: topk=%d not in [1,16]", K);
  FGVC_CHECK_ARG(n_lanes >= 1 && n_lanes <= 65535 && H > 0 && W > 0 && groups >= 1 && stride > 0 && sigma > 0.f,
                 "fgvc_point_cycle_lanes: bad sizes");
  FGVC_CHECK_ARG(pair_ref == nullptr || groups == 1, "fgvc_point_cycle_lanes: shared lists need groups == 1");
  FGVC_CHECK_ARG(temperature > 0.f, "fgvc_point_cycle_lanes: temperature must be > 0");
  int max_L = 1, max_Lp = 4;
  int64_t n_maps = 0;
  for (int i = 0; i < n_lanes; ++i) {
    const fgvc_lane& ln = lanes_host[i];
    const fgvc_cycle& cy = cycles_host[i];
    FGVC_CHECK_ARG(ln.job_begin >= 0 && ln.job_end > ln.job_begin, "fgvc_point_cycle_lanes: lane %d is empty", i);
    FGVC_CHECK_ARG(ln.L > 0 && ln.Lp >= ln.L && ln.Lp % 4 == 0 && ln.lab_offset >= 0 && ln.lab_offset % 4 == 0 &&
                       ln.coord_offset >= 0 && ln.coord_offset % 2 == 0 && cy.map_offset >= 0 && cy.t >= 0 &&
                       cy.s >= 0 && cy.t != cy.s,
                   "fgvc_point_cycle_lanes: bad label sizes, offsets or frames in lane %d", i);
    for (int j = ln.job_begin; j < ln.job_end; ++j)
      FGVC_CHECK_ARG(jobs_host[j].out_slot == j - ln.job_begin + 1,
                     "fgvc_point_cycle_lanes: the out_slots of lane %d must be 1, 2, ..., n", i);
    max_L = max(max_L, ln.L);
    max_Lp = max(max_Lp, ln.Lp);
    n_maps = max(n_maps, cy.map_offset + ln.L);
  }
  FGVC_CHECK_ARG(n_maps <= 0x7fffffff, "fgvc_point_cycle_lanes: too many maps");
  const int n_pix = H * W;
  cudaStream_t st = (cudaStream_t)stream;
  cycle_seed_kernel<<<dim3((unsigned)(((int64_t)n_pix * max_Lp + 255) / 256), n_lanes), 256, 0, st>>>(
      lanes_dev, cycles_dev, coords, H, W, stride, 2.f * sigma * sigma, lab_bank);
  FGVC_LAUNCH_CHECK();
  int rc = launch_gather_chain_lanes(topk_val, topk_idx, K, groups, jobs_dev, lanes_dev, lanes_host, n_lanes,
                                     mem_label_slot, pair_ref, n_pix, temperature, flags, lab_bank, chain_ws,
                                     chain_ws_bytes, st);
  if (rc) return rc;
  cycle_last_nchw_kernel<<<dim3(cdiv(n_pix, 32), cdiv(max_L, 32), n_lanes), 256, 0, st>>>(lanes_dev, cycles_dev,
                                                                                            lab_bank, n_pix, maps_nchw);
  FGVC_LAUNCH_CHECK();
  rc = fgvc_heatmap_coords(maps_nchw, (int32_t)n_maps, H, W, out_h, out_w, coord_topk, xy_scratch, stream);
  if (rc) return rc;
  cycle_decide_kernel<<<dim3(cdiv(max_L, 128), n_lanes), 128, 0, st>>>(lanes_dev, cycles_dev, xy_scratch, coords,
                                                                      threshold, cycle_coords, vis);
  FGVC_LAUNCH_CHECK();
  return FGVC_OK;
}
