/*
 * fgvc_b200 -- C ABI of the B200-native label-propagation path of FGVC (mmpt).
 *
 * This is the drop-in boundary: plain C, device pointers + sizes, no torch types.
 * The Python host (fgvc_b200/ops.py, tracker.py) binds it with ctypes; a maintainer of
 * the reference would bind exactly these symbols (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns every buffer; the library allocates nothing persistent except a
 *     small cache of TMA descriptors;
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*), never
 *     synchronises, and returns 0 on success or a negative fgvc_status; the message is
 *     available from fgvc_last_error() (thread local);
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Data layout in HBM (all fp32 unless noted)
 *   feature bank  feat[slot][2][H*W][C]   part 0 = "hi", part 1 = "lo" of a two-term split of
 *                 the L2-normalised row (fgvc_bank_format: fp32/TF32 or fp16); pixel-major so
 *                 that the channel (contraction) dimension is contiguous = K-major MMA operands.
 *   label bank    lab[slot][H*W][Lp]      Lp = L rounded up to a multiple of 4 (float4
 *                 rows); pixel-major so that the k winners of a query are k coalesced rows.
 *   top-k lists   val[job][group][Nq][K], idx[job][group][Nq][K] (int32,
 *                 idx = position_in_memory_list * Nk + key_pixel, -1 = empty), sorted
 *                 descending; val is the raw cosine (not yet divided by the temperature).
 *
 * Reference interfaces replaced (paths relative to the FGVC repository):
 *   mmpt/models/common/local_attention.py:267  masked_attention_efficient
 *   mmpt/models/common/local_attention.py:392  masked_attention_efficient_v2
 *   mmpt/models/common/local_attention.py:721  masked_attention_efficient_c2f
 *   mmpt/models/common/affinity_utils.py:75    spatial_neighbor (folded into the kernels)
 *   mmpt/models/trackers/vanilla_tracker.py:172 img2coord, :204 draw_gaussion_map_online,
 *                                           :305 forward_test_main (per-frame loop)
 */
#ifndef FGVC_B200_H_
#define FGVC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FGVC_VERSION 100

#if defined(__GNUC__)
#define FGVC_API __attribute__((visibility("default")))
#else
#define FGVC_API
#endif

typedef enum fgvc_status {
  FGVC_OK = 0,
  FGVC_ERR_INVALID = -1,     /* bad argument / unsupported shape */
  FGVC_ERR_CUDA = -2,        /* a CUDA runtime / driver call failed */
  FGVC_ERR_UNSUPPORTED = -3  /* valid in the reference but not built here */
} fgvc_status;

/* feature-bank formats (both hold an L2-normalised frame as a two-term split, pixel-major):
 *   TF32: fp32 [slot][2][H*W][C], hi = tf32(x), lo = x - hi            -> 3xTF32 tensor engine
 *   F16 : fp16 [slot][2][H*W][C], X = 16 x, hi = fp16(X), lo = fp16(X - hi)  -> 3-term fp16 tensor
 *         engine (same 11 + 11 significant bits per operand, twice the MMA depth per instruction,
 *         half the bytes; the 2^4 scale keeps lo a normal fp16 number so the three products share one
 *         fp32 accumulator).  Needs C % 64 == 0. */
typedef enum fgvc_bank_format { FGVC_BANK_TF32 = 0, FGVC_BANK_F16 = 1 } fgvc_bank_format;

typedef enum fgvc_mask_mode { FGVC_MASK_CIRCLE = 0, FGVC_MASK_SQUARE = 1 } fgvc_mask_mode;

/* affinity engines of K1.  AUTO picks the tcgen05 kernel matching the bank format whenever the
 * shape allows (TF32 bank: C % 32 == 0; F16 bank: C % 64 == 0; K <= 16); SIMT is the fp32
 * CUDA-core kernel for every other shape. */
typedef enum fgvc_engine {
  FGVC_ENGINE_AUTO = 0,
  FGVC_ENGINE_SIMT = 1,
  FGVC_ENGINE_TCGEN05 = 2
} fgvc_engine;

/* One propagation job = one query frame and its memory list (a multiset of frames:
 * frame 0 appears twice while t <= precede_frames, vanilla_tracker.py:346-362). */
typedef struct fgvc_job {
  int32_t q_slot;     /* feature-bank slot of the query frame */
  int32_t mem_begin;  /* memory entries [mem_begin, mem_end) of the mem_* tables */
  int32_t mem_end;
  int32_t out_slot;   /* label-bank slot written by fgvc_gather_labels */
} fgvc_job;

/* One lane of fgvc_point_clip_tail_lanes: one recurrence of a clip (the forward or the backward track of a point group)
 * = the consecutive jobs [job_begin, job_end) in recurrence order, with their out_slots running consecutively up or
 * down, over its own label bank lab_bank + lab_offset ([slot][H*W][Lp]) and its own tracks coords + coord_offset
 * ([slot][L][2]).  Two lanes may share a bank when neither reads a slot the other writes. */
typedef struct fgvc_lane {
  int32_t job_begin;
  int32_t job_end;
  int32_t L;             /* label channels (points) of the lane's bank */
  int32_t Lp;            /* bank row length: L rounded up to a multiple of 4 */
  int64_t lab_offset;    /* floats from lab_bank to the lane's bank */
  int64_t coord_offset;  /* floats from coords to the lane's tracks */
} fgvc_lane;

/* One lane of fgvc_c2f_point_clip_tail_lanes: one coarse-to-fine recurrence of a clip (the forward or the backward
 * track of a point group) = the consecutive jobs [job_begin, job_end) in recurrence order, with their out_slots running
 * consecutively up or down.  Its fine label bank is fine_lab + lab_offset ([slot][Hf*Wf][Lp]), its coarse outputs go
 * to coarse_out + out_offset ([slot][Hc*Wc][Lp]) and its tracks to coords + coord_offset ([slot][L][2]).  Two lanes
 * may share a fine bank when neither reads a slot the other writes. */
typedef struct fgvc_c2f_lane {
  int32_t job_begin;
  int32_t job_end;
  int32_t L;             /* label channels (points) of the lane */
  int32_t Lp;            /* bank row length: L rounded up to a multiple of 4 */
  int64_t lab_offset;    /* floats from fine_lab to the lane's fine label bank */
  int64_t out_offset;    /* floats from coarse_out to the lane's coarse-output bank */
  int64_t coord_offset;  /* floats from coords to the lane's tracks */
} fgvc_c2f_lane;

/* Job-packed query tiles of the fp16 tensor engine (fgvc_affinity_topk_packed): a tile group = up to 4 jobs that
 * share most of their memory frames (consecutive query frames of a clip) and are multiplied against each key box
 * together.  Memory entries [u_begin, u_end) of the union tables list every (frame, mask flag) any job of the group
 * uses; union_pos[entry][i] is the entry's position in job[i]'s own memory list (what the top-k indices refer to)
 * or -1 when job[i] does not have it. */
typedef struct fgvc_tile_group {
  int32_t job[4];   /* indices into jobs[]; unused = -1 */
  int32_t n_jobs;
  int32_t u_begin;
  int32_t u_end;
  int32_t out_group; /* which of the job's output lists this group writes (x split + part, see fgvc_affinity_topk_packed) */
} fgvc_tile_group;

/* fgvc_gather_labels flags */
#define FGVC_WEIGHT_COSINE 1 /* weights = clamp(a, 0)^2 instead of softmax(a)   (mode='cosine', local_attention.py:371) */
#define FGVC_HARD_PROP 4     /* clip tails only: the memory keeps one_hot(argmax) of each propagated frame
                                (hard_prop, vanilla_tracker.py:762-767); predictions still decode the soft labels */
#define FGVC_SIM_L2 2        /* a = (2 cos - 1) / temperature with temperature := sqrt(C)
                                (sim_mode='l2-distance' on normalised features, local_attention.py:324-327) */

/* Local-window ("HR") propagation (HRVanillaTracker.forward_test_main, vanilla_tracker.py:492-585, on
 * mmcv.ops.Correlation + F.unfold(padding=r)): with a SQUARE mask of radius r the window positions outside the image
 * are candidates too, with affinity 0 and value 0; the gather merges them analytically into the winners.  The flag
 * carries the geometry: FGVC_ZERO_PAD | (r << 8) | (W << 16), r <= 255, W <= 65535. */
#define FGVC_ZERO_PAD 8
#define FGVC_ZERO_PAD_FLAGS(radius, W) (FGVC_ZERO_PAD | ((radius) << 8) | ((W) << 16))

#define FGVC_MEM_UNMASKED 0x40000000 /* OR into mem_feat_slot: radius mask not applied
                                        (the first non_mask_len frames, local_attention.py:347) */

FGVC_API const char* fgvc_last_error(void);
FGVC_API int fgvc_version(void);
/* number of CUDA devices visible to the library (0 => every compute call fails) */
FGVC_API int fgvc_device_count(void);
/* kernels launched by this library in this process so far (bench.py's gpu_launches) */
FGVC_API int64_t fgvc_launch_count(void);

/* K0 -- F.normalize(dim=C) + NCHW -> pixel-major + hi/lo split in the bank's format (see fgvc_bank_format)
 * (local_attention.py:308-310).  src: n_frames frames of [C][H*W], consecutive frames
 * src_frame_stride floats apart, channels src_chan_stride floats apart (so a
 * [1,C,T,H,W] key stack can be read in place).  Writes bank slots
 * first_slot .. first_slot+n_frames-1. */
FGVC_API int fgvc_prep_features(const float* src, int64_t src_frame_stride, int64_t src_chan_stride,
                       int32_t n_frames, int32_t C, int32_t H, int32_t W, int32_t normalize,
                       void* feat_bank, int32_t bank_format, int32_t first_slot, void* stream);

/* label layout conversions: NCHW [L][H*W] (channel stride src_chan_stride) <-> pixel-major */
FGVC_API int fgvc_labels_to_pixmajor(const float* src, int64_t src_chan_stride, int32_t L, int32_t n_pix,
                            float* lab_bank, int32_t slot, int32_t Lp, void* stream);
FGVC_API int fgvc_labels_to_nchw(const float* lab_bank, int32_t slot, int32_t Lp, int32_t L, int32_t n_pix,
                        float* dst, void* stream);

/* Bilinear up-sampling of a pixel-major label map src[Hs*Ws][Lp] into slot `slot` of a label bank of Hd x Wd maps,
 * with F.interpolate(mode='bilinear', align_corners=False) taps (vanilla_tracker.py:396-400 applies it to the
 * propagated map; the coarse-to-fine clip driver uses it to turn the coarse output of
 * masked_attention_efficient_c2f, local_attention.py:721-880, into the next frame's fine memory labels). */
FGVC_API int fgvc_upsample_labels(const float* src, int32_t Hs, int32_t Ws, int32_t Lp, float* lab_bank, int32_t slot,
                         int32_t Hd, int32_t Wd, void* stream);

/* draw_gaussion_map_online at feature resolution (vanilla_tracker.py:204-221):
 * lab[slot][y*W+x][p] = exp(-((x*stride-px)^2 + (y*stride-py)^2) / (2 sigma^2)).
 * points_xy: [P][2] (x,y) image pixels. */
FGVC_API int fgvc_gaussian_labels(const float* points_xy, int32_t P, int32_t H, int32_t W, int32_t stride,
                         float sigma, float* lab_bank, int32_t slot, int32_t Lp, void* stream);

/* 1 when the tcgen05 engine of K1 takes this shape, else 0 (AUTO then uses the SIMT engine) */
FGVC_API int fgvc_tc_supported(int32_t bank_format, int32_t H, int32_t W, int32_t C, int32_t K);

/* workspace bytes for the top-k lists of n_jobs jobs */
FGVC_API int64_t fgvc_topk_bytes(int32_t n_jobs, int32_t groups, int32_t n_query, int32_t K);

/* K1 -- affinity + radius mask + running top-K for jobs[0..n_jobs) in ONE launch
 * (local_attention.py:318-356 without materialising the affinity).  The memory list of
 * each job is split into `groups` contiguous parts (load balance for short job lists);
 * fgvc_gather_labels merges them.  K in [1,16]; radius = neighbor_range // 2. */
FGVC_API int fgvc_affinity_topk(const void* feat_bank, int32_t bank_format, int32_t n_slots, int32_t H, int32_t W, int32_t C,
                       const fgvc_job* jobs, int32_t n_jobs, const int32_t* mem_feat_slot,
                       int32_t radius, int32_t mask_mode, int32_t K, int32_t groups,
                       float* topk_val, int32_t* topk_idx, int32_t engine, void* stream);

/* K1 with a starting floor for the lists (F16 bank, fp16 tensor engine; ignored by the other engines): floor[job][query
 * pixel], in accumulator units (256 x cosine) as written by fgvc_topk_floor, must be a value that at least K genuine
 * candidates of EVERY consumer of the job's lists reach -- the lists then hold only candidates above it, which is all
 * a top-K merge needs.  For launches whose lists start cold and stay short: one list per (query frame, memory frame)
 * pair shared between the point groups of a clip (vanilla_tracker.py:262-284 re-runs the whole sub-clip per group),
 * where half of the launch was list insertion.  fgvc_topk_floor scores the 5 x 5 neighbourhood of the query's own
 * position in ONE memory frame per job (seed_feat_slot[job]; < 0 = no floor for the job) exactly, in-image and in-mask
 * keys only, and writes the K-th largest minus a rounding margin (-inf where fewer than K are valid). */
FGVC_API int fgvc_affinity_topk_seeded(const void* feat_bank, int32_t bank_format, int32_t n_slots, int32_t H, int32_t W, int32_t C,
                       const fgvc_job* jobs, int32_t n_jobs, const int32_t* mem_feat_slot,
                       int32_t radius, int32_t mask_mode, int32_t K, int32_t groups, const float* floor,
                       float* topk_val, int32_t* topk_idx, int32_t engine, void* stream);
FGVC_API int fgvc_topk_floor(const void* feat_bank, int32_t bank_format, int32_t H, int32_t W, int32_t C,
                       const fgvc_job* jobs, int32_t n_jobs, const int32_t* seed_feat_slot, int32_t radius,
                       int32_t mask_mode, int32_t K, float* floor_out, void* stream);

/* K1 on job-packed tiles (F16 bank, tcgen05 fp16 three-term engine only; local_attention.py:318-356 for several
 * consecutive frames of the loop vanilla_tracker.py:345-366 at once): same output as fgvc_affinity_topk
 * for the jobs named by the tile groups (lists are written at [job][list][Nq][K] by job index, `groups` lists per
 * job).  A tile group covers the memory entries [u_begin, u_end) of the union tables, cut into `split` contiguous
 * parts (one CTA or CTA pair each); part y writes list  out_group * split + y  of its jobs, so `groups` must be
 * split x (number of distinct out_group values) and every (job, list) must be written by exactly one tile group.
 * jobs_per_tile in {1, 2, 4}: tile rows = jobs_per_tile jobs x a pixel block.  A tile is one CTA (128 rows); with the
 * environment variable FGVC_TC16_PAIR=1 and a map large enough it is a CTA PAIR (256 rows, tcgen05 cta_group::2: both
 * SMs of the pair multiply the same key box and each stages half of it) -- same results, not faster (DESIGN.md 4.1).
 * fgvc_packed_tile_shape reports the pixel block of one job, the key-box height and the CTAs per tile the launcher
 * will use (for costing). */
FGVC_API int fgvc_affinity_topk_packed(const void* feat_bank, int32_t n_slots, int32_t H, int32_t W, int32_t C,
                       const fgvc_job* jobs, const fgvc_tile_group* tile_groups, int32_t n_tile_groups,
                       const int32_t* union_feat_slot, const int32_t* union_pos, int32_t jobs_per_tile,
                       int32_t radius, int32_t mask_mode, int32_t K, int32_t groups, int32_t split,
                       float* topk_val, int32_t* topk_idx, void* stream);
FGVC_API int fgvc_packed_tile_shape(int32_t H, int32_t W, int32_t radius, int32_t mask_mode, int32_t jobs_per_tile,
                       int32_t* tile_h, int32_t* tile_w, int32_t* box_h, int32_t* ctas_per_tile);

/* test hook (tcgen05 engine, groups = 1, use with ONE query tile): additionally dumps the
 * raw 128 x 128 accumulator tile of the first dbg_max_boxes key boxes to
 * dbg[box][query_row][key_col] and (mem entry, box y, box x, N) to dbg_meta[box][4]. */
FGVC_API int fgvc_debug_affinity_boxes(const void* feat_bank, int32_t bank_format, int32_t n_slots, int32_t H, int32_t W, int32_t C,
                       const fgvc_job* jobs, int32_t n_jobs, const int32_t* mem_feat_slot,
                       int32_t radius, int32_t mask_mode, int32_t K, float* topk_val,
                       int32_t* topk_idx, float* dbg, int32_t* dbg_meta, int32_t dbg_max_boxes,
                       void* stream);

/* K1b -- merge groups, /temperature, softmax over the K winners, gather + weighted sum
 * of label rows (local_attention.py:360-374).  Handles jobs[job_begin..job_end) (the
 * jobs of one time step across clips: they must not read each other's out_slot). */
FGVC_API int fgvc_gather_labels(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                       const fgvc_job* jobs, int32_t job_begin, int32_t job_end,
                       const int32_t* mem_label_slot, int32_t n_pix, float temperature, int32_t flags,
                       float* lab_bank, int32_t Lp, void* stream);

/* Dense propagation -- topk = None (local_attention.py:376-383): weights = soft-max (or clamp(a,0)^2 with
 * FGVC_WEIGHT_COSINE) over ALL allowed candidates; flash-style, fp32 on the CUDA cores, writes each job's
 * out_slot of the label bank directly.  jobs[0..n_jobs) must not read each other's out_slot. */
FGVC_API int fgvc_dense_propagate(const void* feat_bank, int32_t bank_format, int32_t H, int32_t W, int32_t C,
                         const fgvc_job* jobs, int32_t n_jobs, const int32_t* mem_feat_slot,
                         const int32_t* mem_label_slot, int32_t radius, int32_t mask_mode, float temperature,
                         int32_t flags, float* lab_bank, int32_t Lp, void* stream);

/* K3 -- F.interpolate(bilinear, align_corners=False) to (out_h,out_w) fused with img2coord
 * (vanilla_tracker.py:396-400, :172-191): top-5 soft-argmax, all-zero map -> -1.
 * maps: n_maps channel-major maps [H*W]; out_xy: [n_maps][2]. */
FGVC_API int fgvc_heatmap_coords(const float* maps, int32_t n_maps, int32_t H, int32_t W, int32_t out_h,
                        int32_t out_w, int32_t topk, float* out_xy, void* stream);
/* same on the analytic full-resolution gaussian of frame 0 (vanilla_tracker.py:321-343) */
FGVC_API int fgvc_gaussian_coords(const float* points_xy, int32_t P, int32_t out_h, int32_t out_w,
                         float sigma, int32_t topk, float* out_xy, void* stream);

/* VOS-style decode (vanilla_tracker.py:769-798): bilinear up-sample, per-channel min-max
 * normalise where max > 0, argmax over channels -> uint8 [out_h][out_w].
 * maps: [L][H*W]; scratch_minmax: [2*L] floats. */
FGVC_API int fgvc_decode_masks(const float* maps, int32_t L, int32_t H, int32_t W, int32_t out_h,
                      int32_t out_w, float* scratch_minmax, uint8_t* out_mask, void* stream);

/* same, reading slot `slot` of the pixel-major label bank directly (no NCHW copy) */
FGVC_API int fgvc_decode_masks_pixmajor(const float* lab_bank, int32_t slot, int32_t Lp, int32_t L, int32_t H,
                               int32_t W, int32_t out_h, int32_t out_w, float* scratch_minmax,
                               uint8_t* out_mask, void* stream);

/* Clip-level tails: the sequential part of the reference loop (vanilla_tracker.py:345-412)
 * enqueued by one call after K0 + K1 ran for the whole clip.  jobs_host = host copy of the
 * job table (the launcher needs each out_slot).
 *  mask tail : the K1b gather chain over jobs [job_begin, job_end) (+ optional NCHW copies into
 *              maps_nchw[slot]), then ONE batched decode of all their frames into
 *              masks[slot][out_h][out_w]; scratch_minmax: (job_end - job_begin) * 2 * L words;
 *  point tail: the K1b gather chain over jobs [job_begin, job_end) with an NCHW copy of every frame
 *              into maps_nchw[slot][L][H*W], then ONE K3 launch over all their (frame, point) maps
 *              into coords[slot][L][2]; the out_slots of the range must be consecutive (ascending, or descending
 *              for a track run backwards in time). */
/* chain_ws (optional, fgvc_chain_workspace_bytes(job_end - job_begin, H*W, K) bytes): with it the gather chain of a
 * range runs as ONE persistent cooperative kernel (label-independent weights for all frames first, then one grid
 * barrier per frame) instead of one launch per frame; NULL keeps the per-frame launches.  Same results. */
FGVC_API int64_t fgvc_chain_workspace_bytes(int32_t n_jobs, int32_t n_pix, int32_t K);
FGVC_API int fgvc_mask_clip_tail(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                        const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                        int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                        float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L,
                        int32_t out_h, int32_t out_w, float* scratch_minmax, uint8_t* masks,
                        float* maps_nchw, void* chain_ws, int64_t chain_ws_bytes, void* stream);
FGVC_API int fgvc_point_clip_tail(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                         const fgvc_job* jobs_dev, const fgvc_job* jobs_host, int32_t job_begin,
                         int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                         float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L,
                         int32_t out_h, int32_t out_w, int32_t coord_topk, float* maps_nchw,
                         float* coords, void* chain_ws, int64_t chain_ws_bytes, void* stream);

/* Point tail on SHARED top-k lists (the grouping loop of VanillaTracker.forward_test, vanilla_tracker.py:249-295, which
 * re-runs forward_test_main per unique query frame).  Jobs of different with_first groups with the same query frame use the same
 * memory frames except their first one, so K1 is run once per query frame over the union of those frames with one
 * group per memory entry (fgvc_affinity_topk, groups = longest union): one list per (query frame, memory frame) pair.
 * pair_ref[e] = index of the list (in units of H*W*K elements of topk_val / topk_idx) for memory entry e of the
 * per-group job table; the tail merges each job's lists, re-basing the positions to the job's own memory list.
 * chain_ws is required. */
FGVC_API int fgvc_point_clip_tail_shared(const float* topk_val, const int32_t* topk_idx, int32_t K,
                         const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                         int32_t job_begin, int32_t job_end, const int32_t* mem_label_slot, int32_t H, int32_t W,
                         float temperature, int32_t flags, float* lab_bank, int32_t Lp, int32_t L,
                         int32_t out_h, int32_t out_w, int32_t coord_topk, float* maps_nchw,
                         float* coords, void* chain_ws, int64_t chain_ws_bytes, void* stream);

/* Point tail of SEVERAL independent recurrences of one clip (bidirectional tracking: every point group is tracked
 * forward from its query frame and, on the time-reversed clip, backward to frame 0).  Each lane (fgvc_lane) is the
 * point tail above over its own job range, bank and tracks, and gives bit for bit what that tail gives; but the
 * chains of all lanes run together: ONE weight launch over the jobs of every lane, then ONE cooperative kernel whose
 * step s gathers job s of every lane still running, with one grid barrier per step -- the longest lane's length of
 * barriers instead of the sum over the lanes.  The NCHW copies and K3 then run per lane.  pair_ref: NULL (lists of
 * `groups` parts per job) or the shared lists of fgvc_point_clip_tail_shared (groups must be 1).
 * lanes_dev / lanes_host: the lane table in device and host memory.  maps_nchw: scratch of (largest out_slot + 1) x
 * (largest L) x H*W floats, reused lane after lane.  chain_ws (required): fgvc_chain_workspace_bytes(je - jb, H*W, K)
 * bytes, [jb, je) = the smallest job range holding every lane. */
FGVC_API int fgvc_point_clip_tail_lanes(const float* topk_val, const int32_t* topk_idx, int32_t K, int32_t groups,
                         const int32_t* pair_ref, const fgvc_job* jobs_dev, const fgvc_job* jobs_host,
                         const fgvc_lane* lanes_dev, const fgvc_lane* lanes_host, int32_t n_lanes,
                         const int32_t* mem_label_slot, int32_t H, int32_t W, float temperature, int32_t flags,
                         float* lab_bank, int32_t out_h, int32_t out_w, int32_t coord_topk, float* maps_nchw,
                         float* coords, void* chain_ws, int64_t chain_ws_bytes, void* stream);

/* K2 -- coarse-to-fine propagation (local_attention.py:721-880), single query frame.
 * Coarse stage = per-memory-frame masked argmax on the coarse bank (K1 with K=1 per
 * frame); fine stage = (2*radius_fine+1)^2 window of the fine bank centred at
 * scale*(ky,kx), zero padded (padded candidates: affinity 0, value 0), top-K over
 * T*R^2, softmax, gather of FINE labels.  Output on the coarse grid: out[Hc*Wc][Lp].
 * job_dev / job_host: the same job in device memory (read by K1) and host memory (read by
 * the launcher); scratch_val / scratch_idx: fgvc_c2f_scratch_elems(n_mem, Hc*Wc) elements each (the coarse per-frame
 * arg-max table, one floor per coarse query, then the fine top-K lists).  With an F16 fine bank (Cf % 64 == 0,
 * Cf <= 256, n_mem <= 64) the fine stage runs on the tensor cores as a window-mode K1 (csrc/topk_tc16.cu) whose lists
 * start from the K-th best of the exactly scored window centres (+ 4 neighbours) of all memory frames; otherwise one
 * warp per candidate. */
FGVC_API int64_t fgvc_c2f_scratch_elems(int32_t n_mem, int32_t n_coarse);
FGVC_API int fgvc_c2f_propagate(const void* coarse_bank, int32_t bank_format, int32_t n_slots, int32_t Hc, int32_t Wc,
                       int32_t C, const void* fine_bank, int32_t Hf, int32_t Wf, int32_t Cf,
                       const fgvc_job* job_dev, const fgvc_job* job_host,
                       const int32_t* mem_feat_slot, const int32_t* mem_label_slot, int32_t radius,
                       int32_t mask_mode, int32_t radius_fine, int32_t K, float temperature,
                       const float* fine_lab_bank, int32_t Lp, float* out, float* scratch_val,
                       int32_t* scratch_idx, int64_t scratch_elems, int32_t engine, void* stream);

/* Coarse-to-fine propagation of a whole clip (C2FPointTracker.track_queries), split where the recurrence is.  The
 * coarse arg-max, the fine window top-K, the zero-padded candidates and the soft-max weights of a job depend on the
 * features only; only the gather of fine label rows and the up-sampling of its result are recurrent.
 *
 * fgvc_c2f_clip_weights: for the jobs [job_begin, job_end) of jobs_host, the label-independent half of
 * fgvc_c2f_propagate, bit for bit what that call computes for each job: (weight, fine label row) pairs
 * weights[job - job_begin][Hc*Wc][K], rows[...] (row = mem_label_slot * Hf*Wf + fine pixel, -1 = zero-padded or empty
 * candidate, weight 0 = unused).  Enqueued as one coarse K1 per distinct memory length (K = 1, groups = length, over a
 * length-sorted copy of the jobs), then for all jobs at once either the floor kernel + one window-mode K1 + one weights
 * kernel (the tensor-core fine stage) or one weights-only launch of the one-warp-per-candidate fine kernel.  The launch
 * count does not depend on the number of jobs.  ws: fgvc_c2f_clip_workspace_bytes(...) bytes (job tables, arg-max
 * tables, floors and fine lists of the range; a caller bounds it by calling in job slices).  jobs_host is read by the
 * call only; the job tables it needs on the device are copied into ws. */
FGVC_API int64_t fgvc_c2f_clip_workspace_bytes(const fgvc_job* jobs_host, int32_t job_begin, int32_t job_end,
                       int32_t Hc, int32_t Wc, int32_t K);
FGVC_API int fgvc_c2f_clip_weights(const void* coarse_bank, int32_t bank_format, int32_t n_slots, int32_t Hc, int32_t Wc,
                       int32_t C, const void* fine_bank, int32_t Hf, int32_t Wf, int32_t Cf,
                       const fgvc_job* jobs_host, int32_t job_begin, int32_t job_end,
                       const int32_t* mem_feat_slot, const int32_t* mem_label_slot, int32_t radius,
                       int32_t mask_mode, int32_t radius_fine, int32_t K, float temperature, float* weights,
                       int32_t* rows, void* ws, int64_t ws_bytes, int32_t engine, void* stream);

/* The recurrent half for several lanes (fgvc_c2f_lane) at once: ONE cooperative kernel whose step s, for every lane
 * still running, (1) gathers job s's coarse output out[q] = sum_k w * fine_lab[row] (the FMA sequence of the gather of
 * fgvc_c2f_propagate) into the lane's coarse-output bank at the job's out_slot, grid barrier, (2) up-samples it into
 * the job's out_slot of the lane's fine bank (the taps of fgvc_upsample_labels), grid barrier -- twice the longest
 * lane's length in barriers.  Then per lane the NCHW copies of its coarse outputs into maps_nchw[slot][L][Hc*Wc] and
 * ONE K3 launch over all its (frame, point) maps into coords[slot][L][2].  weights / rows: fgvc_c2f_clip_weights of
 * the jobs from job_base on (every lane's jobs inside).  maps_nchw: scratch of (largest out_slot + 1) x (largest L) x
 * Hc*Wc floats, reused lane after lane.  barrier_ws: 256 bytes of scratch (zeroed by the call).  Each lane's tracks
 * and coarse outputs are bit for bit what fgvc_c2f_propagate + fgvc_upsample_labels + K3 give frame by frame. */
FGVC_API int fgvc_c2f_point_clip_tail_lanes(const float* weights, const int32_t* rows, int32_t K, int32_t job_base,
                       const fgvc_job* jobs_dev, const fgvc_job* jobs_host, const fgvc_c2f_lane* lanes_dev,
                       const fgvc_c2f_lane* lanes_host, int32_t n_lanes, int32_t Hc, int32_t Wc, int32_t Hf,
                       int32_t Wf, float* fine_lab, float* coarse_out, int32_t out_h, int32_t out_w,
                       int32_t coord_topk, float* maps_nchw, float* coords, void* barrier_ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FGVC_B200_H_ */
