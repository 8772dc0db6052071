// K1 (tcgen05 engine, fp16 three-term split): fused affinity + radius mask + running top-K.  ONE kernel template for
//   * plain tiles (one job per query tile), job-packed tiles (J consecutive jobs x a small pixel block per tile),
//   * single-CTA tiles (128 rows, cta_group::1) and CTA-PAIR tiles (256 rows, cta_group::2: the two SMs of a pair
//     multiply the SAME key box, each staging half of it),
//   * the window mode of the coarse-to-fine fine stage (K2).
//
// Operands are the F16 bank:  X = 16 x,  hi = fp16(X),  lo = fp16(X - hi)  -- 11 + 11 significant bits per
// operand, what the 3xTF32 split carries (rows are unit vectors, the 2^4 scale keeps `lo` a normal fp16 number).
// Three products per K step (16 channels), all into ONE fp32 accumulator in tensor memory:
//     D += hi_q * hi_k;   D += hi_q * lo_k;   D += lo_q * hi_k          (D = 256 * affinity, lo*lo < 2^-22 dropped)
// Both query parts live in tensor memory (2 x C/2 columns, two channels per 32-bit cell), so every MMA is TS-form:
// an M = 128 (per CTA) tcgen05.mma then costs N/2 cycles, +43 if A came from shared memory
// (profiles/r1_mma_issue_rates.md).  TMEM: [0,256) up to four accumulator tiles of N columns (the MMA warp may run
// three boxes ahead of the epilogue), [256,384) hi_q, [384,512) lo_q.
//
// CTA pairs (NCTA = 2) are built and tested but NOT what AUTO runs: a cta_group::2 MMA costs the same N/2 cycles
// per SM as a single-CTA one (profiles/r2_mma_pair_rates.md), a 256-row tile has the larger halo (+17 % tensor
// work on the bench clip), and the kernel is bound by its epilogue, not by the L2 -> SM fabric
// (profiles/r2_a_l2_bound.md, profiles/r2_b_epilogue.md).  FGVC_TC16_PAIR=1 selects them.
//
// CTA anatomy (320 threads): warp 0 = TMA producer (one elected lane), warp 1 = MMA issuer (one elected lane; of
// the leader CTA for a pair), warps 2-9 = epilogue: thread = query row (TMEM lane), warpgroup w owns key rows
// w, w + 2 (, ...) of a box.  A key box is a spatial rectangle (16 x BH pixels of one memory frame): halos are box
// coordinates and out-of-image pixels are zero-filled by the TMA unit.  The boxes a tile needs are listed once per
// CTA (centre-out) and walked by all three roles.  The circle / square mask is one 16-bit interval per (thread, key
// row); a row whose maximum is below the floor of every lane is rejected by one vote, candidates above the thread's
// running K-th value are inserted into a sorted register list in warp-wide rounds; the partial lists of a query
// (one per warpgroup) share their K-th values through shared memory.
#include <stdlib.h>

#include <type_traits>

#include "tc_common.cuh"

namespace fgvc {
namespace tc16 {

constexpr int RING_BYTES = 192 * 1024;
constexpr int MAX_STAGES = 12;
constexpr int MAX_NC = 64;                     // keys of a box staged per CTA (x NCTA = N of the MMA)
constexpr int AHI_COL = 256, ALO_COL = 384;
constexpr int MAX_ACC = 4;                     // accumulator tiles in TMEM columns [0, 256): 256 / N of them, at most 4
constexpr int EPI_WG = 2;                     // epilogue warpgroups: 4 warps per TMEM lane quarter share the rows of a box
constexpr int THREADS = 64 + 128 * EPI_WG;
constexpr int MAX_BOXES = 3840;                // per box list (masked halo / whole frame)
constexpr int THR_BYTES = 128 * EPI_WG * 4;    // running K-th values of the partial lists, shared per query
constexpr int AUX_BYTES = 1024 + THR_BYTES + 2 * MAX_BOXES * 4;
constexpr int SMEM_BYTES = RING_BYTES + AUX_BYTES;
constexpr int TW_MAX_MEM = 64;                 // window mode: memory entries per call

struct Params {
  int H, W, C, n_pix;          // key grid (window mode: the FINE grid)
  int radius, mode, reach;
  int QH, QW, qw_shift;        // pixel block of ONE job inside a tile
  int lpj_shift;               // log2(tile rows per job): rows = J jobs x (128 * NCTA / J) pixels
  int BH, bh_shift;            // key-box height (a power of two): a box = 16 x BH pixels = N keys, BH / NCTA rows
                               // staged per CTA
  int tiles_x;
  int lists_per_job, split, k_out;   // output lists per job; a tile group's memory list is split `split` ways (grid.y)
  const fgvc_job* jobs;
  const fgvc_tile_group* tgroups;   // packed tiles (one per grid.z) or nullptr: one job per grid.z
  const int32_t* ent;               // memory entries: union table (packed) / mem_feat table
  const int32_t* upos;              // packed: [entry][4] position in job i's own list, -1 = not in it
  // window mode (K2 fine stage)
  int HQ, WQ, scale, rf, chunks;
  fgvc_job job;
  const c2f_wjob* wjobs;            // several jobs in one launch (grid.y = their (entry, chunk) CTAs) or nullptr: `job`
  int n_wjobs;
  const int32_t* best;              // [n_mem][HQ * WQ] coarse arg-max key pixel per memory entry
  const float* floor;               // [HQ * WQ] lower bound of the query's final K-th value (accumulator units) or nullptr
  float* tv;
  int32_t* ti;
  float* dbg;
  int32_t* dbg_meta;
  int dbg_max_boxes;
  int exp_flags;             // experiments (FGVC_TC16_EXP env): 1 = no candidate scan, 4 = half the TMA bytes
};

// ------------------------------------------------------------------------- PTX wrappers (cta_group aware)
template <int NCTA>
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  if (NCTA == 1)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// completion of all prior MMAs of this thread -> one arrival on `bar` (in both CTAs of a pair)
template <int NCTA>
__device__ __forceinline__ void umma_commit_all(uint64_t* bar) {
  if (NCTA == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  else
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
}
__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint4& a, const uint4& b, const uint4& c,
                                           const uint4& d) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w), "r"(c.x), "r"(c.y),
        "r"(c.z), "r"(c.w), "r"(d.x), "r"(d.y), "r"(d.z), "r"(d.w)
      : "memory");
}
// kind::f16 instruction descriptor: c_format F32 = 1 [4,6), a/b_format F16 = 0, K-major, N>>3 [17,23), M>>4 [24,29)
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of `p` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
// (default semantics, as CUTLASS's umma_arrive_2x1SM_sm0: the .release.cluster form costs a MEMBAR.ALL.GPU per arrival,
// and what it would order -- the tcgen05.ld results -- is already complete: tcgen05.wait::ld + fence::before_thread_sync)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// one 64-channel chunk of this CTA's part of a key box -> shared memory; completion bytes go to the LEADER's barrier
template <int NCTA>
__device__ __forceinline__ void tma_box(const CUtensorMap* map, uint32_t leader_bar, void* dst, int c0, int c1, int c2,
                                        int c3, int c4) {
  if (NCTA == 1)
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}

// One key row of a box for one warp: r[j] = accumulator (256 x affinity) of this lane's query against key j of the row,
// `bits` = the lane's in-mask keys.  Most rows hold nothing above the running K-th values once the lists are warm:
// a 3-input max tree over the row (8 instructions) and one vote reject those.  Otherwise candidates (in-mask and above
// the lane's K-th value) are inserted into the sorted register list in warp-wide rounds: in every round each lane that
// still has a candidate takes its next one, so a round serves several lanes at once.
// experiment counters (build with -DFGVC_TC16_STATS, run with FGVC_TC16_EXP & 16): row scans, rows past the quick reject, insertion rounds, list insertions
__device__ unsigned long long g_stats[8];

template <int K>
__device__ __forceinline__ void scan_row(const uint32_t (&r)[16], uint32_t bits, TopK<K>& top, int kbase, float floor_,
                                         int stats) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
  const float thr = fmaxf(top.thr(), floor_);
  float mx = fmaxf(fmaxf(v[0], v[1]), v[2]);
#pragma unroll
  for (int j = 3; j < 15; j += 2) mx = fmaxf(fmaxf(mx, v[j]), v[j + 1]);
  mx = fmaxf(mx, v[15]);
#ifdef FGVC_TC16_STATS
  if (stats && (threadIdx.x & 31) == 0) atomicAdd(&g_stats[0], 1ull);
#endif
  if (!__any_sync(0xffffffffu, bits != 0 && mx > thr)) return;
#ifdef FGVC_TC16_STATS
  if (stats && (threadIdx.x & 31) == 0) atomicAdd(&g_stats[1], 1ull);
#endif
  uint32_t cand = 0;
#pragma unroll
  for (int j = 0; j < 16; ++j) cand |= (v[j] > thr) ? (1u << j) : 0u;
  cand &= bits;
  while (__any_sync(0xffffffffu, cand != 0)) {
#ifdef FGVC_TC16_STATS
    if (stats && (threadIdx.x & 31) == 0) atomicAdd(&g_stats[2], 1ull);
#endif
    if (cand) {
      const int j = __ffs(cand) - 1;
      cand &= cand - 1;
      const float x = select16(v, j);
      if (x > fmaxf(top.thr(), floor_)) {
        top.push(x, kbase + j);
#ifdef FGVC_TC16_STATS
        if (stats) atomicAdd(&g_stats[3], 1ull);
#endif
      }
    }
  }
}

template <int K, int NCTA, bool WIN>
__global__ void __launch_bounds__(THREADS, 1)
affinity_topk_tc16_kernel(const __grid_constant__ CUtensorMap tmap_k, const __half* __restrict__ bank, const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + RING_BYTES);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tfull_bar = empty_bar + MAX_STAGES;   // [MAX_ACC]
  uint64_t* tempty_bar = tfull_bar + MAX_ACC;     // [MAX_ACC]
  uint64_t* a_bar = tempty_bar + MAX_ACC;         // query operand written to TMEM
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_bar + 1);
  int* nbox = reinterpret_cast<int*>(tmem_slot + 2);      // [2] number of boxes in each list
  int* halfw = reinterpret_cast<int*>(tmem_slot + 4);     // [reach + 2] <= 130 entries, then rect[4] (window mode)
  // box lists (by | bx << 16): [0] = radius halo of this query tile minus boxes no query can see,
  // [1] = every box of the frame (unmasked memory entries).  Identical for all memory entries, so
  // the three warp roles just walk a list instead of re-deriving the geometry per box.
  // Window mode: ONE list (this CTA's chunk of its entry's rectangle) over both areas.
  float* thr_sh = reinterpret_cast<float*>(ring + RING_BYTES + 1024);      // [128 queries][EPI_WG lists]
  uint32_t* boxes = reinterpret_cast<uint32_t*>(ring + RING_BYTES + 1024 + THR_BYTES);
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u)) __trap();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = NCTA == 2 ? cluster_ctarank() : 0u;
  const int tile = blockIdx.x / NCTA;
  const int qy0 = (tile / p.tiles_x) * p.QH, qx0 = (tile % p.tiles_x) * p.QW;

  // ---- this CTA's jobs and memory entries
  fgvc_tile_group tg;
  int e_lo, e_hi, og = 0;
  // window mode: this CTA's job, memory entry (position in the job's list), chunk of the entry's boxes, and the
  // job's arg-max table, floors and lists -- from the job table when the launch has several jobs
  fgvc_job wjob = p.job;
  int went = blockIdx.y, wchunk = blockIdx.z, wchunks = p.chunks;
  const int32_t* wbest = p.best;
  const float* wfloor = p.floor;
  float* wtv = p.tv;
  int32_t* wti = p.ti;
  if (WIN && p.wjobs != nullptr) {
    int lo = 0, hi = p.n_wjobs - 1;
    while (lo < hi) {                                        // last job with y_begin <= blockIdx.y
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(&p.wjobs[mid].y_begin) <= (int)blockIdx.y) lo = mid; else hi = mid - 1;
    }
    const c2f_wjob& wj = p.wjobs[lo];
    wjob = wj.job;
    wchunks = wj.chunks;
    went = ((int)blockIdx.y - wj.y_begin) / wchunks;
    wchunk = ((int)blockIdx.y - wj.y_begin) - went * wchunks;
    wbest = p.best + wj.best_off;
    wfloor = p.floor != nullptr ? p.floor + wj.floor_off : nullptr;
    wtv = p.tv + wj.list_off;
    wti = p.ti + wj.list_off;
  }
  if (WIN) {
    tg.job[0] = 0; tg.n_jobs = 1;
    e_lo = wjob.mem_begin + went; e_hi = e_lo + 1;
  } else {
    if (p.tgroups) {
      // heaviest groups first: in clip order the late jobs have the longest memory lists, and a launch that ends
      // with its longest CTAs pays for them in the tail
      tg = p.tgroups[gridDim.z - 1 - blockIdx.z];
    } else {
      const fgvc_job job = p.jobs[blockIdx.z];
      tg.job[0] = blockIdx.z; tg.job[1] = tg.job[2] = tg.job[3] = -1;
      tg.n_jobs = 1; tg.u_begin = job.mem_begin; tg.u_end = job.mem_end; tg.out_group = 0;
    }
    const int n_mem = tg.u_end - tg.u_begin;
    const int per = (n_mem + p.split - 1) / p.split;
    e_lo = tg.u_begin + blockIdx.y * per;
    e_hi = min(tg.u_end, e_lo + per);
    og = tg.out_group * p.split + blockIdx.y;
  }
  const int nq_c = WIN ? p.HQ * p.WQ : 0;
  const int qH = WIN ? p.HQ : p.H, qW = WIN ? p.WQ : p.W;       // query grid

  if (!WIN && e_lo >= e_hi) {
    // This (tile group, part) has no memory entry (more parts than entries).  Uniform over the CTA pair and before
    // any barrier / tensor-memory allocation: write the empty lists and leave.
    if (threadIdx.x < 128) {
      const int R = (int)rank * 128 + (int)threadIdx.x;
      const int jm = R >> p.lpj_shift, rm = R & ((1 << p.lpj_shift) - 1);
      const int jb = jm < tg.n_jobs ? tg.job[jm] : -1;
      const int qy = qy0 + (rm >> p.qw_shift), qx = qx0 + (rm & (p.QW - 1));
      if (jb >= 0 && qy < p.H && qx < p.W) {
        const int64_t o = (((int64_t)jb * p.lists_per_job + og) * p.n_pix + qy * p.W + qx) * p.k_out;
        for (int i = 0; i < p.k_out; ++i) { p.tv[o + i] = -INFINITY; p.ti[o + i] = -1; }
      }
    }
    return;
  }

  const int NC = 16 * p.BH / NCTA;             // keys of a box staged by this CTA
  const int N = 16 * p.BH;                     // keys of a box = accumulator columns
  // The MMA warp may run n_acc - 1 boxes ahead of the epilogue's loads: the scan time of a box varies a lot (list
  // insertions), and with only two tiles both sides kept waiting for each other (profiles/r2_b_epilogue.md)
  const int n_acc = min(MAX_ACC, 256 / N);
  const uint32_t acc_cols = 256u / (uint32_t)n_acc;
  const int n_kc = p.C / 64;
  // one stage = this CTA's part of one whole key box (all C channels: n_kc chunks of [hi rows ; lo rows] x 128 B),
  // so the single issuing threads pay one barrier round trip per box instead of one per 64 channels
  const int chunk_bytes = 2 * NC * 128;
  const int stage_bytes = n_kc * chunk_bytes;
  const int n_stages = min(MAX_STAGES, RING_BYTES / stage_bytes);
  const uint32_t stage_tx = (uint32_t)(NCTA * stage_bytes);      // bytes that complete on the leader's barrier

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_k) : "memory");
    for (int s = 0; s < n_stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    for (int b = 0; b < MAX_ACC; ++b) { mbar_init(tfull_bar + b, 1); mbar_init(tempty_bar + b, 4 * EPI_WG * NCTA); }
    mbar_init(a_bar, 4 * EPI_WG * NCTA);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    if (NCTA == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
  }
  // half width of the mask at row distance d (d = 0 .. reach), -1 beyond (one sentinel entry)
  if constexpr (WIN) {
    for (int d = threadIdx.x; d <= p.rf + 1; d += THREADS) halfw[d] = d <= p.rf ? p.rf : -1;
  } else {
    for (int d = threadIdx.x; d <= p.reach + 1; d += THREADS) {
      int hw = -1;
      if (d <= p.reach) {
        if (p.mode == FGVC_MASK_CIRCLE) {
          while (hw + 1 <= p.reach && (hw + 1) * (hw + 1) + d * d < p.radius * p.radius) ++hw;
        } else {
          hw = p.radius;
        }
      }
      halfw[d] = hw;
    }
  }
  if constexpr (!WIN) {
    if (warp == 2 || warp == 3) {          // one warp per list
      const int li = warp - 2;
      const Walk w = make_walk(p, li ? FGVC_MEM_UNMASKED : 0, qy0, qx0);
      const int ncols = (w.x_hi - w.x_lo) / 16 + 1, nrows = (w.y_hi - w.y_lo) / p.BH + 1;
      uint32_t* list = boxes + li * MAX_BOXES;
      int cnt = 0;
      for (int base = 0; base < nrows * ncols; base += 32) {
        const int i = base + lane;
        const int by = w.y_lo + (i / ncols) * p.BH, bx = w.x_lo + (i % ncols) * 16;
        const bool keep = i < nrows * ncols && !box_skipped(p, w, by, bx, qy0, qx0);
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        const int pos = cnt + __popc(bal & ((1u << lane) - 1u));
        if (keep && pos < MAX_BOXES) list[pos] = (uint32_t)by | ((uint32_t)bx << 16);
        cnt += __popc(bal);
      }
      cnt = min(cnt, MAX_BOXES);
      __syncwarp();
      // Centre-out order for the halo list: the best matches of a query sit near its own position, so
      // walking the boxes nearest to the tile first raises the running K-th values early and the
      // (divergent, ~80-instruction) list insertions become rare.  Rank sort, n is a few dozen.
      if (li == 0 && cnt > 1 && cnt <= 128) {
        const int cy2 = 2 * qy0 + p.QH, cx2 = 2 * qx0 + p.QW;          // twice the tile centre
        uint32_t mine[4]; int rnk[4];
        for (int t = 0; t < 4; ++t) {
          const int i = lane + 32 * t;
          mine[t] = i < cnt ? list[i] : 0u;
          rnk[t] = 0;
        }
        for (int j = 0; j < cnt; ++j) {
          const uint32_t o = list[j];
          const int oy = 2 * (int)(o & 0xffffu) + p.BH - cy2, ox = 2 * (int)(o >> 16) + 16 - cx2;
          const int od = oy * oy + ox * ox;
          for (int t = 0; t < 4; ++t) {
            const int i = lane + 32 * t;
            const int my = 2 * (int)(mine[t] & 0xffffu) + p.BH - cy2, mx = 2 * (int)(mine[t] >> 16) + 16 - cx2;
            const int md = my * my + mx * mx;
            rnk[t] += (od < md || (od == md && j < i)) ? 1 : 0;
          }
        }
        __syncwarp();
        for (int t = 0; t < 4; ++t)
          if (lane + 32 * t < cnt) list[rnk[t]] = mine[t];
      }
      if (lane == 0) nbox[li] = cnt;
    }
  } else if (warp >= 2 && warp < 6) {
    // ---- window mode: bounding rectangle of the tile's window centres in this CTA's memory entry (lane = query)
    int* rect = halfw + 132;                                // (the table above holds <= 130 entries)
    const int m = (warp - 2) * 32 + lane;
    const int qy = qy0 + (m >> p.qw_shift), qx = qx0 + (m & (p.QW - 1));
    const bool qvalid = qy < p.HQ && qx < p.WQ;
    int cy_lo = 1 << 30, cy_hi = -1, cx_lo = 1 << 30, cx_hi = -1;
    int my_cy = 0, my_cx = 0;
    if (qvalid) {
      const int b = max(__ldg(wbest + (int64_t)went * nq_c + qy * p.WQ + qx), 0) % nq_c;
      my_cy = cy_lo = cy_hi = (b / p.WQ) * p.scale;
      my_cx = cx_lo = cx_hi = (b % p.WQ) * p.scale;
    }
    cy_lo = __reduce_min_sync(0xffffffffu, cy_lo); cy_hi = __reduce_max_sync(0xffffffffu, cy_hi);
    cx_lo = __reduce_min_sync(0xffffffffu, cx_lo); cx_hi = __reduce_max_sync(0xffffffffu, cx_hi);
    if (warp == 2 && lane < 4) rect[lane] = lane == 0 ? cy_lo : (lane == 1 ? cy_hi : (lane == 2 ? cx_lo : cx_hi));
    asm volatile("bar.sync 2, 128;" ::: "memory");
    if (warp != 2 && lane == 0) {
      atomicMin(rect + 0, cy_lo); atomicMax(rect + 1, cy_hi);
      atomicMin(rect + 2, cx_lo); atomicMax(rect + 3, cx_hi);
    }
    asm volatile("bar.sync 2, 128;" ::: "memory");
    // The boxes of the rectangle grown by rf, clipped to the map -- minus those no window of the tile touches (a few
    // far-away arg-max keys stretch the rectangle over most of the frame): every lane marks the boxes of its own
    // window in a bitmap (scratch: the start of the ring, idle until the producer starts), warp 2 lists this CTA's
    // chunk of the marked boxes.
    uint32_t* cover = reinterpret_cast<uint32_t*>(ring);
    int cnt = 0;
    if (rect[1] >= 0) {                                         // (else: no valid query in the tile)
      const int y_lo = max(0, rect[0] - p.rf), y_hi = min(p.H - 1, rect[1] + p.rf);
      const int x_lo = max(0, rect[2] - p.rf), x_hi = min(p.W - 1, rect[3] + p.rf);
      const int ncols = (x_hi - x_lo) / 16 + 1, nrows = (y_hi - y_lo) / p.BH + 1;
      const int total = nrows * ncols, words = (total + 31) / 32;
      for (int i = m; i < words; i += 128) cover[i] = 0u;
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (qvalid) {
        const int r0 = (max(my_cy - p.rf, 0) - y_lo) >> p.bh_shift, r1 = (min(my_cy + p.rf, p.H - 1) - y_lo) >> p.bh_shift;
        const int c0 = (max(my_cx - p.rf, 0) - x_lo) >> 4, c1 = (min(my_cx + p.rf, p.W - 1) - x_lo) >> 4;
        for (int r = r0; r <= r1; ++r)
          for (int c = c0; c <= c1; ++c) {
            const int i = r * ncols + c;
            atomicOr(cover + (i >> 5), 1u << (i & 31));
          }
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (warp == 2) {
        int kept = 0;
        for (int i = lane; i < words; i += 32) kept += __popc(cover[i]);
        kept = __reduce_add_sync(0xffffffffu, kept);
        const int k_lo = (int)((int64_t)kept * wchunk / wchunks), k_hi = (int)((int64_t)kept * (wchunk + 1) / wchunks);
        int seen = 0;
        for (int base = 0; base < total; base += 32) {
          const int i = base + lane;
          const bool keep = i < total && ((cover[i >> 5] >> (i & 31)) & 1u);
          const uint32_t bal = __ballot_sync(0xffffffffu, keep);
          const int pos = seen + __popc(bal & ((1u << lane) - 1u));
          if (keep && pos >= k_lo && pos < k_hi && pos - k_lo < 2 * MAX_BOXES) {
            const int by = y_lo + (i / ncols) * p.BH, bx = x_lo + (i % ncols) * 16;
            boxes[pos - k_lo] = (uint32_t)by | ((uint32_t)bx << 16);
          }
          seen += __popc(bal);
        }
        cnt = min(k_hi - k_lo, 2 * MAX_BOXES);
      }
    }
    if (warp == 2 && lane == 0) { nbox[0] = cnt; nbox[1] = 0; }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic accesses to the ring before the TMA writes
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    // ================================ TMA producer ====================================
    // one elected lane runs the whole loop (the compiler then keeps everything in uniform registers)
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const int n_ld = (p.exp_flags & 4) ? max(1, n_kc / 2) : n_kc;     // experiment: half the L2 -> SM bytes
      const int row_off = (int)rank * (p.BH / NCTA);                     // this CTA's key rows of a box
      for (int e = e_hi - 1; e >= e_lo; --e) {       // newest memory frame first: thresholds rise early
        const int raw = p.ent[e];
        const int slot = raw & ~FGVC_MEM_UNMASKED;
        const int li = (!WIN && (raw & FGVC_MEM_UNMASKED)) ? 1 : 0;
        const int nb = nbox[li];
        for (int b = 0; b < nb; ++b) {
          const uint32_t bb = boxes[li * MAX_BOXES + b];
          const int by = (int)(bb & 0xffffu), bx = (int)(bb >> 16);
          mbar_wait(empty_bar + stage, phase ^ 1);
          const uint32_t fb = NCTA == 2 ? map_to_rank(smem_u32(full_bar + stage), 0) : smem_u32(full_bar + stage);
          if (rank == 0) mbar_expect_tx(full_bar + stage, stage_tx / n_kc * n_ld);
          // per 64-channel chunk one TMA box = (64 channels, 16 x BH/NCTA pixels, both parts): hi rows then lo rows
          for (int kc = 0; kc < n_ld; ++kc)
            tma_box<NCTA>(&tmap_k, fb, ring + stage * stage_bytes + kc * chunk_bytes, kc * 64, bx, by + row_off, 0, slot);
          if (++stage == n_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================= MMA issuer (leader CTA of the pair) =====================================
    if (rank == 0) {
      mbar_wait(a_bar, 0);
      tc_fence_after();
      int n_total = 0;                                 // boxes this CTA processes
      for (int e = e_lo; e < e_hi; ++e) n_total += nbox[(!WIN && (p.ent[e] & FGVC_MEM_UNMASKED)) ? 1 : 0];
      if (elect_one()) {
        const uint32_t idesc = make_idesc_f16(128 * NCTA, N);
        int stage = 0, buf = 0;
        uint32_t phase = 0, tpar = 0;                  // tpar: bit b = parity of accumulator b's next "drained" phase
        const uint32_t ring_u32 = smem_u32(ring);
        const uint64_t desc_hi = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61) | ((uint64_t)1 << 16);
        const uint64_t lo_off = (uint64_t)((NC * 128) >> 4);           // lo rows follow the hi rows of a chunk
        // The barrier probes of box it+1 are issued while the last MMAs of box it are still queued in
        // the tensor pipe, so the pipe does not drain during the ~100-cycle try_wait round trips.
        if (n_total > 0) {
          mbar_wait(tempty_bar + 0, 1);
          mbar_wait(full_bar + 0, phase);
          tc_fence_after();
        }
        for (int it = 0; it < n_total; ++it) {
          const uint32_t d_tmem = tmem_base + (uint32_t)buf * acc_cols;
          const uint32_t sa = ring_u32 + (uint32_t)(stage * stage_bytes);
          for (int kc = 0; kc < n_kc; ++kc) {
            const uint64_t b = desc_hi | (uint64_t)((sa + (uint32_t)(kc * chunk_bytes)) >> 4);
            const uint32_t a_hi = tmem_base + AHI_COL + kc * 32, a_lo = tmem_base + ALO_COL + kc * 32;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {       // 4 x (K = 16 fp16 = 32 B) per 128 B swizzle row
              if (ks == 3 && kc == n_kc - 1) break;  // the last K step is issued after the probes below
              const uint64_t o = (uint64_t)(ks * 2);
              umma_f16_ts<NCTA>(d_tmem, a_hi + ks * 8, b + o, idesc, (kc | ks) != 0);     // hi*hi
              umma_f16_ts<NCTA>(d_tmem, a_hi + ks * 8, b + lo_off + o, idesc, 1);         // hi*lo
              umma_f16_ts<NCTA>(d_tmem, a_lo + ks * 8, b + o, idesc, 1);                  // lo*hi
            }
          }
          const int nstage = (stage + 1 == n_stages) ? 0 : stage + 1;
          const uint32_t nphase = phase ^ (nstage == 0 ? 1u : 0u);
          const int nbuf = (buf + 1 == n_acc) ? 0 : buf + 1;
          tpar ^= 1u << buf;                              // this tile's next drain completes the following phase
          if (it + 1 < n_total) {
            mbar_wait(tempty_bar + nbuf, ((tpar >> nbuf) & 1u) ^ 1u);       // epilogue drained the next accumulator
            mbar_wait(full_bar + nstage, nphase);                           // next key box landed
            tc_fence_after();
          }
          {
            const int kc = n_kc - 1;
            const uint64_t b = desc_hi | (uint64_t)((sa + (uint32_t)(kc * chunk_bytes)) >> 4);
            const uint32_t a_hi = tmem_base + AHI_COL + kc * 32 + 24, a_lo = tmem_base + ALO_COL + kc * 32 + 24;
            umma_f16_ts<NCTA>(d_tmem, a_hi, b + 6, idesc, 1);
            umma_f16_ts<NCTA>(d_tmem, a_hi, b + lo_off + 6, idesc, 1);
            umma_f16_ts<NCTA>(d_tmem, a_lo, b + 6, idesc, 1);
          }
          umma_commit_all<NCTA>(empty_bar + stage);     // smem stage free (in both CTAs) once these MMAs retire
          umma_commit_all<NCTA>(tfull_bar + buf);       // accumulator complete
          buf = nbuf; stage = nstage; phase = nphase;
        }
      }
    }
    __syncwarp();
  } else {
    // ================================== epilogue ======================================
    const int wg = (warp - 2) >> 2;
    const int lg = warp & 3;
    const int m = lg * 32 + lane;
    const int R = (int)rank * 128 + m;                      // row of the (pair's) tile
    const int jm = R >> p.lpj_shift;                        // which job of the group this lane (this whole warp) serves
    const int rm = R & ((1 << p.lpj_shift) - 1);            // pixel of the block
    const int jb = WIN ? 0 : (jm < tg.n_jobs ? tg.job[jm] : -1);
    const int qy = qy0 + (rm >> p.qw_shift), qx = qx0 + (rm & (p.QW - 1));
    const bool qvalid = jb >= 0 && qy < qH && qx < qW;
    const uint32_t tempty_leader = NCTA == 2 ? map_to_rank(smem_u32(tempty_bar), 0) : 0u;   // the leader's barriers
    {
      // both query parts -> tensor memory, two fp16 channels per 32-bit cell (lower channel in the low half).  The four
      // warps that share a TMEM lane quarter split the channels: 16 cells (64 B of the row) per tcgen05.st.
      // Window mode: the row is the FINE query feature at (scale * qy, scale * qx)   (local_attention.py:785)
      const int q_slot = WIN ? wjob.q_slot : (jb >= 0 ? p.jobs[jb].q_slot : 0);
      const int qpix = !qvalid ? 0 : (WIN ? (qy * p.scale) * p.W + qx * p.scale : qy * p.W + qx);
      const int64_t part = (int64_t)p.n_pix * p.C;
      const __half* row = bank + (int64_t)q_slot * 2 * part + (int64_t)qpix * p.C;
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      const int n_c16 = p.C / 32;                          // 16-cell groups per part
      for (int i = wg; i < 2 * n_c16; i += EPI_WG) {
        const int prt = i >= n_c16 ? 1 : 0, c = (i - prt * n_c16) * 16;
        const uint4* src = reinterpret_cast<const uint4*>(row + prt * part) + c / 4;
        uint4 a = z, b = z, c4 = z, d = z;
        if (qvalid) { a = __ldg(src); b = __ldg(src + 1); c4 = __ldg(src + 2); d = __ldg(src + 3); }
        tmem_st16u(tmem_base + ((uint32_t)(lg * 32) << 16) + (prt ? ALO_COL : AHI_COL) + c, a, b, c4, d);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NCTA == 2) mbar_arrive_cluster(map_to_rank(smem_u32(a_bar), 0)); else mbar_arrive(a_bar);
      }
    }
    TopK<K> top;
    top.init();
    volatile float* thr_mine = thr_sh + m * EPI_WG + wg;
    // every list of this query may start from a floor that K genuine candidates are known to reach (the caller's
    // guarantee): [coarse query] in window mode, [job][query pixel] otherwise
    *thr_mine = (wfloor != nullptr && qvalid)
                    ? __ldg(wfloor + (WIN ? (int64_t)qy * p.WQ + qx : (int64_t)jb * p.n_pix + qy * p.W + qx))
                    : -INFINITY;
    asm volatile("bar.sync 1, %0;" ::"n"(128 * EPI_WG) : "memory");
    // Warpgroup wg owns the key rows wg (and wg + 4 when a box has 8 rows) of every box: a static assignment, so the
    // order in which a query's candidates reach its lists -- and with it the choice among exactly tied values -- does
    // not depend on timing.  (Drawing row tickets from a shared counter balanced the warps a little better, 7.35 ->
    // 7.09 ms on the bench clip, but made tied results vary from run to run: profiles/r2_b_epilogue.md.)
    const int hw_n = WIN ? p.rf : p.reach;                 // halfw[0 .. hw_n], halfw[hw_n + 1] = -1
    const uint32_t lane_base = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(wg * 16);
    int n_total = 0;                                       // boxes of this CTA
    for (int e = e_lo; e < e_hi; ++e) n_total += nbox[(!WIN && (p.ent[e] & FGVC_MEM_UNMASKED)) ? 1 : 0];
    auto run = [&](auto rows_c) {
      constexpr int ROWS = decltype(rows_c)::value;        // key rows of a box per thread
      uint32_t buf = 0, tpar = 0, seq = 0;                 // accumulator of the next box; bit b = parity of its "full" phase
      bool in_flight = false;                              // the rows of box `seq` were requested by the previous box
      // The rows of box i+1 are requested from tensor memory BEFORE box i is scanned (when its accumulator is already
      // complete), into the other of two register sets: the ~100s of cycles of tcgen05.ld latency and the barrier
      // round trip then overlap the scan instead of heading every box (profiles/r2_b_epilogue.md: long-scoreboard
      // and fixed-latency waits dominated the epilogue's stalls at ~4.5 warps per scheduler).
      constexpr bool PREFETCH = ROWS <= 2;                 // (4 rows x 2 sets would not fit the register budget)
      uint32_t ra[ROWS][16], rb[PREFETCH ? ROWS : 1][16];
      auto issue_rows = [&](uint32_t b_, uint32_t (&r)[ROWS][16]) {
        const uint32_t taddr = lane_base + b_ * acc_cols;
#pragma unroll
        for (int rr = 0; rr < ROWS; ++rr) tmem_ld16_issue(taddr + 16 * EPI_WG * rr, r[rr]);
      };
      (void)issue_rows;
      auto box = [&](uint32_t (&rc)[ROWS][16], uint32_t (&rn)[PREFETCH ? ROWS : 1][16], int e, int by, int bx,
                     bool masked, bool mine, int pos_base, int cy, int cx) {
        // 16-bit interval masks of the in-mask, in-image keys of this thread's key rows: the half width at
        // |ky - cy| comes from the table (-1 = row out of reach; unmasked entries: the whole row)
        uint32_t bits[ROWS];
        bool hot[ROWS];
        const bool dump = !WIN && p.dbg != nullptr && (int)seq < p.dbg_max_boxes;
        // per box: the lane's centre relative to the box, the last in-image column of the box, the rows of the box
        // that exist (in the box and in the image).  With bx >= 0: max(max(cx - hw, 0) - bx, 0) = max(cx - bx - hw, 0),
        // and a sentinel half width of -1 gives hi < lo by itself.
        const int cbx = cx - bx, wlim = min(p.W - 1 - bx, 15), rows_ok = min(p.BH, p.H - by), dy0 = by + wg - cy;
#pragma unroll
        for (int rr = 0; rr < ROWS; ++rr) {
          const int row = wg + EPI_WG * rr;
          int hw = p.W;
          if (masked) hw = halfw[min(abs(dy0 + EPI_WG * rr), hw_n + 1)];
          const int lo = max(cbx - hw, 0);
          const int hi = min(cbx + hw, wlim);
          const bool ok = row < rows_ok;                                    // warp-uniform
          bits[rr] = (ok && mine && hi >= lo) ? ((2u << hi) - (1u << lo)) : 0u;
          hot[rr] = ok && (__any_sync(0xffffffffu, bits[rr] != 0) || dump);    // warp-uniform
        }
        if (!in_flight) {
          mbar_wait_sleep(tfull_bar + buf, (tpar >> buf) & 1u);
          tc_fence_after();
          issue_rows(buf, rc);
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int rr = 0; rr < ROWS; ++rr) reg_fence16(rc[rr]);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {                                   // accumulator is in registers: hand the tile back
          if (NCTA == 2) mbar_arrive_cluster(tempty_leader + 8u * buf); else mbar_arrive(tempty_bar + buf);
        }
        if (dump) {
#pragma unroll
          for (int rr = 0; rr < ROWS; ++rr) {
            if (!hot[rr]) continue;
            const int row = wg + EPI_WG * rr;
            float* d = p.dbg + ((int64_t)seq * 128 + m) * 128 + row * 16;
#pragma unroll
            for (int j = 0; j < 16; ++j) d[j] = __uint_as_float(rc[rr][j]) * FGVC_F16_ACC_INV;
            if (p.dbg_meta != nullptr && m == 0 && row == 0) {
              p.dbg_meta[4 * seq + 0] = e; p.dbg_meta[4 * seq + 1] = by;
              p.dbg_meta[4 * seq + 2] = bx; p.dbg_meta[4 * seq + 3] = N;
            }
          }
        }
        tpar ^= 1u << buf;
        buf = (buf + 1 == (uint32_t)n_acc) ? 0u : buf + 1;
        ++seq;
        // request the next box's rows now if its accumulator is already complete (non-blocking probe)
        in_flight = false;
        if constexpr (PREFETCH) {
          if ((int)seq < n_total && mbar_test_wait(tfull_bar + buf, (tpar >> buf) & 1u)) {
            tc_fence_after();
            issue_rows(buf, rn);
            in_flight = true;
          }
        }
        if (p.exp_flags & 1) return;
        // The K-th value of ANY partial list of this query bounds the final K-th value from below, so no list
        // needs candidates under the largest of them: the warpgroups publish theirs when it changes (a stale value
        // is only a weaker bound).  Without this each of the lists climbs to the final threshold on its own.
        float floor_ = -INFINITY;
        if (!(p.exp_flags & 8)) {
#pragma unroll
          for (int w2 = 0; w2 < EPI_WG; ++w2) floor_ = fmaxf(floor_, thr_mine[w2 - wg]);
        }
        const float thr_before = top.thr();
        const int kbase = pos_base + (by + wg) * p.W + bx;
#pragma unroll
        for (int rr = 0; rr < ROWS; ++rr)
          if (hot[rr]) scan_row<K>(rc[rr], bits[rr], top, kbase + EPI_WG * rr * p.W, floor_, p.exp_flags & 16);
        if (top.thr() != thr_before) *thr_mine = top.thr();
      };
      bool flip = false;
      for (int e = e_hi - 1; e >= e_lo; --e) {           // newest memory frame first: thresholds rise early
        const int raw = p.ent[e];
        const bool masked = WIN || !(raw & FGVC_MEM_UNMASKED);
        const int li = masked ? 0 : 1;
        const int nb = nbox[li];
        const uint32_t* blist = boxes + li * MAX_BOXES;
        int upos_e, cy = qy, cx = qx;
        if constexpr (WIN) {
          upos_e = qvalid ? e - wjob.mem_begin : -1;
          // this lane's window centre in this memory entry: scale * (coarse arg-max key)   (local_attention.py:835-845)
          if (qvalid) {
            const int bq = max(__ldg(wbest + (int64_t)(e - wjob.mem_begin) * nq_c + qy * p.WQ + qx), 0) % nq_c;
            cy = (bq / p.WQ) * p.scale;
            cx = (bq % p.WQ) * p.scale;
          }
        } else if (p.tgroups) {
          upos_e = qvalid ? p.upos[4 * e + jm] : -1;     // warp-uniform up to the image border
        } else {
          upos_e = qvalid ? e - tg.u_begin : -1;
        }
        const bool mine = upos_e >= 0;                     // does this lane's job have this memory entry at all?
        const int pos_base = upos_e * p.n_pix;
        for (int b = 0; b < nb; ++b) {
          const uint32_t bb = blist[b];
          const int by = (int)(bb & 0xffffu), bx = (int)(bb >> 16);
          if constexpr (PREFETCH) {
            if (flip) box(rb, ra, e, by, bx, masked, mine, pos_base, cy, cx);
            else box(ra, rb, e, by, bx, masked, mine, pos_base, cy, cx);
            flip = !flip;
          } else {
            box(ra, rb, e, by, bx, masked, mine, pos_base, cy, cx);
          }
        }
      }
    };
    if (p.BH <= EPI_WG) run(std::integral_constant<int, 1>{});
    else if (p.BH <= 2 * EPI_WG) run(std::integral_constant<int, 2>{});
    else run(std::integral_constant<int, 4>{});
    // ---- merge the partial lists of the warpgroups through the (now idle) ring
    asm volatile("bar.sync 1, %0;" ::"n"(128 * EPI_WG) : "memory");
    float* mv = reinterpret_cast<float*>(ring);
    int* mi = reinterpret_cast<int*>(ring + EPI_WG * 128 * K * 4);
    if (wg > 0) {
#pragma unroll
      for (int i = 0; i < K; ++i) { mv[(wg * 128 + m) * K + i] = top.v[i]; mi[(wg * 128 + m) * K + i] = top.id[i]; }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(128 * EPI_WG) : "memory");
    if (wg == 0 && qvalid) {
      for (int w2 = 1; w2 < EPI_WG; ++w2)
        for (int i = 0; i < K; ++i) {
          const float v = mv[(w2 * 128 + m) * K + i];
          if (!(v > top.thr())) break;
          top.push(v, mi[(w2 * 128 + m) * K + i]);
        }
      const int q = qy * qW + qx;
      int64_t o;
      if (WIN) o = ((int64_t)q * ((wjob.mem_end - wjob.mem_begin) * wchunks) + (went * wchunks + wchunk)) * p.k_out;
      else o = (((int64_t)jb * p.lists_per_job + og) * p.n_pix + q) * p.k_out;
#pragma unroll
      for (int i = 0; i < K; ++i)
        if (i < p.k_out) { wtv[o + i] = top.v[i] * FGVC_F16_ACC_INV; wti[o + i] = top.id[i]; }
    }
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (NCTA == 1)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// ------------------------------------------------------------------------------ host
// 5-D map over feat16[slot][part][H][W][C]; box = (64 channels, 16, rows per CTA, both parts, 1), 128B swizzle
static int make_map16(CUtensorMap* map, const void* bank, int n_slots, int H, int W, int C, int rows) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return FGVC_ERR_CUDA;
  }
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, 2, (cuuint64_t)n_slots};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                           (cuuint64_t)2 * H * W * C * 2};
  cuuint32_t box[5] = {64, 16, (cuuint32_t)rows, 2, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(bank), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (f16) failed with %d (H=%d W=%d C=%d rows=%d)", (int)r, H, W, C, rows);
    return FGVC_ERR_CUDA;
  }
  return FGVC_OK;
}

// all MMAs are TS-form: a box costs ~N plus a small fixed hand-shake.  Pair tiles stage BH / 2 rows per CTA: BH even.
static int box_cost16(int rows, int bh) { return cdiv(rows, bh) * (16 * bh + 24); }
static int pick_bh16(int rows, int ncta) {
  const int max_bh = MAX_NC / 16 * ncta;       // powers of two: the epilogue splits row tickets with a shift
  int best = max_bh;
  for (int bh = max_bh / 2; bh >= ncta; bh /= 2)
    if (box_cost16(rows, bh) < box_cost16(rows, best)) best = bh;
  return best;
}

template <int K, int NCTA, bool WIN>
static int launch_k(const CUtensorMap& mk, const void* bank, const Params& p, dim3 grid, cudaStream_t st) {
  auto kern = affinity_topk_tc16_kernel<K, NCTA, WIN>;
  FGVC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(THREADS, 1, 1);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  FGVC_CUDA(cudaLaunchKernelEx(&cfg, kern, mk, reinterpret_cast<const __half*>(bank), p));
  FGVC_LAUNCH_CHECK();
#ifdef FGVC_TC16_STATS
  if (p.exp_flags & 16) {      // experiment: print and reset the scan counters (synchronises!)
    unsigned long long h[8] = {0};
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(h, g_stats, sizeof(h));
    fprintf(stderr, "[tc16 stats] grid=(%u,%u,%u) row_scans=%llu hot_rows=%llu rounds=%llu pushes=%llu\n", grid.x, grid.y,
            grid.z, h[0], h[1], h[2], h[3]);
    unsigned long long z[8] = {0};
    cudaMemcpyToSymbol(g_stats, z, sizeof(z));
  }
#endif
  return FGVC_OK;
}
template <int NCTA, bool WIN>
static int launch_by_k(const CUtensorMap& mk, const void* bank, const Params& p, dim3 grid, int K, cudaStream_t st) {
  if (K <= 4) return launch_k<4, NCTA, WIN>(mk, bank, p, grid, st);
  if (K <= 10) return launch_k<10, NCTA, WIN>(mk, bank, p, grid, st);
  return launch_k<16, NCTA, WIN>(mk, bank, p, grid, st);
}

// pixel block of one job for `rows_per_job` tile rows: as square as the count allows, orientation by halo cost
static void block_shape(int H, int W, int reach, int rows_per_job, int ncta, int* QH, int* QW, int* BH) {
  auto halo_cost = [&](int qh, int qw) {
    int rows = min(H, qh + 2 * reach), cols = min(W, qw + 2 * reach);
    double tiles = (double)cdiv(H, qh) * cdiv(W, qw);
    return tiles * box_cost16(rows, pick_bh16(rows, ncta)) * cdiv(cols, 16);
  };
  int a = 16, b = 16;
  switch (rows_per_job) {
    case 256: a = 16; b = 16; break;
    case 128: a = 16; b = 8; break;
    case 64: a = 8; b = 8; break;
    default: a = 8; b = 4; break;      // 32
  }
  if (a != b && halo_cost(b, a) < halo_cost(a, b)) { int t = a; a = b; b = t; }
  *QH = a; *QW = b;
  *BH = pick_bh16(min(H, a + 2 * reach), ncta);
}

static int ilog2(int v) { int s = 0; while ((1 << s) < v) ++s; return s; }

}  // namespace tc16

bool tc16_supported(int H, int W, int C, int K) {
  return C % 64 == 0 && C >= 64 && C <= 256 && K >= 1 && K <= 16 && H >= 1 && W >= 1;
}

// CTA pairs (cta_group::2) halve the L2 -> shared-memory bytes per MAC, but a 256-row tile has a larger pixel block
// per job and so a larger halo (bench clip: 2.82x the in-mask pairs against 2.41x for single-CTA tiles).  Measured
// (profiles/r2_b_epilogue.md) K1 is bound by the epilogue's candidate scan, not by the L2 fabric, so pairs do not pay
// yet: they are built and tested, and selected with FGVC_TC16_PAIR=1.
static bool use_pairs(int H, int W, int jobs_per_tile) {
  const int force = getenv("FGVC_TC16_PAIR") ? atoi(getenv("FGVC_TC16_PAIR")) : -1;   // experiments / tests
  (void)jobs_per_tile; (void)W;
  return force == 1 && H >= 2;
}

// tile = jobs_per_tile jobs x (128 * ncta / jobs_per_tile) pixels.  Exposed so that the host can cost the packings
// before building the tables.
void packed_tile_shape(int H, int W, int reach, int jobs_per_tile, int* QH, int* QW, int* BH, int* ncta_out) {
  const int ncta = use_pairs(H, W, jobs_per_tile) ? 2 : 1;
  tc16::block_shape(H, W, reach, 128 * ncta / jobs_per_tile, ncta, QH, QW, BH);
  if (ncta_out) *ncta_out = ncta;
}

static int launch_k1(const void* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs, int n_z,
                     const fgvc_tile_group* tgroups, const int32_t* ent, const int32_t* upos, int jobs_per_tile,
                     int radius, int mode, int K, int lists_per_job, int split, float* tv, int32_t* ti, float* dbg,
                     int32_t* dbg_meta, int dbg_max_boxes, cudaStream_t st, const float* floor = nullptr) {
  using namespace tc16;
  Params p = {};
  p.floor = floor;
  p.H = H; p.W = W; p.C = C; p.n_pix = H * W;
  p.radius = radius; p.mode = mode; p.reach = mask_reach(radius, mode);
  int ncta = 1;
  packed_tile_shape(H, W, p.reach, jobs_per_tile, &p.QH, &p.QW, &p.BH, &ncta);
  if (dbg) {                    // the debug dump describes single-CTA tiles
    ncta = 1;
    block_shape(H, W, p.reach, 128 / jobs_per_tile, 1, &p.QH, &p.QW, &p.BH);
  }
  static const int force_bh = getenv("FGVC_TC16_BH") ? atoi(getenv("FGVC_TC16_BH")) : 0;   // timing experiments only
  if (force_bh >= ncta && force_bh <= MAX_NC / 16 * ncta && (force_bh & (force_bh - 1)) == 0) p.BH = force_bh;
  p.bh_shift = ilog2(p.BH);
  p.qw_shift = ilog2(p.QW);
  p.lpj_shift = ilog2(128 * ncta / jobs_per_tile);
  p.lists_per_job = lists_per_job; p.split = split; p.k_out = K;
  p.tiles_x = cdiv(W, p.QW);
  p.jobs = jobs; p.tgroups = tgroups; p.ent = ent; p.upos = upos; p.tv = tv; p.ti = ti;
  p.dbg = dbg; p.dbg_meta = dbg_meta; p.dbg_max_boxes = dbg_max_boxes;
  static const int exp_flags = getenv("FGVC_TC16_EXP") ? atoi(getenv("FGVC_TC16_EXP")) : 0;   // perf experiments only
  p.exp_flags = exp_flags;
  FGVC_CHECK_ARG(p.reach + 1 <= 128, "tcgen05 f16 engine: radius %d too large", radius);
  if (cdiv(H, p.BH) * cdiv(W, 16) > MAX_BOXES || H >= 65536 || W >= 65536) {
    set_error("tcgen05 f16 engine: a %dx%d map has more than %d key boxes", H, W, MAX_BOXES);
    return FGVC_ERR_UNSUPPORTED;      // AUTO falls back to the CUDA-core engine
  }
  CUtensorMap mk;
  int rc = make_map16(&mk, bank, n_slots, H, W, C, p.BH / ncta);
  if (rc) return rc;
  dim3 grid(cdiv(H, p.QH) * p.tiles_x * ncta, split, n_z);
  if (ncta == 2) return launch_by_k<2, false>(mk, bank, p, grid, K, st);
  return launch_by_k<1, false>(mk, bank, p, grid, K, st);
}

int launch_affinity_topk_tc16(const void* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs, int n_jobs,
                              const int32_t* mem_feat, int radius, int mode, int K, int groups, float* tv, int32_t* ti,
                              float* dbg, int32_t* dbg_meta, int dbg_max_boxes, cudaStream_t st, const float* floor) {
  return launch_k1(bank, n_slots, H, W, C, jobs, n_jobs, nullptr, mem_feat, nullptr, 1, radius, mode, K, groups, groups,
                   tv, ti, dbg, dbg_meta, dbg_max_boxes, st, floor);
}

// A floor for the lists of every (job, query pixel): the K-th largest of the exactly scored 5 x 5 neighbourhood of the
// query's own position in ONE memory frame of the job (seed_slot[job], e.g. the previous frame), restricted to
// in-image, in-mask keys -- K genuine candidates of the job reach it.  For launches whose lists start cold and stay
// short (one list per (query frame, memory frame) pair, shared between the point groups of a clip): without a floor
// half of such a launch is lock-step list insertion.  One warp per query pixel, 8 channels per lane, accumulator
// units (256 x affinity), the same three products as the MMA; -inf where fewer than K samples are valid.
__global__ void __launch_bounds__(256)
topk_floor_kernel(const __half* __restrict__ bank, int H, int W, int C, const fgvc_job* __restrict__ jobs,
                  const int32_t* __restrict__ seed_slot, int radius, int mode, int K, float* __restrict__ floor_out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_pix = H * W;
  const int q = blockIdx.x * 8 + warp;
  if (q >= n_pix) return;
  const int job = blockIdx.y;
  const int ss = __ldg(seed_slot + job);
  float* out = floor_out + (int64_t)job * n_pix + q;
  if (ss < 0) { if (lane == 0) *out = -INFINITY; return; }
  const int qy = q / W, qx = q - qy * W;
  const int64_t part = (int64_t)n_pix * C;
  const bool act = 8 * lane < C;
  float hq[8], lq[8];
  {
    const __half* row = bank + (int64_t)jobs[job].q_slot * 2 * part + (int64_t)q * C + 8 * lane;
    uint4 a = make_uint4(0u, 0u, 0u, 0u), b = a;
    if (act) { a = __ldg(reinterpret_cast<const uint4*>(row)); b = __ldg(reinterpret_cast<const uint4*>(row + part)); }
    const __half2* ah = reinterpret_cast<const __half2*>(&a);
    const __half2* bh = reinterpret_cast<const __half2*>(&b);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 x = __half22float2(ah[i]), y = __half22float2(bh[i]);
      hq[2 * i] = x.x; hq[2 * i + 1] = x.y; lq[2 * i] = y.x; lq[2 * i + 1] = y.y;
    }
  }
  float acc[32];
#pragma unroll
  for (int s = 0; s < 32; ++s) {
    acc[s] = 0.f;
    if (s >= 25) continue;
    const int py = qy + s / 5 - 2, px = qx + s % 5 - 2;
    if (py < 0 || py >= H || px < 0 || px >= W || !act) continue;          // (validity is applied after the reduction)
    const __half* row = bank + (int64_t)ss * 2 * part + ((int64_t)py * W + px) * C + 8 * lane;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(row)), b = __ldg(reinterpret_cast<const uint4*>(row + part));
    const __half2* ah = reinterpret_cast<const __half2*>(&a);
    const __half2* bh = reinterpret_cast<const __half2*>(&b);
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 hk = __half22float2(ah[i]), lk = __half22float2(bh[i]);
      t += hq[2 * i] * hk.x + hq[2 * i] * lk.x + lq[2 * i] * hk.x;
      t += hq[2 * i + 1] * hk.y + hq[2 * i + 1] * lk.y + lq[2 * i + 1] * hk.y;
    }
    acc[s] = t;
  }
  // transposing reduction: 31 shuffles; afterwards lane s holds the full sum of sample s in acc[0]
#pragma unroll
  for (int off = 16, n = 32; off >= 1; off >>= 1, n >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (i < n / 2) {
        const float send = upper ? acc[i] : acc[i + n / 2];
        const float keep = upper ? acc[i + n / 2] : acc[i];
        acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
  }
  float mine = -INFINITY;
  if (lane < 25) {
    const int dy = lane / 5 - 2, dx = lane % 5 - 2;
    const int py = qy + dy, px = qx + dx;
    const bool in_mask = mode == FGVC_MASK_CIRCLE ? dy * dy + dx * dx < radius * radius : (abs(dy) <= radius && abs(dx) <= radius);
    if (py >= 0 && py < H && px >= 0 && px < W && in_mask) mine = acc[0];
  }
  const int n_valid = __popc(__ballot_sync(0xffffffffu, mine > -INFINITY));
  int ahead = 0;
#pragma unroll
  for (int j = 0; j < 25; ++j) {
    const float u = __shfl_sync(0xffffffffu, mine, j);
    ahead += (u > mine || (u == mine && j < lane)) ? 1 : 0;
  }
  const uint32_t pick = __ballot_sync(0xffffffffu, lane < 25 && mine > -INFINITY && ahead == K - 1);
  float kth = -INFINITY;
  if (n_valid >= K && pick) kth = __shfl_sync(0xffffffffu, mine, __ffs(pick) - 1);
  if (kth > -INFINITY) kth -= 0.05f + 1e-5f * fabsf(kth);        // summation order of the MMA vs this loop
  if (lane == 0) *out = kth;
}

int launch_topk_floor16(const void* bank, int H, int W, int C, const fgvc_job* jobs, int n_jobs, const int32_t* seed_slot,
                        int radius, int mode, int K, float* floor_out, cudaStream_t st) {
  if (!tc16_supported(H, W, C, K)) {
    set_error("fgvc_topk_floor: needs the F16 bank with C %% 64 == 0, C <= 256 (C=%d)", C);
    return FGVC_ERR_UNSUPPORTED;
  }
  for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
    dim3 grid(cdiv(H * W, 8), min(65535, n_jobs - j0));
    topk_floor_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(bank), H, W, C, jobs + j0, seed_slot + j0, radius,
                                           mode, K, floor_out + (int64_t)j0 * H * W);
    FGVC_LAUNCH_CHECK();
  }
  return FGVC_OK;
}

int launch_affinity_topk_tc16_packed(const void* bank, int n_slots, int H, int W, int C, const fgvc_job* jobs,
                                     const fgvc_tile_group* tgroups, int n_tgroups, const int32_t* uent,
                                     const int32_t* upos, int jobs_per_tile, int radius, int mode, int K, int groups,
                                     int split, float* tv, int32_t* ti, cudaStream_t st) {
  FGVC_CHECK_ARG(jobs_per_tile == 1 || jobs_per_tile == 2 || jobs_per_tile == 4,
                 "packed tcgen05 engine: jobs_per_tile=%d must be 1, 2 or 4", jobs_per_tile);
  FGVC_CHECK_ARG(split >= 1 && groups % split == 0, "packed tcgen05 engine: groups=%d is not a multiple of split=%d",
                 groups, split);
  return launch_k1(bank, n_slots, H, W, C, jobs, n_tgroups, tgroups, uent, upos, jobs_per_tile, radius, mode, K, groups,
                   split, tv, ti, nullptr, nullptr, 0, st);
}

// ------------------------------------------------------------------------------ window mode (K2 fine stage)
// masked_attention_efficient_c2f (local_attention.py:721-880): every coarse query looks, in every memory frame, at
// the (2 rf + 1)^2 window of the FINE key map centred at scale * (coarse arg-max key) -- a data-dependent centre per
// (query, frame).  Same engine with three changes of geometry: a tile = 128 COARSE queries whose operand rows are
// the fine query features at the strided positions; one CTA = (tile, memory entry, chunk of that entry's boxes),
// the boxes covering the bounding rectangle of the tile's 128 window centres grown by rf; the mask of a lane is
// its own window around ITS centre of this entry.  Zero-padded window positions (affinity 0, value 0 in the
// reference's F.unfold) are counted analytically and inserted by the tail kernel (c2f.cu).
bool c2f_window_supported(int Hf, int Wf, int Cf, int K, int n_mem) {
  return tc16_supported(Hf, Wf, Cf, K) && n_mem >= 1 && n_mem <= tc16::TW_MAX_MEM && Hf < 65536 && Wf < 65536 &&
         (int64_t)n_mem * Hf * Wf < (1ll << 31);
}

// c2f fine stage: a lower bound of every coarse query's final K-th fine affinity that holds across ALL the CTAs
// (memory entries x box chunks) working on the query.  The fine lists of a (tile, entry, chunk) CTA start cold and see
// only a few hundred candidates, so without it ~45 of them are inserted per list, 5-16 lock-step insertion rounds per
// key row (profiles/r2_d_point_tail.md).  Exactly scored here: the window centre and its 4 neighbours in every memory
// entry (in-image, in-window, distinct candidates); the K-th largest of them, minus a rounding margin, is reached by
// K genuine candidates.  One warp per coarse query, accumulator units (256 x affinity), same three products as the MMA.
constexpr int FLOOR_SAMPLES = 5;
__global__ void __launch_bounds__(256)
c2f_floor_kernel(const __half* __restrict__ bank, int Hf, int Wf, int Cf, int HQ, int WQ, int scale, int rf,
                 fgvc_job job, const c2f_wjob* __restrict__ wjobs, const int32_t* __restrict__ ent,
                 const int32_t* __restrict__ best, int K, float* __restrict__ floor_out) {
  // several jobs (wjobs): job = blockIdx.y of the table
  // one CTA per coarse query, one warp per memory entry (8 at a time), the 5 samples of an entry in flight together
  __shared__ float samp[tc16::TW_MAX_MEM * FLOOR_SAMPLES];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = blockIdx.x, nq = HQ * WQ;
  const int qy = q / WQ, qx = q - qy * WQ;
  const int64_t n_pix = (int64_t)Hf * Wf;
  if (wjobs != nullptr) {
    job = wjobs[blockIdx.y].job;
    best += wjobs[blockIdx.y].best_off;
    floor_out += wjobs[blockIdx.y].floor_off;
  }
  const __half* qrow = bank + ((int64_t)job.q_slot * 2 * n_pix + (int64_t)(qy * scale) * Wf + qx * scale) * Cf;
  const __half* qlo = qrow + n_pix * Cf;
  const int n_mem = job.mem_end - job.mem_begin;
  float2 hq[4], lq[4];                                  // Cf <= 256: <= 4 channel pairs per lane
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = 2 * lane + 64 * i;
    hq[i] = c < Cf ? __half22float2(*reinterpret_cast<const __half2*>(qrow + c)) : make_float2(0.f, 0.f);
    lq[i] = c < Cf ? __half22float2(*reinterpret_cast<const __half2*>(qlo + c)) : make_float2(0.f, 0.f);
  }
  for (int e = warp; e < n_mem; e += 8) {
    const int b = max(__ldg(best + (int64_t)e * nq + q), 0) % nq;
    const int cy = (b / WQ) * scale, cx = (b % WQ) * scale;
    const int slot = __ldg(ent + job.mem_begin + e) & ~FGVC_MEM_UNMASKED;
    float acc[FLOOR_SAMPLES];
    bool ok[FLOOR_SAMPLES];
#pragma unroll
    for (int sidx = 0; sidx < FLOOR_SAMPLES; ++sidx) {
      const int dy = sidx == 3 ? 1 : (sidx == 4 ? -1 : 0), dx = sidx == 1 ? 1 : (sidx == 2 ? -1 : 0);
      const int py = cy + dy, px = cx + dx;
      ok[sidx] = py >= 0 && py < Hf && px >= 0 && px < Wf && abs(dy) <= rf && abs(dx) <= rf;      // warp-uniform
      acc[sidx] = 0.f;
      if (!ok[sidx]) continue;
      const __half* krow = bank + ((int64_t)slot * 2 * n_pix + (int64_t)py * Wf + px) * Cf;
      const __half* klo = krow + n_pix * Cf;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = 2 * lane + 64 * i;
        if (c < Cf) {
          const float2 hk = __half22float2(*reinterpret_cast<const __half2*>(krow + c));
          const float2 lk = __half22float2(*reinterpret_cast<const __half2*>(klo + c));
          acc[sidx] += hq[i].x * hk.x + hq[i].x * lk.x + lq[i].x * hk.x + hq[i].y * hk.y + hq[i].y * lk.y + lq[i].y * hk.y;
        }
      }
    }
#pragma unroll
    for (int sidx = 0; sidx < FLOOR_SAMPLES; ++sidx) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[sidx] += __shfl_xor_sync(0xffffffffu, acc[sidx], o);
      if (lane == 0) samp[e * FLOOR_SAMPLES + sidx] = ok[sidx] ? acc[sidx] : -INFINITY;
    }
  }
  __syncthreads();
  if (warp != 0) return;
  // the K-th largest sample: the one with exactly K - 1 samples ahead of it (ties broken by position);
  // -inf (invalid positions, or fewer than K valid samples) = no floor
  const int n = n_mem * FLOOR_SAMPLES;
  float kth = -INFINITY;
  for (int i = lane; i < n; i += 32) {
    const float v = samp[i];
    int ahead = 0;
    for (int j = 0; j < n; ++j) {
      const float u = samp[j];
      ahead += (u > v || (u == v && j < i)) ? 1 : 0;
    }
    if (ahead == K - 1) kth = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kth = fmaxf(kth, __shfl_xor_sync(0xffffffffu, kth, o));
  if (kth > -INFINITY) kth -= 0.05f + 1e-5f * fabsf(kth);           // summation order of the MMA vs this loop
  if (lane == 0) floor_out[q] = kth;
}

// how many CTAs share one (tile, entry): fill the chip, at most 4 (the tail merges n_mem * chunks lists per query)
int c2f_window_chunks(int Hc, int Wc, int n_mem) {
  const long tiles = (long)cdiv(Hc, 8) * cdiv(Wc, 16);
  long c = 148 / (tiles * n_mem > 0 ? tiles * n_mem : 1);
  return (int)(c < 1 ? 1 : (c > 4 ? 4 : c));
}

// fine stage of c2f as a window-mode K1: top-K lists tv / ti [Hc * Wc][n_mem * chunks][K] over the in-window, in-image
// fine keys (idx = memory position * Hf * Wf + fine key pixel).  best: [n_mem][Hc * Wc] coarse arg-max keys.
// wjobs_dev == nullptr: the one job `job`, grid (tiles, n_mem, chunks); else the n_wjobs jobs of the table (the device
// copy of wjobs_host), grid (tiles, n_y): best / floor_ws / tv / ti are then bases that the table's offsets add to.
static int launch_window(const void* fine_bank, int n_slots, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                         const fgvc_job& job, const c2f_wjob* wjobs_dev, int n_wjobs, int n_y, const int32_t* mem_feat,
                         const int32_t* best, int rf, int K, int chunks, float* floor_ws, float* tv, int32_t* ti,
                         cudaStream_t st) {
  using namespace tc16;
  Params p = {};
  p.H = Hf; p.W = Wf; p.C = Cf; p.n_pix = Hf * Wf;
  p.HQ = Hc; p.WQ = Wc; p.scale = scale; p.rf = rf;
  // coarse tile 8 x 16 or 16 x 8: whichever leaves fewer idle lanes on this grid
  const long waste_a = (long)cdiv(Hc, 8) * cdiv(Wc, 16), waste_b = (long)cdiv(Hc, 16) * cdiv(Wc, 8);
  if (waste_b < waste_a) { p.QH = 16; p.QW = 8; p.qw_shift = 3; }
  else { p.QH = 8; p.QW = 16; p.qw_shift = 4; }
  p.lpj_shift = 7;
  p.BH = MAX_NC / 16;
  p.bh_shift = ilog2(p.BH);
  p.k_out = K;
  p.chunks = chunks;
  p.tiles_x = cdiv(Wc, p.QW);
  p.job = job; p.ent = mem_feat; p.best = best; p.tv = tv; p.ti = ti;
  p.wjobs = wjobs_dev; p.n_wjobs = n_wjobs;
  static const int exp_win = getenv("FGVC_TC16_EXP_WIN") ? atoi(getenv("FGVC_TC16_EXP_WIN")) : 0;   // perf experiments only
  p.exp_flags = exp_win;
  // worst case (scattered arg-max keys): the entry lists every box of the frame
  FGVC_CHECK_ARG(rf >= 0 && rf <= 126, "c2f window engine: radius_fine %d too large", rf);
  if ((int64_t)cdiv(Hf, p.BH) * cdiv(Wf, 16) > 2 * MAX_BOXES) {
    set_error("c2f window engine: a %dx%d map exceeds %d key boxes", Hf, Wf, 2 * MAX_BOXES);
    return FGVC_ERR_UNSUPPORTED;
  }
  CUtensorMap mk;
  int rc = make_map16(&mk, fine_bank, n_slots, Hf, Wf, Cf, p.BH);
  if (rc) return rc;
  static const bool no_floor = getenv("FGVC_C2F_NOFLOOR") != nullptr;     // perf experiments only
  if (floor_ws != nullptr && !no_floor) {
    c2f_floor_kernel<<<dim3(Hc * Wc, wjobs_dev != nullptr ? n_wjobs : 1), 256, 0, st>>>(
        reinterpret_cast<const __half*>(fine_bank), Hf, Wf, Cf, Hc, Wc, scale, rf, job, wjobs_dev, mem_feat, best, K,
        floor_ws);
    FGVC_LAUNCH_CHECK();
    p.floor = floor_ws;
  }
  dim3 grid(cdiv(Hc, p.QH) * p.tiles_x, job.mem_end - job.mem_begin, chunks);
  if (wjobs_dev != nullptr) grid = dim3(cdiv(Hc, p.QH) * p.tiles_x, n_y, 1);
  return launch_by_k<1, true>(mk, fine_bank, p, grid, K, st);
}

int launch_c2f_window_tc16(const void* fine_bank, int n_slots, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                           const fgvc_job& job, const int32_t* mem_feat, const int32_t* best, int rf, int K, int chunks,
                           float* floor_ws, float* tv, int32_t* ti, cudaStream_t st) {
  return launch_window(fine_bank, n_slots, Hc, Wc, Hf, Wf, Cf, scale, job, nullptr, 0, 0, mem_feat, best, rf, K, chunks,
                       floor_ws, tv, ti, st);
}

// the fine stage of the jobs of a c2f_wjob table in one window-mode K1 launch (and one floor launch): every job gets
// the lists, chunk for chunk, that launch_c2f_window_tc16 gives it alone
int launch_c2f_window_tc16_jobs(const void* fine_bank, int n_slots, int Hc, int Wc, int Hf, int Wf, int Cf, int scale,
                                const c2f_wjob* wjobs_dev, int n_wjobs, int n_y, const int32_t* mem_feat,
                                const int32_t* best, int rf, int K, float* floor_ws, float* tv, int32_t* ti,
                                cudaStream_t st) {
  FGVC_CHECK_ARG(n_wjobs >= 1 && n_wjobs <= 65535 && n_y >= 1 && n_y <= 65535,
                 "c2f window engine: %d jobs / %d (job, entry, chunk) CTAs per tile, at most 65535", n_wjobs, n_y);
  fgvc_job none = {0, 0, 1, 0};
  return launch_window(fine_bank, n_slots, Hc, Wc, Hf, Wf, Cf, scale, none, wjobs_dev, n_wjobs, n_y, mem_feat, best, rf,
                       K, 1, floor_ws, tv, ti, st);
}

}  // namespace fgvc
