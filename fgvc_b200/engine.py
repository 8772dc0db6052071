"""Device-side state of the propagation path: feature bank, label bank, job tables, and
thin wrappers that enqueue the CUDA kernels through the C ABI (fgvc_b200/_lib.py).

Vocabulary follows the reference (``feat_bank`` / ``seg_bank`` of
mmpt/models/trackers/vanilla_tracker.py:318-394): a *slot* holds one frame.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._lib import Job, call, ptr, stream_ptr

_NUM_SMS = {}


def num_sms(device=None):
    """SM count of ``device`` (grid sizing of the host-side planners); 148 on a B200."""
    idx = torch.device(device).index if device is not None and torch.device(device).index is not None \
        else (torch.cuda.current_device() if torch.cuda.is_available() else -1)
    if idx < 0:
        return 148
    if idx not in _NUM_SMS:
        _NUM_SMS[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _NUM_SMS[idx]


def pad4(n):
    return (n + 3) // 4 * 4


def default_split(C):
    """'f16' (three-term fp16 split, all-TMEM operands: the fast tensor engine) when the channel
    count allows, else 'tf32' (3xTF32)."""
    return "f16" if (C % 64 == 0 and C <= 256) else "tf32"


class FeatureBank:
    """feat[slot][2][H*W][C]: L2-normalised, pixel-major two-term split (K0 output).
    ``split='tf32'``: fp32 cells, hi = tf32(x), lo = x - hi (3xTF32 engine);
    ``split='f16'``: fp16 cells, X = 16 x, hi = fp16(X), lo = fp16(X - hi) (fp16 three-term engine)."""

    def __init__(self, n_slots, C, H, W, device, split=None):
        _lib.require_cuda()
        self.n_slots, self.C, self.H, self.W = n_slots, C, H, W
        self.split = split or default_split(C)
        assert self.split in ("tf32", "f16")
        if self.split == "f16" and C % 4:
            raise ValueError("the f16 bank needs C % 4 == 0")
        self.fmt = _lib.BANK_F16 if self.split == "f16" else _lib.BANK_TF32
        dt = torch.float16 if self.split == "f16" else torch.float32
        self.buf = torch.empty(n_slots, 2, H * W, C, dtype=dt, device=device)
        self.unit_rows = True          # until a frame is loaded without normalisation

    def dense(self):
        """fp32 [slot, H*W, C] view of what the split encodes (tests / diagnostics)."""
        if self.split == "f16":
            return (self.buf[:, 0].float() + self.buf[:, 1].float()) / 16.0
        return self.buf[:, 0] + self.buf[:, 1]

    def load(self, src, first_slot, n_frames, frame_stride, chan_stride, normalize=True):
        """src: fp32 CUDA tensor; frame f / channel c / pixel p at
        ``src.data_ptr + 4*(f*frame_stride + c*chan_stride + p)``."""
        assert src.is_cuda and src.dtype == torch.float32
        assert 0 <= first_slot and first_slot + n_frames <= self.n_slots
        if not normalize:
            self.unit_rows = False
        call("fgvc_prep_features", ptr(src), frame_stride, chan_stride, n_frames, self.C, self.H, self.W,
             int(bool(normalize)), ptr(self.buf), self.fmt, first_slot, stream_ptr())

    def load_frames(self, feats, first_slot=0, normalize=True):
        """feats [n,C,H,W] contiguous."""
        feats = feats.contiguous()
        n, C, H, W = feats.shape
        assert (C, H, W) == (self.C, self.H, self.W)
        self.load(feats, first_slot, n, C * H * W, H * W, normalize)


class LabelBank:
    """lab[slot][H*W][Lp], Lp = L padded to a multiple of 4."""

    def __init__(self, n_slots, L, H, W, device, buf=None):
        """``buf``: a flat fp32 CUDA tensor of n_slots * H*W * Lp elements to hold the bank (several banks carved out of
        one allocation); default: a new one."""
        _lib.require_cuda()
        self.n_slots, self.L, self.Lp, self.H, self.W = n_slots, L, pad4(L), H, W
        if buf is None:
            self.buf = torch.empty(n_slots, H * W, self.Lp, dtype=torch.float32, device=device)
        else:
            self.buf = buf.view(n_slots, H * W, self.Lp)

    def put_nchw(self, src, slot, chan_stride=None):
        """src: [L,H,W] view whose pixels are contiguous; chan_stride in floats."""
        assert src.is_cuda and src.dtype == torch.float32
        if chan_stride is None:
            src = src.contiguous()
            chan_stride = self.H * self.W
        call("fgvc_labels_to_pixmajor", ptr(src), chan_stride, self.L, self.H * self.W, ptr(self.buf), slot,
             self.Lp, stream_ptr())

    def get_nchw(self, slot, out=None):
        if out is None:
            out = torch.empty(self.L, self.H, self.W, dtype=torch.float32, device=self.buf.device)
        call("fgvc_labels_to_nchw", ptr(self.buf), slot, self.Lp, self.L, self.H * self.W, ptr(out), stream_ptr())
        return out

    def put_gaussians(self, points_xy, slot, stride, sigma=6.0):
        """draw_gaussion_map_online at feature resolution (vanilla_tracker.py:204-221)."""
        pts = points_xy.to(device=self.buf.device, dtype=torch.float32).contiguous()
        assert pts.shape == (self.L, 2)
        call("fgvc_gaussian_labels", ptr(pts), self.L, self.H, self.W, int(stride), float(sigma), ptr(self.buf),
             slot, self.Lp, stream_ptr())


class JobTable:
    """Propagation jobs: (query slot, memory list, output slot).  Host lists -> device int32."""

    def __init__(self):
        self.jobs, self.mem_feat, self.mem_label = [], [], []
        self._dev = None
        self._packed = {}

    def add(self, q_slot, mem_feat_slots, mem_label_slots, out_slot, unmasked=0):
        """``unmasked``: number of leading memory entries without the radius mask
        (``non_mask_len``, local_attention.py:347)."""
        assert len(mem_feat_slots) == len(mem_label_slots) >= 1
        b = len(self.mem_feat)
        for i, s in enumerate(mem_feat_slots):
            self.mem_feat.append(int(s) | (_lib.MEM_UNMASKED if i < unmasked else 0))
        self.mem_label.extend(int(s) for s in mem_label_slots)
        self.jobs.append((int(q_slot), b, b + len(mem_feat_slots), int(out_slot)))
        self._dev = None
        self._packed = {}
        return len(self.jobs) - 1

    def add_raw(self, q_slot, raw_feat_entries, out_slot):
        """A job whose memory entries already carry their FGVC_MEM_UNMASKED flags (label slots = feature slots)."""
        b = len(self.mem_feat)
        self.mem_feat.extend(int(r) for r in raw_feat_entries)
        self.mem_label.extend(int(r) & ~_lib.MEM_UNMASKED for r in raw_feat_entries)
        self.jobs.append((int(q_slot), b, b + len(raw_feat_entries), int(out_slot)))
        self._dev = None
        self._packed = {}
        return len(self.jobs) - 1

    def __len__(self):
        return len(self.jobs)

    @property
    def max_mem(self):
        return max(j[2] - j[1] for j in self.jobs)

    def device(self, device):
        if self._dev is None or self._dev[0].device != torch.device(device):
            j = torch.tensor(self.jobs, dtype=torch.int32).reshape(-1, 4).to(device)
            mf = torch.tensor(self.mem_feat, dtype=torch.int32).to(device)
            ml = torch.tensor(self.mem_label, dtype=torch.int32).to(device)
            self._dev = (j, mf, ml)
        return self._dev

    def host_job(self, i):
        return Job(*self.jobs[i])

    def _tile_groups(self, j0, j1, J, aligned):
        """[(out_group, [job indices])]: J consecutive jobs per group; ``aligned``: one set of groups per class a of
        memory frames (slot % J == a), the jobs grouped with phase a (query slots a+1 .. a+J together) so that a
        sliding memory window is used by all J jobs of a group or by none."""
        if not aligned:
            return [(0, list(range(a, min(a + J, j1)))) for a in range(j0, j1, J)]
        out = []
        for a in range(J):
            groups = {}
            for i in range(j0, j1):
                groups.setdefault((self.jobs[i][0] - a - 1) // J, []).append(i)
            out.extend((a, groups[g]) for g in sorted(groups))
        return out

    def sequential(self, j0, j1):
        """jobs [j0, j1) are consecutive query frames (what the aligned packing assumes)"""
        return all(self.jobs[i + 1][0] == self.jobs[i][0] + 1 for i in range(j0, j1 - 1))

    def _group_table(self, members, J, cls):
        """union entries of a tile group: {(raw entry, occurrence): [position in member i's own list or -1] * 4}"""
        table = {}
        for li, i in enumerate(members):
            seen = {}
            b, e = self.jobs[i][1], self.jobs[i][2]
            for pos, raw in enumerate(self.mem_feat[b:e]):
                occ = seen.get(raw, 0)
                seen[raw] = occ + 1
                if cls is None or (raw & ~_lib.MEM_UNMASKED) % J == cls:
                    table.setdefault((raw, occ), [-1, -1, -1, -1])[li] = pos
        return table

    def union_sizes(self, j0, j1, J, aligned=False):
        """sizes of the union memory lists of the tile groups of jobs [j0, j1) (cost model)."""
        return [len(self._group_table(m, J, a if aligned else None)) for a, m in self._tile_groups(j0, j1, J, aligned)]

    def packed_cuts(self, cuts, J, device, aligned=False):
        """``packed`` of the consecutive job ranges ``cuts`` [(j0, j1), ...] concatenated: no tile group spans two
        ranges, so the tile groups of each range are the ones ``packed`` gives for it alone."""
        parts = [self.packed(a, b, J, device, aligned) for a, b in cuts if b > a]
        if len(parts) == 1:
            return parts[0]
        groups, uents, upos, u = [], [], [], 0
        for g, ue, up in parts:
            g = g.clone()
            g[:, 5:7] += u
            n = int(g[:, 6].max()) - u if g.shape[0] else 0
            groups.append(g)
            uents.append(ue[:n])
            upos.append(up[:n])
            u += n
        return torch.cat(groups), torch.cat(uents), torch.cat(upos)

    def packed(self, j0, j1, J, device, aligned=False):
        """Tile groups of jobs [j0, j1) for fgvc_affinity_topk_packed: (groups [n,8] int32, union entries [U] int32,
        union positions [U,4] int32) on ``device``.  A memory list is a multiset (frame 0 twice while
        t <= precede_frames): the k-th occurrence of a frame in one job is matched with the k-th occurrence in the
        others.  Union entries are ordered oldest frame first -- the kernel walks them backwards."""
        key = (j0, j1, J, bool(aligned), str(device))
        hit = self._packed.get(key)
        if hit is not None:
            return hit
        groups, uent, upos = [], [], []
        for cls, members in self._tile_groups(j0, j1, J, aligned):
            assert len(members) <= 4
            table = self._group_table(members, J, cls if aligned else None)
            order = sorted(table, key=lambda k: (k[0] & ~_lib.MEM_UNMASKED, 0 if (k[0] & _lib.MEM_UNMASKED) else 1, k[1]))
            u0 = len(uent)
            for k in order:
                uent.append(k[0])
                upos.append(table[k])
            groups.append(members + [-1] * (4 - len(members)) + [len(members), u0, len(uent), cls])
        out = (torch.tensor(groups, dtype=torch.int32).reshape(-1, 8).to(device),
               torch.tensor(uent if uent else [0], dtype=torch.int32).to(device),
               torch.tensor(upos if upos else [[-1] * 4], dtype=torch.int32).reshape(-1, 4).to(device))
        self._packed[key] = out
        return out


def pick_groups(n_jobs, H, W, max_mem, max_groups=4):
    """Number of memory groups per job for one K1 launch.  A CTA is one (query tile, job, group);
    one CTA runs per SM, so a launch takes ceil(ctas / 148) rounds of (1/groups) of a job's memory
    list.  Pick the split with the fewest effective rounds (short launches suffer most from a
    partially filled last wave); ties go to fewer groups (less per-CTA set-up and merging)."""
    ctas = n_jobs * (-(-H // 8)) * (-(-W // 16))          # 128-query tiles (8x16 or 16x8 pixels)
    best, best_cost = 1, None
    for g in range(1, max(1, min(max_groups, max_mem)) + 1):
        rounds = -(-ctas * g // num_sms())
        cost = rounds / g + 0.02 * (g - 1)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = g, cost
    return best


def plan_chunks(n_jobs, tiles, copy_ratio=0.75, launch_cost=0.4):
    """Split jobs 0..n_jobs-1 into consecutive chunks for the host pipeline.  Chunk i's K1 launch
    (chunk_jobs * tiles CTAs, one CTA per SM => whole rounds) can start once its frames have been copied
    (copies are issued back to back on the copy stream) and the previous chunk has finished.  Dynamic
    programme over cut positions minimising the finish time; unit = compute time of one job at full
    efficiency, ``copy_ratio`` = copy time of one frame in that unit, ``launch_cost`` = per-chunk overhead
    (K0 + tail launches, pipeline fill)."""
    jobs_per_round = num_sms() / float(tiles)

    def compute(n):
        return -(-n * tiles // num_sms()) * jobs_per_round + launch_cost

    INF = float("inf")
    best = [(INF, None)] * (n_jobs + 1)
    best[0] = (0.0, None)
    for end in range(1, n_jobs + 1):
        copied = copy_ratio * (end + 1)                    # frames 0..end are on the device
        for start in range(0, end):
            c = max(copied, best[start][0]) + compute(end - start)
            if c < best[end][0]:
                best[end] = (c, start)
    cuts, e = [], n_jobs
    while e > 0:
        s0 = best[e][1]
        cuts.append((s0, e))
        e = s0
    cuts.reverse()
    return cuts


def plan_overlap_chunks(n_jobs, tiles, max_chunks=6):
    """Split the jobs of a resident clip into the largest number of K1 launches (<= max_chunks) that
    costs no extra round compared with one launch, so that the gather chain of chunk i (second stream)
    can overlap K1 of chunk i+1 for free.  Falls back to a single launch."""
    def rounds(n):
        return -(-n * tiles // num_sms())

    single = rounds(n_jobs)
    best = [(0, n_jobs)]
    for k in range(2, max_chunks + 1):
        if k > n_jobs:
            break
        base, extra = divmod(n_jobs, k)
        sizes = [base + (1 if i < extra else 0) for i in range(k)]
        if sum(rounds(n) for n in sizes) <= single:
            cuts, s0 = [], 0
            for n in sizes:
                cuts.append((s0, s0 + n))
                s0 += n
            best = cuts
    return best


class TopKLists:
    def __init__(self, n_jobs, groups, n_query, K, device):
        self.n_jobs, self.groups, self.n_query, self.K = n_jobs, groups, n_query, K
        self.val = torch.empty(n_jobs, groups, n_query, K, dtype=torch.float32, device=device)
        self.idx = torch.empty(n_jobs, groups, n_query, K, dtype=torch.int32, device=device)


_CHAIN_WS = {}


def _ws_key(dev):
    dev = torch.device(dev)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    return (idx, torch.cuda.current_stream(dev).cuda_stream)


_COVER = {}


def tile_shape(H, W, radius, mode, J):
    """(QH, QW, BH, ncta) of the fp16 tensor engine for J jobs per tile: pixel block of one job, key-box height, CTAs
    per tile (2 = CTA pair, 256 tile rows)."""
    import ctypes as ct
    qh, qw, bh, nc = ct.c_int32(), ct.c_int32(), ct.c_int32(), ct.c_int32()
    call("fgvc_packed_tile_shape", H, W, int(radius), int(mode), int(J), ct.byref(qh), ct.byref(qw), ct.byref(bh),
         ct.byref(nc))
    return qh.value, qw.value, bh.value, nc.value


BOX_FIXED = 24        # per-box hand-shake of the engine in key units (csrc/topk_tc16.cu: box_cost16)
TILE_SETUP = 160      # per (tile, tile group) set-up in key units: barriers, TMEM, query rows, box lists, list merge


def _cover_keys(H, W, radius, mode, J):
    """Keys a query tile multiplies (whole key boxes of its radius halo that some query can see), summed over
    the tiles of a map, for J jobs per tile -- the geometry of csrc/topk_tc16.cu.  Every tile is a full M = 128
    (x 2 for CTA pairs) MMA, so the tensor work of a launch is  sum over tile groups of |union memory list| x this
    number x tile rows."""
    env = os.environ.get("FGVC_TC16_PAIR", "")
    key = (H, W, radius, mode, J, env)
    if key in _COVER:
        return _COVER[key]
    QH, QW, BH, ncta = tile_shape(H, W, radius, mode, J)
    reach = radius - 1 if mode == _lib.MASK_CIRCLE else radius

    def seen(dy, dx):
        return dy * dy + dx * dx < radius * radius if mode == _lib.MASK_CIRCLE else (dy <= radius and dx <= radius)

    total = keys = tiles = 0
    for qy0 in range(0, H, QH):
        for qx0 in range(0, W, QW):
            tiles += 1
            y_lo, y_hi = max(0, qy0 - reach), min(H - 1, qy0 + QH - 1 + reach)
            x_lo, x_hi = max(0, qx0 - reach), min(W - 1, qx0 + QW - 1 + reach)
            qy1, qx1 = min(H - 1, qy0 + QH - 1), min(W - 1, qx0 + QW - 1)
            for by in range(y_lo, y_hi + 1, BH):
                dy = max(0, by - qy1, qy0 - min(H - 1, by + BH - 1))
                for bx in range(x_lo, x_hi + 1, 16):
                    dx = max(0, bx - qx1, qx0 - min(W - 1, bx + 15))
                    if seen(dy, dx):
                        total += 16 * BH + BOX_FIXED
                        keys += 16 * BH
    _COVER[key] = dict(cost=total, keys=keys, tiles=tiles, rows=128 * ncta)
    return _COVER[key]


def dense_pairs(table, j0, j1, H, W, radius, mode, J, aligned=False):
    """(query row, key) pairs the tensor engine multiplies for jobs [j0, j1) packed J per tile: every tile is a
    full MMA against every key box of its halo, for every entry of the group's union memory list."""
    c = _cover_keys(H, W, radius, mode, J)
    return c["rows"] * c["keys"] * sum(table.union_sizes(j0, j1, J, aligned))


def packing_cost(table, j0, j1, H, W, radius, mode, J, aligned=False):
    """tensor time of one K1 launch in key units x tile rows (the cost model behind pick_packing)."""
    c = _cover_keys(H, W, radius, mode, J)
    u = table.union_sizes(j0, j1, J, aligned)
    return c["rows"] * (sum(u) * c["cost"] + len(u) * c["tiles"] * TILE_SETUP)


def pick_packing(table, j0, j1, H, W, radius, mode):
    """(jobs per tile, aligned) with the least tensor work for jobs [j0, j1).  ``aligned`` = memory frames are
    divided into J classes by slot index mod J and the query frames of class a are grouped with phase a, so that
    every job of a tile group uses every memory entry of the group (no wasted rows at the ends of the sliding
    window); each job then has J partial lists, merged by the gather.  FGVC_PACK = "J" or "Ja" forces it."""
    forced = os.environ.get("FGVC_PACK")
    seq = table.sequential(j0, j1)
    if forced is not None:
        return int(forced.rstrip("a")), forced.endswith("a") and seq
    if j1 - j0 < 2:
        return 1, False
    ckey = ("pick", j0, j1, H, W, radius, mode, os.environ.get("FGVC_TC16_PAIR", ""))
    if ckey in table._packed:
        return table._packed[ckey]
    best, best_cost = (1, False), None
    # The aligned packings issue 11 % fewer tensor MACs on a precede-20 clip, but every tile then covers ~5 memory
    # entries instead of ~25 and K1 is bound by the epilogue's list insertions, which are most frequent while the
    # lists are cold: measured 8.1 ms against 7.0 ms (profiles/r2_b_epilogue.md).  AUTO therefore keeps the plain
    # packings; FGVC_PACK="4a" selects an aligned one.
    for J, aligned in ((1, False), (2, False), (4, False)):
        if aligned and not seq:
            continue
        cost = packing_cost(table, j0, j1, H, W, radius, mode, J, aligned)
        if best_cost is None or cost < 0.97 * best_cost:      # a more complex packing must pay for itself
            best, best_cost = (J, aligned), cost
    table._packed[ckey] = best
    return best


def pair_key(table, job):
    """(query frame, backward) of a job of ``table``: the memory frames of a job run backwards in time (the forward
    tracker on the time-reversed clip) all lie after its query frame, those of a forward job before it."""
    q_slot, b = job[0], job[1]
    return q_slot, (table.mem_feat[b] & ~_lib.MEM_UNMASKED) > q_slot


def shared_pair_table(table, spans, T, decide_jobs=None, max_entries=None):
    """Several ``with_first`` groups of one clip: the jobs (group g, query frame t) of different groups see the same
    memory frames except their first one, so the label-independent K1 work is shared -- run it once per query frame
    and direction over the UNION of the groups' memory entries, one list per (query frame, direction, memory entry),
    and let the tail merge each job's lists.  Forward and backward jobs of a query frame are not merged: their
    memories have no frame in common, and the list floor of the shared launch needs one.  Returns (utable, Gmax,
    pair_ref) or None when sharing would not pay:
      utable   : JobTable with one job per (query frame, direction), entries = sorted unique (frame, mask flag) of all
                 groups;
      pair_ref : for every memory entry of ``table`` the index (u_job * Gmax + position in the union) of its list.
    ``decide_jobs``: whether sharing pays is judged on the first ``decide_jobs`` jobs only (the tracking jobs, when the
    cycle checks follow them: adding the checks must not change how the tracks are computed).  ``max_entries``: a
    (query frame, direction) with more entries is split over several utable jobs of at most that many (K1 takes at
    most 64 lists per job); default: no split, None when a union has more than 64 entries."""
    by_key = {}
    for job in table.jobs:
        by_key.setdefault(pair_key(table, job), set()).update(table.mem_feat[job[1]:job[2]])
    dec = by_key
    if decide_jobs is not None:
        dec = {}
        for job in table.jobs[:decide_jobs]:
            dec.setdefault(pair_key(table, job), set()).update(table.mem_feat[job[1]:job[2]])
    if not dec or len(table.jobs[:decide_jobs]) < 1.8 * len(dec) or max(len(v) for v in dec.values()) > 64:
        return None
    gmax = max(len(v) for v in by_key.values())
    if max_entries is None and gmax > 64:
        return None
    gmax = min(gmax, max_entries or gmax)
    utable, where = JobTable(), {}
    for key in sorted(by_key):
        ent = sorted(by_key[key], key=lambda r: (r & ~_lib.MEM_UNMASKED, 0 if (r & _lib.MEM_UNMASKED) else 1))
        for c in range(0, len(ent), gmax):
            u = len(utable)
            utable.add_raw(key[0], ent[c:c + gmax], key[0])
            for i, r in enumerate(ent[c:c + gmax]):
                where[(key, r)] = u * gmax + i
    pair_ref = []
    for job in table.jobs:
        key = pair_key(table, job)
        pair_ref.extend(where[(key, r)] for r in table.mem_feat[job[1]:job[2]])
    return utable, gmax, pair_ref


def frame_runs(table, j0, j1):
    """Maximal runs [a, b) of feature slots that the jobs [j0, j1) of ``table`` read (their query frames and memory
    frames): what a rank of the two-phase split has to upload and prepare."""
    need = set()
    for (q_slot, b, e, _) in table.jobs[j0:j1]:
        need.add(q_slot)
        need.update(r & ~_lib.MEM_UNMASKED for r in table.mem_feat[b:e])
    need = sorted(need)
    runs, i = [], 0
    while i < len(need):
        j = i
        while j + 1 < len(need) and need[j + 1] == need[j] + 1:
            j += 1
        runs.append((need[i], need[j] + 1))
        i = j + 1
    return runs


def chain_workspace(dev, n_jobs, n_pix, K, flags=0, force=False):
    """(pointer, bytes) of the scratch that lets a clip tail run its gather chain as one persistent kernel;
    (None, 0) = per-frame launches (hard propagation decodes between frames, single-frame ranges gain nothing)."""
    if not force and (n_jobs <= 1 or (flags & _lib.HARD_PROP) or os.environ.get("FGVC_NO_CHAIN") == "1"):
        return None, 0
    nbytes = int(_lib.load().fgvc_chain_workspace_bytes(int(n_jobs), int(n_pix), int(K)))
    ws = _CHAIN_WS.get(_ws_key(dev))
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _CHAIN_WS[_ws_key(dev)] = ws
    return ptr(ws), nbytes


def point_tail_lanes(lists, pair_ref, table, lanes, lab, maps, coords, H, W, out_hw, temperature, flags, coord_topk=5):
    """fgvc_point_clip_tail_lanes: the point tails of several independent recurrences of a clip in one multi-lane
    gather chain.  ``lanes``: list of (job_begin, job_end, L, lab_offset, coord_offset), offsets in floats into the
    flat tensors ``lab`` (label banks) and ``coords`` (tracks); ``maps``: NCHW scratch of every lane;
    ``pair_ref``: device int32 tensor of the shared lists or None."""
    dev = lab.device
    jobs_dev, _, mem_label = table.device(dev)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4).contiguous()
    host = (_lib.Lane * len(lanes))(*[_lib.Lane(jb, je, L, pad4(L), lo, co) for (jb, je, L, lo, co) in lanes])
    lanes_dev = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(dev)
    jb, je = min(ln[0] for ln in lanes), max(ln[1] for ln in lanes)
    call("fgvc_point_clip_tail_lanes", ptr(lists.val), ptr(lists.idx), lists.K, 1 if pair_ref is not None else lists.groups,
         ptr(pair_ref) if pair_ref is not None else None, ptr(jobs_dev), ptr(jobs_host), ptr(lanes_dev), ctypes.c_void_p(ctypes.addressof(host)), len(lanes),
         ptr(mem_label), H, W, float(temperature), int(flags), ptr(lab), int(out_hw[0]), int(out_hw[1]), int(coord_topk),
         ptr(maps), ptr(coords), *chain_workspace(dev, je - jb, H * W, lists.K, flags, force=True), stream_ptr())


def point_cycle_lanes(lists, pair_ref, table, lanes, coords, cycle_coords, vis, H, W, out_hw, stride, temperature,
                      flags, threshold, sigma=6.0, coord_topk=5):
    """fgvc_point_cycle_lanes: the cycle checks ``lanes`` [(job_begin, job_end, L, coord_offset, t, s)] in one call.
    Their banks, the NCHW maps of their last slots, the K3 output and the chain workspace are allocated here, for this
    call only: a caller bounds the memory by the checks it passes (VanillaTracker._cycle_tail)."""
    dev = coords.device
    n_pix = H * W
    jobs_dev, _, mem_label = table.device(dev)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4).contiguous()
    hl, hc, lab_off, map_off = [], [], 0, 0
    for jb, je, L, c_off, t, s in lanes:
        hl.append(_lib.Lane(jb, je, L, pad4(L), lab_off, c_off))
        hc.append(_lib.Cycle(t, s, map_off))
        lab_off += (je - jb + 1) * n_pix * pad4(L)
        map_off += L
    host_l, host_c = (_lib.Lane * len(hl))(*hl), (_lib.Cycle * len(hc))(*hc)
    lanes_dev = torch.frombuffer(bytearray(host_l), dtype=torch.uint8).to(dev)
    cycles_dev = torch.frombuffer(bytearray(host_c), dtype=torch.uint8).to(dev)
    lab = torch.empty(lab_off, dtype=torch.float32, device=dev)
    maps = torch.empty(map_off * n_pix, dtype=torch.float32, device=dev)
    xy = torch.empty(map_off * 2, dtype=torch.float32, device=dev)
    jb, je = min(ln[0] for ln in lanes), max(ln[1] for ln in lanes)
    ws_bytes = int(_lib.load().fgvc_chain_workspace_bytes(je - jb, n_pix, lists.K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    call("fgvc_point_cycle_lanes", ptr(lists.val), ptr(lists.idx), lists.K, 1 if pair_ref is not None else lists.groups,
         ptr(pair_ref) if pair_ref is not None else None, ptr(jobs_dev), ptr(jobs_host), ptr(lanes_dev),
         ctypes.c_void_p(ctypes.addressof(host_l)), ptr(cycles_dev), ctypes.c_void_p(ctypes.addressof(host_c)),
         len(lanes), ptr(mem_label), H, W, int(stride), float(sigma), float(temperature), int(flags), ptr(lab),
         int(out_hw[0]), int(out_hw[1]), int(coord_topk), float(threshold), ptr(coords), ptr(maps), ptr(xy),
         ptr(cycle_coords), ptr(vis), ptr(ws), ws_bytes, stream_ptr())


def cycle_lane_bytes(n_jobs, L, n_pix, K):
    """device bytes point_cycle_lanes allocates for a check of n_jobs jobs over L points: its bank of n_jobs + 1 slots,
    its share of the chain workspace, its NCHW maps and K3 output"""
    return 4 * (n_jobs + 1) * n_pix * pad4(L) + int(_lib.load().fgvc_chain_workspace_bytes(n_jobs, n_pix, K)) - 256 + \
        4 * L * n_pix + 8 * L


K1_TIMING = None       # bench.py: a list -> affinity_topk appends (start, end) CUDA events of every K1 launch


class K1Plan:
    """How one K1 launch is tiled: J jobs per query tile, ``aligned`` memory classes (pick_packing), ``split`` parts
    per tile group (load balance of short launches).  A job gets ``lists_per_job`` partial top-k lists."""

    def __init__(self, J=1, aligned=False, split=1):
        self.J, self.aligned, self.split = int(J), bool(aligned), int(split)

    @property
    def lists_per_job(self):
        return (self.J if self.aligned else 1) * self.split

    def __repr__(self):
        return f"K1Plan(J={self.J}, aligned={self.aligned}, split={self.split})"


def tensor16_ok(bank, K, engine):
    return engine in (_lib.ENGINE_AUTO, _lib.ENGINE_TCGEN05) and bank.fmt == _lib.BANK_F16 and \
        bool(_lib.load().fgvc_tc_supported(bank.fmt, bank.H, bank.W, bank.C, int(K)))


def plan_k1(bank, table, radius, K, mask_mode="circle", job_range=None, engine=_lib.ENGINE_AUTO, groups=None, pack=True):
    """Tiling of a K1 launch over ``job_range`` of ``table``.  ``groups`` fixes the lists per job (no aligned classes)."""
    j0, j1 = job_range if job_range is not None else (0, len(table))
    mode = _lib.MASK_CIRCLE if mask_mode == "circle" else _lib.MASK_SQUARE
    J, aligned = 1, False
    if pack and tensor16_ok(bank, K, engine):
        J, aligned = pick_packing(table, j0, j1, bank.H, bank.W, int(radius), mode)
        if groups is not None and aligned:
            aligned = False
    if groups is None:
        groups = 1 if aligned else pick_groups(j1 - j0, bank.H, bank.W, table.max_mem)
    return K1Plan(J, aligned, groups)


def affinity_topk(bank, table, radius, K, mask_mode="circle", groups=None, engine=_lib.ENGINE_AUTO, lists=None,
                  job_range=None, pack=True, plan=None, floor=None, cuts=None):
    """K1 over every job of ``table`` (or the jobs ``job_range=(begin, end)``) in one launch.  ``AUTO``
    = the tensor engine of the bank format when the shape allows, else the CUDA-core engine.  ``plan`` (plan_k1)
    fixes the tiling; the lists hold ``plan.lists_per_job`` partial lists per job, merged by the gather.
    ``floor`` [jobs, Nq] (topk_floor): starting value of the lists, un-packed launches only (see the header).
    ``cuts``: consecutive sub-ranges of the launch whose jobs are packed into query tiles only with each other
    (JobTable.packed_cuts): a range then gets the lists it gets in a launch of its own with the same plan."""
    dev = bank.buf.device
    jobs, mem_feat, _ = table.device(dev)
    j0, j1 = job_range if job_range is not None else (0, len(table))
    if plan is None:
        if groups is None and lists is not None:
            groups = lists.groups
        plan = plan_k1(bank, table, radius, K, mask_mode, (j0, j1), engine, groups, pack)
    groups = plan.lists_per_job
    if lists is None:
        lists = TopKLists(len(table), groups, bank.H * bank.W, K, dev)
    assert lists.groups == groups and lists.K == K and lists.n_jobs >= len(table), (lists.groups, plan)
    mode = _lib.MASK_CIRCLE if mask_mode == "circle" else _lib.MASK_SQUARE
    per_job = groups * lists.n_query * K * 4      # bytes of one job's lists
    if K1_TIMING is not None:
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev[0].record()
        try:
            return _affinity_topk_launch(bank, table, radius, K, mode, groups, engine, lists, j0, j1, plan, per_job,
                                         jobs, mem_feat, dev, floor, cuts)
        finally:
            ev[1].record()
            K1_TIMING.append(ev)
    return _affinity_topk_launch(bank, table, radius, K, mode, groups, engine, lists, j0, j1, plan, per_job, jobs,
                                 mem_feat, dev, floor, cuts)


def topk_floor(bank, table, seed_slots, radius, K, mask_mode="circle"):
    """fgvc_topk_floor: per (job, query pixel) the K-th best of the exactly scored 5 x 5 neighbourhood of the query's own
    position in frame ``seed_slots[job]`` (< 0: none).  F16 bank with a tensor-engine shape only, else None."""
    if bank.fmt != _lib.BANK_F16 or not tensor16_ok(bank, K, _lib.ENGINE_AUTO):
        return None
    dev = bank.buf.device
    jobs, _, _ = table.device(dev)
    seeds = torch.tensor(list(seed_slots), dtype=torch.int32, device=dev)
    assert seeds.numel() == len(table)
    out = torch.empty(len(table), bank.H * bank.W, dtype=torch.float32, device=dev)
    mode = _lib.MASK_CIRCLE if mask_mode == "circle" else _lib.MASK_SQUARE
    call("fgvc_topk_floor", ptr(bank.buf), bank.fmt, bank.H, bank.W, bank.C, ptr(jobs), len(table), ptr(seeds), int(radius),
         mode, int(K), ptr(out), stream_ptr())
    return out


def _affinity_topk_launch(bank, table, radius, K, mode, groups, engine, lists, j0, j1, plan, per_job, jobs, mem_feat, dev,
                          floor=None, cuts=None):
    # fp16 tensor engine: J consecutive jobs per query tile when that saves tensor work (csrc/topk_tc16.cu)
    if (plan.J > 1 or plan.aligned) and tensor16_ok(bank, K, engine):
        tg, uent, upos = table.packed(j0, j1, plan.J, dev, plan.aligned) if cuts is None else \
            table.packed_cuts([(max(a, j0), min(b, j1)) for a, b in cuts], plan.J, dev, plan.aligned)
        try:
            call("fgvc_affinity_topk_packed", ptr(bank.buf), bank.n_slots, bank.H, bank.W, bank.C, ptr(jobs), ptr(tg),
                 int(tg.shape[0]), ptr(uent), ptr(upos), int(plan.J), int(radius), mode, int(K), int(groups),
                 int(plan.split), ptr(lists.val), ptr(lists.idx), stream_ptr())
            return lists
        except _lib.FgvcError as err:
            # a shape the tensor kernel does not take (e.g. a huge map): AUTO goes on to the un-packed entry point,
            # which falls back to the CUDA-core engine
            if err.rc != _lib.ERR_UNSUPPORTED or engine != _lib.ENGINE_AUTO:
                raise
    if floor is not None:
        call("fgvc_affinity_topk_seeded", ptr(bank.buf), bank.fmt, bank.n_slots, bank.H, bank.W, bank.C,
             ctypes.c_void_p(jobs.data_ptr() + 16 * j0), j1 - j0, ptr(mem_feat), int(radius), mode, int(K), int(groups),
             ctypes.c_void_p(floor.data_ptr() + 4 * lists.n_query * j0),
             ctypes.c_void_p(lists.val.data_ptr() + per_job * j0), ctypes.c_void_p(lists.idx.data_ptr() + per_job * j0),
             int(engine), stream_ptr())
        return lists
    call("fgvc_affinity_topk", ptr(bank.buf), bank.fmt, bank.n_slots, bank.H, bank.W, bank.C,
         ctypes.c_void_p(jobs.data_ptr() + 16 * j0), j1 - j0, ptr(mem_feat), int(radius), mode, int(K), int(groups),
         ctypes.c_void_p(lists.val.data_ptr() + per_job * j0), ctypes.c_void_p(lists.idx.data_ptr() + per_job * j0),
         int(engine), stream_ptr())
    return lists


def sim_params(cfg_or_none, C, temperature, mode="softmax", sim_mode="dot_product", normalize=True):
    """(temperature, flags) for fgvc_gather_labels.  ``sim_mode='l2-distance'`` (local_attention.py:324-327)
    is (2ab - |a|^2)/sqrt(C): on L2-normalised features |a|^2 = 1, so it is a monotone map of the cosine --
    same top-k -- applied to the winners only; without normalisation it would need key norms: not built."""
    flags = 0
    if mode == "cosine":
        flags |= _lib.WEIGHT_COSINE
    elif mode != "softmax":
        raise ValueError(mode)
    if sim_mode == "l2-distance":
        if not normalize:
            raise NotImplementedError("sim_mode='l2-distance' needs normalize=True (unit vectors)")
        flags |= _lib.SIM_L2
        temperature = float(C) ** 0.5
    elif sim_mode != "dot_product":
        raise AssertionError(sim_mode)
    return float(temperature), flags


def gather_labels(lists, table, job_begin, job_end, labels, temperature, flags=0):
    """K1b for jobs [job_begin, job_end): writes each job's out_slot of ``labels``."""
    dev = labels.buf.device
    jobs, _, mem_label = table.device(dev)
    call("fgvc_gather_labels", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, ptr(jobs), int(job_begin),
         int(job_end), ptr(mem_label), labels.H * labels.W, float(temperature), int(flags), ptr(labels.buf),
         labels.Lp, stream_ptr())


def dense_propagate(bank, table, job_begin, job_end, labels, radius, temperature, flags=0, mask_mode="circle"):
    """topk=None (local_attention.py:376-383): soft-max / clamp^2 over ALL allowed candidates, written straight
    into each job's out_slot of ``labels``."""
    dev = labels.buf.device
    jobs, mem_feat, mem_label = table.device(dev)
    mode = _lib.MASK_CIRCLE if mask_mode == "circle" else _lib.MASK_SQUARE
    call("fgvc_dense_propagate", ptr(bank.buf), bank.fmt, bank.H, bank.W, bank.C,
         ctypes.c_void_p(jobs.data_ptr() + 16 * int(job_begin)), int(job_end - job_begin), ptr(mem_feat), ptr(mem_label),
         int(radius), mode, float(temperature), int(flags), ptr(labels.buf), labels.Lp, stream_ptr())


def heatmap_coords(maps, out_hw, topk=5):
    """K3: maps [n,H,W] fp32 CUDA -> [n,2] (x,y) after bilinear up-sampling to out_hw."""
    maps = maps.contiguous()
    n, H, W = maps.shape
    out = torch.empty(n, 2, dtype=torch.float32, device=maps.device)
    call("fgvc_heatmap_coords", ptr(maps), n, H, W, int(out_hw[0]), int(out_hw[1]), int(topk), ptr(out), stream_ptr())
    return out


def gaussian_coords(points_xy, out_hw, sigma=6.0, topk=5):
    pts = points_xy.to(dtype=torch.float32).contiguous()
    out = torch.empty(pts.shape[0], 2, dtype=torch.float32, device=pts.device)
    call("fgvc_gaussian_coords", ptr(pts), pts.shape[0], int(out_hw[0]), int(out_hw[1]), float(sigma), int(topk),
         ptr(out), stream_ptr())
    return out


def decode_masks(maps, out_hw):
    """VOS-style decode: maps [L,H,W] -> uint8 [h,w] (vanilla_tracker.py:769-798)."""
    maps = maps.contiguous()
    L, H, W = maps.shape
    scratch = torch.empty(2 * L, dtype=torch.float32, device=maps.device)
    out = torch.empty(out_hw[0], out_hw[1], dtype=torch.uint8, device=maps.device)
    call("fgvc_decode_masks", ptr(maps), L, H, W, int(out_hw[0]), int(out_hw[1]), ptr(scratch), ptr(out), stream_ptr())
    return out


def memory_frames(t, precede_frames, with_first=True, first=0):
    """Memory multiset of query frame t for a clip starting at ``first``
    (vanilla_tracker.py:346-362): the first frame is prepended even when the window
    already holds it."""
    win = list(range(max(first, t - precede_frames), t))
    return ([first] + win) if with_first else win


def query_job_table(t0s, T, precede_frames, with_first, bidirectional, unmasked):
    """Jobs of point groups queried at frames ``t0s`` of a T-frame clip (the grouping of VanillaTracker.forward_test,
    vanilla_tracker.py:249-295).  Per group the forward jobs t0+1 .. T-1 (memory_frames with first = t0), then with
    ``bidirectional`` the backward jobs t0-1 .. 0: the forward tracker on the time-reversed clip (query frame T-1-t0)
    mapped back to frame indices, memory [t0] + [min(t0, t + precede), ..., t + 1].  ``unmasked(mem)``: leading
    memory entries without the radius mask.  Returns (JobTable, spans) with spans[i] = (first job, t0) of group i."""
    table = JobTable()
    spans = []
    for t0 in t0s:
        spans.append((len(table), t0))
        for t in range(t0 + 1, T):
            mem = track_memory(t, t0, T, precede_frames, with_first)
            table.add(t, mem, mem, t, unmasked=unmasked(mem))
        if bidirectional:
            for t in range(t0 - 1, -1, -1):
                mem = track_memory(t, t0, T, precede_frames, with_first)
                table.add(t, mem, mem, t, unmasked=unmasked(mem))
    return table, spans


def track_memory(t, t0, T, precede_frames, with_first):
    """Memory frames of query frame t != t0 of a track that starts at t0 (query_job_table): forward (t > t0) the
    reference's memory_frames with first = t0, backward (t < t0) the same on the time-reversed clip."""
    if t > t0:
        return memory_frames(t, precede_frames, with_first, first=t0)
    return [T - 1 - r for r in memory_frames(T - 1 - t, precede_frames, with_first, first=T - 1 - t0)]


def cycle_end(t, t0, frames):
    """Frame where the cycle check of a prediction at t != t0 (test_cfg.cycle_occlusion) stops: ``frames`` steps from
    t toward the query frame t0, not past it; ``frames=None``: t0."""
    if frames is None:
        return t0
    return max(t0, t - frames) if t > t0 else min(t0, t + frames)


def cycle_job_table(table, spans, T, precede_frames, with_first, bidirectional, frames, unmasked):
    """Append the jobs of the cycle checks of every group of ``spans`` (query_job_table's (first job, t0) pairs) to
    ``table``.  The check of (group, t) re-tracks the prediction at t toward t0 with the tracker that starts at t --
    the backward one for t > t0, the forward one for t < t0 -- over the query frames between t and s = cycle_end(t, t0,
    frames): the jobs query_job_table([t], ..., bidirectional=True) has for those frames, in recurrence order.  Their
    label slots are local to the check's own bank: slot 0 = frame t, slot k = the frame of the k-th job (out_slot k).
    Returns the checks as (group index, t, s, first job, end job), longest first (consecutive checks then have similar
    lengths, which keeps the grid barriers of a chunk of them few)."""
    checks = []
    for g, (_, t0) in enumerate(spans):
        ts = list(range(t0 + 1, T)) + (list(range(t0 - 1, -1, -1)) if bidirectional else [])
        checks.extend((g, t, cycle_end(t, t0, frames)) for t in ts)
    checks.sort(key=lambda c: -abs(c[1] - c[2]))
    out = []
    for g, t, s in checks:
        step = -1 if s < t else 1
        jb = len(table)
        for q in range(t + step, s + step, step):
            mem = track_memory(q, t, T, precede_frames, with_first)
            table.add(q, mem, [abs(m - t) for m in mem], abs(q - t), unmasked=unmasked(mem))
        out.append((g, t, s, jb, len(table)))
    return out


def c2f_propagate(coarse, fine, table, job_index, fine_labels, radius, radius_fine, K, temperature,
                  mask_mode="circle", engine=_lib.ENGINE_AUTO):
    dev = coarse.buf.device
    jobs, mem_feat, mem_label = table.device(dev)
    hj = table.host_job(job_index)
    n_mem = hj.mem_end - hj.mem_begin
    nq = coarse.H * coarse.W
    out = torch.empty(nq, fine_labels.Lp, dtype=torch.float32, device=dev)
    n_scr = int(_lib.load().fgvc_c2f_scratch_elems(n_mem, nq))
    sv = torch.empty(n_scr, dtype=torch.float32, device=dev)
    si = torch.empty(n_scr, dtype=torch.int32, device=dev)
    mode = _lib.MASK_CIRCLE if mask_mode == "circle" else _lib.MASK_SQUARE
    jptr = ctypes.c_void_p(jobs.data_ptr() + 16 * job_index)
    call("fgvc_c2f_propagate", ptr(coarse.buf), coarse.fmt, coarse.n_slots, coarse.H, coarse.W, coarse.C, ptr(fine.buf),
         fine.fmt, fine.H, fine.W, fine.C,
         jptr, ctypes.byref(hj), ptr(mem_feat), ptr(mem_label), int(radius), mode, int(radius_fine), int(K),
         float(temperature), ptr(fine_labels.buf), fine_labels.Lp, ptr(out), ptr(sv), ptr(si), n_scr, int(engine),
         stream_ptr())
    return out


def check_ref_frame(ref_frame, T):
    """``ref_frame`` of a T-frame mask clip as an int in [0, T); ValueError otherwise."""
    if isinstance(ref_frame, bool) or not isinstance(ref_frame, (int, np.integer)) or not 0 <= int(ref_frame) < T:
        raise ValueError(f"ref_frame must be an int in [0, {T}), got {ref_frame!r}")
    return int(ref_frame)


class MaskClipPropagator:
    """VOS-style propagation of one clip with pre-allocated banks (the loop of
    vanilla_tracker.py:345-412 / :730-798 for mask labels): K0 over all frames, ONE K1 launch
    over all frames' jobs, then per frame K1b gather -> NCHW -> decode (bilinear up-sample,
    min-max normalise, argmax).  ``events=True`` records CUDA events around K1.

    ``ref_frame`` = t0: the annotated frame.  The masks of frames t0+1 .. T-1 are the propagation of the clip from t0
    on (memory_frames with first = t0), those of frames t0-1 .. 0 the propagation of the time-reversed clip from t0
    (track_memory); each half is bit for bit the run of this class with ref_frame = 0 on the sliced / the flipped clip
    when that run tiles K1 the same way (a shorter clip may pick more partial lists per job, plan_k1; exactly tied
    affinities may then be merged in another order).
    K1 runs once over both directions (no query tile mixes them), and the two tails are the two lanes of one
    fgvc_mask_clip_tail_lanes call: max(t0, T-1-t0) grid barriers instead of T-1.  ref_frame = 0 is the plain forward
    propagation through fgvc_mask_clip_tail."""

    def __init__(self, T, C, H, W, L, out_hw, cfg, device, engine_id=_lib.ENGINE_AUTO, split=None, ref_frame=0):
        self.T, self.C, self.H, self.W, self.L, self.out_hw, self.cfg = T, C, H, W, L, tuple(out_hw), cfg
        self.ref_frame = t0 = check_ref_frame(ref_frame, T)
        self.engine_id = engine_id
        self.device = device
        self.bank = FeatureBank(T, C, H, W, device, split=split or cfg.get("split"))
        self.labels = LabelBank(T, L, H, W, device)
        nr = cfg.get("neighbor_range", None)
        unmasked_first = 0 if cfg.get("with_first_neighbor", True) else 1
        # forward jobs t0+1 .. T-1, then backward jobs t0-1 .. 0 (with t0 = 0: today's jobs 1 .. T-1)
        self.table, _ = query_job_table([t0], T, cfg["precede_frames"], cfg.get("with_first", True), True,
                                        lambda mem: len(mem) if nr is None else unmasked_first)
        self.n_fwd = T - 1 - t0
        # the lanes of the tail: (job_begin, job_end) of each non-empty direction
        self.lanes = [(a, b) for a, b in ((0, self.n_fwd), (self.n_fwd, len(self.table))) if b > a]
        self.radius = (nr // 2) if nr is not None else 1
        # the tiling of K1 (jobs per tile, aligned memory classes, parts) is fixed per clip: it sizes the lists
        self.plan = plan_k1(self.bank, self.table, self.radius, cfg["topk"], cfg.get("mask_mode", "circle"),
                            engine=engine_id) if T > 1 else K1Plan()
        self.groups = self.plan.lists_per_job
        self.lists = TopKLists(max(1, len(self.table)), self.groups, H * W, cfg["topk"], device) if T > 1 else None
        self.table.device(device)
        self.maps = torch.empty(T, L, H, W, dtype=torch.float32, device=device)
        self.masks = torch.empty(T, out_hw[0], out_hw[1], dtype=torch.uint8, device=device)
        self.scratch = torch.empty(max(T, 1) * 2 * L, dtype=torch.float32, device=device)
        self.k1_events = None
        self._tail_stream = None
        # optional: K1 in a few launches with the gather chain of chunk i on a side stream under K1 of chunk
        # i+1.  Measured on config 2 it does not pay (the tail is real SM work, not latency): off by default, and
        # forward propagation (ref_frame = 0) only.
        self._overlap = (plan_overlap_chunks(len(self.table), (-(-H // 8)) * (-(-W // 16)))
                         if (T > 1 and t0 == 0 and cfg.get("overlap_tail", False)) else [])
        self._lanes_dev = None
        if t0 > 0:
            host = (_lib.Lane * len(self.lanes))(*[_lib.Lane(a, b, L, self.labels.Lp, 0, 0) for a, b in self.lanes])
            self._lanes_host = host
            self._lanes_dev = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(device)
        self.temperature, self.flags = sim_params(cfg, C, cfg["temperature"], sim_mode=cfg.get("sim_mode", "dot_product"),
                                                  normalize=cfg.get("with_norm", True))
        if cfg.get("hard_prop", False):
            self.flags |= _lib.HARD_PROP
        if cfg.get("local_window", False):       # HRVanillaTracker: square window, zero-padded candidates
            self.flags |= _lib.zero_pad_flags(self.radius, W)
        self.jobs_host = torch.tensor(self.table.jobs, dtype=torch.int32).reshape(-1, 4).contiguous()

    def _decode(self, t, masks=None):
        masks = self.masks if masks is None else masks
        call("fgvc_decode_masks_pixmajor", ptr(self.labels.buf), t, self.labels.Lp, self.L, self.H, self.W,
             self.out_hw[0], self.out_hw[1], ptr(self.scratch), ptr(masks[t]), stream_ptr())

    def _tail_lanes(self, want_maps):
        """both directions from ref_frame > 0: the two lanes of one fgvc_mask_clip_tail_lanes call over the one bank"""
        lists = self.lists
        jobs, _, mem_label = self.table.device(self.device)
        call("fgvc_mask_clip_tail_lanes", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, None, ptr(jobs),
             ptr(self.jobs_host), ptr(self._lanes_dev), ctypes.c_void_p(ctypes.addressof(self._lanes_host)),
             len(self.lanes), ptr(mem_label), self.H, self.W, self.temperature, self.flags, ptr(self.labels.buf),
             self.out_hw[0], self.out_hw[1], ptr(self.scratch), ptr(self.masks),
             ptr(self.maps) if want_maps else None,
             *chain_workspace(self.device, len(self.table), self.H * self.W, lists.K, self.flags,
                              force=not (self.flags & _lib.HARD_PROP)), stream_ptr())

    def _tail(self, j0, j1, want_maps, lists=None, masks=None):
        lists = lists or self.lists
        masks = self.masks if masks is None else masks
        jobs, _, mem_label = self.table.device(self.device)
        call("fgvc_mask_clip_tail", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups,
             ptr(jobs), ptr(self.jobs_host), j0, j1, ptr(mem_label), self.H, self.W,
             self.temperature, self.flags, ptr(self.labels.buf), self.labels.Lp, self.L, self.out_hw[0],
             self.out_hw[1], ptr(self.scratch), ptr(masks), ptr(self.maps) if want_maps else None,
             *chain_workspace(self.device, j1 - j0, self.H * self.W, lists.K, self.flags), stream_ptr())

    def _k1(self, j0, j1, lists=None):
        cfg = self.cfg
        lists = lists or self.lists
        # both directions: no query tile mixes them, so each gets the lists (and the K1 cost) of a run of its own
        affinity_topk(self.bank, self.table, self.radius, cfg["topk"], cfg.get("mask_mode", "circle"),
                      engine=self.engine_id, lists=lists, job_range=(j0, j1), plan=self.plan,
                      cuts=self.lanes if self.ref_frame > 0 else None)

    def run(self, feats, onehot, events=False, want_maps=True):
        """feats [T,C,H,W] fp32 CUDA; onehot [L,H,W] fp32 CUDA, the labels of frame ``ref_frame``.  Returns (maps,
        masks); ``want_maps=False`` skips the NCHW copies of the propagated label maps."""
        cfg = self.cfg
        t0 = self.ref_frame
        self.bank.load_frames(feats, 0, normalize=cfg.get("with_norm", True))
        self.labels.put_nchw(onehot, t0)
        if want_maps:
            self.maps[t0].copy_(onehot)
        self._decode(t0)
        if self.T > 1:
            if events:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            if t0 > 0:
                self._k1(0, len(self.table))
                if events:
                    e1.record()
                self._tail_lanes(want_maps)
            elif len(self._overlap) <= 1:
                self._k1(0, len(self.table))
                if events:
                    e1.record()
                self._tail(0, len(self.table), want_maps)
            else:
                # K1 in a few launches on this stream; the sequential gather chain + decode of chunk i run
                # on a high-priority side stream while K1 of chunk i+1 keeps the SMs busy
                if self._tail_stream is None:
                    self._tail_stream = torch.cuda.Stream(device=self.device, priority=-1)
                cur = torch.cuda.current_stream()
                side = self._tail_stream
                side.wait_stream(cur)                      # label bank slot 0 / previous use of the buffers
                for (j0, j1) in self._overlap:
                    self._k1(j0, j1)
                    ev = torch.cuda.Event()
                    ev.record(cur)
                    with torch.cuda.stream(side):
                        side.wait_event(ev)
                        self._tail(j0, j1, want_maps)
                if events:
                    e1.record()
                cur.wait_stream(side)
            if events:
                self.k1_events = (e0, e1)
        return (self.maps if want_maps else None), self.masks

    def run_host(self, feats_host, onehot_host, masks_host, chunks=None):
        """End-to-end form: PINNED host features [T,C,H,W] / one-hot [L,H,W] in, uint8 masks
        [T,h,w] out to pinned host memory.  Two levels of overlap, nothing synchronises the host:
          * within a clip the host->device copy of job chunk i+1 (copy stream) overlaps K0 + K1 + tail of chunk
            i -- a frame's jobs only need earlier frames.  ``chunks``: list of (job_begin, job_end); default =
            :func:`plan_chunks` (best latency of ONE clip);
          * across clips the staging buffers are double-buffered, so the copies of the NEXT call start while this
            call still computes (they only wait for the K0 launches that read the same staging buffer two calls
            ago).  For a stream of clips ``chunks=[(0, n_jobs)]`` is then the fastest plan: the copies are
            hidden behind the previous clip and K1 runs as one launch.
        The chunked upload relies on every job reading earlier frames only: ``ref_frame > 0`` (backward jobs read
        later frames) raises NotImplementedError; use ``run`` for it."""
        if self.ref_frame != 0:
            raise NotImplementedError("run_host propagates from frame 0 only; use run() for ref_frame > 0")
        cfg = self.cfg
        if not hasattr(self, "_stage"):
            self._stage = [torch.empty(self.T, self.C, self.H, self.W, dtype=torch.float32, device=self.device)
                           for _ in range(2)]
            self._onehot = [torch.empty(self.L, self.H, self.W, dtype=torch.float32, device=self.device)
                            for _ in range(2)]
            self._stage_free = [None, None]                         # last K0 that read the buffer
            self._masks2 = [self.masks, torch.empty_like(self.masks)]   # device masks, one per call in flight
            self._masks_free = [None, None]                         # last device->host copy that read the buffer
            self._flip = 0
            self._copy = torch.cuda.Stream(device=self.device)
            self._back = torch.cuda.Stream(device=self.device)      # device->host copies of finished masks
            self._chunks = plan_chunks(len(self.table), (-(-self.H // 8)) * (-(-self.W // 16))) if self.T > 1 else []
        chunks = chunks or self._chunks
        cur = torch.cuda.current_stream()
        b = self._flip
        self._flip ^= 1
        stage, onehot, masks_dev = self._stage[b], self._onehot[b], self._masks2[b]
        if self._masks_free[b] is not None:
            cur.wait_event(self._masks_free[b])           # (two calls ago: long done)
        if self._stage_free[b] is not None:
            self._copy.wait_event(self._stage_free[b])    # staging buffer b free again
        else:
            self._copy.wait_stream(cur)
        evs = []
        with torch.cuda.stream(self._copy):
            onehot.copy_(onehot_host, non_blocking=True)
            f0 = 0
            for (j0, j1) in (chunks or [(0, 0)]):
                f1 = j1 + 1 if j1 > j0 else self.T          # job j propagates frame j + 1
                stage[f0:f1].copy_(feats_host[f0:f1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy)
                evs.append((f0, f1, j0, j1, ev))
                f0 = f1
        for n, (f0, f1, j0, j1, ev) in enumerate(evs):
            cur.wait_event(ev)
            self.bank.load_frames(stage[f0:f1], f0, normalize=cfg.get("with_norm", True))
            if f0 == 0:
                self.labels.put_nchw(onehot, 0)
                self._decode(0, masks_dev)
            if n == len(evs) - 1:
                free = torch.cuda.Event()
                free.record(cur)
                self._stage_free[b] = free
            if j1 > j0:
                self._k1(j0, j1)
                self._tail(j0, j1, False, masks=masks_dev)
            # ship the masks of this chunk while the next chunk / the next clip computes (PCIe is full duplex)
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(self._back):
                self._back.wait_event(done)
                m0 = 0 if f0 == 0 else f0
                masks_host[m0:f1].copy_(masks_dev[m0:f1], non_blocking=True)
                if n == len(evs) - 1:
                    mf = torch.cuda.Event()
                    mf.record(self._back)
                    self._masks_free[b] = mf
        return masks_host

    def join_host(self):
        """Make the current stream wait for the device->host copies of every ``run_host`` call so far (the
        caller synchronises that stream, or the device, before reading ``masks_host``)."""
        if hasattr(self, "_back"):
            torch.cuda.current_stream().wait_stream(self._back)
