"""Drop-in test-time tracker: same constructor and ``forward_test`` contract as the
reference's ``VanillaTracker`` (mmpt/models/trackers/vanilla_tracker.py:75-412,
``BaseModel.forward`` mmpt/models/trackers/base.py:44-60), label propagation on the
B200 kernels.

What changes relative to the reference loop (results identical, see tests):
  * the clip is encoded ONCE for all ``with_first`` groups and the features stay in HBM
    (reference: re-encodes per group and parks features on the CPU, :133-153, :262-284);
  * affinity + mask + top-k of EVERY (group, frame) job is one kernel launch -- it does
    not depend on the propagated labels (SURVEY.md section 8e); only the cheap gather is
    sequential in time;
  * heat-maps are never up-sampled into a [T,P,h,w] tensor nor shipped to the host:
    K3 fuses the bilinear up-sampling with the top-5 soft-argmax (:396-406, :172-191).
"""
import os

import torch
import torch.nn as nn

from . import _lib, engine
from .encoder import build_backbone
from .engine import FeatureBank, LabelBank


class _Cfg(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


class VanillaTracker(nn.Module):
    """Pixel tracker; ``eval_arc='B200VanillaTracker'`` selects it in tools/test.py when
    registered in mmpt's MODELS registry (see INTEGRATION.md)."""

    def __init__(self, backbone, head=None, train_cfg=None, test_cfg=None, init_cfg=None):
        super().__init__()
        self.backbone = build_backbone(backbone)
        # The reference runs self.head(x) in extract_feat when a head is configured and concatenates every block with
        # test_cfg.all_blocks (vanilla_tracker.py:86-124).  Neither is built: fail loudly instead of silently feeding
        # different features (the shipped eval config, res18_d1_eval, uses neither).
        if head is not None:
            raise NotImplementedError("VanillaTracker(head=...) is not built: the encoder side is plain PyTorch and "
                                      "only the head-less eval configuration is mirrored")
        if test_cfg is not None and (test_cfg.get("all_blocks", False) if hasattr(test_cfg, "get") else False):
            raise NotImplementedError("test_cfg.all_blocks is not built")
        self.head = head
        self.train_cfg = train_cfg
        self.test_cfg = test_cfg if hasattr(test_cfg, "get") and hasattr(test_cfg, "precede_frames") \
            else _Cfg(test_cfg or {})
        self.stride_sample = self.test_cfg.get("stride_sample", False)
        self.engine_id = self.test_cfg.get("engine", _lib.ENGINE_AUTO)
        self.cycle_cfg()                              # a malformed cycle_occlusion fails here, not after the encoder
        self.register_buffer("iteration", torch.tensor(0, dtype=torch.float))

    def init_weights(self):
        if hasattr(self.backbone, "init_weights"):
            self.backbone.init_weights()

    # ------------------------------------------------------------------ BaseModel.forward
    def forward(self, test_mode=False, **kwargs):
        if test_mode:
            return self.forward_test(**kwargs)
        return self.forward_train(**kwargs)

    def forward_train(self, imgs, labels=None):
        raise NotImplementedError

    # ------------------------------------------------------------------------- encoder
    def extract_feat(self, imgs):
        x = self.backbone(imgs)
        if self.stride_sample:
            x = x[:, :, ::self.stride_sample, ::self.stride_sample]
        return x

    @torch.no_grad()
    def get_feats(self, frames):
        """frames [T,3,h,w] -> [T,C,Hf,Wf] on the device, in chunks of ``batch_step``
        (vanilla_tracker.py:133-153 without the round trip through host memory)."""
        step = self.test_cfg.get("batch_step", 5)
        outs = []
        for s in range(0, frames.shape[0], step):
            f = self.extract_feat(frames[s:s + step])
            if isinstance(f, (tuple, list)):
                f = f[0]
            outs.append(f.float())
        return torch.cat(outs, dim=0)

    @torch.no_grad()
    def encode_to_bank(self, frames, n_levels=1):
        """frames [T,3,h,w] -> FeatureBank of the clip, encoder and K0 overlapped: the (PyTorch) encoder runs on the
        current stream in chunks of ``batch_step`` frames (vanilla_tracker.py:133-153), and K0 (normalise + split +
        pixel-major) of chunk i runs on a side stream while the encoder works on chunk i + 1.  Features go straight
        into the bank: the [T,C,Hf,Wf] fp32 tensor of the whole clip (the reference moves it to the host and back)
        is never assembled.  ``test_cfg.encoder_channels_last`` runs the encoder in channels-last memory format.

        ``n_levels > 1``: the encoder returns that many output levels (a tuple, in ``out_indices`` order), each goes
        into a bank of its own (with its own ``engine.default_split`` unless ``test_cfg.split`` forces one), and the
        list of banks is returned."""
        cfg = self.test_cfg
        step = cfg.get("batch_step", 5)
        T = frames.shape[0]
        cur = torch.cuda.current_stream()
        if getattr(self, "_k0_stream", None) is None:
            self._k0_stream = torch.cuda.Stream(device=frames.device)
        side = self._k0_stream
        side.wait_stream(cur)
        banks = None
        for s0 in range(0, T, step):
            x = frames[s0:s0 + step]
            if cfg.get("encoder_channels_last", False):
                x = x.contiguous(memory_format=torch.channels_last)
            f = self.extract_feat(x)
            fs = list(f) if isinstance(f, (tuple, list)) else [f]
            fs = [t.float().contiguous() for t in fs[:n_levels]]
            if banks is None:
                banks = [FeatureBank(T, t.shape[1], t.shape[2], t.shape[3], frames.device, split=cfg.get("split"))
                         for t in fs]
            ready = torch.cuda.Event()
            ready.record(cur)
            with torch.cuda.stream(side):
                side.wait_event(ready)
                for bank, t in zip(banks, fs):
                    bank.load_frames(t, s0, normalize=cfg.get("with_norm", cfg.get("withnorm", True)))
            for t in fs:
                t.record_stream(side)
        cur.wait_stream(side)
        return banks[0] if n_levels == 1 else banks

    def _stream_in(self, feats_host, bank, table, t0, radius, mask_mode, normalize, n_chunks=6):
        """Host features of ONE clip -> feature bank and top-k lists, pipelined: the frames are copied in chunks on a
        side stream (two staging buffers); on the compute stream K0 of a chunk and K1 of the jobs whose query frame
        lies in it follow as soon as it has landed (a job only reads frames before its own), so the host link and the
        kernels overlap inside a single clip.  Same lists as one K1 launch over the whole table."""
        cfg = self.test_cfg
        dev = bank.buf.device
        T = feats_host.shape[0]
        cur = torch.cuda.current_stream()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        cp = self._copy_stream
        plan = engine.plan_k1(bank, table, radius, cfg.topk, mask_mode, engine=self.engine_id)
        lists = engine.TopKLists(len(table), plan.lists_per_job, bank.H * bank.W, cfg.topk, dev)
        step = -(-T // n_chunks)
        # the two staging buffers live across calls (a stream of clips): the first copy of the next clip then only waits
        # for the K0 that last read its buffer, not for the previous clip's whole tail
        key = (step,) + tuple(feats_host.shape[1:]) + (dev.index,)
        if getattr(self, "_stage_key", None) != key:
            self._stage = [torch.empty(key[:-1], dtype=torch.float32, device=dev) for _ in range(2)]
            self._stage_free, self._stage_key = [None, None], key
            cp.wait_stream(cur)                           # fresh memory: earlier kernels of this stream may still use it
        stage, free = self._stage, self._stage_free
        for i, a in enumerate(range(0, T, step)):
            b = min(T, a + step)
            buf = stage[i % 2][:b - a]
            with torch.cuda.stream(cp):
                if free[i % 2] is not None:
                    cp.wait_event(free[i % 2])            # K0 of the chunk that used this buffer has read it
                buf.copy_(feats_host[a:b], non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(cp)
            cur.wait_event(ready)
            bank.load_frames(buf, a, normalize=normalize)
            free[i % 2] = torch.cuda.Event()
            free[i % 2].record(cur)
            j0, j1 = max(a, t0 + 1) - (t0 + 1), b - (t0 + 1)   # jobs of this group: job j <-> query frame t0 + 1 + j
            if j1 > j0:
                engine.affinity_topk(bank, table, radius, cfg.topk, mask_mode, engine=self.engine_id, lists=lists,
                                     job_range=(j0, j1), plan=plan)
        return lists

    # --------------------------------------------------------------------- propagation
    two_phase_sharding = True      # apis.sharded_forward_test: forward_test(..., shard=(rank, world))
    local_window = False           # HRVanillaTracker: square window + zero-padded candidates

    @torch.no_grad()
    def propagate_points(self, feats, groups, image_hw, shard=None, return_cycle=False):
        """feats [T,C,Hf,Wf] (CUDA); groups: list of (t0, points_xy [P',2]).
        Returns list of [T,P',2] float64 CUDA tensors (zeros before t0).
        ``shard=(rank, world)``: two-phase split of ONE video over the default process group (SURVEY 8e): K1 runs for
        this rank's frame range only and the top-k lists are all-gathered; the recurrent tail runs for this rank's
        slice of every group's points and the tracks are all-gathered.  Every rank returns the full result.

        ``test_cfg.cycle_occlusion = dict(frames=H, threshold=delta)``: forward-backward cycle check of every
        prediction (INTEGRATION.md section 2).  Returns (tracks, visibility) then: visibility = per group a [T,P'] bool
        tensor, True at the query frame and where the prediction at t, re-tracked from t toward t0 for H frames
        (None: back to t0) and stopping at s, lands within delta image pixels of the track at s; False where there
        is no prediction (t < t0 without ``bidirectional``).  ``return_cycle=True`` adds per group the [T,P',2]
        float64 re-tracked positions (row t holds the one at s, zeros where there is no check)."""
        cfg = self.test_cfg
        cyc = self.cycle_cfg()
        host_feats = False
        if isinstance(feats, FeatureBank):               # encode_to_bank: K0 already ran, overlapped with the encoder
            pre_bank = feats
            T, C, Hf, Wf, dev = pre_bank.n_slots, pre_bank.C, pre_bank.H, pre_bank.W, pre_bank.buf.device
        else:
            pre_bank = None
            T, C, Hf, Wf = feats.shape
            dev = feats.device
            if not feats.is_cuda:                        # host features (pinned): staged in frame chunks, see below
                _lib.require_cuda()
                host_feats, dev = True, torch.device("cuda", torch.cuda.current_device())
        h, w = image_hw
        stride = h // Hf
        precede = cfg.precede_frames
        with_first_mem = cfg.get("with_first", True)
        v1 = cfg.get("test_mode", "v1") == "v1"
        nr = cfg.get("neighbor_range", None)
        if nr is None and not v1:
            raise TypeError("test_mode v2 needs neighbor_range (the reference computes neighbor_range//2)")
        unmasked_first = 0 if (cfg.get("with_first_neighbor", True) or not v1) else 1
        # masked_attention_efficient_v2 always uses the circular dist < radius mask and has no sim_mode
        # (local_attention.py:392-508): a v2 config with other settings must not change the result
        mask_mode = cfg.get("mask_mode", "circle") if v1 else "circle"
        if self.local_window:
            mask_mode, unmasked_first = "square", 0          # (2r+1)^2 window around the query position, every frame
        temperature, flags = engine.sim_params(cfg, C, cfg.temperature,
                                               sim_mode=cfg.get("sim_mode", "dot_product") if v1 else "dot_product",
                                               normalize=cfg.get("with_norm", True))

        if self.local_window:
            if nr is None:
                raise TypeError("the local-window tracker needs neighbor_range")
            # window positions outside the image stay candidates (affinity 0, value 0): merged by the gather
            flags |= _lib.zero_pad_flags(nr // 2, Wf)
        normalize = cfg.get("with_norm", cfg.get("withnorm", True))
        if pre_bank is not None:
            bank = pre_bank
        else:
            bank = FeatureBank(T, C, Hf, Wf, dev, split=cfg.get("split"))
            if not host_feats and (shard is None or shard[1] == 1):
                bank.load_frames(feats, 0, normalize=normalize)

        bidirectional = bool(cfg.get("bidirectional", False))
        # per group: (first job, t0); forward jobs t0+1 .. T-1, then (bidirectional) backward jobs t0-1 .. 0
        unmasked = lambda mem: len(mem) if nr is None else unmasked_first       # noqa: E731
        table, spans = engine.query_job_table([t0 for t0, _ in groups], T, precede, with_first_mem, bidirectional,
                                              unmasked)
        n_track = len(table)
        # cycle checks: their jobs follow the tracking jobs in the same table, so one K1 launch covers both and a list
        # the tracks need already is not scored twice
        checks = None
        if cyc is not None and n_track:
            checks = engine.cycle_job_table(table, spans, T, precede, with_first_mem, bidirectional, cyc["frames"],
                                            unmasked)
        radius = (nr // 2) if nr is not None else 1
        rank, world = shard if shard is not None else (0, 1)
        # several groups: the label-independent K1 work is shared between the groups (one list per (query frame,
        # memory frame) pair); FGVC_NO_SHARE=1 keeps one K1 job per (group, frame).  Whether it is shared is decided
        # on the tracking jobs alone, so that the cycle checks leave the tracks bit for bit as they are
        shared = None
        if len(groups) > 1 and n_track > 0 and os.environ.get("FGVC_NO_SHARE") != "1":
            shared = engine.shared_pair_table(table, spans, T, decide_jobs=n_track,
                                              max_entries=64 if checks is not None else None)
        # (the streamed path needs every job to read only earlier frames: forward jobs only)
        streamed = host_feats and len(groups) == 1 and world == 1 and len(table) > 0 and not bidirectional and \
            checks is None
        if host_feats and not streamed and world == 1:
            bank.load_frames(feats.to(dev, non_blocking=True), 0, normalize=normalize)
        if streamed:
            lists = self._stream_in(feats, bank, table, groups[0][0], radius, mask_mode, normalize)
        elif len(table) == 0:
            lists = None
        elif world > 1:
            from . import apis
            ktable = shared[0] if shared is not None else table
            plan = engine.plan_k1(bank, ktable, radius, cfg.topk, mask_mode, engine=self.engine_id,
                                  groups=shared[1] if shared is not None else None, pack=shared is None,
                                  job_range=(0, n_track) if (shared is None and checks is not None) else None)
            lo, hi, per = apis.frame_shard(len(ktable), rank, world)
            lists = engine.TopKLists(per * world, plan.lists_per_job, Hf * Wf, cfg.topk, dev)
            if pre_bank is None:
                # phase 1 only reads the frames of this rank's jobs (query frames + their memories) and phase 2 reads no
                # features at all: a rank uploads (host features) and prepares ~T / world + precede frames instead of
                # the whole clip
                for a, b_ in engine.frame_runs(ktable, lo, hi):
                    bank.load_frames(feats[a:b_].to(dev, non_blocking=True), a, normalize=normalize)
            if hi > lo:
                engine.affinity_topk(bank, ktable, radius, cfg.topk, mask_mode, engine=self.engine_id, lists=lists,
                                     job_range=(lo, hi), plan=plan,
                                     cuts=[(0, n_track), (n_track, len(ktable))] if shared is None else None)
            apis.gather_job_lists(lists.val, per, rank, world)
            apis.gather_job_lists(lists.idx, per, rank, world)
        else:
            if shared is not None:
                utable, gmax, _ = shared
                # every list of a query frame t starts from the K-th best of the query's 5 x 5 neighbourhood in frame
                # t - 1 (t + 1 for the backward jobs), which is in the memory of every group that is alive at t: without
                # it the per-pair lists start cold and half of the launch is list insertion
                floor = None
                if os.environ.get("FGVC_NO_FLOOR") != "1" and radius >= 3:
                    # the frame nearest to t that EVERY job of a (query frame, direction) has in its memory (-1: none,
                    # no floor)
                    common = {}
                    for job in table.jobs:
                        key = engine.pair_key(table, job)
                        mem = {r & ~_lib.MEM_UNMASKED for r in table.mem_feat[job[1]:job[2]]}
                        common[key] = mem if key not in common else (common[key] & mem)
                    seeds = []
                    for job in utable.jobs:
                        key = engine.pair_key(utable, job)
                        seeds.append((min if key[1] else max)(common.get(key, set()), default=-1))
                    floor = engine.topk_floor(bank, utable, seeds, radius, cfg.topk, mask_mode)
                lists = engine.affinity_topk(bank, utable, radius, cfg.topk, mask_mode, groups=gmax,
                                             engine=self.engine_id, pack=False, floor=floor)
            elif checks is not None:
                # the tiling of the tracking jobs alone (jobs per tile, lists per job), and no query tile mixes them
                # with the checks' jobs: the tracks get the lists they get without the checks
                plan = engine.plan_k1(bank, table, radius, cfg.topk, mask_mode, job_range=(0, n_track),
                                      engine=self.engine_id)
                lists = engine.affinity_topk(bank, table, radius, cfg.topk, mask_mode, engine=self.engine_id, plan=plan,
                                             cuts=[(0, n_track), (n_track, len(table))])
            else:
                lists = engine.affinity_topk(bank, table, radius, cfg.topk, mask_mode, engine=self.engine_id)
        pair_ref = torch.tensor(shared[2], dtype=torch.int32, device=dev) if shared is not None else None
        # coordinates of the query frames (soft-argmax of the analytic gaussian, :321-343): one launch for all groups
        all_pts = torch.cat([pts.to(device=dev, dtype=torch.float32) for _, pts in groups], dim=0) if groups else None
        all_c0 = engine.gaussian_coords(all_pts, (h, w)) if groups and all_pts.shape[0] else None
        outs, coords, parts = self._point_tail(lists, pair_ref, table, spans, groups, all_pts, all_c0, rank, world, T,
                                               Hf, Wf, (h, w), stride, temperature, flags, bidirectional, dev)
        if cyc is not None:
            # per group [T, P_rank, 2] positions and flags of the checks, cycle position in channels 2-3, flag in 4
            cyc_xy, vis = self._cycle_tail(lists, pair_ref, table, checks, parts, coords, T, Hf, Wf, (h, w), stride,
                                           temperature, flags, cyc["threshold"], dev)
            outs = [torch.cat([o.double(), c.double(), v[..., None].double()], dim=-1) for o, c, v in zip(outs, cyc_xy, vis)]
        else:
            outs = [o.double() for o in outs]
        if world > 1:
            from . import apis
            sizes = [int(pts.shape[0]) for _, pts in groups]
            pads = [-(-n // world) for n in sizes]
            local = torch.zeros(T, sum(pads), outs[0].shape[-1] if outs else 2, dtype=torch.float64, device=dev)
            off = 0
            for o, pad in zip(outs, pads):
                local[:, off:off + o.shape[1]] = o
                off += pad
            outs = apis.gather_point_tracks(local, sizes, rank, world)
        if cyc is None:
            return outs
        tracks, vis = [o[..., :2].contiguous() for o in outs], [o[..., 4] != 0 for o in outs]
        if return_cycle:
            return tracks, vis, [o[..., 2:4].contiguous() for o in outs]
        return tracks, vis

    def cycle_cfg(self):
        """``test_cfg.cycle_occlusion`` checked: dict(frames=positive int or None, threshold=float >= 0,
        max_bytes=device bytes the checks of one chain call may use, default half of what is free), or None."""
        c = self.test_cfg.get("cycle_occlusion")
        if c is None:
            return None
        unknown = set(c) - {"frames", "threshold", "max_bytes"}
        if unknown or "threshold" not in c:
            raise TypeError(f"test_cfg.cycle_occlusion takes frames, threshold (required) and max_bytes, got {dict(c)}")
        frames = c.get("frames")
        if frames is not None and (isinstance(frames, bool) or int(frames) != frames or frames < 1):
            raise ValueError(f"cycle_occlusion.frames must be a positive int or None, got {frames!r}")
        if not float(c["threshold"]) >= 0:
            raise ValueError(f"cycle_occlusion.threshold must be >= 0, got {c['threshold']!r}")
        return dict(frames=None if frames is None else int(frames), threshold=float(c["threshold"]),
                    max_bytes=c.get("max_bytes"))

    def _cycle_tail(self, lists, pair_ref, table, checks, parts, coords, T, Hf, Wf, image_hw, stride, temperature, flags,
                    threshold, dev):
        """Cycle checks of this rank's points after the tracking tail (they start from its tracks): per check one lane
        of a multi-lane gather chain over its own bank (engine.point_cycle_lanes), in chunks of checks whose buffers
        fit ``max_bytes`` -- one chain call per chunk.  Returns per group the [T, P_rank, 2] float32 cycle positions and
        the [T, P_rank] uint8 flags (1 at the query frame)."""
        cyc_coords = torch.zeros_like(coords)
        vis = torch.zeros(coords.numel() // 2, dtype=torch.uint8, device=dev)
        c_offs, off = [], 0
        for _, t0, _, P in parts:
            c_offs.append(off)
            vis[off // 2 + t0 * P:off // 2 + (t0 + 1) * P] = 1            # visible at the query frame
            off += T * P * 2
        lanes = [(jb, je, parts[g][3], c_offs[g], t, s) for g, t, s, jb, je in (checks or []) if parts[g][3]]
        budget = self.cycle_cfg()["max_bytes"]
        if budget is None:
            free, _ = torch.cuda.mem_get_info(dev)
            budget = (free + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)) // 2
        n_pix = Hf * Wf
        i = 0
        while i < len(lanes):
            # a chunk: consecutive checks (consecutive jobs) while they fit the budget (at least one)
            j, used = i, 0
            while j < len(lanes):
                jb, je, L = lanes[j][:3]
                need = engine.cycle_lane_bytes(je - jb, L, n_pix, lists.K)
                if j > i and (used + need > budget or je - lanes[i][0] > 65535):
                    break
                used += need
                j += 1
            engine.point_cycle_lanes(lists, pair_ref, table, lanes[i:j], coords, cyc_coords, vis, Hf, Wf,
                                     image_hw, stride, temperature, flags, threshold)
            i = j
        cyc_out, vis_out = [], []
        for (_, t0, _, P), c in zip(parts, c_offs):
            cyc_out.append(cyc_coords[c:c + T * P * 2].view(T, P, 2))
            vis_out.append(vis[c // 2:c // 2 + T * P].view(T, P))
        return cyc_out, vis_out

    def _point_tail(self, lists, pair_ref, table, spans, groups, all_pts, all_c0, rank, world, T, Hf, Wf, image_hw, stride,
                    temperature, flags, bidirectional, dev):
        """Recurrent tail: every group of this rank's points is tracked forward from its query frame and, with
        ``test_cfg.bidirectional``, backward to frame 0 -- a lane per direction over the group's label bank (both read
        slot t0 and write disjoint slots).  All banks and tracks are carved out of one allocation each, and every lane
        of the clip runs in ONE gather chain (engine.point_tail_lanes).  Returns per group the [T, P_rank, 2] float32
        tracks (rows that no lane writes stay zero), the flat buffer they are views of, and per group (first job, t0,
        first point in all_pts, points of this rank)."""
        n_pix = Hf * Wf
        parts, p_off = [], 0               # per group: (first job, t0, first point in all_pts, points of this rank)
        for (j0, t0), (_, pts) in zip(spans, groups):
            P_all = int(pts.shape[0])
            lo_p, hi_p = (0, P_all) if world == 1 else ((P_all * rank) // world, (P_all * (rank + 1)) // world)
            parts.append((j0, t0, p_off + lo_p, hi_p - lo_p))
            p_off += P_all
        lab = torch.empty(sum(T * n_pix * engine.pad4(P) for *_, P in parts), dtype=torch.float32, device=dev)
        coords = torch.zeros(sum(T * P * 2 for *_, P in parts), dtype=torch.float32, device=dev)
        lanes, outs, lab_off, c_off = [], [], 0, 0
        for j0, t0, a, P in parts:
            track = coords[c_off:c_off + T * P * 2].view(T, P, 2)
            outs.append(track)
            if P:
                labels = LabelBank(T, P, Hf, Wf, dev, buf=lab[lab_off:lab_off + T * n_pix * engine.pad4(P)])
                labels.put_gaussians(all_pts[a:a + P], t0, stride)
                track[t0] = all_c0[a:a + P]
                n_fw = T - t0 - 1
                # the forward lane, then (bidirectional: the table holds the group's backward jobs) the backward lane
                for jb, je in ((j0, j0 + n_fw), (j0 + n_fw, j0 + T - 1))[:2 if bidirectional else 1]:
                    if je > jb:
                        lanes.append((jb, je, P, lab_off, c_off))
            lab_off += T * n_pix * engine.pad4(P)
            c_off += T * P * 2
        if lanes:
            maps = torch.empty(T * max(ln[2] for ln in lanes) * n_pix, dtype=torch.float32, device=dev)   # NCHW scratch
            engine.point_tail_lanes(lists, pair_ref, table, lanes, lab, maps, coords, Hf, Wf, image_hw, temperature, flags)
        return outs, coords, parts

    def forward_test(self, rgbs, query_points, trajectories, visibilities, save_image=False, save_path=None,
                     iteration=None, shard=None):
        """rgbs [1,T,3,h,w]; query_points [1,P,3] (t,x,y); trajectories [1,T,P,2];
        visibilities [1,T,P].  Returns the reference's 5-tuple
        (traj_gt, vis_gt, traj_pred, vis_pred, query_points), re-ordered by query frame
        when ``test_cfg.with_first`` is set (vanilla_tracker.py:227-303)."""
        _lib.require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        rgbs, query_points = rgbs.to(dev), query_points.to(dev)
        trajectories, visibilities = trajectories.to(dev), visibilities.to(dev)
        assert rgbs.shape[0] == 1
        B, T = rgbs.shape[:2]
        h, w = rgbs.shape[-2:]
        feats = self.encode_to_bank(rgbs[0])           # FeatureBank: encoder chunks overlapped with K0
        cycle = self.cycle_cfg() is not None
        if not self.test_cfg.get("with_first", False):
            out = self.propagate_points(feats, [(0, query_points[0, :, 1:])], (h, w), shard=shard)
            traj, vis_pred = (out[0][0], out[1][0][None].to(visibilities.dtype)) if cycle else \
                (out[0], torch.zeros_like(visibilities))
            return trajectories, visibilities, traj[None], vis_pred, query_points
        qt = query_points[0, :, 0]
        ts = torch.unique(qt).tolist()
        order = [torch.nonzero(qt == t).flatten() for t in ts]
        groups = [(int(t), query_points[0, idx, 1:]) for t, idx in zip(ts, order)]
        out = self.propagate_points(feats, groups, (h, w), shard=shard)
        trajs = out[0] if cycle else out
        perm = torch.cat(order)
        pred = torch.cat(trajs, dim=1).to(trajectories.dtype)[None]
        vis_pred = torch.cat(out[1], dim=1)[None].to(visibilities.dtype) if cycle else torch.zeros_like(visibilities)
        return (trajectories[:, :, perm], visibilities[:, :, perm], pred, vis_pred, query_points[:, perm])

    # -------------------------------------------------- VOS-style entry (mask labels)
    @torch.no_grad()
    def propagate_masks(self, feats, ref_seg, out_hw, num_classes=None, ref_frame=0):
        """feats [T,C,Hf,Wf]; ref_seg int [Hf,Wf]: the mask of frame ``ref_frame`` (default: the first frame), already
        at feature resolution.  Returns (label maps [T,L,Hf,Wf], uint8 masks [T,h,w]) with the decode of
        vanilla_tracker.py:769-798.  With ref_frame = t0 > 0 the frames after t0 are propagated forward from t0 and
        the frames before it backward (the forward propagation of the time-reversed clip from t0), in one call."""
        T, C, Hf, Wf = feats.shape
        ref_frame = engine.check_ref_frame(ref_frame, T)
        dev = feats.device
        onehot = torch.nn.functional.one_hot(ref_seg.long().to(dev), num_classes).permute(2, 0, 1).float().contiguous()
        clip = engine.MaskClipPropagator(T, C, Hf, Wf, onehot.shape[0], out_hw, self.test_cfg, dev, self.engine_id,
                                         ref_frame=ref_frame)
        return clip.run(feats.float().contiguous(), onehot)


def nearest_resize(seg, size):
    """``pil_nearest_interpolate`` (mmpt/models/common/utils.py:39-56) on the device: PIL's NEAREST picks the source
    pixel floor((dst + 0.5) * in / out).  seg [H,W] integer tensor -> [size[0], size[1]]."""
    H, W = seg.shape[-2:]
    dev = seg.device
    ys = ((torch.arange(size[0], device=dev, dtype=torch.float64) + 0.5) * H / size[0]).floor().clamp_(0, H - 1).long()
    xs = ((torch.arange(size[1], device=dev, dtype=torch.float64) + 0.5) * W / size[1]).floor().clamp_(0, W - 1).long()
    return seg[..., ys, :][..., xs]


def pad_divide_by(x, d):
    """mmpt/models/common/utils.py:397-412: zero-pad the last two dims symmetrically to multiples of d."""
    h, w = x.shape[-2:]
    nh, nw = -(-h // d) * d, -(-w // d) * d
    lh, lw = (nh - h) // 2, (nw - w) // 2
    pad = (lw, nw - w - lw, lh, nh - h - lh)
    return torch.nn.functional.pad(x, pad), pad


class HRVanillaTracker(VanillaTracker):
    """Local-window ("HR") tracker: ``HRVanillaTracker`` of the reference (vanilla_tracker.py:415-831) without
    mmcv.ops.Correlation.  Per frame every query pixel correlates with the (2r+1)^2 window around its own position in
    each memory frame (r = neighbor_range // 2); window positions outside the image are candidates with affinity 0
    and value 0; top-k over all frames, temperature after the top-k, soft-max, weighted sum (:541-563).  On the GPU
    this is K1 with the square mask (the R^2-fold correlation volume and the unfolded labels never exist) plus the
    analytic zero candidates in the gather (FGVC_ZERO_PAD).

    ``forward_test`` is the point entry (:492-585); ``forward_test_vos`` the mask entry
    ``forward_test_backward_save_mem(imgs, ref_seg_map, img_meta)`` (:663-831)."""

    local_window = True

    def __init__(self, stride=2, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.stride = stride
        self.hard_prop = self.test_cfg.get("hard_prop", False)

    @torch.no_grad()
    def forward_test_vos(self, imgs, ref_seg_map, img_meta, save_image=False, save_path=None, iteration=None,
                         ref_frame=0):
        """imgs [1, n, 3, T, h, w] (or [1, 3, T, h, w]); ref_seg_map [1, h, w] integer labels of frame ``ref_frame``
        (default 0); img_meta[0]['original_shape'].  Returns a list with one uint8/int array [T, H0, W0] of per-frame
        label masks (frame ``ref_frame`` = the given mask), as the reference's ``list(all_seg_preds)`` for integer
        input.  With ref_frame = t0 > 0 the frames after t0 are propagated forward from t0 and the frames before it
        backward, as the reference does on the time-reversed clip from t0."""
        _lib.require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        imgs = imgs.to(dev)
        if imgs.ndim == 6:
            imgs = imgs.reshape((-1,) + imgs.shape[2:])
        assert imgs.shape[0] == 1 and ref_seg_map.ndim == 3, "one clip, integer reference mask"
        ref_frame = engine.check_ref_frame(ref_frame, imgs.shape[2])
        h, w = imgs.shape[-2:]
        imgs, _ = pad_divide_by(imgs, self.stride)
        seg, pa = pad_divide_by(ref_seg_map.to(dev), self.stride)
        pad_shape = tuple(seg.shape[-2:])
        oh, ow = (int(x) for x in img_meta[0]["original_shape"][:2])
        frames = imgs[0].transpose(0, 1).contiguous()              # [T,3,H,W]
        feats = self.get_feats(frames)
        T, C, Hf, Wf = feats.shape
        small = nearest_resize(seg[0], (Hf, Wf)).long()
        onehot = torch.nn.functional.one_hot(small).permute(2, 0, 1).float().contiguous()
        L = onehot.shape[0]
        first = torch.nn.functional.interpolate(ref_seg_map[None].float().to(dev), size=(oh, ow), mode="nearest")[0, 0]
        cfg = dict(self.test_cfg)
        cfg.update(mask_mode="square", local_window=True, with_first_neighbor=True,
                   with_norm=self.test_cfg.get("with_norm", True))
        direct = sum(pa) == 0 and (oh, ow) == (h, w)
        clip = engine.MaskClipPropagator(T, C, Hf, Wf, L, (oh, ow) if direct else pad_shape, cfg, dev, self.engine_id,
                                         ref_frame=ref_frame)
        maps, masks = clip.run(feats.float().contiguous(), onehot, want_maps=not direct)
        if direct:
            out = masks.clone()
        else:
            # padded input or a different original size: the reference's exact resize chain on the label maps
            # (:769-798: bilinear to the padded size, un-pad, bilinear to the original size, min-max, arg-max)
            F = torch.nn.functional
            p = F.interpolate(maps, size=pad_shape, mode="bilinear", align_corners=False)
            p = p[:, :, pa[2]:pad_shape[0] - pa[3], pa[0]:pad_shape[1] - pa[1]]
            p = F.interpolate(p, size=(oh, ow), mode="bilinear", align_corners=False)
            lo, hi = p.amin(dim=(2, 3), keepdim=True), p.amax(dim=(2, 3), keepdim=True)
            p = torch.where(hi > 0, (p - lo) / (hi - lo + 1e-12), p)
            out = p.argmax(dim=1).to(torch.uint8)
        out[ref_frame] = first.to(out.dtype)
        return [out.cpu().numpy()]


B200VanillaTracker = VanillaTracker
B200HRVanillaTracker = HRVanillaTracker


def register_in_mmpt():
    """Inside an mmpt installation: make ``eval_arc='B200VanillaTracker'`` (and the HR and coarse-to-fine trackers)
    resolvable."""
    from mmpt.models.registry import MODELS
    from .c2f_tracker import C2FTracker
    MODELS.register_module(name="B200VanillaTracker", module=VanillaTracker)
    MODELS.register_module(name="B200HRVanillaTracker", module=HRVanillaTracker)
    MODELS.register_module(name="B200C2FTracker", module=C2FTracker)
    return MODELS
