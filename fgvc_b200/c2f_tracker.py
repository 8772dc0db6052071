"""Coarse-to-fine point tracking of a clip: the recurrent driver around ``masked_attention_efficient_c2f``
(mmpt/models/common/local_attention.py:721-880) that BASELINE config 3-(ii) names.

The reference defines the operator but no driver (SURVEY.md section 8, row a8): its output lives on the COARSE query
grid while its memory labels are consumed at FINE resolution.  This module closes the loop in the simplest way the
reference's own tracker suggests (vanilla_tracker.py:305-412); the test harness restates the same loop step by step
around the genuine operator (tests/golden/c2f_driver.npz):

    S_fine[0]  = gaussian heat-maps of the query points at the fine stride          (vanilla_tracker.py:204-221)
    for t = 1 .. T-1:
        mem       = [0] + [max(0, t - precede) .. t-1]                                (:346-362)
        out_c     = c2f(q = Fc[t], k = Fc[mem], q_fine = Ff[t], k_fine = Ff[mem], v = S_fine[mem])   -> [L, Hc, Wc]
        S_fine[t] = bilinear(out_c -> (Hf, Wf), align_corners=False)                 the next frames' memory labels
        traj[t]   = img2coord(bilinear(out_c -> (h, w)))                              (:396-406)

Everything stays resident in HBM across frames: both feature banks are built once per clip (two K0 launches), the fine
label bank holds every frame, a frame costs one coarse K1 (k = 1 per memory frame), one window-mode K1 on the tensor
cores, the c2f tail, one up-sampling kernel and K3.

``C2FTracker`` is the drop-in model around it (``eval_arc='B200C2FTracker'``): one encoder pass feeds a coarse and a
fine bank, each in its own format, and ``C2FPointTracker.track_banks`` tracks the clip's query groups.
"""
import ctypes

import torch

from . import _lib, apis, engine
from .engine import FeatureBank, JobTable, LabelBank
from .tracker import VanillaTracker

# bound of the list workspace of one fgvc_c2f_clip_weights call (the host calls it in job slices beyond): ~1.5 MB per
# job at 32^2 coarse / 128^2 fine, precede 5, K 10 -- a strided 50-frame clip tracked both ways fits one slice
_CLIP_WS_BUDGET = 2 << 30


class C2FPointTracker:
    """cfg keys: precede_frames, topk, temperature, neighbor_range (coarse), radius_fine, with_first (memory),
    with_first_neighbor, with_norm, split, mask_mode; bidirectional (track_queries only)."""

    def __init__(self, cfg, engine_id=_lib.ENGINE_AUTO):
        if cfg.get("cycle_occlusion") is not None:
            raise NotImplementedError("C2FPointTracker: cycle_occlusion is not built")
        self.cfg = cfg
        self.engine_id = engine_id

    def _stage(self, feats_coarse, feats_fine, coarse, fine, normalize, n_chunks=6):
        """K0 of both feature stacks.  Device tensors: two launches, returns a no-op.  Host (pinned) tensors: chunked
        copies on a side stream + K0 per chunk on a second one; returns ``landed(t)``, which makes the current stream
        wait for the chunk frame t is in."""
        if feats_coarse.is_cuda and feats_fine.is_cuda:
            coarse.load_frames(feats_coarse.float(), 0, normalize=normalize)
            fine.load_frames(feats_fine.float(), 0, normalize=normalize)
            return lambda t: None
        dev = coarse.buf.device
        T = feats_coarse.shape[0]
        cur = torch.cuda.current_stream()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream, self._k0_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        cp, k0 = self._copy_stream, self._k0_stream
        step = -(-T // n_chunks)
        # two persistent staging buffers per stack (kept across calls): a copy waits only for the K0 that last read its buffer
        key = (step,) + tuple(feats_coarse.shape[1:]) + tuple(feats_fine.shape[1:]) + (dev.index,)
        if getattr(self, "_stage_key", None) != key:
            self._stage_c = [torch.empty((step,) + tuple(feats_coarse.shape[1:]), dtype=torch.float32, device=dev) for _ in range(2)]
            self._stage_f = [torch.empty((step,) + tuple(feats_fine.shape[1:]), dtype=torch.float32, device=dev) for _ in range(2)]
            self._stage_free, self._stage_key = [None, None], key
            cp.wait_stream(cur)                           # fresh memory: earlier kernels of this stream may still use it
        k0.wait_stream(cur)                               # the banks may still be read by the previous call's kernels
        done = []
        for i, a in enumerate(range(0, T, step)):
            b = min(T, a + step)
            fc, ff = self._stage_c[i % 2][:b - a], self._stage_f[i % 2][:b - a]
            with torch.cuda.stream(cp):
                if self._stage_free[i % 2] is not None:
                    cp.wait_event(self._stage_free[i % 2])
                fc.copy_(feats_coarse[a:b], non_blocking=True)
                ff.copy_(feats_fine[a:b], non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(cp)
            with torch.cuda.stream(k0):
                k0.wait_event(ready)
                coarse.load_frames(fc, a, normalize=normalize)
                fine.load_frames(ff, a, normalize=normalize)
                ev = torch.cuda.Event()
                ev.record(k0)
            self._stage_free[i % 2] = ev
            done.append((b, ev))
        state = {"i": 0}

        def landed(t):
            while state["i"] < len(done) and done[state["i"]][0] <= t:
                state["i"] += 1                      # chunks wholly before frame t: already waited for, or implied
            # frame t lies in chunk i (its end is the first one > t): wait for it (events of earlier chunks precede it
            # on the same stream)
            if state["i"] < len(done) and not state.get(state["i"]):
                cur.wait_event(done[state["i"]][1])
                state[state["i"]] = True
        return landed

    @torch.no_grad()
    def track(self, feats_coarse, feats_fine, points_xy, image_hw):
        """feats_coarse [T,C,Hc,Wc], feats_fine [T,Cf,Hf,Wf] (CUDA fp32, Hf = s * Hc); points_xy [P,2] (x, y) image
        pixels of the points at frame 0.  Returns (traj [T,P,2] float32 CUDA, out_coarse list of [Nq_c, Lp])."""
        _lib.require_cuda()
        cfg = self.cfg
        T, C, Hc, Wc = feats_coarse.shape
        Tf, Cf, Hf, Wf = feats_fine.shape
        assert T == Tf and Hf % Hc == 0 and Wf % Wc == 0 and Hf // Hc == Wf // Wc, "fine grid must be s x the coarse grid"
        h, w = image_hw
        dev = feats_coarse.device if feats_coarse.is_cuda else torch.device("cuda", torch.cuda.current_device())
        stride_f = h // Hf
        split = cfg.get("split") or ("f16" if (engine.default_split(C) == "f16" and Cf % 4 == 0) else "tf32")
        normalize = cfg.get("with_norm", True)
        coarse = FeatureBank(T, C, Hc, Wc, dev, split=split)
        fine = FeatureBank(T, Cf, Hf, Wf, dev, split=split)
        # host features: copied in frame chunks on a side stream; the frame loop below waits for the chunk a frame is in
        # (frame t only reads frames <= t), so the host link overlaps the propagation of the frames already there
        landed = self._stage(feats_coarse, feats_fine, coarse, fine, normalize)
        P = points_xy.shape[0]
        pts = points_xy.to(device=dev, dtype=torch.float32).contiguous()
        labels = LabelBank(T, P, Hf, Wf, dev)
        labels.put_gaussians(pts, 0, stride_f)
        table = JobTable()
        unmasked_first = 0 if cfg.get("with_first_neighbor", True) else 1
        for t in range(1, T):
            mem = engine.memory_frames(t, cfg["precede_frames"], cfg.get("with_first", True))
            table.add(t, mem, mem, t, unmasked=unmasked_first)
        radius = cfg["neighbor_range"] // 2
        traj = torch.zeros(T, P, 2, dtype=torch.float32, device=dev)
        traj[0] = engine.gaussian_coords(pts, (h, w))
        maps = torch.empty(P, Hc, Wc, dtype=torch.float32, device=dev)
        outs = []
        for t in range(1, T):
            landed(t)
            out = engine.c2f_propagate(coarse, fine, table, t - 1, labels, radius, cfg.get("radius_fine", 12),
                                       cfg["topk"], cfg["temperature"], cfg.get("mask_mode", "circle"), self.engine_id)
            # the coarse output becomes (a) the fine memory labels of the following frames, (b) this frame's coordinates
            _lib.call("fgvc_upsample_labels", _lib.ptr(out), Hc, Wc, labels.Lp, _lib.ptr(labels.buf), t, Hf, Wf,
                      _lib.stream_ptr())
            _lib.call("fgvc_labels_to_nchw", _lib.ptr(out), 0, labels.Lp, P, Hc * Wc, _lib.ptr(maps), _lib.stream_ptr())
            traj[t] = engine.heatmap_coords(maps, (h, w))
            outs.append(out)
        landed(T - 1)            # (a one-frame clip: the banks must not be released under the staging stream)
        return traj, outs

    @torch.no_grad()
    def track_queries(self, feats_coarse, feats_fine, query_points, image_hw):
        """TAP-Vid queries: query_points [P, 3] (t, x, y) as ``forward_test``'s ``query_points[0]`` (and
        ``metrics.tapvid_sample``).  Returns traj [T, P, 2] float32 CUDA in the input point order.

        The points are grouped by query frame t0.  Frames t >= t0 of a group are what ``track(feats_coarse[t0:],
        feats_fine[t0:], points)`` gives; with the cfg key ``bidirectional`` frames t < t0 are what ``track()`` gives on
        the time-reversed prefix ``feats[:t0 + 1].flip(0)``, mapped back (memory [t0] + [min(t0, t + precede) .. t + 1]),
        else they are zero.  The label-independent stages of every job of the clip (coarse arg-max, fine window top-K,
        zero-padded candidates, soft-max weights) run in a few launches whose number does not grow with the groups
        (fgvc_c2f_clip_weights), and every forward and backward recurrence runs as a lane of one cooperative chain
        (fgvc_c2f_point_clip_tail_lanes).  Host features (pinned) are uploaded whole, then take the same path."""
        _lib.require_cuda()
        cfg = self.cfg
        T, C, Hc, Wc = feats_coarse.shape
        Tf, Cf, Hf, Wf = feats_fine.shape
        assert T == Tf and Hf % Hc == 0 and Wf % Wc == 0 and Hf // Hc == Wf // Wc, "fine grid must be s x the coarse grid"
        h, w = image_hw
        dev = feats_coarse.device if feats_coarse.is_cuda else torch.device("cuda", torch.cuda.current_device())
        stride_f = h // Hf
        split = cfg.get("split") or ("f16" if (engine.default_split(C) == "f16" and Cf % 4 == 0) else "tf32")
        normalize = cfg.get("with_norm", True)
        coarse = FeatureBank(T, C, Hc, Wc, dev, split=split)
        fine = FeatureBank(T, Cf, Hf, Wf, dev, split=split)
        coarse.load_frames(feats_coarse.to(dev, non_blocking=True).float(), 0, normalize=normalize)
        fine.load_frames(feats_fine.to(dev, non_blocking=True).float(), 0, normalize=normalize)
        return self.track_banks(coarse, fine, query_points, image_hw)

    @torch.no_grad()
    def track_banks(self, coarse, fine, query_points, image_hw, shard=None):
        """The clip path of ``track_queries`` over two loaded ``FeatureBank``s, each in its own format: coarse
        [T, C, Hc, Wc], fine [T, Cf, s Hc, s Wc] (e.g. a TF32 coarse bank at C = 512 and an F16 fine bank at Cf = 256,
        as ``C2FTracker`` encodes them).  query_points [P, 3] (t, x, y); returns traj [T, P, 2] float32 CUDA in the
        input point order, with the semantics of ``track_queries``.

        ``shard=(rank, world)``: the two-phase split of ``VanillaTracker.propagate_points`` over the default process
        group.  Phase 1 runs fgvc_c2f_clip_weights for this rank's job range (``apis.frame_shard``) into its slot of the
        (weight, row) buffers, which are all-gathered; phase 2 runs the lanes chain for this rank's slice of every
        group's points (``apis.point_shard``), and the tracks are all-gathered.  Every rank returns the full result,
        bit for bit that of ``world = 1``."""
        cfg = self.cfg
        T, Hc, Wc, Hf, Wf = coarse.n_slots, coarse.H, coarse.W, fine.H, fine.W
        assert fine.n_slots == T and Hf % Hc == 0 and Wf % Wc == 0 and Hf // Hc == Wf // Wc, \
            "fine grid must be s x the coarse grid"
        h, w = image_hw
        dev = coarse.buf.device
        stride_f = h // Hf
        rank, world = shard if shard is not None else (0, 1)

        qp = query_points.to(device=dev, dtype=torch.float32)
        qt = qp[:, 0].round().long()
        t0s = torch.unique(qt).tolist()
        order = [torch.nonzero(qt == t).flatten() for t in t0s]
        bidirectional = bool(cfg.get("bidirectional", False))
        unmasked_first = 0 if cfg.get("with_first_neighbor", True) else 1
        table, spans = engine.query_job_table(t0s, T, cfg["precede_frames"], cfg.get("with_first", True), bidirectional,
                                              lambda mem: unmasked_first)
        K = int(cfg["topk"])
        n_c, n_f = Hc * Wc, Hf * Wf
        # phase 1: the (weight, fine label row) pairs of this rank's jobs, then of every job
        lo, hi, per = apis.frame_shard(len(table), rank, world)
        weights = torch.empty(per * world, n_c, K, dtype=torch.float32, device=dev)
        rows = torch.empty(per * world, n_c, K, dtype=torch.int32, device=dev)
        if hi > lo:
            self._clip_weights(coarse, fine, table, lo, hi, K, weights, rows, dev)
        apis.gather_job_lists(weights, per, rank, world)
        apis.gather_job_lists(rows, per, rank, world)

        # phase 2: per group, this rank's slice of its points (all of them at world = 1)
        sizes = [int(o.numel()) for o in order]
        parts = [apis.point_shard(P, rank, world) for P in sizes]
        mine = [b - a for a, b in parts]
        perm = torch.cat(order) if order else torch.zeros(0, dtype=torch.long, device=dev)
        pts_all = qp[perm, 1:].contiguous()
        c0_all = engine.gaussian_coords(pts_all, (h, w)) if pts_all.shape[0] else None
        lab = torch.empty(sum(T * n_f * engine.pad4(P) for P in mine), dtype=torch.float32, device=dev)
        cout = torch.empty(sum(T * n_c * engine.pad4(P) for P in mine), dtype=torch.float32, device=dev)
        coords = torch.zeros(sum(T * P * 2 for P in mine), dtype=torch.float32, device=dev)
        lanes, tracks = [], []
        lab_off = out_off = c_off = p_off = 0
        for (j0, t0), P_all, (a, _), P in zip(spans, sizes, parts, mine):
            track = coords[c_off:c_off + T * P * 2].view(T, P, 2)
            tracks.append(track)
            if P:
                labels = LabelBank(T, P, Hf, Wf, dev, buf=lab[lab_off:lab_off + T * n_f * engine.pad4(P)])
                labels.put_gaussians(pts_all[p_off + a:p_off + a + P], t0, stride_f)
                track[t0] = c0_all[p_off + a:p_off + a + P]
                n_fw, n_bw = T - t0 - 1, (t0 if bidirectional else 0)
                # forward lane, backward lane: they share the group's banks (both read slot t0, they write disjoint
                # slots)
                for jb, je in ((j0, j0 + n_fw), (j0 + n_fw, j0 + n_fw + n_bw)):
                    if je > jb:
                        lanes.append(_lib.C2FLane(jb, je, P, engine.pad4(P), lab_off, out_off, c_off))
            lab_off += T * n_f * engine.pad4(P)
            out_off += T * n_c * engine.pad4(P)
            c_off += T * P * 2
            p_off += P_all
        if lanes:
            self._chain(weights, rows, table, lanes, coarse, fine, lab, cout, coords, K, (h, w), dev)
        if world > 1:
            pads = [-(-n // world) for n in sizes]
            local = torch.zeros(T, sum(pads), 2, dtype=torch.float32, device=dev)
            off = 0
            for tr, pad in zip(tracks, pads):
                local[:, off:off + tr.shape[1]] = tr
                off += pad
            tracks = apis.gather_point_tracks(local, sizes, rank, world)
        traj = torch.zeros(T, qp.shape[0], 2, dtype=torch.float32, device=dev)
        if perm.numel():
            traj[:, perm] = torch.cat(tracks, dim=1)
        return traj

    def _clip_weights(self, coarse, fine, table, lo, hi, K, weights, rows, dev):
        """fgvc_c2f_clip_weights over the jobs [lo, hi) of ``table``, in job slices of bounded workspace, into rows
        [lo, hi) of ``weights`` / ``rows``."""
        cfg = self.cfg
        n_c = coarse.H * coarse.W
        _, mem_feat, mem_label = table.device(dev)
        jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4).contiguous()
        lib = _lib.load()
        total = int(lib.fgvc_c2f_clip_workspace_bytes(_lib.ptr(jobs_host), lo, hi, coarse.H, coarse.W, K))
        # slices: bounded workspace, and at most 65535 window CTAs per coarse tile (<= 4 per memory entry)
        n_mem = sum(j[2] - j[1] for j in table.jobs[lo:hi])
        n = hi - lo
        n_slices = max(-(-total // _CLIP_WS_BUDGET), -(-4 * n_mem // 65535), -(-n // 65535))
        mode = _lib.MASK_CIRCLE if cfg.get("mask_mode", "circle") == "circle" else _lib.MASK_SQUARE
        ws = None
        for i in range(n_slices):
            a, b = lo + (n * i) // n_slices, lo + (n * (i + 1)) // n_slices
            need = int(lib.fgvc_c2f_clip_workspace_bytes(_lib.ptr(jobs_host), a, b, coarse.H, coarse.W, K))
            if ws is None or ws.numel() < need:
                ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.call("fgvc_c2f_clip_weights", _lib.ptr(coarse.buf), coarse.fmt, coarse.n_slots, coarse.H, coarse.W,
                      coarse.C, _lib.ptr(fine.buf), fine.fmt, fine.H, fine.W, fine.C, _lib.ptr(jobs_host), a, b,
                      _lib.ptr(mem_feat), _lib.ptr(mem_label), int(cfg["neighbor_range"] // 2), mode,
                      int(cfg.get("radius_fine", 12)), K, float(cfg["temperature"]),
                      ctypes.c_void_p(weights.data_ptr() + 4 * a * n_c * K),
                      ctypes.c_void_p(rows.data_ptr() + 4 * a * n_c * K), _lib.ptr(ws), need, int(self.engine_id),
                      _lib.stream_ptr())

    def _chain(self, weights, rows, table, lanes, coarse, fine, lab, cout, coords, K, image_hw, dev):
        """fgvc_c2f_point_clip_tail_lanes over ``lanes`` (the weights and rows of every job of ``table``)."""
        n_c = coarse.H * coarse.W
        jobs_dev, _, _ = table.device(dev)
        jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4).contiguous()
        host = (_lib.C2FLane * len(lanes))(*lanes)
        lanes_dev = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(dev)
        maps = torch.empty(coarse.n_slots * max(ln.L for ln in lanes) * n_c, dtype=torch.float32, device=dev)  # NCHW scratch
        barrier = torch.empty(256, dtype=torch.uint8, device=dev)
        _lib.call("fgvc_c2f_point_clip_tail_lanes", _lib.ptr(weights), _lib.ptr(rows), K, 0, _lib.ptr(jobs_dev),
                  _lib.ptr(jobs_host), _lib.ptr(lanes_dev), ctypes.c_void_p(ctypes.addressof(host)), len(lanes),
                  coarse.H, coarse.W, fine.H, fine.W, _lib.ptr(lab), _lib.ptr(cout), int(image_hw[0]), int(image_hw[1]), 5,
                  _lib.ptr(maps), _lib.ptr(coords), _lib.ptr(barrier), _lib.stream_ptr())


_EXPECTED_BACKBONE = "backbone=dict(type='ResNet', depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3), pool_type='none')"


class C2FTracker(VanillaTracker):
    """Coarse-to-fine point tracker as a drop-in model (``eval_arc='B200C2FTracker'``, BASELINE config 3-(ii)):
    VanillaTracker's constructor and ``forward_test`` contract, the clip path of ``C2FPointTracker.track_banks``.

    One encoder pass gives both levels: the backbone returns exactly two, the lower ``out_index`` is the fine level and
    the higher the coarse level, with fine H, W = s x coarse H, W.  With the shipped eval backbone (ResNet-18,
    ``strides=(1, 1, 1, 4)``, ``pool_type='none'``) and ``out_indices=(2, 3)``, a 256^2 clip gives layer 3 at 128^2 x
    256 channels and layer 4 at 32^2 x 512 channels: s = 4.  Each level goes into its own FeatureBank, K0 of encoder
    chunk i overlapped with the encoder of chunk i + 1 (``encode_to_bank``), and each bank takes its own
    ``engine.default_split``: the coarse bank TF32 at C = 512 (the 3xTF32 engine), the fine bank F16 at Cf = 256 (the
    tensor-core window-mode fine stage); ``test_cfg.split`` forces one format for both.

    test_cfg keys: those of ``C2FPointTracker`` (precede_frames, topk, temperature, neighbor_range -- the coarse
    radius --, radius_fine, with_first, with_first_neighbor, with_norm, split, mask_mode, bidirectional) and
    VanillaTracker's batch_step, encoder_channels_last, engine.  ``with_first`` is also the grouping key of
    ``forward_test``, as in VanillaTracker.  Keys of VanillaTracker that the c2f path does not implement raise
    NotImplementedError when set to a non-default value."""

    def __init__(self, backbone, head=None, train_cfg=None, test_cfg=None, init_cfg=None):
        super().__init__(backbone, head=head, train_cfg=train_cfg, test_cfg=test_cfg, init_cfg=init_cfg)
        cfg = self.test_cfg
        if cfg.get("test_mode", "v1") != "v1":
            raise NotImplementedError("C2FTracker: test_mode v2 is not built (the c2f operator is a v1 operator)")
        if cfg.get("sim_mode", "dot_product") != "dot_product":
            raise NotImplementedError("C2FTracker: only sim_mode='dot_product' is built")
        for key in ("hard_prop", "stride_sample"):
            if cfg.get(key, False):
                raise NotImplementedError(f"C2FTracker: test_cfg.{key} is not built")
        if cfg.get("cycle_occlusion") is not None:
            raise NotImplementedError("C2FTracker: test_cfg.cycle_occlusion is not built (the coarse-to-fine recurrence "
                                      "is another operator; VanillaTracker and HRVanillaTracker have it)")
        for key in ("topk", "neighbor_range"):
            if cfg.get(key) is None:
                raise NotImplementedError(f"C2FTracker needs test_cfg.{key} (the c2f path has no {key}=None form)")

    def extract_feat(self, imgs):
        """imgs [n,3,h,w] -> [fine, coarse] encoder levels; raises ValueError unless the backbone gives exactly two
        levels with fine H, W = s x coarse H, W for one integer s."""
        x = self.backbone(imgs)
        levels = list(x) if isinstance(x, (tuple, list)) else [x]
        if len(levels) != 2:
            raise ValueError(f"C2FTracker needs a backbone with exactly two output levels (fine, coarse), got "
                             f"{len(levels)}: use e.g. {_EXPECTED_BACKBONE}")
        (Hf, Wf), (Hc, Wc) = levels[0].shape[-2:], levels[1].shape[-2:]
        if Hf % Hc or Wf % Wc or Hf // Hc != Wf // Wc:
            raise ValueError(f"C2FTracker: the fine level ({Hf}x{Wf}, lower out_index) must be s times the coarse level "
                             f"({Hc}x{Wc}) in H and W for one integer s: use e.g. {_EXPECTED_BACKBONE}")
        return levels

    def forward_test(self, rgbs, query_points, trajectories, visibilities, save_image=False, save_path=None,
                     iteration=None, shard=None):
        """rgbs [1,T,3,h,w]; query_points [1,P,3] (t,x,y); trajectories [1,T,P,2]; visibilities [1,T,P].  Returns
        VanillaTracker's 5-tuple (traj_gt, vis_gt, traj_pred, vis_pred, query_points): with ``test_cfg.with_first``
        the points are grouped by query frame and re-ordered by group (with ``bidirectional`` each group is also
        tracked backwards), else every point is tracked from frame 0 in input order.  ``shard=(rank, world)``: the
        two-phase split of ``C2FPointTracker.track_banks``."""
        _lib.require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        rgbs, query_points = rgbs.to(dev), query_points.to(dev)
        trajectories, visibilities = trajectories.to(dev), visibilities.to(dev)
        assert rgbs.shape[0] == 1
        h, w = rgbs.shape[-2:]
        fine, coarse = self.encode_to_bank(rgbs[0], n_levels=2)
        c2f = C2FPointTracker(self.test_cfg, self.engine_id)
        qp = query_points[0]
        if not self.test_cfg.get("with_first", False):
            qp = torch.cat([torch.zeros_like(qp[:, :1]), qp[:, 1:]], dim=1)
            traj = c2f.track_banks(coarse, fine, qp, (h, w), shard=shard)
            return trajectories, visibilities, traj.double()[None], torch.zeros_like(visibilities), query_points
        traj = c2f.track_banks(coarse, fine, qp, (h, w), shard=shard)
        qt = qp[:, 0]
        perm = torch.cat([torch.nonzero(qt == t).flatten() for t in torch.unique(qt).tolist()])
        return (trajectories[:, :, perm], visibilities[:, :, perm], traj[:, perm].to(trajectories.dtype)[None],
                torch.zeros_like(visibilities), query_points[:, perm])

    def propagate_points(self, *args, **kwargs):
        raise NotImplementedError("C2FTracker tracks points through forward_test (C2FPointTracker.track_banks)")

    def propagate_masks(self, *args, **kwargs):
        raise NotImplementedError("C2FTracker has no mask propagation")


B200C2FTracker = C2FTracker
