"""C2FTracker: the coarse-to-fine tracker as a drop-in model.  One encoder pass feeds a TF32 coarse bank (layer 4,
C = 512) and an F16 fine bank (layer 3, Cf = 256); each layer of the path is pinned on its own:
  * the C ABI with one format per bank: the per-frame loop (fgvc_c2f_propagate + up-sampling + K3) and the clip path
    (fgvc_c2f_clip_weights + lanes chain) agree bit for bit on mixed banks, and the mixed clip weights equal those of a
    uniform F16 run (coarse level through the CUDA-core engine) wherever the coarse arg-max is tie-free;
  * the model: with one forced format it is C2FPointTracker.track_queries on the same encoder outputs, its 5-tuple is
    ordered as VanillaTracker's, its tracks are within the c2f driver bound of the oracle loop;
  * launch counts, and the two-phase split (two ranks simulated in one process) against one rank."""
import copy
import os
import threading

import numpy as np
import pytest
import torch

from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

BACKBONE = dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3), pool_type="none")
CFG3 = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12, with_first=True)
SMALL = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=6, radius_fine=5, batch_step=4)


def _coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


def _mixed_banks(seed=21, T=7, C=512, split_coarse=None, split_fine=None):
    """32^2 x C coarse and 128^2 x 256 fine features (config 3-(ii) geometry) in banks of their default formats"""
    from fgvc_b200.engine import FeatureBank
    g = torch.Generator().manual_seed(seed)
    fc, ff = _coherent(g, T, C, 32, 32).cuda(), _coherent(g, T, 256, 128, 128).cuda()
    coarse = FeatureBank(T, C, 32, 32, fc.device, split=split_coarse)
    fine = FeatureBank(T, 256, 128, 128, ff.device, split=split_fine)
    coarse.load_frames(fc)
    fine.load_frames(ff)
    return fc, ff, coarse, fine


def _queries(g, t0s, per_group, h, w):
    P = per_group * len(t0s)
    xy = torch.rand(P, 2, generator=g) * torch.tensor([w - 1.0, h - 1.0])
    t = torch.tensor([t0s[i % len(t0s)] for i in range(P)], dtype=torch.float32)
    return torch.cat([t[:, None], xy], dim=1)


def _per_frame_loop(coarse, fine, qp, hw, cfg):
    """every lane of the clip frame by frame: fgvc_c2f_propagate, fgvc_upsample_labels, NCHW copy + K3"""
    from fgvc_b200 import _lib, engine
    from fgvc_b200.engine import LabelBank
    T, Hc, Wc, Hf, Wf = coarse.n_slots, coarse.H, coarse.W, fine.H, fine.W
    h, w = hw
    qt = qp[:, 0].long()
    t0s = sorted(set(qt.tolist()))
    bidirectional = cfg.get("bidirectional", False)
    table, spans = engine.query_job_table(t0s, T, cfg["precede_frames"], cfg.get("with_first", True), bidirectional,
                                          lambda mem: 0)
    traj = torch.zeros(T, qp.shape[0], 2, dtype=torch.float32, device="cuda")
    for j0, t0 in spans:
        idx = torch.nonzero(qt == t0).flatten()
        pts = qp[idx, 1:].cuda().contiguous()
        P = pts.shape[0]
        labels = LabelBank(T, P, Hf, Wf, "cuda")
        labels.put_gaussians(pts, t0, h // Hf)
        traj[t0, idx.cuda()] = engine.gaussian_coords(pts, hw)
        maps = torch.empty(P, Hc, Wc, dtype=torch.float32, device="cuda")
        for j in range(j0, j0 + (T - 1 - t0) + (t0 if bidirectional else 0)):
            t = table.jobs[j][3]
            out = engine.c2f_propagate(coarse, fine, table, j, labels, cfg["neighbor_range"] // 2, cfg["radius_fine"],
                                       cfg["topk"], cfg["temperature"])
            _lib.call("fgvc_upsample_labels", _lib.ptr(out), Hc, Wc, labels.Lp, _lib.ptr(labels.buf), t, Hf, Wf,
                      _lib.stream_ptr())
            _lib.call("fgvc_labels_to_nchw", _lib.ptr(out), 0, labels.Lp, P, Hc * Wc, _lib.ptr(maps), _lib.stream_ptr())
            traj[t, idx.cuda()] = engine.heatmap_coords(maps, hw)
    return traj


@pytest.mark.parametrize("bidirectional", [False, True])
def test_mixed_banks_per_frame_loop_equals_clip_path(bidirectional):
    import fgvc_b200
    from fgvc_b200 import _lib
    _, _, coarse, fine = _mixed_banks()
    assert (coarse.fmt, fine.fmt) == (_lib.BANK_TF32, _lib.BANK_F16)
    qp = _queries(torch.Generator().manual_seed(4), [0, 3, 6], 8, 256, 256)
    cfg = dict(CFG3, bidirectional=bidirectional)
    got = fgvc_b200.C2FPointTracker(cfg).track_banks(coarse, fine, qp, (256, 256))
    want = _per_frame_loop(coarse, fine, qp, (256, 256), cfg)
    assert torch.equal(got, want), float((got - want).abs().max())


def test_mixed_clip_weights_equal_uniform_f16_where_the_coarse_argmax_is_tie_free():
    """mixed: TF32 coarse bank (the 3xTF32 engine, non-resident above C = 256); uniform F16: the fp16 tensor engine
    covers C <= 256, so its coarse K1 runs on the CUDA cores.  The fine stage reads the same F16 bank in both.  At
    C = 384: the CUDA-core engine stages 2 x 64 x (C + 4) + 64 x 65 floats of shared memory, 280 832 B at C = 512, more
    than a block has, so no engine takes an F16 bank at C = 512 and C = 384 is the widest channel count both runs
    cover."""
    import fgvc_b200
    from fgvc_b200 import _lib, engine
    fc, _, coarse, fine = _mixed_banks(seed=33, C=384)
    _, _, coarse16, _ = _mixed_banks(seed=33, C=384, split_coarse="f16")
    assert (coarse.fmt, coarse16.fmt, fine.fmt) == (_lib.BANK_TF32, _lib.BANK_F16, _lib.BANK_F16)
    T, n_c, K, tau = coarse.n_slots, 32 * 32, CFG3["topk"], CFG3["temperature"]
    cfg = dict(CFG3, bidirectional=True)
    table, _ = engine.query_job_table([0, 3, 6], T, cfg["precede_frames"], True, True, lambda mem: 0)
    n = len(table)
    trk = fgvc_b200.C2FPointTracker(cfg)
    runs = []
    for cb in (coarse, coarse16):
        wts = torch.empty(n, n_c, K, dtype=torch.float32, device="cuda")
        rows = torch.empty(n, n_c, K, dtype=torch.int32, device="cuda")
        trk._clip_weights(cb, fine, table, 0, n, K, wts, rows, torch.device("cuda"))
        runs.append((wts, rows))
    # float64 coarse affinities: a query is tie-free when its masked top-2 gap exceeds gap_eps (affinity / tau units)
    # in every memory entry of its job
    gap_eps = 3e-5
    x = torch.nn.functional.normalize(fc.double().flatten(2), dim=1)          # [T, C, n_c]
    mask = O.neighbor_mask(32, 32, cfg["neighbor_range"]).cuda()             # [key, query]
    tie_free = torch.ones(n, n_c, dtype=torch.bool, device="cuda")
    for j, (q_slot, mb, me, _) in enumerate(table.jobs):
        for m in table.mem_feat[mb:me]:
            a = (x[m & ~_lib.MEM_UNMASKED].t() @ x[q_slot]).masked_fill(~mask, -float("inf"))
            top2 = a.topk(2, dim=0).values
            tie_free[j] &= (top2[0] - top2[1]) / tau > gap_eps
    excluded = 1.0 - float(tie_free.float().mean())
    assert excluded <= 0.02, excluded
    (w1, r1), (w2, r2) = runs
    sel = tie_free[..., None].expand_as(w1)
    assert torch.equal(w1[sel], w2[sel]) and torch.equal(r1[sel], r2[sel])


def _model(cfg, seed=0):
    import fgvc_b200
    torch.manual_seed(seed)
    return fgvc_b200.C2FTracker(backbone=dict(BACKBONE), test_cfg=dict(cfg)).cuda().eval()


def _clip(T=9, h=64, w=64, P=12, seed=3, first_frame_only=False):
    from fgvc_b200 import synthetic as S
    rgbs = S.synthetic_video(T, h, w, seed=seed)[None]
    qp = S.query_points(P, T, h, w, seed=seed + 1, first_frame_only=first_frame_only)[None]
    return rgbs, qp, torch.zeros(1, T, P, 2), torch.zeros(1, T, P)


@torch.no_grad()
def _levels(model, rgbs):
    """the model's own encoder outputs, chunked as encode_to_bank chunks them: (layer 4 [T,512,..], layer 3 [T,256,..])"""
    step = model.test_cfg.get("batch_step", 5)
    frames = rgbs[0].cuda()
    parts = [model.extract_feat(frames[s:s + step]) for s in range(0, frames.shape[0], step)]
    return torch.cat([p[1].float() for p in parts]), torch.cat([p[0].float() for p in parts])


@pytest.mark.parametrize("with_first", [False, True])
@pytest.mark.parametrize("bidirectional", [False, True])
def test_uniform_format_forward_test_equals_track_queries(with_first, bidirectional):
    import fgvc_b200
    cfg = dict(SMALL, split="tf32", with_first=with_first, bidirectional=bidirectional)
    model = _model(cfg)
    rgbs, qp, traj, vis = _clip()
    with torch.no_grad():
        out = model(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
    layer4, layer3 = _levels(model, rgbs)
    q = qp[0].clone()
    if not with_first:
        q[:, 0] = 0
    want = fgvc_b200.C2FPointTracker(cfg).track_queries(layer4, layer3, q, (64, 64))
    if with_first:
        perm = torch.argsort(qp[0, :, 0], stable=True).cuda()
        want = want[:, perm]
    assert torch.equal(out[2][0].float(), want), float((out[2][0].float() - want).abs().max())


@pytest.mark.parametrize("with_first", [False, True])
def test_five_tuple_is_ordered_as_vanilla_tracker(with_first):
    import fgvc_b200
    cfg = dict(SMALL, with_first=with_first, bidirectional=True)
    model = _model(cfg)
    vanilla = fgvc_b200.VanillaTracker(backbone=model.backbone, test_cfg=dict(cfg)).cuda().eval()
    rgbs, qp, _, _ = _clip()
    T, P = rgbs.shape[1], qp.shape[1]
    g = torch.Generator().manual_seed(8)
    traj, vis = torch.rand(1, T, P, 2, generator=g), (torch.rand(1, T, P, generator=g) > 0.3).float()
    with torch.no_grad():
        got = model(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
        want = vanilla(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
    for i in (0, 1, 3, 4):
        assert torch.equal(got[i], want[i]), i
    assert got[2].shape == want[2].shape and got[2].dtype == want[2].dtype
    assert bool((got[3] == 0).all())


class _Lookup(torch.nn.Module):
    """a backbone whose two levels are fixed feature stacks: frame t of the clip is the constant image t"""

    def __init__(self, fine, coarse):
        super().__init__()
        self.fine, self.coarse = fine, coarse

    def forward(self, x):
        t = x[:, 0, 0, 0].round().long().cpu()
        return self.fine[t].to(x.device), self.coarse[t].to(x.device)


def test_default_formats_are_mixed_and_forward_test_is_within_the_oracle_bound():
    """coherent fixture features (those of the c2f driver bound, test_gpu_c2f_queries.py) as the two encoder levels,
    C = 512 coarse and Cf = 256 fine: the default formats are TF32 / F16, and the tracks of a frame-0 group and the
    backward half of a later group are within the driver bound of the oracle loop on the same features"""
    import fgvc_b200
    from fgvc_b200 import _lib
    torch.set_num_threads(os.cpu_count() or 8)
    T, t0, Hc, Wc, s = 6, 4, 8, 10, 4
    h, w = Hc * s * 2, Wc * s * 2
    g = torch.Generator().manual_seed(77)
    fc, ff = _coherent(g, T, 512, Hc, Wc), _coherent(g, T, 256, Hc * s, Wc * s)
    cfg = dict(SMALL, with_first=True, bidirectional=True)
    model = fgvc_b200.C2FTracker(backbone=_Lookup(ff, fc), test_cfg=dict(cfg))
    rgbs = torch.arange(T, dtype=torch.float32).view(1, T, 1, 1, 1).expand(1, T, 3, h, w).contiguous()
    fine, coarse = model.encode_to_bank(rgbs[0].cuda(), n_levels=2)
    assert (coarse.fmt, fine.fmt) == (_lib.BANK_TF32, _lib.BANK_F16)
    pts = torch.rand(12, 2, generator=g) * torch.tensor([w - 1.0, h - 1.0])
    qp = torch.cat([torch.tensor([0.0, float(t0)]).repeat(6)[:, None], pts], dim=1)[None]
    with torch.no_grad():
        out = model(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=torch.zeros(1, T, 12, 2),
                    visibilities=torch.zeros(1, T, 12))
    pred = out[2][0].cpu().numpy()                      # re-ordered by group: the 6 points at frame 0, then t0
    qs = out[4][0].cpu()
    _, fw = O.track_clip_c2f_port(fc, ff, qs[:6, 1:], (h, w), cfg)
    _, bw = O.track_clip_c2f_port(fc[:t0 + 1].flip(0).contiguous(), ff[:t0 + 1].flip(0).contiguous(), qs[6:, 1:],
                                  (h, w), cfg)
    for err in (np.abs(pred[:, :6] - fw).max(axis=-1), np.abs(pred[:t0 + 1, 6:][::-1] - bw).max(axis=-1)):
        assert float((err <= 0.5).mean()) >= 0.9 and float(err.max()) <= 1.0, float(err.max())


def _calls_and_launches(monkeypatch, fn):
    from fgvc_b200 import _lib
    calls, launches = {}, {}
    orig = _lib.call

    def spy(name, *args):
        n0 = _lib.launch_count()
        orig(name, *args)
        calls[name] = calls.get(name, 0) + 1
        launches[name] = launches.get(name, 0) + _lib.launch_count() - n0

    monkeypatch.setattr(_lib, "call", spy)
    fn()
    monkeypatch.setattr(_lib, "call", orig)
    return calls, launches


def test_launch_counts(monkeypatch):
    from fgvc_b200 import _lib
    T = 12
    model = _model(dict(SMALL, with_first=True, bidirectional=True))
    rgbs, _, traj, vis = _clip(T=T, P=16)
    # K0 twice per encoder chunk (one per level) and nothing else of ours: the encoder is PyTorch
    n0 = _lib.launch_count()
    model.encode_to_bank(rgbs[0].cuda(), n_levels=2)
    assert _lib.launch_count() - n0 == 2 * -(-T // SMALL["batch_step"])
    runs = {}
    for t0s in ([0, 1], list(range(8))):
        qp = _queries(torch.Generator().manual_seed(5), t0s, 2, 64, 64)[None]
        P = qp.shape[1]
        with torch.no_grad():
            calls, launches = _calls_and_launches(monkeypatch, lambda: model(
                test_mode=True, rgbs=rgbs, query_points=qp, trajectories=torch.zeros(1, T, P, 2),
                visibilities=torch.zeros(1, T, P)))
        runs[len(t0s)] = (calls["fgvc_c2f_clip_weights"], launches["fgvc_c2f_clip_weights"],
                          calls["fgvc_c2f_point_clip_tail_lanes"])
    assert runs[2] == runs[8] and runs[2][0] == 1 and runs[2][2] == 1, runs


class _FakeGroup:
    """the collectives of apis.gather_job_lists / gather_point_tracks between threads of one process, one per rank"""

    def __init__(self, world):
        self.world, self.bar, self.slots, self.local = world, threading.Barrier(world), {}, threading.local()

    def _exchange(self, t):
        self.slots[self.local.rank] = t.clone()
        self.bar.wait()
        out = [self.slots[r] for r in range(self.world)]
        self.bar.wait()
        return out

    def all_gather(self, parts, t):
        for p, o in zip(parts, self._exchange(t)):
            p.copy_(o)

    def all_gather_into_tensor(self, buf, mine):
        for r, o in enumerate(self._exchange(mine)):
            buf[r * mine.shape[0]:(r + 1) * mine.shape[0]].copy_(o)


@pytest.mark.parametrize("with_first", [False, True])
def test_two_phase_split_equals_one_rank(monkeypatch, with_first):
    """shard=(rank, 2) on two threads with the all-gathers done between them: every rank's 5-tuple is the one-rank
    result bit for bit (strided, bidirectional query groups; more ranks than points in no group)"""
    import torch.distributed as dist
    cfg = dict(SMALL, with_first=with_first, bidirectional=True)
    model = _model(cfg)
    models = [model, copy.deepcopy(model)]
    rgbs, qp, traj, vis = _clip(T=10, P=13, seed=21)
    with torch.no_grad():
        want = model(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
    grp = _FakeGroup(2)
    monkeypatch.setattr(dist, "get_backend", lambda *a: "nccl")
    monkeypatch.setattr(dist, "all_gather", grp.all_gather)
    monkeypatch.setattr(dist, "all_gather_into_tensor", grp.all_gather_into_tensor)
    got, errors = [None, None], []

    def rank_main(r):
        grp.local.rank = r
        try:
            with torch.no_grad():
                got[r] = models[r](test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis,
                                   shard=(r, 2))
            torch.cuda.synchronize()
        except BaseException as e:            # (a failing rank must not leave the other at the barrier)
            errors.append(e)
            grp.bar.abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for out in got:
        for a, b in zip(out, want):
            assert torch.equal(a, b)

