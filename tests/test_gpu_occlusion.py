"""Occlusion flags by forward-backward cycle consistency (test_cfg.cycle_occlusion): every prediction p_t of a query
group is re-tracked from t toward the query frame t0, stopping at s, and the point is visible at t iff the re-track
lands within `threshold` pixels of the group's own p_s.  The checks are lanes of one gather chain per chunk
(csrc/cycle.cu) after the tracking tail.  Needs a B200."""
import copy
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STRIDE = 2
BASE = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=10, with_first=True, with_first_neighbor=False)
DELTA = 4.0


def _coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


def _points(g, P, H, W, margin=0.0):
    lo = torch.tensor([margin, margin])
    return lo + torch.rand(P, 2, generator=g) * (torch.tensor([W * STRIDE - 1.0, H * STRIDE - 1.0]) - 2 * lo)


def _tracker(cfg, hr=False):
    import fgvc_b200
    cls = fgvc_b200.HRVanillaTracker if hr else fgvc_b200.VanillaTracker
    return cls(backbone=torch.nn.Identity(), test_cfg=cfg)


def _hw(feats):
    return (feats.shape[-2] * STRIDE, feats.shape[-1] * STRIDE)


def _checks(t0, T, frames, bidirectional):
    from fgvc_b200 import engine
    ts = [t for t in range(T) if t > t0 or (bidirectional and t < t0)]
    return [(t, engine.cycle_end(t, t0, frames)) for t in ts]


VARIANTS = {
    "circle": (BASE, False),
    "square": (dict(BASE, mask_mode="square"), False),
    "hr": (dict(BASE, with_first_neighbor=True), True),
}


@pytest.mark.parametrize("frames", [1, 3, None])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_cycle_positions_are_the_retracks_and_tracks_are_untouched(monkeypatch, variant, bidirectional, frames):
    """FGVC_NO_SHARE=1: each cycle position is bit for bit what propagate_points from (t, p_t) gives at s, and the flags
    follow from it; shared lists: within the shared-list bound of the bidirectional tests.  The tracks are the run
    without the key bit for bit in both modes."""
    cfg, hr = VARIANTS[variant]
    if hr and not (bidirectional and frames == 3):
        pytest.skip("the HR tracker once")
    cfg = dict(cfg, bidirectional=bidirectional)
    key = dict(cfg, cycle_occlusion=dict(frames=frames, threshold=DELTA))
    g = torch.Generator().manual_seed(61)
    T, C, H, W = 9, 64, 24, 32
    feats = _coherent(g, T, C, H, W).cuda()
    groups = [(t0, _points(g, n, H, W)) for t0, n in ((0, 5), (T // 2, 3), (T - 1, 6))]
    res = {}
    for share in ("1", "0"):
        monkeypatch.setenv("FGVC_NO_SHARE", share)
        plain = _tracker(cfg, hr).propagate_points(feats, groups, _hw(feats))
        tracks, vis, cyc = _tracker(key, hr).propagate_points(feats, groups, _hw(feats), return_cycle=True)
        for a, b in zip(plain, tracks):
            assert torch.equal(a, b), share
        res[share] = (tracks, vis, cyc)
    monkeypatch.setenv("FGVC_NO_SHARE", "1")
    tracks, vis, cyc = res["1"]
    n_checks = 0
    for (t0, pts), tr, v, c in zip(groups, tracks, vis, cyc):
        assert v.dtype == torch.bool and v.shape == (T, pts.shape[0]) and bool(v[t0].all())
        checked = set()
        for t, s in _checks(t0, T, frames, bidirectional):
            ref = _tracker(dict(cfg, bidirectional=True), hr).propagate_points(feats, [(t, tr[t].float())],
                                                                               _hw(feats))[0]
            assert torch.equal(c[t], ref[s]), (t0, t, s)
            d = (c[t] - tr[s]).norm(dim=-1)
            sure = (d - DELTA).abs() > 1e-3
            assert torch.equal(v[t][sure], (d <= DELTA)[sure]), (t0, t, s)
            checked.add(t)
            n_checks += 1
        for t in set(range(T)) - checked - {t0}:                # no prediction (forward-only, before t0): not visible
            assert not bool(v[t].any()) and not bool(c[t].any())
    assert n_checks > 0
    # shared lists: positions within the bound, flags equal where they are not on the threshold
    for (t0, _), a, b, va, vb, ta in zip(groups, res["0"][2], res["1"][2], res["0"][1], res["1"][1], res["0"][0]):
        assert float((a - b).abs().max()) < 1e-3, t0
        for t, s in _checks(t0, T, frames, bidirectional):
            d = (a[t] - ta[s]).norm(dim=-1)
            sure = (d - DELTA).abs() > 1e-3
            assert torch.equal(va[t][sure], vb[t][sure]), (t0, t)


def _k1_and_cycle_launches(monkeypatch, fn):
    from fgvc_b200 import _lib, engine
    launches, calls = {}, {}
    orig = _lib.call

    def spy(name, *args):
        n0 = _lib.launch_count()
        orig(name, *args)
        launches[name] = launches.get(name, 0) + _lib.launch_count() - n0
        calls[name] = calls.get(name, 0) + 1

    monkeypatch.setattr(_lib, "call", spy)
    monkeypatch.setattr(engine, "call", spy)
    out = fn()
    monkeypatch.setattr(_lib, "call", orig)
    monkeypatch.setattr(engine, "call", orig)
    k1 = sum(n for name, n in launches.items() if "topk" in name)
    return out, k1, calls.get("fgvc_point_cycle_lanes", 0), launches.get("fgvc_point_cycle_lanes", 0)


@pytest.mark.parametrize("share", ["1", "0"])
def test_launch_counts_and_chunks(monkeypatch, share):
    """K1 launches are the same with and without the key; a cycle call is 6 launches (seeding, weights, chain, NCHW
    copy, K3, decision) whatever the number of groups; a small max_bytes splits the checks into several calls with the
    same result bit for bit"""
    monkeypatch.setenv("FGVC_NO_SHARE", share)
    g = torch.Generator().manual_seed(62)
    T, C, H, W = 12, 64, 16, 24
    feats = _coherent(g, T, C, H, W).cuda()
    cfg = dict(BASE, bidirectional=True)
    per_call = set()
    for t0s in ((0, 5), (0, 3, 6, 9, 11)):
        groups = [(t0, _points(g, 4, H, W)) for t0 in t0s]
        _, k1_plain, _, _ = _k1_and_cycle_launches(
            monkeypatch, lambda: _tracker(cfg).propagate_points(feats, groups, _hw(feats)))
        key = dict(cfg, cycle_occlusion=dict(frames=None, threshold=DELTA))
        one, k1_key, calls, launches = _k1_and_cycle_launches(
            monkeypatch, lambda: _tracker(key).propagate_points(feats, groups, _hw(feats), return_cycle=True))
        assert k1_key == k1_plain and calls == 1, (t0s, k1_key, k1_plain, calls)
        per_call.add(launches)
        small = dict(cfg, cycle_occlusion=dict(frames=None, threshold=DELTA, max_bytes=12 * H * W * 4 * 8))
        many, _, calls, launches = _k1_and_cycle_launches(
            monkeypatch, lambda: _tracker(small).propagate_points(feats, groups, _hw(feats), return_cycle=True))
        assert calls > 2 and launches == 6 * calls, (calls, launches)
        for a, b in zip(one, many):
            for x, y in zip(a, b):
                assert torch.equal(x, y)
    assert per_call == {6}, per_call


def _flagged(vis, frames):
    return float((~vis[frames]).float().mean())


def test_static_clip_is_visible_everywhere():
    g = torch.Generator().manual_seed(63)
    T, C, H, W = 10, 64, 24, 32
    feats = _coherent(g, 1, C, H, W).expand(T, -1, -1, -1).contiguous().cuda()
    groups = [(t0, _points(g, 12, H, W, margin=16.0)) for t0 in (0, T // 2, T - 1)]
    for hr in (False, True):
        cfg = dict(BASE, with_first_neighbor=hr, bidirectional=True, cycle_occlusion=dict(frames=None, threshold=4.0))
        _, vis = _tracker(cfg, hr).propagate_points(feats, groups, _hw(feats))
        for (t0, _), v in zip(groups, vis):
            assert bool(v.all()), (hr, t0, float((~v).float().mean()))


def test_scene_cut_is_flagged():
    """frames 0..k-1 one static scene, k..T-1 another (another seed): with frames=None every check of a frame after the
    cut re-tracks across it, so its landing point is unrelated to the track at t0 -- the first memory frame is matched
    without the radius mask (with_first_neighbor=False), so it can be anywhere in the image.  A landing point uniform
    over the 48 x 64 image falls within 4 px of a given point with probability ~pi 16 / 3072 = 1.6 %, so at least half
    of the entries after the cut must be flagged; before the cut the clip is static and none is."""
    g = torch.Generator().manual_seed(64)
    T, k, C, H, W = 12, 6, 64, 24, 32
    a, b = _coherent(g, 1, C, H, W), _coherent(torch.Generator().manual_seed(640), 1, C, H, W)
    feats = torch.cat([a.expand(k, -1, -1, -1), b.expand(T - k, -1, -1, -1)]).contiguous().cuda()
    groups = [(0, _points(g, 32, H, W, margin=16.0))]
    cfg = dict(BASE, cycle_occlusion=dict(frames=None, threshold=4.0))
    _, vis = _tracker(cfg).propagate_points(feats, groups, _hw(feats))
    before, after = _flagged(vis[0], slice(1, k)), _flagged(vis[0], slice(k, T))
    msg = f"flagged share before the cut {before:.3f}, after it {after:.3f}"
    print(msg)
    assert before == 0.0 and after >= 0.5, msg


def _model(cfg):
    import fgvc_b200
    torch.manual_seed(0)
    return fgvc_b200.VanillaTracker(backbone=dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2,),
                                                  pool_type="none"), test_cfg=cfg).cuda().eval()


def _sample(T=12, h=48, w=64, N=9, seed=3):
    from fgvc_b200 import metrics, synthetic as S
    video = ((S.synthetic_video(T, h, w, seed=7).permute(0, 2, 3, 1).clamp(-1, 1) + 1) * 127.5).to(torch.uint8).numpy()
    rng = np.random.default_rng(seed)
    points = np.clip(np.cumsum(rng.normal(0, 0.01, (N, T, 2)), axis=1) + rng.uniform(0.2, 0.8, (N, 1, 2)), 0, 1)
    occluded = rng.random((N, T)) < 0.2
    return metrics.tapvid_sample(dict(video=video, points=points, occluded=occluded), (h, w), query_mode="strided")


CFG_MODEL = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=12, with_first=True, with_first_neighbor=True,
                 bidirectional=True, cycle_occlusion=dict(frames=3, threshold=4.0))


def test_forward_test_fills_vis_pred_and_the_metrics_use_it():
    from fgvc_b200 import metrics
    sample = _sample()
    key = _model(CFG_MODEL)
    plain = _model({k: v for k, v in CFG_MODEL.items() if k != "cycle_occlusion"})
    with torch.no_grad():
        traj, vis, pred, vis_pred, qp = key(test_mode=True, **sample)
        out_plain = plain(test_mode=True, **sample)
    assert torch.equal(pred, out_plain[2]) and bool((out_plain[3] == 0).all())
    assert vis_pred.dtype == vis.dtype and vis_pred.shape == vis.shape
    T, P = vis.shape[1:]
    for i in range(P):
        assert bool(vis_pred[0, int(qp[0, i, 0]), i])                  # visible at the query frame
    q_tyx = qp[..., [0, 2, 1]]
    gt_occ, pred_occ = ~vis.permute(0, 2, 1).bool(), ~vis_pred.permute(0, 2, 1).bool()
    out = metrics.compute_tapvid_metrics(q_tyx, gt_occ, traj.permute(0, 2, 1, 3), pred_occ, pred.permute(0, 2, 1, 3),
                                         "strided")
    assert out and all(bool(torch.isfinite(v).all()) for v in out.values())
    ev = torch.ones(P, T, dtype=torch.bool, device=vis.device)
    ev[torch.arange(P), qp[0, :, 0].long()] = False
    want = float(((pred_occ[0] == gt_occ[0]) & ev).sum()) / float(ev.sum())
    assert abs(float(out["occlusion_accuracy"][0]) - want) < 1e-12


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


def test_two_phase_split_equals_one_rank(monkeypatch):
    """shard=(rank, 2) on two threads: the checks' jobs in the frame-sharded K1, the checks over each rank's points, the
    flags gathered with the tracks -- every rank's 5-tuple is the one-rank result bit for bit"""
    import torch.distributed as dist
    model = _model(CFG_MODEL)
    models = [model, copy.deepcopy(model)]
    sample = _sample(T=10, N=13, seed=21)
    with torch.no_grad():
        want = model(test_mode=True, **sample)
    grp = _FakeGroup(2)
    monkeypatch.setattr(dist, "get_backend", lambda *a: "nccl")
    monkeypatch.setattr(dist, "all_gather", grp.all_gather)
    monkeypatch.setattr(dist, "all_gather_into_tensor", grp.all_gather_into_tensor)
    got, errors = [None, None], []

    def rank_main(r):
        grp.local.rank = r
        try:
            with torch.no_grad():
                got[r] = models[r](test_mode=True, shard=(r, 2), **sample)
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


def test_c2f_tracker_rejects_the_key():
    from fgvc_b200.c2f_tracker import C2FTracker
    with pytest.raises(NotImplementedError):
        C2FTracker(backbone=torch.nn.Identity(), test_cfg=dict(BASE, radius_fine=5, cycle_occlusion=dict(
            frames=1, threshold=4.0)))


@pytest.mark.parametrize("frames", [1, None])
def test_one_group_tracks_are_untouched(frames):
    """one group: no shared lists; the checks' K1 jobs join the tracking launch with the tracking jobs' tiling"""
    g = torch.Generator().manual_seed(65)
    T, C, H, W = 20, 64, 32, 48
    feats = _coherent(g, T, C, H, W).cuda()
    groups = [(4, _points(g, 40, H, W))]
    cfg = dict(BASE, with_first_neighbor=True, bidirectional=True)
    plain = _tracker(cfg).propagate_points(feats, groups, _hw(feats))
    tracks, _ = _tracker(dict(cfg, cycle_occlusion=dict(frames=frames, threshold=DELTA))).propagate_points(
        feats, groups, _hw(feats))
    assert torch.equal(plain[0], tracks[0])
