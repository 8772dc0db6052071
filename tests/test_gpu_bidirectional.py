"""Bidirectional point tracking (test_cfg.bidirectional): every group is also tracked to the frames before its query
frame, as the forward tracker does on the time-reversed clip, and all forward and backward recurrences of a clip run
as lanes of one multi-lane gather chain (csrc/gather.cu).  Needs a B200."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402

STRIDE = 2


def _coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


def _points(g, P, H, W):
    return torch.rand(P, 2, generator=g) * torch.tensor([W * STRIDE - 1.0, H * STRIDE - 1.0])


def _tracker(cfg, hr=False, bidirectional=True):
    import fgvc_b200
    cls = fgvc_b200.HRVanillaTracker if hr else fgvc_b200.VanillaTracker
    return cls(backbone=torch.nn.Identity(), test_cfg=dict(cfg, bidirectional=bidirectional))


def _run(cfg, feats, groups, hr=False, bidirectional=True):
    H, W = feats.shape[-2:]
    return _tracker(cfg, hr, bidirectional).propagate_points(feats, groups, (H * STRIDE, W * STRIDE))


BASE = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=10, with_first=True, with_first_neighbor=False)
VARIANTS = {
    "with_first": (BASE, False),
    "no_first": (dict(BASE, with_first=False), False),
    "v2": (dict(BASE, test_mode="v2"), False),
    "square": (dict(BASE, mask_mode="square"), False),
    "hr": (dict(BASE, with_first_neighbor=True), True),
}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_backward_half_is_the_forward_track_of_the_reversed_clip(variant):
    """Frames before t0 equal the forward tracker on feats.flip(0) from T-1-t0 bit for bit; frames from t0 on equal the
    forward-only run bit for bit."""
    cfg, hr = VARIANTS[variant]
    g = torch.Generator().manual_seed(51)
    T, C, H, W = 9, 64, 24, 32
    feats = _coherent(g, T, C, H, W).cuda()
    pts = _points(g, 6, H, W)
    for t0 in (0, 4, T - 1):
        both = _run(cfg, feats, [(t0, pts)], hr)[0]
        fwd = _run(cfg, feats, [(t0, pts)], hr, bidirectional=False)[0]
        rev = _run(cfg, feats.flip(0).contiguous(), [(T - 1 - t0, pts)], hr, bidirectional=False)[0]
        assert torch.equal(both[t0:], fwd[t0:]), (variant, t0)
        assert torch.equal(both[:t0], rev.flip(0)[:t0]), (variant, t0)
        if t0 > 0:
            assert bool((both[:t0] != 0).any(dim=-1).all())            # no zero-filled frame before the query


def test_many_groups_on_shared_lists(monkeypatch):
    """Queries at 0, 2, 5 and 7 of a 10-frame clip: K1 shared per (query frame, direction).  Each backward half equals
    the reversed single-group run, and the whole result the per-group K1 run, up to the order of exact ties."""
    g = torch.Generator().manual_seed(52)
    T, C, H, W = 10, 64, 24, 32
    feats = _coherent(g, T, C, H, W).cuda()
    groups = [(t0, _points(g, 3 + t0, H, W)) for t0 in (0, 2, 5, 7)]
    monkeypatch.delenv("FGVC_NO_SHARE", raising=False)
    shared = _run(BASE, feats, groups)
    monkeypatch.setenv("FGVC_NO_SHARE", "1")
    plain = _run(BASE, feats, groups)
    monkeypatch.delenv("FGVC_NO_SHARE", raising=False)
    for (t0, pts), a, b in zip(groups, shared, plain):
        assert a.shape == (T, pts.shape[0], 2)
        assert float((a - b).abs().max()) < 1e-3
        if t0 > 0:
            rev = _run(BASE, feats.flip(0).contiguous(), [(T - 1 - t0, pts)], bidirectional=False)[0]
            assert float((a[:t0] - rev.flip(0)[:t0]).abs().max()) < 1e-3, t0


def test_tracks_match_the_oracle_on_both_sides():
    g = torch.Generator().manual_seed(53)
    T, C, H, W = 8, 64, 24, 32
    feats = _coherent(g, T, C, H, W)
    cfg = dict(BASE, with_first_neighbor=True, step=64)
    groups = [(t0, _points(g, 5, H, W)) for t0 in (0, 3, T - 1)]
    got = _run(cfg, feats.cuda(), groups)
    hw = (H * STRIDE, W * STRIDE)
    for (t0, pts), tr in zip(groups, got):
        tr = tr.cpu().numpy()
        _, fwd = O.track_clip_port(feats[t0:], pts, hw, cfg)
        _, bwd = O.track_clip_port(feats.flip(0)[T - 1 - t0:], pts, hw, cfg)
        want = np.concatenate([bwd[::-1][:t0], fwd], axis=0)
        assert np.abs(tr - want).max() <= 0.5, t0


# lanes of unequal length and unequal Lp (3, 7 and 13 points); a 200 x 200 map puts more than 64 queries on every CTA
# of the lane chain (multi-pass branch); 2 points keep every lane's rows at one float4
GEOMS = {"one_pass": (9, 24, 32, (3, 7, 13)), "short_rows": (9, 24, 32, (2, 2, 2)), "large_map": (5, 200, 200, (2, 5, 3))}


def _per_lane(real):
    """engine.point_tail_lanes with one call, hence one gather chain, per lane"""
    def tail(lists, pair_ref, table, lanes, *a, **kw):
        for lane in lanes:
            real(lists, pair_ref, table, [lane], *a, **kw)
    return tail


@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("share", ["1", "0"])
@pytest.mark.parametrize("geom", sorted(GEOMS))
def test_lanes_are_an_exact_rescheduling(monkeypatch, geom, share, bidirectional):
    from fgvc_b200 import engine
    T, H, W, sizes = GEOMS[geom]
    g = torch.Generator().manual_seed(54)
    feats = _coherent(g, T, 64, H, W).cuda()
    t0s = (0, T // 2, T - 1)
    groups = [(t0, _points(g, n, H, W)) for t0, n in zip(t0s, sizes)]
    monkeypatch.setenv("FGVC_NO_SHARE", share)
    lanes = _run(BASE, feats, groups, bidirectional=bidirectional)
    monkeypatch.setattr(engine, "point_tail_lanes", _per_lane(engine.point_tail_lanes))
    per_lane = _run(BASE, feats, groups, bidirectional=bidirectional)
    for a, b in zip(lanes, per_lane):
        assert torch.equal(a, b)


def test_chain_is_two_launches_whatever_the_groups_and_length(monkeypatch):
    """weights + lane chain: 2 launches, one tail call per clip, bidirectional and forward-only; only the NCHW copy and
    K3 of every lane (2 each) grow with the lanes."""
    from fgvc_b200 import _lib, engine
    seen = []
    real = engine.point_tail_lanes

    def counted(lists, pair_ref, table, lanes, *a, **kw):
        before = _lib.launch_count()
        real(lists, pair_ref, table, lanes, *a, **kw)
        seen.append((_lib.launch_count() - before, len(lanes)))

    monkeypatch.setattr(engine, "point_tail_lanes", counted)
    # forward-only: no lane for a group queried at the last frame
    for bidirectional, n_lanes in ((True, [3, 8, 6]), (False, [2, 4, 3])):
        seen.clear()
        g = torch.Generator().manual_seed(55)
        for T, t0s in ((6, (0, 3)), (12, (0, 3, 6, 9, 11)), (20, (2, 9, 17))):
            feats = _coherent(g, T, 64, 16, 24).cuda()
            _run(BASE, feats, [(t0, _points(g, 4, 16, 24)) for t0 in t0s], bidirectional=bidirectional)
        assert [n for _, n in seen] == n_lanes, bidirectional
        assert all(d - 2 * n == 2 for d, n in seen), (bidirectional, seen)


def test_pinned_host_features_equal_the_resident_run():
    g = torch.Generator().manual_seed(56)
    T, C, H, W = 9, 64, 24, 32
    feats = _coherent(g, T, C, H, W)
    for groups in ([(4, _points(g, 5, H, W))], [(0, _points(g, 3, H, W)), (6, _points(g, 4, H, W))]):
        res = _run(BASE, feats.cuda(), groups)
        host = _run(BASE, feats.pin_memory(), groups)
        for a, b in zip(res, host):
            assert torch.equal(a, b)


def test_forward_test_on_a_strided_tapvid_sample():
    import fgvc_b200
    from fgvc_b200 import metrics, synthetic as S
    T, h, w, N = 12, 48, 64, 9
    video = ((S.synthetic_video(T, h, w, seed=7).permute(0, 2, 3, 1).clamp(-1, 1) + 1) * 127.5).to(torch.uint8).numpy()
    g = np.random.default_rng(3)
    points = np.clip(np.cumsum(g.normal(0, 0.01, (N, T, 2)), axis=1) + g.uniform(0.2, 0.8, (N, 1, 2)), 0, 1)
    occluded = g.random((N, T)) < 0.2
    sample = metrics.tapvid_sample(dict(video=video, points=points, occluded=occluded), (h, w), query_mode="strided")
    cfg = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=12, with_first=True, with_first_neighbor=True,
               bidirectional=True)
    torch.manual_seed(0)
    trk = fgvc_b200.VanillaTracker(backbone=dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2,),
                                                 pool_type="none"), test_cfg=cfg).cuda().eval()
    traj, vis, pred, vis_pred, qp = trk(test_mode=True, **sample)
    P = qp.shape[1]
    assert pred.shape == (1, T, P, 2) and bool((vis_pred == 0).all())
    assert sorted(set(qp[0, :, 0].tolist())) == [0, 5, 10]
    for i in range(P):
        t0 = int(qp[0, i, 0])
        assert bool((pred[0, :t0, i] != 0).any(dim=-1).all()), i          # no (0, 0) row before the query frame
    q_tyx = qp[..., [0, 2, 1]]
    out = metrics.compute_tapvid_metrics(q_tyx, ~vis.permute(0, 2, 1), traj.permute(0, 2, 1, 3),
                                         ~vis.permute(0, 2, 1), pred.permute(0, 2, 1, 3), "strided")
    assert out and all(bool(torch.isfinite(v).all()) for v in out.values())
