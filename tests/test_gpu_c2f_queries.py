"""C2FPointTracker.track_queries: TAP-Vid query groups through the coarse-to-fine tracker, forward and backward, with
the label-independent stages of the clip in a few launches (fgvc_c2f_clip_weights) and every recurrence as a lane of
one cooperative chain (fgvc_c2f_point_clip_tail_lanes).  The reference is track() itself, group by group, on the sliced
and on the time-reversed clip: bit for bit."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


def _coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


BASE = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=6, radius_fine=5, with_first=True)


def _case(seed, T, t0s, per_group=4, C=64, Hc=8, Wc=12, s=4):
    g = torch.Generator().manual_seed(seed)
    fc, ff = _coherent(g, T, C, Hc, Wc).cuda(), _coherent(g, T, C, Hc * s, Wc * s).cuda()
    h, w = Hc * s * 2, Wc * s * 2
    P = per_group * len(t0s)
    xy = torch.rand(P, 2, generator=g) * torch.tensor([w - 1.0, h - 1.0])
    t = torch.tensor([t0s[i % len(t0s)] for i in range(P)], dtype=torch.float32)   # groups interleaved in the input
    return fc, ff, torch.cat([t[:, None], xy], dim=1), (h, w)


def _per_group_track(trk, fc, ff, qp, hw, bidirectional):
    """what a user gets from track() by hand: per query frame the sliced clip forward, the flipped prefix backward"""
    T = fc.shape[0]
    want = torch.zeros(T, qp.shape[0], 2, dtype=torch.float32, device="cuda")
    for t0 in sorted(set(int(v) for v in qp[:, 0].tolist())):
        idx = torch.nonzero(qp[:, 0] == t0).flatten().cuda()
        pts = qp[idx.cpu(), 1:]
        want[t0:, idx] = trk.track(fc[t0:], ff[t0:], pts, hw)[0]
        if bidirectional and t0 > 0:
            want[:t0 + 1, idx] = trk.track(fc[:t0 + 1].flip(0), ff[:t0 + 1].flip(0), pts, hw)[0].flip(0)
    return want


VARIANTS = {
    "base": {},
    "no_first": dict(with_first=False),
    "no_first_neighbor": dict(with_first_neighbor=False),
    "square": dict(mask_mode="square"),
    "k4": dict(topk=4),
    "k16": dict(topk=16),
    "tf32_fallback": dict(split="tf32"),                 # fine stage: one warp per candidate, weights-only form
    "long_memory": dict(precede_frames=11),              # 12 entries x 4 chunks = 48 lists: the serial merge branch
}
# (every other window variant has <= 4 entries x 4 chunks = 16 lists per query: the warp merge branch; the 8 x 12
# coarse map is one tile, so c2f_window_chunks gives 4 chunks)


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("bidirectional", [False, True])
def test_groups_equal_track_on_sliced_and_flipped_clips(variant, bidirectional):
    import fgvc_b200
    T = 14 if variant == "long_memory" else 9
    fc, ff, qp, hw = _case(11, T, [0, T // 2, T - 1])
    cfg = dict(BASE, bidirectional=bidirectional, **VARIANTS[variant])
    trk = fgvc_b200.C2FPointTracker(cfg)
    got = trk.track_queries(fc, ff, qp, hw)
    want = _per_group_track(trk, fc, ff, qp, hw, bidirectional)
    assert got.shape == (T, qp.shape[0], 2) and got.dtype == torch.float32
    assert torch.equal(got, want), float((got - want).abs().max())
    if not bidirectional:
        for i in range(qp.shape[0]):
            assert bool((got[:int(qp[i, 0]), i] == 0).all())


@pytest.mark.parametrize("bidirectional", [False, True])
def test_single_group_at_frame_0_equals_track(bidirectional):
    import fgvc_b200
    fc, ff, qp, hw = _case(5, 9, [0], per_group=7)
    trk = fgvc_b200.C2FPointTracker(dict(BASE, bidirectional=bidirectional))
    assert torch.equal(trk.track_queries(fc, ff, qp, hw), trk.track(fc, ff, qp[:, 1:], hw)[0])


def test_cfg3_geometry_groups_equal_track():
    """config-3-(ii) geometry: coarse 32 x 32 (r = 12), fine 128 x 128 (radius_fine 12), 256 x 256 image, precede 5"""
    import fgvc_b200
    g = torch.Generator().manual_seed(3302)
    T, C = 7, 256
    fc, ff = _coherent(g, T, C, 32, 32).cuda(), _coherent(g, T, C, 128, 128).cuda()
    xy = torch.rand(64, 2, generator=g) * 236 + 10
    qp = torch.cat([torch.tensor([0.0, 3.0, 6.0, 3.0]).repeat(16)[:, None], xy], dim=1)
    cfg = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12, with_first=True,
               bidirectional=True)
    trk = fgvc_b200.C2FPointTracker(cfg)
    got = trk.track_queries(fc, ff, qp, (256, 256))
    assert torch.equal(got, _per_group_track(trk, fc, ff, qp, (256, 256), True))


def test_backward_half_matches_oracle_loop():
    """frames before t0 against the oracle's coarse-to-fine loop on the flipped prefix (the bound of the c2f driver
    test: the up-sampled coarse peak is a plateau whose last bit decides img2coord's five pixels)"""
    import fgvc_b200
    torch.set_num_threads(os.cpu_count() or 8)
    g = torch.Generator().manual_seed(77)
    T, C, Hc, Wc, s, t0 = 6, 64, 8, 10, 4, 4
    fc, ff = _coherent(g, T, C, Hc, Wc), _coherent(g, T, C, Hc * s, Wc * s)
    h, w = Hc * s * 2, Wc * s * 2
    pts = torch.rand(6, 2, generator=g) * torch.tensor([w - 1.0, h - 1.0])
    cfg = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=6, radius_fine=5, with_first=True,
               bidirectional=True)
    qp = torch.cat([torch.full((6, 1), float(t0)), pts], dim=1)
    got = fgvc_b200.C2FPointTracker(cfg).track_queries(fc.cuda(), ff.cuda(), qp, (h, w)).cpu().numpy()
    _, want = O.track_clip_c2f_port(fc[:t0 + 1].flip(0).contiguous(), ff[:t0 + 1].flip(0).contiguous(), pts, (h, w), cfg)
    err = np.abs(got[:t0 + 1][::-1] - want).max(axis=-1)
    assert float((err <= 0.5).mean()) >= 0.9 and float(err.max()) <= 1.0, float(err.max())


def _launches_by_entry(monkeypatch, fn):
    from fgvc_b200 import _lib
    counts = {}
    orig = _lib.call

    def spy(name, *args):
        n0 = _lib.launch_count()
        orig(name, *args)
        counts[name] = counts.get(name, 0) + _lib.launch_count() - n0

    monkeypatch.setattr(_lib, "call", spy)
    fn()
    monkeypatch.setattr(_lib, "call", orig)
    return counts


def test_launch_counts_do_not_grow_with_groups(monkeypatch):
    import fgvc_b200
    T = 12
    runs = {}
    for t0s in ([0, 1], list(range(8))):
        fc, ff, qp, hw = _case(3, T, t0s, per_group=2)
        trk = fgvc_b200.C2FPointTracker(dict(BASE, bidirectional=True))
        counts = _launches_by_entry(monkeypatch, lambda: trk.track_queries(fc, ff, qp, hw))
        n_lanes = sum(1 for t0 in t0s if t0 < T - 1) + sum(1 for t0 in t0s if t0 > 0)
        runs[len(t0s)] = (counts["fgvc_c2f_clip_weights"], counts["fgvc_c2f_point_clip_tail_lanes"], n_lanes)
    (w2, c2, l2), (w8, c8, l8) = runs[2], runs[8]
    # coarse K1 per memory length (2 .. precede + 1), floor, window K1, weights: the same for 2 and for 8 groups
    assert w2 == w8 == 3 + 3, runs
    # the chain is one launch; the rest is a fixed number of launches (NCHW copies, K3) per lane
    per_lane = (c8 - c2) // (l8 - l2)
    assert (c8 - c2) % (l8 - l2) == 0 and c2 - per_lane * l2 == 1 and c8 - per_lane * l8 == 1, runs


def test_strided_tapvid_sample_end_to_end():
    import fgvc_b200
    from fgvc_b200 import metrics, synthetic as S
    T, h, w, N = 12, 64, 96, 9
    video = ((S.synthetic_video(T, h, w, seed=7).permute(0, 2, 3, 1).clamp(-1, 1) + 1) * 127.5).to(torch.uint8).numpy()
    g = np.random.default_rng(3)
    points = np.clip(np.cumsum(g.normal(0, 0.01, (N, T, 2)), axis=1) + g.uniform(0.2, 0.8, (N, 1, 2)), 0, 1)
    occluded = g.random((N, T)) < 0.2
    sample = metrics.tapvid_sample(dict(video=video, points=points, occluded=occluded), (h, w), query_mode="strided")
    rgbs = sample["rgbs"][0].cuda()
    fc = S.encode(S.davis_encoder(stride=8).cuda(), rgbs)
    ff = S.encode(S.davis_encoder(stride=2).cuda(), rgbs)
    cfg = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=6, radius_fine=6, with_first=True,
               bidirectional=True)
    qp = sample["query_points"][0]
    pred = fgvc_b200.C2FPointTracker(cfg).track_queries(fc, ff, qp, (h, w))
    assert sorted(set(qp[:, 0].tolist())) == [0, 5, 10]
    for i in range(qp.shape[0]):
        t0 = int(qp[i, 0])
        assert bool((pred[:t0, i] != 0).any(dim=-1).all()), i          # no (0, 0) row before the query frame
    traj, vis = sample["trajectories"].cuda(), sample["visibilities"].cuda()
    out = metrics.compute_tapvid_metrics(qp[None][..., [0, 2, 1]], ~vis.permute(0, 2, 1), traj.permute(0, 2, 1, 3),
                                         ~vis.permute(0, 2, 1), pred[None].permute(0, 2, 1, 3), "strided")
    assert out and all(bool(torch.isfinite(v).all()) for v in out.values())


def test_pinned_host_features_give_the_resident_result():
    import fgvc_b200
    fc, ff, qp, hw = _case(9, 9, [0, 4, 8])
    trk = fgvc_b200.C2FPointTracker(dict(BASE, bidirectional=True))
    want = trk.track_queries(fc, ff, qp, hw)
    got = trk.track_queries(fc.cpu().pin_memory(), ff.cpu().pin_memory(), qp, hw)
    assert torch.equal(got, want)
