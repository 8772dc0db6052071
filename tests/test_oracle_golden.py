"""The oracle restatement vs. the committed outputs of the genuine reference
(tests/golden/*.npz, written by oracle/gen_golden.py).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


PROP = ["rand_small", "rand_nonmask1", "coh_dupframe0", "coh_c256", "tiny_fewcands"]


@pytest.mark.parametrize("name", PROP)
def test_propagate_port_matches_reference(golden_dir, name):
    d = _load(golden_dir, f"prop_{name}.npz")
    q, k, v = (torch.from_numpy(d[x]) for x in "qkv")
    nr, topk, nml = int(d["neighbor_range"]), int(d["topk"]), int(d["non_mask_len"])
    H, W = q.shape[2:]
    mask = O.neighbor_mask(H, W, nr)
    out = O.propagate_port(q, k, v, mask=mask, temperature=0.07, topk=topk, step=64, non_mask_len=nml)
    assert torch.allclose(out, torch.from_numpy(d["out_v1"]), atol=2e-6, rtol=0)
    out2 = O.propagate_port(q, k, v, radius=nr // 2, temperature=0.07, topk=topk, step=64)
    assert torch.allclose(out2, torch.from_numpy(d["out_v2"]), atol=2e-6, rtol=0)


DENSE = [("softmax", {}), ("softmax_nonmask1", dict(non_mask_len=1)), ("cosine", dict(mode="cosine")),
         ("l2", dict(sim_mode="l2-distance")), ("nomask", None)]


@pytest.mark.parametrize("name,kw", DENSE)
def test_dense_port_matches_reference(golden_dir, name, kw):
    """topk=None: weights over ALL allowed candidates (local_attention.py:376-383)."""
    d = _load(golden_dir, "prop_dense.npz")
    q, k, v = (torch.from_numpy(d[x]) for x in "qkv")
    H, W = q.shape[2:]
    if kw is None:
        out = O.propagate_port(q, k, v, mask=None, temperature=0.07, topk=None)
    else:
        out = O.propagate_port(q, k, v, mask=O.neighbor_mask(H, W, int(d["neighbor_range"])), temperature=0.07,
                               topk=None, **kw)
    want = torch.from_numpy(d[name])
    assert torch.allclose(out, want, atol=2e-6, rtol=1e-6)


@pytest.mark.parametrize("name", PROP)
def test_propagate_exact_matches_reference(golden_dir, name):
    d = _load(golden_dir, f"prop_{name}.npz")
    q, k, v = (torch.from_numpy(d[x]) for x in "qkv")
    nr, topk, nml = int(d["neighbor_range"]), int(d["topk"]), int(d["non_mask_len"])
    T = k.shape[2]
    ex = O.propagate_exact(q, k, v, radius=nr // 2, temperature=0.07, topk=topk,
                           masked=[t >= nml for t in range(T)])
    rep = O.compare_labels(d["out_v1"][0], ex["out"], ex["gap"], gap_eps=1e-4)
    assert rep["max_abs_clear"] < 5e-6, rep
    # ambiguous queries are rare and the only place the two may disagree
    assert rep["n_ambiguous"] <= 0.02 * ex["gap"].numel() + 2, rep


def test_masks_match_reference(golden_dir):
    d = _load(golden_dir, "masks.npz")
    for key in d.files:
        mode, H, W, nr = key.split("_")
        got = O.neighbor_mask(int(H), int(W), int(nr), mode).numpy()
        assert (got == d[key]).all(), key


def test_c2f_matches_reference(golden_dir):
    d = _load(golden_dir, "c2f_small.npz")
    t = {k: torch.from_numpy(d[k]) for k in ("q", "k", "qf", "kf", "v")}
    H, W = t["q"].shape[2:]
    mask = O.neighbor_mask(H, W, int(d["neighbor_range"]))
    got = O.c2f_port(t["q"], t["k"], t["qf"], t["kf"], t["v"], mask, temperature=0.07,
                     topk=int(d["topk"]), radius_fine=int(d["radius_fine"]))
    assert torch.allclose(got["out"], torch.from_numpy(d["out"]), atol=5e-6, rtol=0)
    got64 = O.c2f_port(t["q"], t["k"], t["qf"], t["kf"], t["v"], mask, temperature=0.07,
                       topk=int(d["topk"]), radius_fine=int(d["radius_fine"]), dtype=torch.float64)
    assert (got64["out"].float() - torch.from_numpy(d["out"])).abs().max() < 5e-5


def test_img2coord_matches_reference(golden_dir):
    d = _load(golden_dir, "tracker.npz")
    got = O.img2coord_port(d["i2c_maps"])
    assert np.allclose(got, d["i2c_xy"], atol=1e-12)
    assert (got[:, 2, 1] == -1).all()


@pytest.mark.parametrize("tag", ["s8", "s2"])
def test_tracker_driver_matches_reference(golden_dir, tag):
    """forward_test grouping + forward_test_main loop, from the genuine encoder's features."""
    d = _load(golden_dir, "tracker.npz")
    feats = torch.from_numpy(d[f"{tag}_feats"])
    qp = d[f"{tag}_query_points"][0]
    rgbs = d[f"{tag}_rgbs"]
    T, (h, w) = rgbs.shape[1], rgbs.shape[3:]
    cfg = dict(precede_frames=int(d[f"{tag}_precede_frames"]), topk=10, temperature=0.07,
               neighbor_range=int(d[f"{tag}_neighbor_range"]), step=64, with_first=True,
               with_first_neighbor=True)
    pred = np.zeros((T, qp.shape[0], 2))
    remap = np.zeros_like(qp)
    col = 0
    for t0, idx in O.group_by_query_frame(qp):
        _, traj = O.track_clip_port(feats[t0:], torch.from_numpy(qp[idx, 1:]), (h, w), cfg)
        pred[t0:, col:col + len(idx)] = traj
        remap[col:col + len(idx)] = qp[idx]
        col += len(idx)
    assert np.allclose(remap, d[f"{tag}_query_points_remap"][0])
    assert np.abs(pred - d[f"{tag}_traj_pred"][0]).max() < 1e-3


def test_legacy_matches_reference(golden_dir):
    d = _load(golden_dir, "legacy.npz")
    a, b, img = (torch.from_numpy(d[k]) for k in ("a", "b", "img"))
    aff = O.compute_affinity_port(a, b, temperature=0.07, softmax_dim=1)
    assert torch.allclose(aff, torch.from_numpy(d["aff"]), atol=1e-6)
    prop = O.propagate_legacy_port(img, aff, topk=4)
    assert torch.allclose(prop, torch.from_numpy(d["prop"]), atol=1e-5)


def test_sharding_and_collect_order():
    # datasets/samplers/distributed_sampler.py:49-53 and apis/test.py:231-235
    assert O.shard_indices(10, 1, 4) == [1, 5, 9]
    assert O.shard_indices(10, 3, 4) == [3, 7, 1]
    parts = [[f"r{r}i{i}" for i in O.shard_indices(10, r, 4)] for r in range(4)]
    got = O.interleave_results(parts, 10)
    assert got == [f"r{i % 4}i{i}" for i in range(10)]


def test_memory_multiset_duplicates_frame0():
    assert O.memory_frames(1, 5) == [0, 0]
    assert O.memory_frames(3, 5) == [0, 0, 1, 2]
    assert O.memory_frames(8, 5) == [0, 3, 4, 5, 6, 7]
    assert O.memory_frames(3, 5, with_first=False) == [0, 1, 2]


@pytest.mark.parametrize("mode", ["first", "strided"])
def test_tapvid_metrics_match_reference(golden_dir, mode):
    d = _load(golden_dir, "tapvid_metrics.npz")
    got = O.tapvid_metrics_port(d["qp"], d["gt_occ"], d["gt"], d["pred_occ"], d["pred"], mode)
    from fgvc_b200 import metrics
    dev = metrics.compute_tapvid_metrics(*(torch.from_numpy(d[k]) for k in ("qp", "gt_occ", "gt", "pred_occ", "pred")),
                                         query_mode=mode)
    keys = [k[len(mode) + 2:] for k in d.files if k.startswith(mode + "__")]
    assert len(keys) == 13
    for k in keys:
        assert np.allclose(got[k], d[f"{mode}__{k}"], atol=1e-12), k
        assert np.allclose(dev[k].numpy(), d[f"{mode}__{k}"], atol=1e-12), k


def test_c2f_clip_loop_port_matches_genuine_operator_loop(golden_dir):
    """oracle.track_clip_c2f_port (the driver loop of fgvc_b200/c2f_tracker.py restated around c2f_port) against the
    same loop run around the GENUINE masked_attention_efficient_c2f (fixture written by oracle/gen_golden.py)."""
    d = np.load(os.path.join(golden_dir, "c2f_driver.npz"))
    cfg = dict(precede_frames=int(d["precede_frames"]), topk=int(d["topk"]), temperature=float(d["temperature"]),
               neighbor_range=int(d["neighbor_range"]), radius_fine=int(d["radius_fine"]), with_first=True)
    outs, traj = O.track_clip_c2f_port(torch.from_numpy(d["feats_c"]), torch.from_numpy(d["feats_f"]),
                                       torch.from_numpy(d["points"]), tuple(int(x) for x in d["image_hw"]), cfg)
    assert (torch.stack(outs) - torch.from_numpy(d["outs"])).abs().max() < 2e-6
    assert np.abs(traj - d["traj"]).max() < 1e-3


def test_nearest_resize_restatement_matches_pillow():
    """pil_nearest_interpolate (common/utils.py:39-56) goes through PIL's NEAREST: the oracle's index formula and the
    product's device version must pick the same source pixels as Pillow itself."""
    from PIL import Image
    from fgvc_b200.tracker import nearest_resize
    rs = np.random.RandomState(0)
    for (H, W, h, w) in [(48, 86, 24, 43), (37, 53, 18, 26), (20, 20, 7, 9), (480, 854, 240, 427), (9, 7, 9, 7)]:
        seg = rs.randint(0, 6, (H, W)).astype(np.uint8)
        want = np.asarray(Image.fromarray(seg).resize((w, h), Image.NEAREST))
        got = O.nearest_resize_port(torch.from_numpy(seg), (h, w)).numpy()
        assert (got == want).all(), (H, W, h, w)
        assert (nearest_resize(torch.from_numpy(seg), (h, w)).numpy() == want).all()


def test_correlation_unfold_restatement_is_the_windowed_dot_product():
    """oracle.correlation_unfold (the F.unfold restatement of mmcv.ops.Correlation, parity unpinned for that op)
    against an explicit loop over displacements: <q[y,x], k[y+dy,x+dx]>, zero outside the image, (dy, dx) row-major."""
    g = torch.Generator().manual_seed(2)
    q, k = torch.randn(2, 5, 6, 7, generator=g), torch.randn(2, 5, 6, 7, generator=g)
    r = 2
    got = O.correlation_unfold(q, k, r)
    kp = torch.nn.functional.pad(k, (r, r, r, r))
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            want = (q * kp[:, :, r + dy:r + dy + 6, r + dx:r + dx + 7]).sum(1)
            assert (got[:, (dy + r) * (2 * r + 1) + dx + r] - want).abs().max() < 1e-5


def test_davis_jf_pck_and_tapvid_packaging_match_the_genuine_functions(golden_dir):
    """fgvc_b200.metrics (device-side J & F, PCK, TAP-Vid record packaging) against outputs of the genuine
    mmpt functions (metrics.py:11-256, jhmdb_dataset.py:143-233, tapvid_evaluation_datasets.py:297-401)."""
    from fgvc_b200 import metrics as M
    d = np.load(os.path.join(golden_dir, "eval_metrics.npz"))
    got = M.jfm(d["jf_gt"], d["jf_res"])
    for k in ("JM", "JR", "JD", "FM", "FR", "FD"):
        assert np.allclose(np.asarray(got[k]), d[f"jf_{k}"], atol=1e-12, equal_nan=True), k
    assert np.allclose(M.db_eval_iou(d["jf_gt"][0], d["jf_res"][0]).numpy(), d["jf_iou_obj0"], atol=1e-12)
    assert np.allclose(M.db_eval_boundary(d["jf_gt"][0], d["jf_res"][0]).numpy(), d["jf_f_obj0"], atol=1e-12)
    dist = M.pck_distances(d["pck_pred"], d["pck_gt"])
    assert [x.numel() for x in dist] == d["pck_count"].tolist()
    assert np.allclose([float(x.sum()) for x in dist], d["pck_dist"], atol=1e-9)
    assert np.allclose(list(M.pck(dist).values()), d["pck_values"], atol=1e-9)
    h, w = (int(x) for x in d["tv_hw"])
    for mode in ("first", "strided"):
        s = M.tapvid_sample(dict(video=d["tv_video"], points=d["tv_points"], occluded=d["tv_occluded"]), (h, w), mode)
        q = d[f"tv_{mode}_query_points"]                               # [1,n,3] (t, y, x)
        assert np.allclose(s["query_points"].numpy(), q[:, :, [0, 2, 1]], atol=1e-5)
        assert np.allclose(s["trajectories"].numpy(), np.transpose(d[f"tv_{mode}_target_points"], (0, 2, 1, 3)), atol=1e-4)
        assert (s["visibilities"].numpy() == ~np.transpose(d[f"tv_{mode}_occluded"], (0, 2, 1))).all()
        assert s["rgbs"].shape == (1, d["tv_video"].shape[0], 3, h, w) and float(s["rgbs"].abs().max()) <= 1.0
