"""Mask propagation from an annotated frame t0 anywhere in the clip (MaskClipPropagator / propagate_masks /
forward_test_vos with ``ref_frame``): the frames after t0 are the forward propagation of the clip from t0, the frames
before it the forward propagation of the time-reversed clip from t0, and both directions run as the two lanes of one
fgvc_mask_clip_tail_lanes call (csrc/clip.cu).  Needs a B200."""
import ctypes

import numpy as np
import pytest
import torch

from fgvc_b200 import _lib, engine
from fgvc_b200._lib import call, ptr, stream_ptr
from oracle import oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")


def _coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


def _seg(H, W, L):
    """blocks of L labels: every object has pixels, and plenty of boundaries"""
    return (torch.arange(H)[:, None] // 7 * 3 + torch.arange(W)[None, :] // 9) % L


def _tracker(cfg):
    import fgvc_b200
    return fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=cfg)


BASE = dict(precede_frames=4, topk=10, temperature=0.07, neighbor_range=12, with_first=True, with_first_neighbor=True)
VARIANTS = {
    "with_first": BASE,
    "no_first": dict(BASE, with_first=False),
    "first_masked": dict(BASE, with_first_neighbor=False),
    "square": dict(BASE, mask_mode="square"),
    "no_radius": dict(BASE, neighbor_range=None),
    "hard_prop": dict(BASE, hard_prop=True),
    "hard_prop_no_first": dict(BASE, hard_prop=True, with_first=False),
}


def _check_halves(cfg, feats, L, t0, out_hw):
    """propagate_masks(ref_frame=t0) against the sliced (t >= t0) and the flipped (t <= t0) frame-0 runs, bit for bit"""
    T, _, H, W = feats.shape
    seg = _seg(H, W, L)
    trk = _tracker(cfg)
    maps, masks = (x.clone() for x in trk.propagate_masks(feats, seg, out_hw, L, ref_frame=t0))
    fm, fk = trk.propagate_masks(feats[t0:].contiguous(), seg, out_hw, L)
    assert torch.equal(maps[t0:], fm) and torch.equal(masks[t0:], fk), t0
    bm, bk = trk.propagate_masks(feats[:t0 + 1].flip(0).contiguous(), seg, out_hw, L)
    assert torch.equal(maps[:t0 + 1], bm.flip(0)) and torch.equal(masks[:t0 + 1], bk.flip(0)), t0
    assert int(masks[0].unique().numel()) > 1 and int(masks[-1].unique().numel()) > 1     # not a blank end


@pytest.mark.parametrize("where", ["mid", "last"])
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_halves_equal_the_sliced_and_flipped_runs(variant, where):
    g = torch.Generator().manual_seed(61)
    T, C, H, W, L = 20, 64, 32, 48, 4
    feats = _coherent(g, T, C, H, W).cuda()
    t0 = {"mid": 9, "last": T - 1}[where]
    _check_halves(VARIANTS[variant], feats, L, t0, (4 * H, 4 * W))


def test_halves_at_the_config2_map_size():
    """60 x 107 x 256 (the f16 tensor engine of K1, packed query tiles), 11 objects, precede 20, r = 12"""
    g = torch.Generator().manual_seed(62)
    T, C, H, W, L = 24, 256, 60, 107, 11
    feats = _coherent(g, T, C, H, W).cuda()
    cfg = dict(precede_frames=20, topk=10, temperature=0.07, neighbor_range=24, with_first=True,
               with_first_neighbor=True)
    _check_halves(cfg, feats, L, 10, (480, 856))


def test_frame_zero_is_the_call_without_the_argument():
    """ref_frame=0 takes today's path: same maps and masks bit for bit, same number of kernel launches"""
    g = torch.Generator().manual_seed(63)
    T, C, H, W, L = 14, 64, 32, 48, 5
    feats = _coherent(g, T, C, H, W).cuda()
    seg = _seg(H, W, L)
    for cfg in (BASE, dict(BASE, hard_prop=True)):
        trk = _tracker(cfg)
        n0 = _lib.launch_count()
        a = [x.clone() for x in trk.propagate_masks(feats, seg, (4 * H, 4 * W), L)]
        n1 = _lib.launch_count()
        b = trk.propagate_masks(feats, seg, (4 * H, 4 * W), L, ref_frame=0)
        n2 = _lib.launch_count()
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert n1 - n0 == n2 - n1


def test_tail_is_a_fixed_number_of_launches(monkeypatch):
    """weights + lane chain + (one NCHW copy) + min-max + arg-max, whatever T and t0"""
    seen = []
    real = engine.MaskClipPropagator._tail_lanes

    def counted(self, want_maps):
        n0 = _lib.launch_count()
        real(self, want_maps)
        seen.append(_lib.launch_count() - n0)

    monkeypatch.setattr(engine.MaskClipPropagator, "_tail_lanes", counted)
    g = torch.Generator().manual_seed(64)
    C, H, W, L = 64, 24, 32, 4
    for T, t0s in ((6, (3, 5)), (13, (6, 1)), (31, (15, 30))):
        feats = _coherent(g, T, C, H, W).cuda()
        onehot = torch.nn.functional.one_hot(_seg(H, W, L), L).permute(2, 0, 1).float().contiguous().cuda()
        for t0 in t0s:
            clip = engine.MaskClipPropagator(T, C, H, W, L, (2 * H, 2 * W), BASE, torch.device(DEV), ref_frame=t0)
            clip.run(feats, onehot, want_maps=True)
            clip.run(feats, onehot, want_maps=False)
    assert seen == [5, 4] * 6, seen


# ------------------------------------------------------------------ the C entry against one mask tail per lane
def _k1(feats, table, cfg):
    T, C, H, W = feats.shape
    bank = engine.FeatureBank(T, C, H, W, DEV)
    bank.load_frames(feats)
    return engine.affinity_topk(bank, table, cfg["neighbor_range"] // 2, cfg["topk"])


def _single_tail(lists, table, j0, j1, lab, L, Lp, H, W, out_hw, masks, maps, flags=0):
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    nbytes = int(_lib.load().fgvc_chain_workspace_bytes(j1 - j0, H * W, lists.K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    scratch = torch.empty((j1 - j0) * 2 * L, dtype=torch.float32, device=DEV)
    call("fgvc_mask_clip_tail", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, ptr(jobs), ptr(jobs_host), j0, j1,
         ptr(mem_label), H, W, 0.07, flags, ptr(lab), Lp, L, out_hw[0], out_hw[1], ptr(scratch), ptr(masks), ptr(maps),
         ptr(ws), nbytes, stream_ptr())


def _lanes_tail(lists, table, lanes, lab, H, W, out_hw, masks, maps, flags=0):
    """lanes: [(job_begin, job_end, L, lab_offset)]"""
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    host = (_lib.Lane * len(lanes))(*[_lib.Lane(a, b, L, engine.pad4(L), off, 0) for a, b, L, off in lanes])
    lanes_dev = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(DEV)
    jb, je = min(ln[0] for ln in lanes), max(ln[1] for ln in lanes)
    nbytes = int(_lib.load().fgvc_chain_workspace_bytes(je - jb, H * W, lists.K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    scratch = torch.empty(sum((b - a) * 2 * L for a, b, L, _ in lanes), dtype=torch.float32, device=DEV)
    call("fgvc_mask_clip_tail_lanes", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, None, ptr(jobs),
         ptr(jobs_host), ptr(lanes_dev), ctypes.c_void_p(ctypes.addressof(host)), len(lanes), ptr(mem_label), H, W, 0.07,
         flags, ptr(lab), out_hw[0], out_hw[1], ptr(scratch), ptr(masks), ptr(maps) if maps is not None else None, ptr(ws),
         nbytes, stream_ptr())


def _onehot_bank(T, L, H, W, slot, g):
    Lp = engine.pad4(L)
    lab = torch.full((T, H * W, Lp), NAN, device=DEV)
    seg = torch.randint(0, L, (H // 4 + 1, W // 4 + 1), generator=g).repeat_interleave(4, 0).repeat_interleave(4, 1)
    oh = torch.nn.functional.one_hot(seg[:H, :W].reshape(-1), Lp).float()
    oh[:, L:] = 0
    lab[slot] = oh.to(DEV)
    return lab


# name -> (T, H, W): 32 x 48 puts every CTA of the lane chain in its one-pass branch; 200 x 200 has more than 64
# queries per CTA at any occupancy (the multi-pass branch)
GEOMS = {"one_pass": (12, 32, 48), "multi_pass": (5, 200, 200)}


@pytest.mark.parametrize("maps_too", [True, False])
@pytest.mark.parametrize("geom", sorted(GEOMS))
def test_lanes_on_one_bank_equal_one_tail_per_lane(geom, maps_too):
    """the two directions of one annotated frame (unequal lengths, L <= 4 and L > 4) on one shared bank"""
    T, H, W = GEOMS[geom]
    g = torch.Generator().manual_seed(65)
    feats = _coherent(g, T, 64, H, W).cuda()
    t0 = 1 if T < 8 else 3
    table, _ = engine.query_job_table([t0], T, BASE["precede_frames"], True, True, lambda mem: 0)
    lists = _k1(feats, table, BASE)
    n_fwd = T - 1 - t0
    out_hw = (2 * H - 3, 2 * W + 5)
    for L in (3, 6):
        Lp = engine.pad4(L)
        lab0 = _onehot_bank(T, L, H, W, t0, g)
        lab_a, lab_b = lab0.clone(), lab0.clone()
        masks_a = torch.zeros(T, *out_hw, dtype=torch.uint8, device=DEV)
        masks_b = masks_a.clone()
        maps_a = torch.full((T, L, H * W), NAN, device=DEV)
        maps_b = maps_a.clone()
        _lanes_tail(lists, table, [(0, n_fwd, L, 0), (n_fwd, len(table), L, 0)], lab_a, H, W, out_hw, masks_a,
                    maps_a if maps_too else None)
        for j0, j1 in ((0, n_fwd), (n_fwd, len(table))):
            _single_tail(lists, table, j0, j1, lab_b, L, Lp, H, W, out_hw, masks_b, maps_b)
        torch.cuda.synchronize()
        assert torch.equal(masks_a, masks_b), L
        assert torch.equal(lab_a.nan_to_num(7.0), lab_b.nan_to_num(7.0)), L
        if maps_too:
            done = [t for t in range(T) if t != t0]
            assert torch.equal(maps_a[done], maps_b[done]), L


@pytest.mark.parametrize("geom", sorted(GEOMS))
def test_lanes_on_separate_banks_equal_one_tail_per_lane(geom):
    """two lanes with their own banks and label counts (3 and 5 objects): frame 0 forward to k, frame T-1 backward to
    k + 1 (distinct out_slots), one call"""
    T, H, W = GEOMS[geom]
    g = torch.Generator().manual_seed(66)
    feats = _coherent(g, T, 64, H, W).cuda()
    k = T // 2 - 1
    table = engine.JobTable()
    for t in range(1, k + 1):
        mem = engine.track_memory(t, 0, T, BASE["precede_frames"], True)
        table.add(t, mem, mem, t, unmasked=1)
    n_a = len(table)
    for t in range(T - 2, k, -1):
        mem = engine.track_memory(t, T - 1, T, BASE["precede_frames"], True)
        table.add(t, mem, mem, t, unmasked=1)
    lists = _k1(feats, table, BASE)
    LA, LB = 3, 5
    bank_a, bank_b = _onehot_bank(T, LA, H, W, 0, g), _onehot_bank(T, LB, H, W, T - 1, g)
    lab = torch.cat([bank_a.flatten(), bank_b.flatten()])
    out_hw = (3 * H, 3 * W)
    masks = torch.zeros(T, *out_hw, dtype=torch.uint8, device=DEV)
    maps = torch.full((T * LB * H * W,), NAN, device=DEV)
    _lanes_tail(lists, table, [(0, n_a, LA, 0), (n_a, len(table), LB, bank_a.numel())], lab, H, W, out_hw, masks, maps)
    ref_masks = torch.zeros_like(masks)
    ref_a, ref_b = torch.full((T, LA, H * W), NAN, device=DEV), torch.full((T, LB, H * W), NAN, device=DEV)
    _single_tail(lists, table, 0, n_a, bank_a, LA, 4, H, W, out_hw, ref_masks, ref_a)
    _single_tail(lists, table, n_a, len(table), bank_b, LB, 8, H, W, out_hw, ref_masks, ref_b)
    torch.cuda.synchronize()
    assert torch.equal(masks[1:T - 1], ref_masks[1:T - 1])
    assert torch.equal(lab[:bank_a.numel()].nan_to_num(7.0), bank_a.flatten().nan_to_num(7.0))
    assert torch.equal(lab[bank_a.numel():].nan_to_num(7.0), bank_b.flatten().nan_to_num(7.0))
    n = H * W
    for t in range(1, k + 1):
        assert torch.equal(maps[t * LA * n:(t + 1) * LA * n].view(LA, n), ref_a[t]), t
    for t in range(k + 1, T - 1):
        assert torch.equal(maps[t * LB * n:(t + 1) * LB * n].view(LB, n), ref_b[t]), t


def test_bad_lane_tables_are_refused():
    lib = _lib.load()
    H, W, L = 8, 8, 3
    table = engine.JobTable()
    table.add(1, [0], [0], 1)
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    val = torch.zeros(1, 1, H * W, 10, device=DEV)
    idx = torch.zeros(1, 1, H * W, 10, dtype=torch.int32, device=DEV)
    lab = torch.zeros(2, H * W, 4, device=DEV)
    scratch = torch.zeros(64, device=DEV)
    masks = torch.zeros(2, H, W, dtype=torch.uint8, device=DEV)
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    good = (0, 1, L, 4, 0, 0)
    cases = {
        "empty lane": ([(0, 0, L, 4, 0, 0)], 10, 1, None),
        "L > 255": ([(0, 1, 256, 256, 0, 0)], 10, 1, None),
        "Lp % 4": ([(0, 1, L, 6, 0, 0)], 10, 1, None),
        "Lp < L": ([(0, 1, 5, 4, 0, 0)], 10, 1, None),
        "lab_offset alignment": ([(0, 1, L, 4, 2, 0)], 10, 1, None),
        "coord_offset": ([(0, 1, L, 4, 0, 2)], 10, 1, None),
        "K = 17": ([good], 17, 1, None),
        "K = 0": ([good], 0, 1, None),
        "no lanes": ([], 10, 1, None),
        "shared lists with groups": ([good], 10, 2, torch.zeros(1, dtype=torch.int32, device=DEV)),
    }
    for name, (lanes, K, groups, pair_ref) in cases.items():
        host = (_lib.Lane * max(1, len(lanes)))(*[_lib.Lane(*ln) for ln in lanes])
        lanes_dev = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(DEV)
        rc = lib.fgvc_mask_clip_tail_lanes(ptr(val), ptr(idx), K, groups, ptr(pair_ref) if pair_ref is not None else None,
                                           ptr(jobs), ptr(jobs_host), ptr(lanes_dev),
                                           ctypes.c_void_p(ctypes.addressof(host)), len(lanes), ptr(mem_label), H, W,
                                           0.07, 0, ptr(lab), H, W, ptr(scratch), ptr(masks), None, ptr(ws),
                                           ws.numel(), stream_ptr())
        assert rc == _lib.ERR_INVALID, name
        msg = lib.fgvc_last_error().decode()
        assert msg.startswith("fgvc_mask_clip_tail_lanes: "), (name, msg)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ the HR tracker's VOS entry
def _hr_tracker(cfg):
    import fgvc_b200
    torch.manual_seed(0)
    return fgvc_b200.HRVanillaTracker(stride=2, backbone=dict(type="ResNet", depth=18, strides=(1, 1, 1, 4),
                                                              out_indices=(2,), pool_type="none"),
                                      test_cfg=cfg).cuda().eval()


@pytest.mark.parametrize("hard_prop", [False, True])
def test_hr_vos_entry_from_a_middle_frame_matches_the_oracle(hard_prop):
    """forward_test_vos(ref_frame=t0) against oracle.track_masks_hr_port on feats[t0:] and on feats[:t0+1] reversed,
    with the tolerance of the frame-0 entry's oracle test; then the padded / resized branch against the entry's own
    frame-0 runs on the sliced and the reversed clip."""
    from fgvc_b200 import synthetic as S
    cfg = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=10, with_first=True, hard_prop=hard_prop)
    trk = _hr_tracker(cfg)
    T, h, w, t0 = 9, 48, 64, 4
    frames = S.synthetic_video(T, h, w, seed=4)
    imgs = frames.transpose(0, 1)[None, None]                          # [1,1,3,T,h,w]
    seg = S.voronoi_mask(h, w, 4, seed=2)
    out = trk.forward_test_vos(imgs, seg[None], [dict(original_shape=(h, w, 3))], ref_frame=t0)[0]
    assert out.shape == (T, h, w)
    feats = trk.get_feats(frames.cuda()).cpu()
    _, fwd = O.track_masks_hr_port(feats[t0:], seg, (h, w), cfg)
    _, bwd = O.track_masks_hr_port(feats[:t0 + 1].flip(0), seg, (h, w), cfg)
    want = torch.cat([bwd.flip(0)[:t0], fwd])
    agree = (torch.from_numpy(out.astype(np.int64)) == want).float().mean(dim=(1, 2))
    assert float(agree.min()) >= 0.995, agree
    assert bool((torch.from_numpy(out[t0].astype(np.int64)) == seg).all())
    # padded input, another original size: the reference's resize chain on the label maps of both directions
    ip, sp, meta = imgs[..., :47, :63], seg[None, :47, :63], [dict(original_shape=(60, 80, 3))]
    out2 = trk.forward_test_vos(ip, sp, meta, ref_frame=t0)[0]
    assert out2.shape == (T, 60, 80)
    f2 = trk.forward_test_vos(ip[:, :, :, t0:], sp, meta)[0]
    b2 = trk.forward_test_vos(ip[:, :, :, :t0 + 1].flip(3), sp, meta)[0]
    want2 = np.concatenate([b2[::-1][:t0], f2])
    agree2 = (out2 == want2).reshape(T, -1).mean(axis=1)
    assert float(agree2.min()) >= 0.995, agree2
    assert (out2[t0] == f2[0]).all()


def test_hr_vos_entry_single_frame():
    from fgvc_b200 import synthetic as S
    trk = _hr_tracker(dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=10, with_first=True))
    frames = S.synthetic_video(1, 32, 32, seed=5)
    seg = S.voronoi_mask(32, 32, 3, seed=1)
    out = trk.forward_test_vos(frames.transpose(0, 1)[None, None], seg[None], [dict(original_shape=(32, 32, 3))],
                               ref_frame=0)[0]
    assert out.shape == (1, 32, 32) and bool((torch.from_numpy(out[0].astype(np.int64)) == seg).all())
    with pytest.raises(ValueError):
        trk.forward_test_vos(frames.transpose(0, 1)[None, None], seg[None], [dict(original_shape=(32, 32, 3))],
                             ref_frame=1)
