"""The label-side kernels, each called directly through the C ABI on inputs built by hand (top-k lists, job tables,
label banks) and pinned to a float64 reference: the gather of the top-k winners and the persistent gather chain
(csrc/gather.cu), the label layout transforms, up-sampling, hardening and Gaussian labels (csrc/prep.cu) and the three
mask decode entry points (csrc/coords.cu).  No affinity kernel runs, so every expectation is exact or float64.

Source coordinates of the bilinear kernels: like ATen's fp32 kernel they compute s = max((d + 0.5) * (in / out) - 0.5, 0)
in fp32 (in / out rounded once, then one fused multiply-add).  A float64 coordinate moves the weights by up to ulp(s),
8e-6 at s = 100, far more than the fp32 rounding of the values, so the references take the coordinate as the kernels
compute it and do everything after it in float64.
"""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fgvc_b200 import _lib, engine
from fgvc_b200._lib import call, ptr, stream_ptr

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
PAD_ID = -2          # index of a zero-padded window position in the references


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ----------------------------------------------------------------------------------------------- top-k lists
def _lists(g, n_mems, groups, n_pix, K, lo, hi, empty=0.25):
    """Flat lists [n_jobs, n_pix, groups * K] (``_pack`` gives the [job][group][query][K] layout): per query, distinct
    values in [lo, hi) in no particular order, empty slots (-inf / -1) anywhere, and now and then an index -1 with a
    large value (empty as well: the index decides).  Key positions are drawn from each job's memory list."""
    n_jobs, N = len(n_mems), groups * K
    shape = (n_jobs, n_pix, N)
    rank = torch.argsort(torch.rand(shape, generator=g), dim=-1).double()
    val = lo + (hi - lo) * (rank + 0.5 + 0.4 * torch.rand(n_jobs, n_pix, 1, generator=g, dtype=torch.float64)) / (N + 1)
    pos = (torch.rand(shape, generator=g, dtype=torch.float64) * torch.tensor(n_mems).view(-1, 1, 1)).long()
    idx = pos * n_pix + torch.randint(0, n_pix, shape, generator=g)
    u = torch.rand(shape, generator=g)
    val, idx = torch.where(u < empty, -math.inf, val), torch.where(u < empty, -1, idx)
    junk = u > 0.97
    val, idx = torch.where(junk, 3.0, val), torch.where(junk, -1, idx)
    return val.float(), idx.int()


def _pack(val, idx, groups, K):
    n_jobs, n_pix, _ = val.shape
    lists = engine.TopKLists(n_jobs, groups, n_pix, K, DEV)
    lists.val.copy_(val.view(n_jobs, n_pix, groups, K).permute(0, 2, 1, 3))
    lists.idx.copy_(idx.view(n_jobs, n_pix, groups, K).permute(0, 2, 1, 3))
    return lists


def _gather64(val, idx, job, mem_label, lab, temperature, flags):
    """float64 restatement of the gather for one job: oracle.propagate_port after its top-k, plus the zero-padded
    window positions of oracle.hr_propagate_port.  Merge the job's lists, keep the K largest values (a real key ahead of
    a zero-padded position of equal value), similarity a = v / temperature or (2 v - 1) / temperature -- formed in fp32
    as the kernels do, the rounding of a is part of the input --, soft-max or clamp(a, 0)^2 weights (a padded position
    has a = 0 and label 0), weighted sum of the label rows reached through mem_label.
    val / idx [groups, n_pix, K]; lab [n_slots, n_pix, Lp] float64.  Returns (labels [n_pix, Lp], weight sum [n_pix])."""
    dev = lab.device
    G, n_pix, K = val.shape
    _, mb, me, _ = job
    v = val.to(dev).permute(1, 0, 2).reshape(n_pix, G * K)
    i = idx.to(dev).permute(1, 0, 2).reshape(n_pix, G * K).long()
    v = torch.where(i >= 0, v, -math.inf)
    if flags & _lib.ZERO_PAD:
        r, W = (flags >> 8) & 0xff, flags >> 16
        H = n_pix // W
        q = torch.arange(n_pix, device=dev)
        qy, qx = q // W, q % W
        cy = (qy + r).clamp(max=H - 1) - (qy - r).clamp(min=0) + 1
        cx = (qx + r).clamp(max=W - 1) - (qx - r).clamp(min=0) + 1
        n_oob = (me - mb) * ((2 * r + 1) ** 2 - cy * cx)
        padv = torch.where(torch.arange(K, device=dev)[None] < n_oob[:, None], 0.0, -math.inf).float()
        v = torch.cat([v, padv], 1)
        i = torch.cat([i, torch.full((n_pix, K), PAD_ID, device=dev)], 1)
    order = torch.sort(v, dim=1, descending=True, stable=True).indices[:, :K]
    tv, ti = v.gather(1, order), i.gather(1, order)
    real, zpad = ti >= 0, (ti == PAD_ID) & torch.isfinite(tv)
    t32 = torch.tensor(temperature, dtype=torch.float32, device=dev)
    a = ((2 * tv - 1) / t32 if flags & _lib.SIM_L2 else tv / t32).double()
    a = torch.where(zpad, 0.0, torch.where(real, a, -math.inf))
    if flags & _lib.WEIGHT_COSINE:
        w = a.clamp(min=0) ** 2
    else:
        m = a.max(1, keepdim=True).values
        w = torch.exp(a - torch.where(torch.isfinite(m), m, 0.0))
        w = w / w.sum(1, keepdim=True).clamp_min(1e-300)
    w = torch.where(real, w, 0.0)
    key = ti.clamp(min=0)
    slot = torch.tensor(mem_label[mb:me], device=dev)[key // n_pix]
    return (w[..., None] * lab[slot, key % n_pix]).sum(1), w.sum(1)


# ------------------------------------------------------------------------------------- 1. gather on fixed lists
# name -> (zero padding, flags, temperature, value range of the lists)
GATHER_CASES = {
    "softmax": (False, 0, 0.07, -1.0, 1.0),
    "softmax-large": (False, 0, 0.07, 45.0, 50.0),         # a = 700: needs the max subtraction
    "cosine": (False, _lib.WEIGHT_COSINE, 0.07, -1.0, 1.0),
    "l2": (False, _lib.SIM_L2, 8.0, -1.0, 1.0),             # temperature sqrt(C), C = 64
    "zeropad-softmax": (True, 0, 0.07, -1.0, 0.5),
    "zeropad-cosine": (True, _lib.WEIGHT_COSINE, 0.07, -1.0, 0.5),
}


@pytest.mark.parametrize("case", list(GATHER_CASES))
@pytest.mark.parametrize("L", [1, 3, 5, 70])
@pytest.mark.parametrize("groups", [1, 3])
@pytest.mark.parametrize("K", [1, 4, 7, 10, 16])
def test_gather_matches_float64(K, groups, L, case):
    """fgvc_gather_labels on hand-made lists: K = 7 runs in the K = 10 kernel with fewer list entries, empty slots
    inside the lists, queries with fewer real candidates than K or none, memory slot 1 listed twice (its tied keys
    reach the same label row, so the result does not depend on which one wins), label slots permuted against the
    memory order, and on the zero-padded window (every pixel of the map is a query: corners, edges, interior) real
    winners of exactly 0 that the padded positions must not displace."""
    zp, flags, tau, lo, hi = GATHER_CASES[case]
    H, W = 9, 13
    n_pix, N = H * W, groups * K
    flags |= _lib.zero_pad_flags(2, W) if zp else 0
    g = torch.Generator().manual_seed(K * 1000 + groups * 100 + L + 7 * list(GATHER_CASES).index(case))
    table = engine.JobTable()
    table.add(7, [3, 1, 4, 1], [3, 1, 4, 1], 6)
    table.add(8, [0, 5, 2], [5, 0, 2], 7)
    val, idx = _lists(g, [4, 3], groups, n_pix, K, lo, hi)
    q = torch.arange(n_pix)
    if N > 1:
        t = q[q % 4 == 1]
        vt = torch.where(idx[0, t, 0] >= 0, val[0, t, 0], (lo + hi) / 2)
        p = torch.randint(0, n_pix, (t.numel(),), generator=g, dtype=torch.int32)
        val[0, t, 0] = val[0, t, N - 1] = vt
        idx[0, t, 0], idx[0, t, N - 1] = 1 * n_pix + p, 3 * n_pix + p
    if zp:
        z = q[q % 4 == 2]
        val[:, z, N // 2] = 0.0
        idx[:, z, N // 2] = z.int()
    val[:, [5, 50]] = -math.inf
    idx[:, [5, 50]] = -1
    lists = _pack(val, idx, groups, K)
    bank = engine.LabelBank(8, L, H, W, DEV)
    lab = torch.rand(8, n_pix, bank.Lp, generator=g, dtype=torch.float64).float()
    lab[:, :, L:] = 0
    lab[6:] = NAN
    bank.buf.copy_(lab)
    engine.gather_labels(lists, table, 0, 2, bank, tau, flags)
    got = bank.buf[6:8].double().cpu()
    lab64 = lab.double()
    for j in range(2):
        want, wsum = _gather64(lists.val[j].cpu(), lists.idx[j].cpu(), table.jobs[j], table.mem_label, lab64, tau, flags)
        err = (got[j] - want).abs().amax(1)
        # labels in [0, 1]: 2e-6 for soft-max weights; 'cosine' weights are not normalised (up to 204 at this
        # temperature), so the bound scales with their sum
        bound = 2e-6 * wsum.clamp(min=1)
        assert bool((err <= bound).all()), (j, float((err - bound).max()), int((err > bound).sum()))
        assert bool((got[j][:, L:] == 0).all())
    if not zp and not flags & _lib.WEIGHT_COSINE:
        bank.buf[:6, :, :L] = 1.0
        engine.gather_labels(lists, table, 0, 2, bank, tau, flags)
        ones = bank.buf[6:8, :, :L].double().cpu()
        for j in range(2):
            _, wsum = _gather64(lists.val[j].cpu(), lists.idx[j].cpu(), table.jobs[j], table.mem_label, lab64, tau, flags)
            has = (wsum > 0)[:, None].expand_as(ones[j])
            assert float((ones[j][has] - 1).abs().max()) <= 1e-6
            assert bool((ones[j][~has] == 0).all())


# ----------------------------------------------------------------------------------------------- 2. the chain
def _chain_grid(n_pix, Lp, max_ctas):
    """(CTAs, queries per CTA) of the gather chain: the launch rule of launch_chain_t (csrc/gather.cu)"""
    ctas = min(max_ctas, max(1, (n_pix * (Lp // 4) + 63) // 64))
    return ctas, -(-n_pix // ctas)


# name -> (zero padding, flags, temperature, value range); 'cosine' at temperature 1 with values <= 0.25 keeps the
# recurrence bounded (weights <= 1 / 16)
CHAIN_CASES = {
    "softmax": (False, 0, 0.07, -1.0, 1.0),
    "cosine": (False, _lib.WEIGHT_COSINE, 1.0, -1.0, 0.25),
    "l2": (False, _lib.SIM_L2, 8.0, -1.0, 1.0),
    "zeropad": (True, 0, 0.07, -1.0, 0.5),
}


def _run_tail(kind, lists, table, lab0, H, W, L, tau, flags, chain, out_hw):
    """one clip tail over all jobs of ``table``; ``chain`` passes the chain workspace (one persistent kernel),
    otherwise one gather launch per frame.  Returns (label bank, NCHW maps, masks or coordinates)."""
    T, n_pix, Lp = lab0.shape
    n = len(table)
    lab = lab0.clone()
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    ws, nbytes = None, 0
    if chain:
        nbytes = int(_lib.load().fgvc_chain_workspace_bytes(n, n_pix, lists.K))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    maps = torch.full((T, L, n_pix), NAN, device=DEV)
    head = (ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, ptr(jobs), ptr(jobs_host), 0, n, ptr(mem_label), H, W,
            float(tau), int(flags), ptr(lab), Lp, L, out_hw[0], out_hw[1])
    if kind == "mask":
        out = torch.zeros(T, out_hw[0], out_hw[1], dtype=torch.uint8, device=DEV)
        scratch = torch.empty(n * 2 * L, dtype=torch.float32, device=DEV)
        call("fgvc_mask_clip_tail", *head, ptr(scratch), ptr(out), ptr(maps), ptr(ws) if chain else None, nbytes,
             stream_ptr())
    else:
        out = torch.zeros(T, L, 2, dtype=torch.float32, device=DEV)
        call("fgvc_point_clip_tail", *head, 5, ptr(maps), ptr(out), ptr(ws) if chain else None, nbytes, stream_ptr())
    torch.cuda.synchronize()
    return lab, maps, out


def _run_lanes(n_lanes, lists, table, lab0, H, W, L, tau, flags, out_hw):
    """fgvc_point_clip_tail_lanes with ``n_lanes`` lanes over all jobs of ``table``, each on its own copy of the bank.
    Returns (label banks [n_lanes, T, n_pix, Lp], NCHW maps of the last lane, coordinates [n_lanes, T, L, 2])."""
    T, n_pix, Lp = lab0.shape
    n = len(table)
    lab = lab0.repeat(n_lanes, 1, 1)
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    nbytes = int(_lib.load().fgvc_chain_workspace_bytes(n, n_pix, lists.K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    maps = torch.full((T, L, n_pix), NAN, device=DEV)
    out = torch.zeros(n_lanes, T, L, 2, dtype=torch.float32, device=DEV)
    host = (_lib.Lane * n_lanes)(*[_lib.Lane(0, n, L, Lp, i * T * n_pix * Lp, i * T * L * 2) for i in range(n_lanes)])
    lanes = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(DEV)
    call("fgvc_point_clip_tail_lanes", ptr(lists.val), ptr(lists.idx), lists.K, lists.groups, None, ptr(jobs),
         ptr(jobs_host), ptr(lanes), ctypes.c_void_p(ctypes.addressof(host)), n_lanes, ptr(mem_label), H, W, float(tau),
         int(flags), ptr(lab), out_hw[0], out_hw[1], 5, ptr(maps), ptr(out), ptr(ws), nbytes, stream_ptr())
    torch.cuda.synchronize()
    return lab.view(n_lanes, T, n_pix, Lp), maps, out


def _check_chain(seed, T, H, W, L, K, groups, case):
    zp, flags, tau, lo, hi = CHAIN_CASES[case]
    flags |= _lib.zero_pad_flags(2, W) if zp else 0
    n_pix, Lp = H * W, engine.pad4(L)
    g = torch.Generator().manual_seed(seed)
    table = engine.JobTable()
    for t in range(1, T):
        mem = engine.memory_frames(t, 2)                  # frame 0 twice while t <= 2
        table.add(t, mem, mem, t)
    val, idx = _lists(g, [j[2] - j[1] for j in table.jobs], groups, n_pix, K, lo, hi, empty=0.15)
    lists = _pack(val, idx, groups, K)
    lab0 = torch.full((T, n_pix, Lp), NAN)
    lab0[0] = torch.rand(n_pix, Lp, generator=g)
    lab0[0, :, L:] = 0
    lab0 = lab0.to(DEV)
    # float64 recurrence: frame t's labels are gathered from the labels computed for its memory frames
    ref = lab0.double()
    for j, job in enumerate(table.jobs):
        ref[job[3]] = _gather64(lists.val[j], lists.idx[j], job, table.mem_label, ref, tau, flags)[0]
    for kind, out_hw in (("mask", (2 * H + 1, 3 * W)), ("point", (2 * H, 2 * W))):
        lab, maps, out = _run_tail(kind, lists, table, lab0, H, W, L, tau, flags, True, out_hw)
        lab1, maps1, out1 = _run_tail(kind, lists, table, lab0, H, W, L, tau, flags, False, out_hw)
        assert torch.equal(lab, lab1), kind
        assert torch.equal(maps[1:], maps1[1:]) and bool(maps[0].isnan().all()), kind
        assert torch.equal(out, out1), kind
        for t in range(1, T):
            scale = max(1.0, float(ref[t].abs().max()))
            err = float((lab[t].double() - ref[t]).abs().max())
            assert err <= 1e-5 * scale, (kind, t, err)
            assert torch.equal(maps[t], lab[t, :, :L].t())
        if kind == "point":
            # the lanes entry, which the trackers call: one lane, and two lanes on two copies of the bank, give what the
            # chained point tail gives
            for n_lanes in (1, 2):
                labs, maps2, outs = _run_lanes(n_lanes, lists, table, lab0, H, W, L, tau, flags, out_hw)
                assert torch.equal(maps2[1:], maps[1:]), n_lanes
                for i in range(n_lanes):
                    assert torch.equal(labs[i], lab) and torch.equal(outs[i], out), (n_lanes, i)


@pytest.mark.parametrize("case", list(CHAIN_CASES))
@pytest.mark.parametrize("K", [1, 7, 16])
@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 11, 70])
def test_gather_chain_matches_per_frame_and_float64(L, K, case):
    """Mask and point clip tails with and without the chain workspace, and the point tail's lanes entry with one and
    two lanes: label bank, NCHW maps, masks and coordinates bit-identical, every frame within 1e-5 of the float64
    recurrence (later frames read earlier out_slots, so a missing barrier or a stale read shows).  On this 13 x 17 map L <= 4 takes the multi-pass branch with a ragged last chunk
    and L >= 5 the one-pass branch; both follow from the launch rule without an occupancy figure."""
    H, W, T = 13, 17, 5
    ctas, per = _chain_grid(H * W, engine.pad4(L), _sms())
    assert ctas < _sms()              # the grid is the rule's own size, whatever the occupancy allows
    if L <= 4:
        assert per > 32 and per % 32 != 0, per
    else:
        assert per <= 32, per
    _check_chain(100 * L + K, T, H, W, L, K, 1 if K == 16 else 2, case)


@pytest.mark.parametrize("L", [1, 11])
def test_gather_chain_large_map(L):
    """More pixels than 32 x (resident CTAs): a 256-thread CTA allows at most 8 resident per SM, so every CTA of the
    chain owns more than 32 queries and runs several passes -- for L = 11 too."""
    H, W, T = 240, 200, 4
    assert H * W > 32 * 8 * _sms()
    _check_chain(7 + L, T, H, W, L, 7, 2, "softmax")


# -------------------------------------------------------------------------------------------- 3. layouts
@pytest.mark.parametrize("strided", [False, True])
@pytest.mark.parametrize("L", [1, 3, 31, 32, 33, 70, 255])
def test_put_get_nchw_roundtrip(L, strided):
    """put_nchw -> get_nchw is exact, the pad channels of the bank are exactly 0, the neighbouring slots are untouched;
    ``strided``: channels chan_stride floats apart, as the operators read a [1, C, T, H, W] stack in place."""
    H, W = 13, 17
    g = torch.Generator().manual_seed(L)
    bank = engine.LabelBank(3, L, H, W, DEV)
    bank.buf.fill_(NAN)
    if strided:
        stack = torch.rand(L, 3, H, W, generator=g).to(DEV)
        src = stack[:, 1]
        bank.put_nchw(src, 1, chan_stride=3 * H * W)
    else:
        src = torch.rand(L, H, W, generator=g).to(DEV)
        bank.put_nchw(src, 1)
    row = bank.buf[1]
    assert torch.equal(row[:, :L], src.reshape(L, H * W).t())
    assert bool((row[:, L:] == 0).all())
    assert bool(bank.buf[0].isnan().all() and bank.buf[2].isnan().all())
    assert torch.equal(bank.get_nchw(1), src)


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("npix_mod4", [0, 2])
@pytest.mark.parametrize("L", [31, 32, 33, 64, 65, 70, 255])
def test_labels_to_nchw_jobs_equals_per_slot_copy(L, npix_mod4, aligned):
    """The NCHW copies of the chained mask tail (labels_to_nchw_jobs, its wide form when L >= 32, n_pix % 4 == 0 and the
    destination is 16-byte aligned) equal the per-slot copy and the bank, bit for bit; an output 4 bytes off alignment
    takes the narrow kernel where the wide one would otherwise run."""
    H, W = (12, 17) if npix_mod4 == 0 else (13, 14)
    n_pix, T = H * W, 4
    assert n_pix % 4 == npix_mod4
    g = torch.Generator().manual_seed(L + npix_mod4)
    table = engine.JobTable()
    for t in range(1, T):
        table.add(t, [0, t - 1], [0, t - 1], t)
    lists = _pack(*_lists(g, [2] * (T - 1), 1, n_pix, 4, -1.0, 1.0), 1, 4)
    Lp = engine.pad4(L)
    lab = torch.full((T, n_pix, Lp), NAN, device=DEV)
    lab[0] = torch.rand(n_pix, Lp, generator=g).to(DEV)
    lab[0, :, L:] = 0
    jobs, _, mem_label = table.device(DEV)
    jobs_host = torch.tensor(table.jobs, dtype=torch.int32).reshape(-1, 4)
    nbytes = int(_lib.load().fgvc_chain_workspace_bytes(T - 1, n_pix, 4))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    size = T * L * n_pix
    buf = torch.full((size + 8,), NAN, device=DEV)
    off = 0 if aligned else 1
    maps = buf[off:off + size].view(T, L, n_pix)
    masks = torch.zeros(T, 2 * H, 2 * W, dtype=torch.uint8, device=DEV)
    scratch = torch.empty((T - 1) * 2 * L, dtype=torch.float32, device=DEV)
    call("fgvc_mask_clip_tail", ptr(lists.val), ptr(lists.idx), 4, 1, ptr(jobs), ptr(jobs_host), 0, T - 1, ptr(mem_label),
         H, W, 0.07, 0, ptr(lab), Lp, L, 2 * H, 2 * W, ptr(scratch), ptr(masks), ptr(maps), ptr(ws), nbytes, stream_ptr())
    torch.cuda.synchronize()
    wide = n_pix % 4 == 0 and L >= 32 and aligned
    for t in range(1, T):
        one = torch.full((L, n_pix), NAN, device=DEV)
        call("fgvc_labels_to_nchw", ptr(lab), t, Lp, L, n_pix, ptr(one), stream_ptr())
        torch.cuda.synchronize()
        assert torch.equal(maps[t], one), (t, wide)
        assert torch.equal(maps[t], lab[t, :, :L].t()), (t, wide)
    assert bool(maps[0].isnan().all())
    assert bool(buf[:off].isnan().all() and buf[off + size:].isnan().all())


# ------------------------------------------------------------------------------------------ 4. up-sampling
def _src_coord(n_out, n_in, dev):
    """(i0, i1, w1 in fp32) of F.interpolate(bilinear, align_corners=False) as the kernels compute them: in / out rounded
    to fp32, then s = max((d + 0.5) * scale - 0.5, 0) rounded once (the product and difference are exact in float64,
    like the fused multiply-add), i0 = floor(s), i1 = min(i0 + 1, in - 1), w1 = s - i0 (exact)."""
    scale = float(np.float32(n_in) / np.float32(n_out))
    d = torch.arange(n_out, dtype=torch.float64, device=dev)
    s = ((d + 0.5) * scale - 0.5).float().clamp(min=0)
    i0 = s.long().clamp(max=n_in - 1)
    return i0, (i0 + 1).clamp(max=n_in - 1), s - i0.float()


def _bilinear64(m, out_h, out_w, w0_fp32):
    """m [C, H, W] float64 -> [C, out_h, out_w]: wy0 * (wx0 * a + wx1 * b) + wy1 * (wx0 * c + wx1 * d) in float64 with
    the kernels' fp32 source coordinates; ``w0_fp32``: w0 = 1 - w1 rounded to fp32 as the kernel computes it, else exact."""
    y0, y1, wy1 = _src_coord(out_h, m.shape[1], m.device)
    x0, x1, wx1 = _src_coord(out_w, m.shape[2], m.device)
    wy0, wx0 = ((1 - wy1).double(), (1 - wx1).double()) if w0_fp32 else (1 - wy1.double(), 1 - wx1.double())
    wy1, wx1 = wy1.double()[:, None], wx1.double()
    wy0 = wy0[:, None]
    r0, r1 = m[:, y0], m[:, y1]
    return wy0 * (wx0 * r0[:, :, x0] + wx1 * r0[:, :, x1]) + wy1 * (wx0 * r1[:, :, x0] + wx1 * r1[:, :, x1])


@pytest.mark.parametrize("Lp", [4, 8, 72])
@pytest.mark.parametrize("shape", [((15, 27), (60, 108)), ((15, 27), (37, 100)), ((33, 33), (128, 128)),
                                   ((40, 40), (24, 30)), ((1, 1), (5, 7))],
                         ids=["x4", "15x27-37x100", "33-128", "down", "1x1"])
def test_upsample_labels_matches_float64(shape, Lp, record_property):
    """fgvc_upsample_labels into slot 2 of a bank: within 2 ulp of the map's max |value| of the float64 interpolation
    (the four products and three sums of the kernel, two of them fused, round at most 2 ulp of the largest value), the
    neighbouring slots keep their canary.  Whether the result is bit-identical to torch's fp32 CUDA interpolate is
    recorded, not asserted."""
    (Hs, Ws), (Hd, Wd) = shape
    g = torch.Generator().manual_seed(Hs * Wd + Lp)
    src = (torch.rand(Hs * Ws, Lp, generator=g) * 5 - 2).to(DEV)
    bank = torch.full((4, Hd * Wd, Lp), 7.25, device=DEV)
    call("fgvc_upsample_labels", ptr(src), Hs, Ws, Lp, ptr(bank), 2, Hd, Wd, stream_ptr())
    torch.cuda.synchronize()
    got = bank[2].view(Hd, Wd, Lp).permute(2, 0, 1)
    m = src.t().reshape(Lp, Hs, Ws)
    want = _bilinear64(m.double(), Hd, Wd, True)
    ulp = float(np.spacing(np.float32(float(src.abs().max()))))
    err = float((got.double() - want).abs().max())
    assert err <= 2 * ulp, (err, ulp)
    assert bool((bank[[0, 1, 3]] == 7.25).all())
    ref32 = F.interpolate(m[None], size=(Hd, Wd), mode="bilinear", align_corners=False)[0]
    same = float((ref32 == got).float().mean())
    record_property("bit_identical_to_torch_fp32", same)
    print(f"upsample {shape} Lp={Lp}: max err {err / ulp:.2f} ulp, {100 * same:.2f} % bit-identical to torch fp32")


# ------------------------------------------------------------------------------------ 5. hard propagation
@pytest.mark.parametrize("L", [2, 3, 5, 11])
def test_hard_propagation_first_maximum(L):
    """fgvc_mask_clip_tail with FGVC_HARD_PROP: after each frame its slot holds one_hot(argmax) of the soft labels with
    torch's first-maximum rule (channel 1 is a copy of channel 0 in frame 0, so the propagated frame 1 ties them exactly
    where they are largest), pad channels 0; the soft labels are the float64 gather of the hardened memory, and the
    masks decoded before hardening equal the NCHW decode of the soft labels."""
    H, W, T, K = 13, 17, 5, 4
    n_pix, Lp = H * W, engine.pad4(L)
    g = torch.Generator().manual_seed(L)
    table = engine.JobTable()
    for t in range(1, T):
        mem = engine.memory_frames(t, 2)
        table.add(t, mem, mem, t)
    lists = _pack(*_lists(g, [j[2] - j[1] for j in table.jobs], 1, n_pix, K, -1.0, 1.0, empty=0.1), 1, K)
    base = torch.rand(L, n_pix, generator=g) * 0.5
    base[0, : n_pix // 2] += 0.5
    base[1] = base[0]
    if L >= 5:
        base[3, n_pix // 2:] += 0.6
        base[4] = base[3]
    lab0 = torch.full((T, n_pix, Lp), NAN)
    lab0[0] = 0
    lab0[0, :, :L] = base.t()
    lab0 = lab0.to(DEV)
    out_hw = (3 * H, 2 * W + 5)
    lab, maps, masks = _run_tail("mask", lists, table, lab0, H, W, L, 0.07, _lib.HARD_PROP, False, out_hw)
    top2 = maps[1].topk(2, dim=0).values
    assert int((top2[0] == top2[1]).sum()) > n_pix // 4          # exact ties between channels are exercised
    for j, job in enumerate(table.jobs):
        t = job[3]
        soft = maps[t]
        hard = F.one_hot(soft.cpu().argmax(0), Lp).float().to(DEV)
        assert torch.equal(lab[t], hard), t
        want = _gather64(lists.val[j], lists.idx[j], job, table.mem_label, lab.double(), 0.07, 0)[0]
        assert float((soft.t().double() - want[:, :L]).abs().max()) <= 2e-6, t
        dec = engine.decode_masks(soft.view(L, H, W), out_hw)
        assert torch.equal(masks[t], dec), t


# ------------------------------------------------------------------------------------------- 6. mask decode
KINDS = ["signed", "small", "large", "zero", "const", "pos", "neg"]


def _decode_maps(g, L, H, W):
    """channels of every kind, in turn: signed with max > 0, small and large ranges (the normalisation decides the
    winner), all zero (not normalised), constant 1 (range 0; bilinear weights reproduce a power of two exactly),
    positive, negative (not normalised)."""
    out = torch.empty(L, H, W)
    for l in range(L):
        u = torch.rand(H, W, generator=g)
        out[l] = {"signed": u * 1.3 - 0.5, "small": u * 0.01, "large": u * 10 - 2, "zero": u * 0, "const": u * 0 + 1,
                  "pos": u, "neg": -u - 0.1}[KINDS[l % len(KINDS)]]
    return out


def _decode64(maps, out_hw):
    """float64 decode (oracle.decode_masks_port): up-sample, min / max over the whole output, normalise where max > 0,
    arg-max.  Returns (arg-max, margin best - second, channels within 1e-5 of the best)."""
    p = _bilinear64(maps.double(), out_hw[0], out_hw[1], False)
    lo, hi = p.amin(dim=(1, 2), keepdim=True), p.amax(dim=(1, 2), keepdim=True)
    p = torch.where(hi > 0, (p - lo) / (hi - lo + 1e-12), p)
    best = p.max(0).values
    margin = best - p.topk(2, dim=0).values[1] if p.shape[0] > 1 else torch.full_like(best, math.inf)
    return p.argmax(0), margin, p >= best - 1e-5


def _assert_decode(got, want, what):
    arg, margin, near = want
    clear = margin > 1e-5
    bad = int(((got.long() != arg) & clear).sum())
    assert bad == 0, (what, bad, int(clear.sum()))
    assert bool(near.gather(0, got.long()[None]).all()), what


@pytest.mark.parametrize("L", [1, 2, 4, 11, 70, 255])
@pytest.mark.parametrize("shape", [((60, 107), (480, 854)), ((16, 16), (17, 33)), ((40, 40), (24, 30)),
                                   ((1, 1), (6, 70))], ids=["bench", "16-17x33", "down", "1x1"])
def test_decode_entry_points_match_float64(shape, L, record_property):
    """fgvc_decode_masks (NCHW), fgvc_decode_masks_pixmajor (a bank slot) and the batched decode of fgvc_mask_clip_tail
    (two frames, each with its own min / max) against the float64 decode: every pixel whose best normalised channel
    leads the second by more than 1e-5 agrees, every other one picks a channel within 1e-5 of the best.  The batched
    decode (min / max from the corner outputs of each source cell, pruned arg-max) equals the pixel-major one outside
    that band; the number of pixels inside it is recorded."""
    (H, W), out_hw = shape
    n_pix = H * W
    g = torch.Generator().manual_seed(L * 31 + H)
    a, b = _decode_maps(g, L, H, W).to(DEV), _decode_maps(g, L, H, W).to(DEV)
    want = [_decode64(a, out_hw), _decode64(b, out_hw)]
    nchw = engine.decode_masks(a, out_hw)
    _assert_decode(nchw, want[0], "nchw")
    bank = engine.LabelBank(4, L, H, W, DEV)
    bank.put_nchw(a, 0)
    bank.put_nchw(b, 1)
    pm = []
    for s in (0, 1):
        out = torch.empty(out_hw, dtype=torch.uint8, device=DEV)
        scratch = torch.empty(2 * L, dtype=torch.float32, device=DEV)
        call("fgvc_decode_masks_pixmajor", ptr(bank.buf), s, bank.Lp, L, H, W, out_hw[0], out_hw[1], ptr(scratch),
             ptr(out), stream_ptr())
        _assert_decode(out, want[s], ("pixmajor", s))
        pm.append(out)
    assert torch.equal(pm[0], nchw)
    # the tail's gather copies slot 0 -> 2 and 1 -> 3 exactly (one candidate per query: weight exp(0) / exp(0) = 1)
    table = engine.JobTable()
    table.add(2, [0], [0], 2)
    table.add(3, [1], [1], 3)
    val = torch.full((2, n_pix, 1), 0.5)
    idx = torch.arange(n_pix, dtype=torch.int32).view(1, -1, 1).repeat(2, 1, 1)
    lists = _pack(val, idx, 1, 1)
    lab, _, masks = _run_tail("mask", lists, table, bank.buf, H, W, L, 1.0, 0, False, out_hw)
    assert torch.equal(lab[2], lab[0]) and torch.equal(lab[3], lab[1])
    band = 0
    for s in (0, 1):
        _assert_decode(masks[2 + s], want[s], ("batched", s))
        clear = want[s][1] > 1e-5
        assert torch.equal(masks[2 + s][clear], pm[s][clear]), s
        band += int((~clear).sum())
    record_property("pixels_in_margin_band", band)


# --------------------------------------------------------------------------------------------- 7. gaussians
@pytest.mark.parametrize("stride", [2, 4, 8])
def test_gaussian_labels_match_float64(stride):
    """put_gaussians (draw_gaussion_map_online at feature resolution) for points on and off the image, within 1e-6
    of float64; pad channels 0, neighbouring slots untouched."""
    H, W = 11, 13
    pts = torch.tensor([[0.0, 0.0], [17.3, 9.6], [-6.5, 30.25], [W * stride + 3.7, -4.1],
                        [W * stride * 0.5, H * stride + 12.0]])
    bank = engine.LabelBank(3, 5, H, W, DEV)
    bank.buf.fill_(NAN)
    bank.put_gaussians(pts, 1, stride)
    p = pts.double()
    x = (torch.arange(W, dtype=torch.float64) * stride).view(1, 1, W)
    y = (torch.arange(H, dtype=torch.float64) * stride).view(1, H, 1)
    want = torch.exp(-((x - p[:, 0, None, None]) ** 2 + (y - p[:, 1, None, None]) ** 2) / (2 * 6.0 ** 2))
    got = bank.buf[1].view(H, W, 8).cpu()
    assert float((got[..., :5].permute(2, 0, 1).double() - want).abs().max()) <= 1e-6
    assert bool((got[..., 5:] == 0).all())
    assert bool(bank.buf[0].isnan().all() and bank.buf[2].isnan().all())
