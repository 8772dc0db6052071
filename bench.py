#!/usr/bin/env python
"""bench.py -- propagated frames/s of the label-propagation hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload = "davis2017_vos"): BASELINE config 2 -- VOS-style mask
propagation on a synthetic DAVIS-2017-shaped clip: 480x854 frames, random-init ResNet-18
stride-8 features (60x107x256, encoder untimed and out of scope), 64 frames per clip,
memory = first frame + 20 preceding frames, radius 12 (neighbor_range 24), top-k 10,
temperature 0.07, 11 objects.  One step = one clip = 63 propagated frames through
K0 (normalise/split) -> K1 (tcgen05 affinity + mask + top-k, one launch) -> 63 x
[K1b gather, NCHW, decode to a 480x854 uint8 mask].

value    : frames/s with the clip's features already resident in HBM.
e2e      : same through the public clip API with HOST (pinned) features in and HOST masks out.
roofline : K1 against the tensor pipe: algorithmic FLOPs 2*C*sum(in-mask pairs) per launch
           over the CUDA-event duration of the K1 launch; peak = measured bf16 dense / 2 (tf32)
           / 3 (3xTF32 issues three tensor MACs per fp32-faithful MAC).
N > 1    : one process per GPU (torchrun), one clip per rank per step (weak scaling, videos
           are independent: no data-path collective); the per-step masks are gathered with one
           NCCL all_gather inside the timed region; time = max over ranks.
--impl reference : the oracle port of the reference's op sequence (torch CPU, all host
           threads) on a bounded sample of the same workload: one full-memory frame per step.
--dump-outputs DIR : after the timed steps, what the last timed step returned to its caller, as DIR/<name>.npy
           (float32 / float64; see dump_outputs).  The inputs are seeded, so two builds run with the same
           arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORK = dict(workload="davis2017_vos", image_hw=(480, 854), stride=8, feat_hw=(60, 107), channels=256,
            clip_frames=64, precede_frames=20, neighbor_range=24, topk=10, temperature=0.07, objects=11)
CFG = dict(precede_frames=WORK["precede_frames"], topk=WORK["topk"], temperature=WORK["temperature"],
           neighbor_range=WORK["neighbor_range"], with_first=True, with_first_neighbor=True)


def in_mask_pairs(H, W, r, square=False):
    """sum over queries of in-mask keys = |{(q,k): dy^2+dx^2 < r^2}| (exact); square: |dy|, |dx| <= r."""
    n = 0
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if (square or dy * dy + dx * dx < r * r):
                n += max(0, H - abs(dy)) * max(0, W - abs(dx))
    return n


def algorithmic_work():
    H, W = WORK["feat_hw"]
    C, T, L = WORK["channels"], WORK["clip_frames"], WORK["objects"]
    pairs = in_mask_pairs(H, W, WORK["neighbor_range"] // 2)
    entries = sum(min(t, WORK["precede_frames"]) + 1 for t in range(1, T))     # memory entries incl. duplicate
    flops = 2.0 * C * pairs * entries
    return dict(flops_per_step=flops, in_mask_pairs=pairs, mem_entries=entries)


def dense_pairs(H, W, r, split="f16"):
    """(query, key) pairs the tensor engine actually multiplies: 128-query tiles x the key boxes (16 x BH pixels)
    of their radius halo that some query of the tile can see.  Same geometry choices as the launcher
    (csrc/topk_tc16.cu: tile orientation and BH by halo cost; corner boxes skipped)."""
    reach = r - 1
    max_bh = 4 if split == "f16" else 8

    def box_cost(rows, bh):
        return -(-rows // bh) * (16 * bh + 24)

    def pick_bh(rows):
        best = max_bh
        for bh in range(max_bh - 1, 0, -1):
            if box_cost(rows, bh) < box_cost(rows, best):
                best = bh
        return best

    def halo_cost(qh, qw):
        rows, cols = min(H, qh + 2 * reach), min(W, qw + 2 * reach)
        return (-(-H // qh)) * (-(-W // qw)) * box_cost(rows, pick_bh(rows)) * (-(-cols // 16))

    QH, QW = (16, 8) if halo_cost(16, 8) < halo_cost(8, 16) else (8, 16)
    bh = pick_bh(min(H, QH + 2 * reach))
    total = 0
    for qy0 in range(0, H, QH):
        for qx0 in range(0, W, QW):
            y_lo, y_hi = max(0, qy0 - reach), min(H - 1, qy0 + QH - 1 + reach)
            x_lo, x_hi = max(0, qx0 - reach), min(W - 1, qx0 + QW - 1 + reach)
            qy1, qx1 = min(H - 1, qy0 + QH - 1), min(W - 1, qx0 + QW - 1)
            for by in range(y_lo, y_hi + 1, bh):
                for bx in range(x_lo, x_hi + 1, 16):
                    by1, bx1 = min(H - 1, by + bh - 1), min(W - 1, bx + 15)
                    dy = max(0, by - qy1, qy0 - by1)
                    dx = max(0, bx - qx1, qx0 - bx1)
                    if dy * dy + dx * dx < r * r:
                        total += 128 * 16 * bh
    return total


def k1_profile(split):
    """numbers of one K1 launch of this workload from the committed ncu capture (profiles/k1_traffic.json): DRAM
    bytes, tensor-pipe and ALU-pipe activity; {} when there is none."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))[split]
    except (OSError, KeyError, ValueError):
        return {}


def k1_traffic(split):
    d = k1_profile(split)
    return d.get("bytes"), d.get("source")


def algorithmic_bytes():
    """SURVEY 8d: per propagated frame 4*[C*Nq + C*Nk*T_u] feature bytes (fp32-equivalent: every unique
    memory frame and the query frame read once) -- summed over the clip's 63 jobs; the top-k lists
    (8*k*Nq per job) are what K1 writes."""
    H, W = WORK["feat_hw"]
    C, T, k = WORK["channels"], WORK["clip_frames"], WORK["topk"]
    n = H * W
    total = 0
    for t in range(1, T):
        uniq = min(t, WORK["precede_frames"]) + (0 if t <= WORK["precede_frames"] else 1)
        total += 4 * (C * n + C * n * uniq) + 8 * k * n
    return total


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d.get("bf16_tflops_sustained", d.get("bf16_tflops")), bf16_burst=d.get("bf16_tflops"),
                    hbm=d.get("hbm_gbs"), src="measured")
    return dict(bf16=1400.0, bf16_burst=1590.0, hbm=6650.0, src="fallback")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))


def build_inputs(device, seed):
    from fgvc_b200 import synthetic as S
    h, w = WORK["image_hw"]
    T = WORK["clip_frames"]
    enc = S.davis_encoder(WORK["stride"], seed=0).to(device)
    frames = S.synthetic_video(T, h, w, seed=seed).to(device)
    feats = S.encode(enc, frames, batch=8).contiguous()
    assert tuple(feats.shape[1:]) == (WORK["channels"],) + WORK["feat_hw"], feats.shape
    seg = S.voronoi_mask(*WORK["feat_hw"], WORK["objects"], seed=seed)
    onehot = torch.nn.functional.one_hot(seg, WORK["objects"]).permute(2, 0, 1).float().contiguous().to(device)
    del enc, frames
    torch.cuda.empty_cache()
    return feats, onehot


DUMP_BYTES = 64 * 1000 * 1000          # all arrays of one --dump-outputs directory together


def dump_outputs(out_dir, arrays, seed=0):
    """Write each tensor of ``arrays`` (name -> tensor) as ``out_dir/<name>.npy``: float64 stays float64, every other
    dtype becomes float32.  An array larger than its even share of DUMP_BYTES is replaced by a sample of its flattened
    elements: the positions are drawn without replacement from a generator seeded with ``seed`` and kept in ascending
    order, so they are the same in every run that dumps an array of that size."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays)) - 4096           # room for the .npy header
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
        n_max = share // a.itemsize
        if a.size > n_max:
            pos = np.random.default_rng(seed).choice(a.size, n_max, replace=False)
            pos.sort()
            a = a.reshape(-1)[pos]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


CONFIG_NOTES = dict(l2="inputs (420 MB features + 840 MB feature bank per clip) exceed the 126 MB L2",
                    clips_per_step_per_gpu=1, parallelism="videos sharded (one clip per GPU per step), results gathered "
                    "to rank 0")


def _dist():
    import torch.distributed as dist
    return dist


def _max_over_ranks(ms, dev, world):
    t = torch.tensor([ms], device=dev)
    if world > 1:
        _dist().all_reduce(t, op=_dist().ReduceOp.MAX)
    return float(t.item())


def measure_h2d(dev, world, nbytes=256 << 20, reps=4):
    """Host -> device bandwidth of THIS rank while every rank copies at once (the e2e ceiling of the platform: the
    GPU boxes are VMs with one NUMA node and a shared host link, so the per-rank rate drops as ranks are added)."""
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    devb = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    devb.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        _dist().barrier()
    best = 0.0
    for _ in range(3):                         # a ceiling: the best of three rounds (the link rate varies by ~15 %)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            devb.copy_(host, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
        best = max(best, nbytes * reps / (ms / 1e3) / 1e9)
    return best


class MaskGather:
    """Per-step masks of every rank -> rank 0 (NCCL gather), on a side stream so that it overlaps the next clip's
    compute; the send buffer is double-buffered (the clip's own mask buffer is rewritten by the next step)."""

    def __init__(self, masks, rank, world, dev):
        self.rank, self.world = rank, world
        self.side = torch.cuda.Stream(device=dev)
        self.send = [torch.empty_like(masks) for _ in range(2)]
        self.recv = [[torch.empty_like(masks) for _ in range(world)] for _ in range(2)] if rank == 0 else [None, None]
        self.free = [None, None]
        self.i = 0

    def push(self, masks):
        cur = torch.cuda.current_stream()
        b = self.i & 1
        self.i += 1
        if self.free[b] is not None:
            cur.wait_event(self.free[b])
        self.send[b].copy_(masks)
        ready = torch.cuda.Event()
        ready.record(cur)
        with torch.cuda.stream(self.side):
            self.side.wait_event(ready)
            work = _dist().gather(self.send[b], self.recv[b], dst=0, async_op=True)
            work.wait()
            done = torch.cuda.Event()
            done.record(self.side)
        self.free[b] = done

    def join(self):
        torch.cuda.current_stream().wait_stream(self.side)


def run_ours(args):
    from fgvc_b200 import _lib, engine
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        _dist().init_process_group("nccl", device_id=dev)
    feats, onehot = build_inputs(dev, seed=1000 + rank)
    T = WORK["clip_frames"]
    H, W = WORK["feat_hw"]
    clip = engine.MaskClipPropagator(T, WORK["channels"], H, W, WORK["objects"], WORK["image_hw"], CFG, dev,
                                     engine_id=_lib.ENGINE_AUTO, split=args.split)
    split = clip.bank.split
    gather = MaskGather(clip.masks, rank, world, dev) if world > 1 else None

    def step(ev=False):
        clip.run(feats, onehot, events=ev, want_maps=False)
        if gather is not None:
            gather.push(clip.masks)

    def barrier():
        if world > 1:
            _dist().barrier()
        torch.cuda.synchronize()

    n_warm = args.warmup if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        step()
    if gather is not None:
        gather.join()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    k1_ev = []
    for _ in range(args.steps):
        step(ev=True)
        k1_ev.append(clip.k1_events)
    if gather is not None:
        gather.join()                   # the last gathers are inside the timed region
    e1.record()
    barrier()
    launches = _lib.launch_count() - launches0
    k1_ms = [a.elapsed_time(b) for a, b in k1_ev]
    clocks = sampler.stop() if sampler else None
    ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
    frames_per_step = (T - 1) * world
    value = frames_per_step * args.steps / (ms / 1e3)

    if args.dump_outputs and rank == 0:
        # [T, 480, 854] object id per pixel of every frame; written before the e2e steps reuse the buffer
        dump_outputs(args.dump_outputs, dict(masks=clip.masks))
    if args.profile:      # under ncu: kernels only, no e2e / CPU legs, no JSON line worth keeping
        if rank == 0:
            print(json.dumps(dict(profile_run=True, ms_per_step=ms / args.steps, k1_ms=k1_ms, plan=repr(clip.plan))))
        return
    # ---- end to end: pinned host features in, host masks out, through the public clip API
    feats_host = feats.cpu().pin_memory()
    onehot_host = onehot.cpu().pin_memory()
    masks_host = torch.empty(tuple(clip.masks.shape), dtype=torch.uint8).pin_memory()

    # a stream of clips: the staging buffers are double-buffered, so the copies of clip i + 1 run under the compute
    # of clip i and K1 stays one launch per clip (engine.MaskClipPropagator.run_host)
    whole = [(0, len(clip.table))]

    def e2e_step():
        clip.run_host(feats_host, onehot_host, masks_host, chunks=whole)

    for _ in range(2):
        e2e_step()
    clip.join_host()
    barrier()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    clip.join_host()                      # the device->host copies of every step are inside the timed region
    e1.record()
    barrier()
    e2e_ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
    e2e_value = frames_per_step * args.steps / (e2e_ms / 1e3)
    h2d = feats_host.numel() * 4 + onehot_host.numel() * 4
    d2h = masks_host.numel()
    h2d_gbs = measure_h2d(dev, world)
    del feats_host, masks_host

    plan, table = clip.plan, clip.table
    secondary = None
    if not args.no_secondary:
        del clip, gather
        torch.cuda.empty_cache()
        secondary = run_secondary(dev, rank, world, args)

    if rank == 0:
        work = algorithmic_work()
        pk = peaks()
        k1 = statistics.mean(k1_ms)
        achieved = work["flops_per_step"] / (k1 / 1e3) / 1e12
        # three tensor MACs per fp32-faithful MAC; the tf32 pipe runs at half the 16-bit rate
        div = 3.0 if split == "f16" else 6.0
        peak = pk["bf16"] / div
        prof = k1_profile(split)
        mode_id = _lib.MASK_CIRCLE
        r = WORK["neighbor_range"] // 2
        J, aligned = (plan.J, plan.aligned) if split == "f16" else (1, False)
        if split == "f16":
            dense = engine.dense_pairs(table, 0, len(table), H, W, r, mode_id, J, aligned)
        else:
            dense = dense_pairs(H, W, r, split) * work["mem_entries"]
        kname = "tc16::affinity_topk_tc16_kernel (K1, tcgen05 fp16 three-term split, one fp32 accumulator" + \
            (f", {J} jobs packed per query tile" if J > 1 else "") + (", aligned memory classes" if aligned else "") + ")" \
            if split == "f16" else "affinity_topk_tc_kernel (K1, tcgen05 3xTF32)"
        overhead = dense / (work["in_mask_pairs"] * work["mem_entries"])
        out = dict(metric="propagated frames/sec", value=value, unit="frames/s", n_gpus=world, steps=args.steps,
                   warmup=n_warm, ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak",
                   vs_baseline=None, dtype=("f16x3" if split == "f16" else "tf32x3") + " split, fp32 accumulate (fp32-faithful)",
                   data="synthetic", config=dict(WORK, **CONFIG_NOTES),
                   e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                            # what the host link allows: every rank copying at once, measured in this run
                            h2d_gbs_per_rank_all_ranks_copying=h2d_gbs,
                            ceiling_frames_per_s=frames_per_step / (h2d / (h2d_gbs * 1e9)),
                            note="bound by the host->device copy of the fp32 features (421 MB per clip); the copies of "
                                 "clip i+1 overlap the compute of clip i"),
                   gpu_launches=int(launches),
                   roofline=dict(bound="tensor", kernel=kname, achieved=achieved, peak=peak,
                                 unit="TFLOP/s", frac=achieved / peak,
                                 frac_vs_burst_peak=achieved / (pk["bf16_burst"] / div) if pk.get("bf16_burst") else None,
                                 traffic=prof.get("bytes"), traffic_source=prof.get("source"),
                                 tensor_pipe_active_pct=prof.get("tensor_pipe_active_pct"),
                                 alu_pipe_active_pct=prof.get("alu_pipe_active_pct"),
                                 algorithmic_bytes=algorithmic_bytes(),
                                 algorithmic_bytes_note="sum over the 63 jobs of a launch of each job's compulsory bytes "
                                                        "(a memory frame is counted once per job that uses it), not a "
                                                        "floor for the launch: the clip's unique data is 420 MB",
                                 k1_ms=k1, k1_share_of_step=k1 / (ms / args.steps),
                                 peak_source=f"{pk['src']} bf16 sustained {pk['bf16']} TF/s" + (" / 3 (three fp16 MMAs per MAC)" if split == "f16"
                                             else " / 2 (tf32) / 3 (3xTF32)"),
                                 flops_per_launch=work["flops_per_step"],
                                 # geometry: a query tile multiplies the union of its queries' circles, in whole key
                                 # boxes, for the union of its jobs' memory lists
                                 tile_overhead=overhead, jobs_per_tile=J, aligned=aligned,
                                 # SURVEY 8d / north_star state the roofline as dense TF32 peak / 3 (3xTF32):
                                 frac_vs_3xtf32_roofline=achieved / (pk["bf16"] / 2.0 / 3.0)),
                   clocks=clocks)
        if secondary is not None:
            out["secondary"] = secondary
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline_sample(frames=3)
        print(json.dumps(out))
    if world > 1:
        _dist().destroy_process_group()


# ----------------------------------------------------------------------------- secondary configurations
# BASELINE.json configs 3, 4, 5 through the tracker API, measured in the same run (bounded: a few seconds in all).
SECONDARY = {
    # TAP-Vid-DAVIS shape: 256x256 at stride 2 -> 128x128, 50 frames, 256 points, r = 15, precede 5; one clip per rank
    "cfg3_tapvid_davis": dict(hw=(256, 256), T=50, P=256, nr=30, precede=[5], clips=None, scaling="weak"),
    # JHMDB shape: 32 clips of 32 frames, 320x320 at stride 2 -> 160x160, 15 key-points; clips sharded over the ranks
    "cfg4_jhmdb_32clips": dict(hw=(320, 320), T=32, P=15, nr=30, precede=[5], clips=32, scaling="strong"),
    # TAP-Vid-Kinetics shape: ONE 250-frame clip, 1024 points, two-phase split over the ranks, memory-length sweep
    "cfg5_tapvid_kinetics": dict(hw=(256, 256), T=250, P=1024, nr=30, precede=[5, 10, 20, 40], clips=None,
                                 scaling="strong"),
    # local-window ("HR", correlation) tracker on the TAP-Vid-DAVIS shape: (2r + 1)^2 window, r = 12, zero-padded borders
    "hr_local_window": dict(hw=(256, 256), T=50, P=256, nr=24, precede=[5], clips=None, scaling="weak", tracker="hr"),
}


def _secondary_feats(c, dev, n_clips, seed0):
    from fgvc_b200 import synthetic as S
    h, w = c["hw"]
    enc = S.davis_encoder(2, seed=0).to(dev)
    out = []
    for i in range(n_clips):
        frames = S.synthetic_video(min(c["T"], 50), h, w, seed=seed0 + i).to(dev)
        f = S.encode(enc, frames, batch=4)
        if f.shape[0] < c["T"]:                          # long clips: tile the encoded frames
            f = f.repeat((c["T"] + f.shape[0] - 1) // f.shape[0], 1, 1, 1)[: c["T"]]
        out.append(f.contiguous())
    del enc
    torch.cuda.empty_cache()
    return out


def run_secondary(dev, rank, world, args):
    import fgvc_b200
    from fgvc_b200 import apis, engine, synthetic as S
    res = {}
    pk = peaks()
    for name, c in SECONDARY.items():
        if args.only and name.split("_")[0] not in args.only and name not in args.only:
            continue
        h, w = c["hw"]
        Hf, Wf = h // 2, w // 2
        n_distinct = 1 if c["clips"] is None else min(4, c["clips"])
        feats_list = _secondary_feats(c, dev, n_distinct, seed0=2000 + (rank if c["scaling"] == "weak" else 0))
        feats_host = [f.cpu().pin_memory() for f in feats_list]
        qp = S.query_points(c["P"], c["T"], h, w, seed=1)
        groups = [(0, qp[:, 1:].to(dev))]
        pairs = in_mask_pairs(Hf, Wf, c["nr"] // 2, square=c.get("tracker") == "hr")
        sweep = []
        for precede in c["precede"]:
            cfg = dict(precede_frames=precede, topk=10, temperature=0.07, neighbor_range=c["nr"], with_first=True,
                       with_first_neighbor=True)
            cls = fgvc_b200.HRVanillaTracker if c.get("tracker") == "hr" else fgvc_b200.VanillaTracker
            trk = cls(backbone=torch.nn.Identity(), test_cfg=cfg)
            my_clips = [0] if c["clips"] is None else list(range(rank, c["clips"], world))
            shard = (rank, world) if (c["clips"] is None and c["scaling"] == "strong" and world > 1) else None

            def one_pass(from_host):
                outs = []
                for ci in my_clips:
                    if from_host:
                        # pinned host tensor: staged in chunks by the tracker (two-phase split: a rank uploads only the
                        # frames its K1 jobs read)
                        f = feats_host[ci % n_distinct]
                    else:
                        f = feats_list[ci % n_distinct]
                    traj = trk.propagate_points(f, groups, (h, w), shard=shard)[0]
                    outs.append((ci, traj.float()))
                if c["clips"] is not None and world > 1:
                    # mmpt/apis/test.py:62-128: rank-strided shards, results interleaved back into dataset order
                    pad = -(-c["clips"] // world) - len(outs)
                    allr = apis.collect_results_gpu(outs + outs[:pad], c["clips"])
                    if rank == 0:
                        assert [i for i, _ in allr] == list(range(c["clips"])), "result order"
                if from_host:
                    return [o[1].cpu() for o in outs]         # device -> host read of the tracks
                return outs

            one_pass(False)
            torch.cuda.synchronize()
            if world > 1:
                _dist().barrier()
            engine.K1_TIMING = []
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 2
            e0.record()
            for _ in range(reps):
                one_pass(False)
            e1.record()
            torch.cuda.synchronize()
            k1_ev, engine.K1_TIMING = engine.K1_TIMING, None
            ms = _max_over_ranks(e0.elapsed_time(e1), dev, world) / reps
            k1_ms = sum(a.elapsed_time(b) for a, b in k1_ev) / reps
            k1_ms = _max_over_ranks(k1_ms, dev, world)
            one_pass(True)                                   # untimed: first-touch of the staging buffers
            torch.cuda.synchronize()
            if world > 1:
                _dist().barrier()
            e0.record()
            one_pass(True)
            e1.record()
            torch.cuda.synchronize()
            e2e_ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
            n_clips_total = world if c["clips"] is None and c["scaling"] == "weak" else (c["clips"] or 1)
            frames = (c["T"] - 1) * n_clips_total
            entries = sum(min(t, precede) + 1 for t in range(1, c["T"]))
            # K1 flops executed by THIS rank's launches (max over ranks of the time): its share of the jobs
            clips_here = len(my_clips) if c["clips"] is not None else 1
            share = (1.0 / world) if shard is not None else 1.0
            flops = 2.0 * 256 * pairs * entries * clips_here * share
            ach = flops / (k1_ms / 1e3) / 1e12 if k1_ms > 0 else None
            sweep.append(dict(precede_frames=precede, frames_per_s=frames / (ms / 1e3), ms_per_pass=ms,
                              e2e_frames_per_s=frames / (e2e_ms / 1e3), k1_ms=k1_ms,
                              k1_tflops_algorithmic=ach, k1_roofline_frac=(ach / (pk["bf16"] / 3.0)) if ach else None))
            del trk
            torch.cuda.empty_cache()
        res[name] = dict(feat_hw=(Hf, Wf), frames=c["T"], points=c["P"], neighbor_range=c["nr"], clips=c["clips"] or
                         ("1 per rank" if c["scaling"] == "weak" else 1), scaling=c["scaling"],
                         parallelism=("two-phase split of one video: K1 sharded over frame ranges, lists all-gathered, "
                                      "tail sharded over points" if c["clips"] is None and c["scaling"] == "strong"
                                      else "clips sharded rank-strided, results gathered in dataset order"),
                         e2e_note="host features in (pinned, copied inside the timed pass in frame chunks that overlap K0 / K1 of the frames already on the device), host tracks out",
                         results=sweep if len(sweep) > 1 else sweep[0])
        del feats_list, feats_host
        torch.cuda.empty_cache()
    if not args.only or "cfg3ii" in args.only:
        res["cfg3ii_c2f_tapvid_davis"] = run_c2f_clip(dev, rank, world)
    order = ["cfg3_tapvid_davis", "cfg3ii_c2f_tapvid_davis"]
    return {k: res[k] for k in order + [k for k in res if k not in order] if k in res}


def run_c2f_clip(dev, rank, world):
    """BASELINE config 3-(ii): coarse-to-fine tracking of one 50-frame 256 x 256 clip per rank, 256 points, coarse
    stride 8 (32 x 32, r = 12) + fine stride 2 (128 x 128, radius_fine 12), through fgvc_b200.C2FPointTracker."""
    import fgvc_b200
    from fgvc_b200 import synthetic as S
    T, P, h, w = 50, 256, 256, 256
    frames = S.synthetic_video(T, h, w, seed=3000 + rank).to(dev)
    fc = S.encode(S.davis_encoder(8, seed=0).to(dev), frames, batch=8).contiguous()
    ff = S.encode(S.davis_encoder(2, seed=0).to(dev), frames, batch=4).contiguous()
    del frames
    torch.cuda.empty_cache()
    pts = S.query_points(P, T, h, w, seed=2)[:, 1:]
    cfg = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12, with_first=True)
    trk = fgvc_b200.C2FPointTracker(cfg)
    trk.track(fc, ff, pts, (h, w))
    torch.cuda.synchronize()
    if world > 1:
        _dist().barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    reps = 2
    for _ in range(reps):
        trk.track(fc, ff, pts, (h, w))
    e1.record()
    torch.cuda.synchronize()
    ms = _max_over_ranks(e0.elapsed_time(e1), dev, world) / reps
    fc_h, ff_h = fc.cpu().pin_memory(), ff.cpu().pin_memory()
    trk.track(fc_h, ff_h, pts, (h, w))                 # untimed: first touch of the staging path
    torch.cuda.synchronize()
    e0.record()
    traj_h = trk.track(fc_h, ff_h, pts, (h, w))[0].cpu()   # pinned host features: staged in chunks by the tracker
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
    return dict(coarse_hw=tuple(fc.shape[2:]), fine_hw=tuple(ff.shape[2:]), frames=T, points=P, radius_fine=12,
                clips="1 per rank", scaling="weak", frames_per_s=(T - 1) * world / (ms / 1e3), ms_per_clip=ms,
                e2e_frames_per_s=(T - 1) * world / (e2e_ms / 1e3),
                ms_per_frame=ms / (T - 1), tracks_shape=list(traj_h.shape),
                note="recurrent driver around masked_attention_efficient_c2f (fgvc_b200/c2f_tracker.py); both "
                     "feature banks and the fine label bank stay resident across frames")


# ------------------------------------------------------------------- CPU baseline / reference
def _cpu_inputs(T):
    """features + soft labels of the first T frames of the bench clip (CPU)."""
    from fgvc_b200 import synthetic as S
    h, w = WORK["image_hw"]
    torch.manual_seed(0)
    enc = S.davis_encoder(WORK["stride"], seed=0)
    frames = S.synthetic_video(T, h, w, seed=1000)
    feats = S.encode(enc, frames, batch=4)
    g = torch.Generator().manual_seed(1)
    labels = torch.rand(T, WORK["objects"], *WORK["feat_hw"], generator=g)
    labels = labels / labels.sum(1, keepdim=True)
    return feats, labels


def _cpu_frame(O, feats, labels, mask, t):
    mem = O.memory_frames(t, WORK["precede_frames"])
    k = feats[mem].permute(1, 0, 2, 3)[None]
    v = labels[mem].permute(1, 0, 2, 3)[None]
    return O.propagate_port(feats[t][None], k, v, mask=mask, temperature=WORK["temperature"], topk=WORK["topk"],
                            step=512)


def _sample_frames(n):
    """n query frames spread evenly over the clip's 63 propagated frames, so that the sample's memory lengths are
    in the clip's proportion (frames 1..20 have t + 1 entries, the rest 21; mean 18.0)."""
    T = WORK["clip_frames"]
    return [1 + int((i + 0.5) * (T - 1) / n) for i in range(n)]


def _cpu_sample(n_frames, warmup=1):
    """Reference CPU path (oracle port of the reference's op sequence, all host threads) on n_frames query frames of
    the bench clip.  The neighbourhood mask is built once per video by the reference (affinity_utils.py:75-112): its
    build time is measured and charged at 1/63 per propagated frame.  Returns (frames/s, ms per frame, cores,
    description, propagated labels of the last frame)."""
    from oracle import oracle as O        # the CPU legs of bench.py are the one place it runs the oracle
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    ts = _sample_frames(n_frames)
    feats, labels = _cpu_inputs(max(ts) + 1)
    s = time.perf_counter()
    mask = O.neighbor_mask(*WORK["feat_hw"], WORK["neighbor_range"])
    t_mask = time.perf_counter() - s
    for i in range(warmup):
        _cpu_frame(O, feats, labels, mask, ts[i % len(ts)])
    s = time.perf_counter()
    for t in ts:
        out = _cpu_frame(O, feats, labels, mask, t)
    dt = time.perf_counter() - s + t_mask * len(ts) / (WORK["clip_frames"] - 1)
    entries = [min(t, WORK["precede_frames"]) + 1 for t in ts]
    desc = (f"{len(ts)} propagated frames of the same clip (query frames {ts}, memory entries {entries}: the clip's "
            f"mean is 18.0), oracle port of the reference op sequence (genuine functions are not on the GPU box), "
            f"torch CPU fp32, {cores} threads; the per-video mask build ({t_mask:.2f} s) is charged at 1/63 per frame")
    return len(ts) / dt, dt / len(ts) * 1e3, cores, desc, out


def cpu_baseline_sample(frames=3):
    value, _, cores, desc, _ = _cpu_sample(frames)
    return dict(value=value, unit="frames/s", cores=cores, kind="port", sample=desc)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, ms, cores, desc, labels = _cpu_sample(args.steps, warmup=max(1, args.warmup))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(labels=labels))       # [1, L, 60, 107] propagated soft labels
    print(json.dumps(dict(impl="reference", metric="propagated frames/sec", value=value, unit="frames/s",
                          n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=args.steps, warmup=max(1, args.warmup),
                          ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None,
                          dtype="f32", data="synthetic", config=dict(WORK, **CONFIG_NOTES),
                          cpu_baseline=dict(value=value, unit="frames/s", cores=cores, kind="port", sample=desc),
                          e2e=dict(value=value, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline sample")
    ap.add_argument("--split", default=None, choices=["f16", "tf32"],
                    help="feature-bank split / tensor engine (default: f16 three-term; tf32 = 3xTF32)")
    ap.add_argument("--profile", action="store_true", help="kernels only (for ncu): no e2e, no CPU baseline")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary block (BASELINE configs 3, 4, 5)")
    ap.add_argument("--only", nargs="*", default=None, help="secondary configs to run (cfg3 cfg4 cfg5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 3
        return run_reference(args)
    if args.steps is None:
        args.steps = 20
    run_ours(args)


if __name__ == "__main__":
    main()
