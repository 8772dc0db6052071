"""Cost of the cycle-consistency occlusion flags (test_cfg.cycle_occlusion) at the config-3 geometry: propagate_points
with bidirectional tracking alone against tracking plus the cycle checks for frames = 1, 5 and None, alternated in one
process.  Per variant: K1 ms (engine.K1_TIMING), the shared K1 lists the checks add (one list per (query frame,
direction, memory frame); without sharing: the K1 jobs they add), the cycle calls' ms (seeding, chain, NCHW copy, K3,
decision; CUDA events from the first fgvc_point_cycle_lanes call to the end of the last), their number (chunks), the
whole call and the peak device memory of the call.  Also checks that the tracks equal the run without the key bit
for bit.  Prints one JSON object with the card name and its power limit.

Clip: 256 x 256 frames -> 128 x 128 x 256 features of a random-init ResNet-18 (strides 1,1,1,4), T = 50, radius 15,
precede 5, top-k 10, temperature 0.07, with_first, with_first_neighbor, bidirectional; TAP-Vid strided queries: 256
points at every 5th frame (10 groups), and one group of 256 points at frame 0.

    python tools/cycle_bench.py [--reps 3]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fgvc_b200  # noqa: E402
from fgvc_b200 import _lib, engine, synthetic as S  # noqa: E402
from bidir_bench import card  # noqa: E402

T, HW, STEP, P = 50, 256, 5, 256
CFG = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=30, with_first=True, with_first_neighbor=True,
           bidirectional=True)
VARIANTS = {"tracking": None, "cycle_H1": 1, "cycle_H5": 5, "cycle_Hnone": None}
DELTA = 4.0


class CycleEvents:
    def __init__(self):
        self.first = self.last = None
        self.calls = 0
        self._call = _lib.call

    def __call__(self, name, *args):
        cyc = name == "fgvc_point_cycle_lanes"
        if cyc and self.first is None:
            self.first = torch.cuda.Event(enable_timing=True)
            self.first.record()
        self._call(name, *args)
        if cyc:
            self.calls += 1
            self.last = torch.cuda.Event(enable_timing=True)
            self.last.record()


def extra_lists(groups, frames):
    """(lists of the tracking jobs, lists the checks add): shared lists with several groups, K1 jobs with one"""
    t0s = [t0 for t0, _ in groups]
    table, spans = engine.query_job_table(t0s, T, CFG["precede_frames"], True, True, lambda mem: 0)
    n_track = len(table)
    engine.cycle_job_table(table, spans, T, CFG["precede_frames"], True, True, frames, lambda mem: 0)
    if len(groups) == 1:
        return n_track, len(table) - n_track
    pairs = [set(), set()]
    for j, job in enumerate(table.jobs):
        key = engine.pair_key(table, job)
        pairs[j >= n_track].update((key, r) for r in table.mem_feat[job[1]:job[2]])
    return len(pairs[0]), len(pairs[1] - pairs[0])


def run(variant, feats, groups):
    cfg = dict(CFG)
    if variant != "tracking":
        cfg["cycle_occlusion"] = dict(frames=VARIANTS[variant], threshold=DELTA)
    trk = fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=cfg)
    ev = CycleEvents()
    _lib.call = engine.call = ev
    engine.K1_TIMING = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    try:
        e0.record()
        out = trk.propagate_points(feats, groups, (HW, HW))
        e1.record()
        torch.cuda.synchronize()
    finally:
        _lib.call = engine.call = ev._call
        k1, engine.K1_TIMING = engine.K1_TIMING, None
    tracks, vis = (out, None) if variant == "tracking" else out
    m = dict(k1_ms=sum(a.elapsed_time(b) for a, b in k1), total_ms=e0.elapsed_time(e1),
             cycle_ms=ev.first.elapsed_time(ev.last) if ev.first is not None else 0.0, cycle_calls=ev.calls,
             peak_memory_gb=torch.cuda.max_memory_allocated() / 1e9)
    if vis is not None:
        m["flagged_share"] = float(sum(float((~v).sum()) for v in vis)) / float(sum(v.numel() for v in vis))
    return tracks, m


def bench(feats, groups, reps):
    outs, times = {}, {v: [] for v in VARIANTS}
    for v in VARIANTS:                                   # warm-up: modules, allocator
        outs[v] = run(v, feats, groups)[0]
        torch.cuda.empty_cache()
    for _ in range(reps):                                # alternated
        for v in VARIANTS:
            times[v].append(run(v, feats, groups)[1])
            torch.cuda.empty_cache()
    res = dict(groups=len(groups), points=sum(int(p.shape[0]) for _, p in groups),
               tracks_equal_without_key={v: all(torch.equal(a, b) for a, b in zip(outs[v], outs["tracking"]))
                                         for v in VARIANTS})
    for v in VARIANTS:
        r = {k: statistics.median(t[k] for t in times[v]) for k in ("k1_ms", "cycle_ms", "total_ms")}
        r["cycle_ms_min_max"] = [min(t["cycle_ms"] for t in times[v]), max(t["cycle_ms"] for t in times[v])]
        r["cycle_calls"] = times[v][0]["cycle_calls"]
        r["peak_memory_gb"] = max(t["peak_memory_gb"] for t in times[v])
        if "flagged_share" in times[v][0]:
            r["flagged_share"] = times[v][0]["flagged_share"]
        if v != "tracking":
            r["track_lists"], r["extra_lists"] = extra_lists(groups, VARIANTS[v])
        res[v] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    enc = S.davis_encoder(stride=2).to(dev)
    feats = S.encode(enc, S.synthetic_video(T, HW, HW, seed=3, device=dev), batch=5).contiguous()
    del enc
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(4)
    strided = [(t0, (torch.rand(P, 2, generator=g) * (HW - 1)).to(dev)) for t0 in range(0, T, STEP)]
    res = dict(card=card(), total_memory_gb=torch.cuda.get_device_properties(dev).total_memory / 1e9,
               feat_hw=list(feats.shape[2:]), channels=feats.shape[1], frames=T, config=CFG, threshold=DELTA,
               reps=args.reps)
    res["strided_10_groups"] = bench(feats, strided, args.reps)
    res["one_group"] = bench(feats, strided[:1], args.reps)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
