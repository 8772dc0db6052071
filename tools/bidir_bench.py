"""Bidirectional point tracking at the config-3 geometry: ms per clip of K1, the recurrent tail and the whole
propagate_points call, for forward-only tracking, bidirectional tracking with one gather chain per lane
(FGVC_NO_LANES=1) and bidirectional tracking with the multi-lane chain, alternated in one process.

Clip: 256 x 256 frames -> 128 x 128 x 256 features of a random-init ResNet-18 (strides 1,1,1,4), T = 50, radius 15,
precede 5, top-k 10, temperature 0.07; TAP-Vid strided queries: 256 points at every 5th frame (10 groups).
K1 = the affinity/top-k launches (engine.K1_TIMING); tail = CUDA events from the first point-tail call to the end of
the last one; total = the whole call.  Prints one JSON object with the card name and its power limit.

    python tools/bidir_bench.py [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fgvc_b200  # noqa: E402
from fgvc_b200 import _lib, engine, synthetic as S  # noqa: E402

T, HW, STEP, P = 50, 256, 5, 256
CFG = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=30, with_first=True, with_first_neighbor=True)
VARIANTS = ("forward", "bidir_no_lanes", "bidir_lanes")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


class TailEvents:
    """CUDA events around the point-tail C calls of one propagate_points call"""

    def __init__(self):
        self.first = self.last = None
        self._call = _lib.call

    def __call__(self, name, *args):
        tail = name.startswith("fgvc_point_clip_tail")
        if tail and self.first is None:
            self.first = torch.cuda.Event(enable_timing=True)
            self.first.record()
        self._call(name, *args)
        if tail:
            self.last = torch.cuda.Event(enable_timing=True)
            self.last.record()


def run(variant, feats, groups):
    os.environ.pop("FGVC_NO_LANES", None)
    if variant == "bidir_no_lanes":
        os.environ["FGVC_NO_LANES"] = "1"
    trk = fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(),
                                   test_cfg=dict(CFG, bidirectional=variant != "forward"))
    tail = TailEvents()
    _lib.call = engine.call = tail
    engine.K1_TIMING = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        e0.record()
        out = trk.propagate_points(feats, groups, (HW, HW))
        e1.record()
        torch.cuda.synchronize()
    finally:
        _lib.call = engine.call = tail._call
        k1, engine.K1_TIMING = engine.K1_TIMING, None
        os.environ.pop("FGVC_NO_LANES", None)
    return out, dict(k1_ms=sum(a.elapsed_time(b) for a, b in k1), tail_ms=tail.first.elapsed_time(tail.last),
                     total_ms=e0.elapsed_time(e1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    enc = S.davis_encoder(stride=2).to(dev)
    feats = S.encode(enc, S.synthetic_video(T, HW, HW, seed=3, device=dev), batch=5).contiguous()
    del enc
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(4)
    groups = [(t0, (torch.rand(P, 2, generator=g) * (HW - 1)).to(dev)) for t0 in range(0, T, STEP)]
    outs, times = {}, {v: [] for v in VARIANTS}
    for v in VARIANTS:                                   # warm-up: modules, workspaces, allocator
        outs[v] = run(v, feats, groups)[0]
    for _ in range(args.reps):                           # alternated
        for v in VARIANTS:
            times[v].append(run(v, feats, groups)[1])
    res = dict(card=card(), feat_hw=list(feats.shape[2:]), channels=feats.shape[1], frames=T, groups=len(groups),
               points=P * len(groups), config=CFG, reps=args.reps,
               lanes_equal_no_lanes=all(torch.equal(a, b) for a, b in zip(outs["bidir_lanes"], outs["bidir_no_lanes"])),
               forward_half_equal=all(torch.equal(a[t0:], b[t0:]) for (t0, _), a, b in
                                      zip(groups, outs["bidir_lanes"], outs["forward"])),
               peak_memory_gb=torch.cuda.max_memory_allocated() / 1e9)
    for v in VARIANTS:
        res[v] = {k: statistics.median(t[k] for t in times[v]) for k in ("k1_ms", "tail_ms", "total_ms")}
        res[v]["tail_ms_min_max"] = [min(t["tail_ms"] for t in times[v]), max(t["tail_ms"] for t in times[v])]
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
