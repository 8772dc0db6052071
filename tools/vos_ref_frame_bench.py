"""Mask propagation from an annotated frame anywhere in the clip, on the config-2 clip of bench.build_inputs (64 frames,
60 x 107 x 256 features, 11 objects, precede 20, r = 12, top-k 10): ms per clip of K1, of the tail (gather chain +
decode) and of the whole MaskClipPropagator.run, and the grid barriers of the chain, at ref_frame = 0, 31 and 63.

At ref_frame = 31 it also times the two-call workaround a user needs without the feature: one frame-0 run on the
frames 31 .. 63, one on the frames 31 .. 0 (a flipped copy of the features), and the stitching of the two mask stacks
-- two K0 passes over frame 31, two K1 launches, two chains, two decodes.  It reports the share of mask pixels on which
the workaround and the one call agree, and whether they are equal bit for bit once the two calls are given the one
call's K1 tiling (a 32-job run on its own splits every memory list into 4 partial lists, the 63-job call does not;
exactly tied affinities may then be merged in another order).

Timing: CUDA events (K1 = MaskClipPropagator.k1_events; tail = end of K1 to the end of the run; run = the whole call,
K0 and the annotated frame's decode included).  Every variant is warmed up once, then the variants are alternated
``--reps`` times; the medians and the min / max are printed as one JSON object with the card name and its power limit.
The feature bank (420 MB) exceeds the 126 MB L2.

    python tools/vos_ref_frame_bench.py [--reps 20]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from fgvc_b200 import _lib, engine  # noqa: E402

REFS = (0, 31, 63)
TWO_CALL_REF = 31


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


def _ev():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def chain_steps(clip):
    """(steps, grid barriers) of the clip's gather chain: the longest lane's jobs, one barrier between two steps"""
    steps = max((b - a for a, b in clip.lanes), default=0)
    return steps, max(steps - 1, 0)


def one_call(clip, feats, onehot):
    e0 = _ev()
    clip.run(feats, onehot, events=True, want_maps=False)
    e2 = _ev()
    torch.cuda.synchronize()
    k0, k1 = clip.k1_events
    return dict(k1_ms=k0.elapsed_time(k1), tail_ms=k1.elapsed_time(e2), run_ms=e0.elapsed_time(e2)), clip.masks.clone()


def two_calls(fwd, bwd, feats, onehot, t0):
    """the workaround: a frame-0 run on feats[t0:] and one on feats[:t0+1] flipped, masks stitched"""
    e0 = _ev()
    fwd.run(feats[t0:], onehot, events=True, want_maps=False)
    rev = feats[:t0 + 1].flip(0).contiguous()
    bwd.run(rev, onehot, events=True, want_maps=False)
    masks = torch.cat([bwd.masks.flip(0)[:t0], fwd.masks])
    e1 = _ev()
    torch.cuda.synchronize()
    k1 = sum(a.elapsed_time(b) for a, b in (fwd.k1_events, bwd.k1_events))
    return dict(k1_ms=k1, run_ms=e0.elapsed_time(e1)), masks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    feats, onehot = bench.build_inputs(dev, seed=0)
    T, C, H, W = feats.shape
    L, out_hw = onehot.shape[0], bench.WORK["image_hw"]
    clips = {t0: engine.MaskClipPropagator(T, C, H, W, L, out_hw, bench.CFG, dev, ref_frame=t0) for t0 in REFS}
    t0 = TWO_CALL_REF
    fwd = engine.MaskClipPropagator(T - t0, C, H, W, L, out_hw, bench.CFG, dev)
    bwd = engine.MaskClipPropagator(t0 + 1, C, H, W, L, out_hw, bench.CFG, dev)
    variants = [f"ref_{r}" for r in REFS] + [f"two_calls_{t0}"]

    def run(v):
        if v.startswith("ref_"):
            return one_call(clips[int(v[4:])], feats, onehot)
        return two_calls(fwd, bwd, feats, onehot, t0)

    outs = {v: run(v)[1] for v in variants}                # warm-up: modules, workspaces, allocator
    times = {v: [] for v in variants}
    for _ in range(args.reps):                              # alternated
        for v in variants:
            times[v].append(run(v)[0])
    one, two = outs[f"ref_{t0}"], outs[f"two_calls_{t0}"]
    # the two calls with the one call's K1 tiling (jobs per tile, lists per job): not timed
    for c in (fwd, bwd):
        c.plan, c.groups = clips[t0].plan, clips[t0].groups
        c.lists = engine.TopKLists(len(c.table), c.groups, H * W, bench.CFG["topk"], dev)
    same_tiling = two_calls(fwd, bwd, feats, onehot, t0)[1]
    res = dict(card=card(), feat_hw=[H, W], channels=C, frames=T, objects=L, config=bench.CFG, reps=args.reps,
               k1_plans=dict(one_call=repr(clips[t0].plan), two_calls=[repr(engine.plan_k1(
                   c.bank, c.table, c.radius, bench.CFG["topk"])) for c in (fwd, bwd)]),
               two_calls_equal_one_call=bool(torch.equal(two, one)),
               two_calls_mask_agreement=float((two == one).float().mean()),
               two_calls_same_tiling_equal_one_call=bool(torch.equal(same_tiling, one)))
    for v in variants:
        res[v] = {k: round(statistics.median(t[k] for t in times[v]), 3) for k in times[v][0]}
        res[v]["run_ms_min_max"] = [round(min(t["run_ms"] for t in times[v]), 3),
                                    round(max(t["run_ms"] for t in times[v]), 3)]
        if v.startswith("ref_"):
            res[v]["tail_ms_min_max"] = [round(min(t["tail_ms"] for t in times[v]), 3),
                                         round(max(t["tail_ms"] for t in times[v]), 3)]
            res[v]["chain_steps"], res[v]["grid_barriers"] = chain_steps(clips[int(v[4:])])
        else:
            res[v]["chain_steps"] = [chain_steps(fwd)[0], chain_steps(bwd)[0]]
            res[v]["grid_barriers"] = chain_steps(fwd)[1] + chain_steps(bwd)[1]
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
