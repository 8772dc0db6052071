"""Coarse-to-fine tracking of TAP-Vid strided query groups at the config-3-(ii) geometry: C2FPointTracker.track_queries
against the per-group track() loop a user would otherwise write, in one process on one GPU.

    python tools/c2f_groups_bench.py [--frames 50] [--reps 5] [--out c2f_groups_bench.json]

Clip: 50 frames, 256 x 256 image, coarse features 32 x 32 x 256 (neighbor_range 24: r = 12), fine features
128 x 128 x 256 (radius_fine 12), precede 5, topk 10, with_first; query frames 0, 5, ..., 45 (TAP-Vid 'strided'),
256 points each.  Timed (median of --reps after one warm-up, host clock around work that ends in a device
synchronise), each with the launch count of one call (fgvc_launch_count):
  loop_fw    per group track(feats[t0:]) -- forward half only
  loop_bidir the same + per group track() on the flipped prefix feats[:t0 + 1].flip(0) (the backward half)
  tq_fw      track_queries, bidirectional off
  tq_bidir   track_queries, bidirectional on
  single_*   one group of 256 points at frame 0: track() against track_queries
and whether each track_queries result equals its loop bit for bit.  The GPU name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import fgvc_b200  # noqa: E402
from fgvc_b200 import _lib  # noqa: E402


def coherent(g, T, C, H, W):
    base = torch.randn(C, H // 2 + 2, W // 2 + 2, generator=g)
    out = []
    for _ in range(T):
        base = base + 0.15 * torch.randn(base.shape, generator=g)
        f = torch.nn.functional.interpolate(base[None], size=(H, W), mode="bilinear", align_corners=False)[0]
        out.append((f + 0.05 * torch.randn(f.shape, generator=g)).relu())
    return torch.stack(out)


def loop(trk, fc, ff, qp, hw, bidirectional):
    T = fc.shape[0]
    out = torch.zeros(T, qp.shape[0], 2, dtype=torch.float32, device="cuda")
    for t0 in sorted(set(int(v) for v in qp[:, 0].tolist())):
        idx = torch.nonzero(qp[:, 0] == t0).flatten()
        pts = qp[idx, 1:]
        out[t0:, idx.cuda()] = trk.track(fc[t0:], ff[t0:], pts, hw)[0]
        if bidirectional and t0 > 0:
            out[:t0 + 1, idx.cuda()] = trk.track(fc[:t0 + 1].flip(0), ff[:t0 + 1].flip(0), pts, hw)[0].flip(0)
    return out


def timed(fn, reps):
    fn()                                           # warm-up: module loads, allocator
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    res = fn()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - n0
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - a) * 1e3)
    ts.sort()
    return res, dict(ms=round(ts[len(ts) // 2], 3), ms_min=round(ts[0], 3), ms_max=round(ts[-1], 3), launches=launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=50)
    ap.add_argument("--points", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    T, P = a.frames, a.points
    g = torch.Generator().manual_seed(50)
    fc = coherent(g, T, 256, 32, 32).cuda()
    ff = coherent(g, T, 256, 128, 128).cuda()
    t0s = list(range(0, T, 5))
    xy = torch.rand(P * len(t0s), 2, generator=g) * 236 + 10
    qp = torch.cat([torch.tensor(t0s, dtype=torch.float32).repeat_interleave(P)[:, None], xy], dim=1)
    hw = (256, 256)
    cfg = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12, with_first=True)
    fw = fgvc_b200.C2FPointTracker(dict(cfg, bidirectional=False))
    bi = fgvc_b200.C2FPointTracker(dict(cfg, bidirectional=True))
    res = {}
    out_loop_fw, res["loop_fw"] = timed(lambda: loop(fw, fc, ff, qp, hw, False), a.reps)
    out_tq_fw, res["tq_fw"] = timed(lambda: fw.track_queries(fc, ff, qp, hw), a.reps)
    out_loop_bi, res["loop_bidir"] = timed(lambda: loop(bi, fc, ff, qp, hw, True), a.reps)
    out_tq_bi, res["tq_bidir"] = timed(lambda: bi.track_queries(fc, ff, qp, hw), a.reps)
    q0 = qp[:P].clone()
    q0[:, 0] = 0
    out_s_track, res["single_track"] = timed(lambda: fw.track(fc, ff, q0[:, 1:], hw)[0], a.reps)
    out_s_tq, res["single_track_queries"] = timed(lambda: fw.track_queries(fc, ff, q0, hw), a.reps)
    res["equal"] = dict(tq_fw=bool(torch.equal(out_tq_fw, out_loop_fw)), tq_bidir=bool(torch.equal(out_tq_bi, out_loop_bi)),
                        single=bool(torch.equal(out_s_tq, out_s_track)))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res["gpu"] = gpu[torch.cuda.current_device()] if gpu else torch.cuda.get_device_name()
    res["clip"] = dict(frames=T, groups=len(t0s), points_per_group=P, coarse="32x32x256", fine="128x128x256",
                       image="256x256", precede=5, topk=10, neighbor_range=24, radius_fine=12)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
