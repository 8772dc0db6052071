"""C2FTracker.forward_test at the config-3-(ii) geometry, mixed bank formats (TF32 coarse, F16 fine) against one
forced format (split='tf32'), in one process on one GPU; with --sharded under torchrun, one clip through
apis.sharded_forward_test at N ranks against the single-rank call.

    python tools/c2f_model_bench.py [--frames 50] [--points 256] [--reps 5] [--out c2f_model_bench.json]
    torchrun --nproc_per_node 2 tools/c2f_model_bench.py --sharded

Clip: 50 frames of 256 x 256 synthetic video through the random-init eval backbone (ResNet-18, strides (1, 1, 1, 4),
pool 'none', out_indices (2, 3)): fine level layer 3, 128 x 128 x 256; coarse level layer 4, 32 x 32 x 512.  precede
5, topk 10, temperature 0.07, neighbor_range 24 (r = 12), radius_fine 12, with_first, bidirectional; encoder chunks of
batch_step 5.  Two query sets: 'strided', 256 tracks queried every 5th frame where visible (metrics.tapvid_sample: 10
groups), and 'first', 256 points queried at frame 0 (one group).  Timed, median of --reps after one warm-up, host
clock around work that ends in a device synchronise:
  forward_test  the whole call (encoder and K0 overlapped on two streams)
  encoder       the backbone over the clip's chunks alone
  k0            K0 of both levels (one launch per level and chunk) alone
  clip_weights  fgvc_c2f_clip_weights over every job of the clip (C2FPointTracker._clip_weights)
  chain         C2FPointTracker.track_banks minus clip_weights: label banks, the lanes chain, NCHW copies, K3
and how far apart the tracks of the two formats are (largest difference, share of (frame, point) entries within 0.5
and 1 px).  The GPU name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import fgvc_b200  # noqa: E402
from fgvc_b200 import _lib, apis, engine, metrics, synthetic as S  # noqa: E402

BACKBONE = dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3), pool_type="none")
CFG = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12, with_first=True,
           bidirectional=True, batch_step=5)


def timed(fn, reps):
    fn()                                           # warm-up: module loads, allocator, cuDNN algorithms
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - a) * 1e3)
    ts.sort()
    return res, round(ts[len(ts) // 2], 3)


def clip(T, P, seed=50):
    h = w = 256
    video = ((S.synthetic_video(T, h, w, seed=seed).permute(0, 2, 3, 1).clamp(-1, 1) + 1) * 127.5).to(torch.uint8)
    g = np.random.default_rng(seed)
    points = np.clip(np.cumsum(g.normal(0, 0.004, (P, T, 2)), axis=1) + g.uniform(0.1, 0.9, (P, 1, 2)), 0, 1)
    occluded = g.random((P, T)) < 0.1
    sample = metrics.tapvid_sample(dict(video=video.numpy(), points=points, occluded=occluded), (h, w),
                                   query_mode="strided")
    rgbs = sample["rgbs"].cuda()
    strided = sample["query_points"].cuda()
    xy = torch.rand(P, 2, generator=torch.Generator().manual_seed(seed)) * 236 + 10
    first = torch.cat([torch.zeros(P, 1), xy], dim=1)[None].cuda()
    return rgbs, dict(strided=strided, first=first)


def model_for(split, seed=0):
    torch.manual_seed(seed)
    cfg = dict(CFG, split=split) if split else dict(CFG)
    return fgvc_b200.C2FTracker(backbone=dict(BACKBONE), test_cfg=cfg).cuda().eval()


@torch.no_grad()
def measure(model, rgbs, qp, reps):
    T = rgbs.shape[1]
    P = qp.shape[1]
    kw = dict(rgbs=rgbs, query_points=qp, trajectories=torch.zeros(1, T, P, 2, device="cuda"),
              visibilities=torch.zeros(1, T, P, device="cuda"))
    out, t_fwd = timed(lambda: model(test_mode=True, **kw), reps)
    frames, step = rgbs[0], model.test_cfg["batch_step"]
    levels, t_enc = timed(lambda: [model.extract_feat(frames[s:s + step]) for s in range(0, T, step)], reps)
    fine, coarse = model.encode_to_bank(frames, n_levels=2)
    levels = [[lv.float().contiguous() for lv in chunk] for chunk in levels]

    def k0():
        for i, chunk in enumerate(levels):
            fine.load_frames(chunk[0], i * step)
            coarse.load_frames(chunk[1], i * step)
    _, t_k0 = timed(k0, reps)
    c2f = fgvc_b200.C2FPointTracker(model.test_cfg, model.engine_id)
    q = qp[0]
    t0s = torch.unique(q[:, 0].round().long()).tolist()
    table, _ = engine.query_job_table(t0s, T, CFG["precede_frames"], True, True, lambda mem: 0)
    K, n_c = CFG["topk"], coarse.H * coarse.W
    wts = torch.empty(len(table), n_c, K, dtype=torch.float32, device="cuda")
    rows = torch.empty(len(table), n_c, K, dtype=torch.int32, device="cuda")
    _, t_w = timed(lambda: c2f._clip_weights(coarse, fine, table, 0, len(table), K, wts, rows, torch.device("cuda")),
                   reps)
    _, t_tb = timed(lambda: c2f.track_banks(coarse, fine, q, (rgbs.shape[-2], rgbs.shape[-1])), reps)
    return out[2], dict(forward_test_ms=t_fwd, encoder_ms=t_enc, k0_ms=t_k0, clip_weights_ms=t_w,
                        chain_ms=round(t_tb - t_w, 3), track_banks_ms=t_tb, groups=len(t0s), points=P,
                        formats=f"coarse {coarse.split} / fine {fine.split}")


def gpu_line():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return gpu[torch.cuda.current_device()] if gpu else torch.cuda.get_device_name()


def sharded(a):
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    rgbs, qps = clip(a.frames, a.points)
    model = model_for(None)
    qp = qps["strided"]
    T, P = rgbs.shape[1], qp.shape[1]
    kw = dict(trajectories=torch.zeros(1, T, P, 2, device="cuda"), visibilities=torch.zeros(1, T, P, device="cuda"))
    with torch.no_grad():
        one, t1 = timed(lambda: model(test_mode=True, rgbs=rgbs, query_points=qp, **kw), a.reps)
        dist.barrier()
        got, tn = timed(lambda: apis.sharded_forward_test(model, rgbs, qp, kw["trajectories"], kw["visibilities"]),
                        a.reps)
    err = float((got[2].double() - one[2].double()).abs().max())
    if rank == 0:
        print(json.dumps(dict(world=world, single_rank_ms=t1, sharded_ms=tn, max_err=err, gpu=gpu_line())))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=50)
    ap.add_argument("--points", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sharded", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    if a.sharded:
        return sharded(a)
    rgbs, qps = clip(a.frames, a.points)
    res = dict(gpu=gpu_line())
    for name, qp in qps.items():
        preds = {}
        for split in (None, "tf32"):
            key = f"{name}_{split or 'mixed'}"
            preds[key], res[key] = measure(model_for(split), rgbs, qp, a.reps)
        d = (preds[f"{name}_mixed"] - preds[f"{name}_tf32"]).abs().amax(dim=-1).flatten()
        res[f"{name}_mixed_vs_tf32"] = dict(max_px=float(d.max()), within_0_5px=float((d <= 0.5).float().mean()),
                                            within_1px=float((d <= 1).float().mean()))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
