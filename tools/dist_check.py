"""Multi-GPU sanity (run under torchrun): two-phase sharded forward_test == single-GPU forward_test, and
multi_gpu_test result collection over NCCL."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, ".")
import fgvc_b200  # noqa: E402
from fgvc_b200 import apis, synthetic as S  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    cfg = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=12, with_first=True, with_first_neighbor=True)
    torch.manual_seed(0)
    trk = fgvc_b200.VanillaTracker(backbone=dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2,),
                                                 pool_type="none"), test_cfg=cfg).cuda().eval()
    T, h, w, P = 8, 64, 96, 11
    rgbs = S.synthetic_video(T, h, w, seed=3)[None]
    qp = S.query_points(P, T, h, w, seed=4, first_frame_only=False)[None]
    traj, vis = torch.zeros(1, T, P, 2), torch.zeros(1, T, P)
    with torch.no_grad():
        got = apis.sharded_forward_test(trk, rgbs, qp, traj, vis)
        want = trk(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
    err = (got[2].double() - want[2].double()).abs().max().item()
    same_order = torch.equal(got[4].cpu(), want[4].cpu())
    # one group (every point queried at frame 0), more points than ranks, longer memory: the packed K1 over frame ranges
    cfg2 = dict(cfg, precede_frames=6, with_first=False)
    trk.test_cfg = type(trk.test_cfg)(cfg2)
    T2, P2 = 14, 37
    rgbs2 = S.synthetic_video(T2, h, w, seed=5)[None]
    qp2 = S.query_points(P2, T2, h, w, seed=6, first_frame_only=True)[None]
    with torch.no_grad():
        got2 = apis.sharded_forward_test(trk, rgbs2, qp2, torch.zeros(1, T2, P2, 2), torch.zeros(1, T2, P2))
        want2 = trk(test_mode=True, rgbs=rgbs2, query_points=qp2, trajectories=torch.zeros(1, T2, P2, 2),
                    visibilities=torch.zeros(1, T2, P2))
    err = max(err, (got2[2].double() - want2[2].double()).abs().max().item())
    # host features through the two-phase split: every rank uploads only the frames its K1 jobs read
    feats = trk.get_feats(rgbs2[0].cuda())
    grp = [(0, qp2[0, :, 1:])]
    with torch.no_grad():
        a = trk.propagate_points(feats.cpu().pin_memory(), grp, (h, w), shard=(rank, world))[0]
        b = trk.propagate_points(feats, grp, (h, w))[0]
    err = max(err, (a - b).abs().max().item())
    # bidirectional tracking (points queried at several frames, tracked both ways): same split, direction-agnostic
    trk.test_cfg = type(trk.test_cfg)(dict(cfg, bidirectional=True))
    with torch.no_grad():
        got3 = apis.sharded_forward_test(trk, rgbs, qp, traj, vis)
        want3 = trk(test_mode=True, rgbs=rgbs, query_points=qp, trajectories=traj, visibilities=vis)
    err = max(err, (got3[2].double() - want3[2].double()).abs().max().item())
    trk.test_cfg = type(trk.test_cfg)(cfg)
    # the coarse-to-fine model (B200C2FTracker): TAP-Vid strided query groups tracked both ways, the same split over
    # the clip weights and the lanes chain
    torch.manual_seed(0)
    c2f = fgvc_b200.B200C2FTracker(backbone=dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3),
                                                 pool_type="none"),
                                   test_cfg=dict(cfg, radius_fine=5, neighbor_range=6, bidirectional=True)).cuda().eval()
    T4, P4 = 12, 5
    qp4 = torch.cat([torch.arange(0, T4, 4).float().repeat_interleave(P4)[:, None],
                     S.query_points(3 * P4, T4, h, w, seed=8)[:, 1:]], dim=1)[None]
    rgbs4 = S.synthetic_video(T4, h, w, seed=9)[None]
    z4 = (torch.zeros(1, T4, 3 * P4, 2), torch.zeros(1, T4, 3 * P4))
    with torch.no_grad():
        got4 = apis.sharded_forward_test(c2f, rgbs4, qp4, *z4)
        want4 = c2f(test_mode=True, rgbs=rgbs4, query_points=qp4, trajectories=z4[0], visibilities=z4[1])
    err_c2f = (got4[2].double() - want4[2].double()).abs().max().item()
    err = max(err, err_c2f)
    same_order = same_order and torch.equal(got4[4].cpu(), want4[4].cpu())
    # video-sharded driver + typed NCCL gather
    ds = [dict(rgbs=S.synthetic_video(4, 32, 48, seed=10 + i)[None], query_points=S.query_points(3, 4, 32, 48, seed=i)[None],
               trajectories=torch.zeros(1, 4, 3, 2), visibilities=torch.zeros(1, 4, 3)) for i in range(2 * world + 1)]
    loader = torch.utils.data.DataLoader(ds, batch_size=None, sampler=apis.DistributedSampler(ds, shuffle=False))
    res = apis.multi_gpu_test(trk, loader, gpu_collect=True)
    if rank == 0:
        ok = len(res) == len(ds) and all(r[2].shape == (1, 4, 3, 2) for r in res)
        ref = [trk(test_mode=True, **d)[2].cpu() for d in ds]
        ok = ok and all(torch.allclose(r[2].cpu().double(), g.double(), atol=1e-4) for r, g in zip(res, ref))
        print(f"dist_check world={world}: sharded max err {err:.2e} (B200C2FTracker {err_c2f:.2e}) "
              f"order_ok={same_order} collect_ok={ok}")
        assert err < 1e-4 and same_order and ok
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
