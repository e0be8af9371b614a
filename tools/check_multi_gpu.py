"""torchrun --nproc-per-node 2 tools/check_multi_gpu.py : tile-band sharded tracking == the unsharded solver, for the
plain loss, Replica's iteration-0 threshold search (10 floats all-reduced) and the frame-wide outlier median (radix-select
histograms all-reduced); keyframe-sharded mapping == the unsharded solver, also with bundle adjustment and re-tie
(`do_ba`, `retie_last`: every rank's means3D and ba_poses() bitwise equal to rank 0's)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from vtgaussian_slam_b200 import synthetic  # noqa: E402
from vtgaussian_slam_b200.fused import MappingSolver, TrackingSolver  # noqa: E402
from vtgaussian_slam_b200.slam_loop import quat_from_matrix  # noqa: E402

rank, world, local = bench.dist_env()
dev = torch.device("cuda", local)
torch.cuda.set_device(dev)
import datetime
dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=60))
pg = dist.group.WORLD
fr = synthetic.make_frame("replica", 400, 240, seed=0)
gt_depth = fr["depth"].copy()
gt_depth[0, 40:70, 100:200] *= 3.0
ok = True
for name, opacity, kw in (("plain", "trained", {}), ("replica_search", "fresh", dict(replica_sil_search=True)),
                          ("outlier_median", "trained", dict(ignore_outlier_depth_loss=True, w_depth=1.0))):
    p = synthetic.view_tied_gaussians(fr, n_edge=4000, opacity=opacity)
    wl = dict(frame=fr, params=p, settings=synthetic.setup_camera(fr["W"], fr["H"], fr["K"], np.eye(4)))
    settings = bench.make_settings(wl, dev)
    params = {k: torch.tensor(v, device=dev) for k, v in p.items()}
    q, t = synthetic.perturbed_pose(seed=1)
    gy = (fr["H"] + 15) // 16
    cut = [0, gy // 2 + 1, gy]
    res = []
    for sharded in (False, True):
        print(f"[rank {rank}] {name} sharded={sharded}", file=sys.stderr, flush=True)
        ts = TrackingSolver(settings, params, device=dev, use_graph=sharded, tile_rows=(cut[rank], cut[rank + 1]) if sharded else (0, 0),
                            process_group=pg if sharded else None, **kw)
        ts.set_frame(torch.tensor(fr["im"]), torch.tensor(gt_depth), q, t)
        best = ts.run_frame(8).numpy()
        res.append((best, ts.loss_terms().cpu().numpy().copy(), float(ts.r._sil[10].item()) if ts.r._sil is not None else 0.0))
    a, b = res
    good = np.allclose(a[0], b[0], rtol=2e-4, atol=1e-6) and abs(a[1][0] - b[1][0]) <= 2e-4 * abs(a[1][0]) and a[2] == b[2]
    ok &= good
    if rank == 0:
        print(name, "OK" if good else "MISMATCH", "best", a[0][:1], b[0][:1], "loss", a[1][0], b[1][0], "thr", a[2], b[2], flush=True)

# keyframe-sharded mapping
p = synthetic.view_tied_gaussians(fr, n_edge=4000, opacity="trained")
wl = dict(frame=fr, params=p, settings=synthetic.setup_camera(fr["W"], fr["H"], fr["K"], np.eye(4)))
settings = bench.make_settings(wl, dev)
poses = synthetic.trajectory(4, step_m=0.02, step_deg=1.0, seed=11)
kfs = []
for k in range(4):
    fk = synthetic.make_frame("replica", 400, 240, seed=50 + k, c2w=poses[k])
    w2c = np.linalg.inv(poses[k])
    kfs.append(dict(cam_q=torch.tensor(quat_from_matrix(w2c[:3, :3]).astype(np.float32), device=dev), cam_t=torch.tensor(w2c[:3, 3].astype(np.float32), device=dev),
                    gt_rgb=torch.tensor(fk["im"], device=dev), gt_depth=torch.tensor(fk["depth"], device=dev)))
out = []
for mode in ("single", "nccl", "fused"):
    print(f"[rank {rank}] mapping {mode}", file=sys.stderr, flush=True)
    sharded = mode != "single"
    ms = MappingSolver(settings, {k: torch.tensor(v, device=dev) for k, v in p.items()}, device=dev, process_group=pg if sharded else None,
                       sharded_step=(mode == "fused") and "auto")
    if mode == "fused" and rank == 0:
        print("fused step (vtgs_sharded_adam over peer memory):", ("ON, NVLS multicast" if ms.sharded["mc"] else "ON, peer loads / stores") if ms.sharded is not None else f"unavailable: {ms.sharded_error}", flush=True)
    mine = kfs[rank::world] if sharded else kfs
    for _ in range(5):
        loss = ms.iteration(mine)
    out.append((float(loss.item()), ms.params["rgb_colors"].cpu().numpy().copy(), ms.params["log_scales"].cpu().numpy().copy()))
good = True
for o in out[1:]:
    good &= abs(out[0][0] - o[0]) <= 1e-4 * abs(out[0][0]) and np.abs(out[0][1] - o[1]).max() <= 2e-3 and np.abs(out[0][2] - o[2]).max() <= 2e-3
ok &= good
if rank == 0:
    print("mapping", "OK" if good else "MISMATCH", [o[0] for o in out], [float(np.abs(out[0][1] - o[1]).max()) for o in out[1:]],
          "fused vs nccl:", float(np.abs(out[1][1] - out[2][1]).max()), flush=True)

# keyframe-sharded mapping with bundle adjustment: the owners step the poses, the records are exchanged and every rank
# re-ties the section's newest Gaussians (two overlapping ranges) to them.  The keyframes are dealt rank-major, so the
# (rank, slot) order of the re-ties is the single run's keyframe order.
lrs = dict(rgb_colors=0.0025, logit_opacities=0.05, log_scales=0.005, cam_unnorm_rots=1e-4, cam_trans=1e-3)
N = p["means3D"].shape[0]
per = (len(kfs) + world - 1) // world
out = []
for mode in ("single", "nccl", "fused"):
    print(f"[rank {rank}] mapping do_ba {mode}", file=sys.stderr, flush=True)
    sharded = mode != "single"
    ms = MappingSolver(settings, {k: torch.tensor(v, device=dev) for k, v in p.items()}, device=dev, lrs=lrs,
                       process_group=pg if sharded else None, sharded_step=(mode == "fused") and "auto")
    if mode == "fused" and rank == 0:
        print("do_ba fused step:", "ON" if ms.sharded is not None else f"unavailable: {ms.sharded_error}", flush=True)
    ba = [dict(kf, cam_q=kf["cam_q"].clone(), cam_t=kf["cam_t"].clone(), id=k) for k, kf in enumerate(kfs)]
    ba[1]["retie_last"], ba[3]["retie_last"] = N // 3, N // 4
    mine = ba[rank * per:(rank + 1) * per] if sharded else ba
    for _ in range(5):
        loss = ms.iteration(mine, do_ba=True)
    poses = ms.ba_poses() if sharded else {kf["id"]: (kf["cam_q"].cpu(), kf["cam_t"].cpu()) for kf in ba}
    pose_vec = torch.cat([torch.cat(poses[k]) for k in sorted(poses)]).to(dev)
    means = ms.params["means3D"]
    same = True
    if sharded:                                           # every replica bitwise equal to rank 0's
        for v in (means.reshape(-1), pose_vec):
            allv = [torch.empty_like(v) for _ in range(world)]
            dist.all_gather(allv, v.contiguous(), group=pg)
            same &= all(torch.equal(allv[0], a) for a in allv)
    out.append((float(loss.item()), ms.params["rgb_colors"].cpu().numpy().copy(), ms.params["log_scales"].cpu().numpy().copy(),
                pose_vec.cpu().numpy(), means.cpu().numpy().copy(), same, sorted(poses)))
good = True
for o in out[1:]:
    good &= o[5] and o[6] == out[0][6] and abs(out[0][0] - o[0]) <= 1e-4 * abs(out[0][0])
    good &= all(np.abs(out[0][i] - o[i]).max() <= 2e-3 for i in (1, 2, 3, 4))
ok &= good
if rank == 0:
    print("mapping do_ba + retie", "OK" if good else "MISMATCH", [o[0] for o in out], "replicas equal:", [o[5] for o in out[1:]],
          "max |d| params / poses / means3D:", [[float(np.abs(out[0][i] - o[i]).max()) for i in (1, 3, 4)] for o in out[1:]],
          flush=True)
flag = torch.tensor([1.0 if ok else 0.0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
passed = flag.item() == 1.0
if rank == 0:
    print("MULTI_GPU_CHECK", "PASS" if passed else "FAIL", flush=True)
sys.stdout.flush()
sys.stderr.flush()
# captured CUDA graphs that hold NCCL kernels are still alive here: skip the orderly teardown (it can wait forever on them)
os._exit(0 if passed else 1)
