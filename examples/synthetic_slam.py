"""Run the compact view-tied SLAM loop on a sequence and print timing + trajectory error as one JSON line.

Synthetic (BASELINE config 4: TUM fr1_desk-shaped 640x480 tracking + mapping over synthetic frames):
    python examples/synthetic_slam.py --shape tum_fr1 --frames 600 --track-iters 200 --map-iters 30 --baseframe-every 30
Add `--align-sections 2` to bundle-adjust every base frame against the two sections it was tracked against (with
`--track-sections 2`; one otherwise): the JSON line then lists each base frame's correction.  At the default
`--align-lr-*` (the tracking rates) this currently raises the ATE (see slam_loop.LoopConfig.align_sections).
On-disk sequences in the reference's layouts (camera parameters from the reference's configs/data/*.yaml):
    python examples/synthetic_slam.py --source replica --basedir data/Replica --sequence room0 --camera-yaml configs/data/replica.yaml
    python examples/synthetic_slam.py --source tum --basedir data/TUM_RGBD --sequence rgbd_dataset_freiburg1_desk \
        --camera-yaml configs/data/TUM/freiburg1_desk.yaml
Frames are decoded ahead of the loop on a worker thread and staged through pinned memory (frames.FrameSource.prefetch).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", default="synthetic", choices=["synthetic", "replica", "tum", "scannetpp"])
    ap.add_argument("--basedir", default=None)
    ap.add_argument("--sequence", default=None)
    ap.add_argument("--camera-yaml", default=None, help="yaml with a camera_params block (reference configs/data/*.yaml)")
    ap.add_argument("--shape", default="tum_fr1")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--frames", type=int, default=60)
    ap.add_argument("--track-iters", type=int, default=40)
    ap.add_argument("--map-iters", type=int, default=15)
    ap.add_argument("--baseframe-every", type=int, default=10)
    ap.add_argument("--map-every", type=int, default=5)
    ap.add_argument("--step-m", type=float, default=0.01)
    ap.add_argument("--step-deg", type=float, default=0.3)
    ap.add_argument("--track-sections", type=int, default=1, help="track against the newest k sections")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--align-sections", type=int, default=0,
                    help="bundle-adjust each base frame against the last N sections it was tracked against (0: off)")
    # the tracking rates: the reference's own mapping pose LRs (1e-8 / 1e-7) leave the pose where it is
    ap.add_argument("--align-lr-rot", type=float, default=4e-4, help="mapping LR of cam_unnorm_rots with --align-sections")
    ap.add_argument("--align-lr-trans", type=float, default=2e-3, help="mapping LR of cam_trans with --align-sections")
    a = ap.parse_args()

    import torch
    from vtgaussian_slam_b200 import synthetic
    from vtgaussian_slam_b200.metrics import ate_after_alignment
    from vtgaussian_slam_b200.slam_loop import LoopConfig, ViewTiedSLAM, ate_rmse

    from vtgaussian_slam_b200 import frames
    if a.source == "synthetic":
        src = frames.SyntheticSource(a.shape, a.frames, a.width, a.height, a.step_m, a.step_deg)
    elif a.source == "scannetpp":
        src = frames.ScannetPPSource(a.basedir, a.sequence, desired_height=a.height or 584, desired_width=a.width or 876,
                                     end=a.frames if a.frames > 0 else -1)         # tracking resolution of configs/scannetpp/*.py
    else:
        import yaml
        with open(a.camera_yaml) as f:
            cam = yaml.safe_load(f)["camera_params"]
        cls = frames.ReplicaSource if a.source == "replica" else frames.TumSource
        src = cls(cam, a.basedir, a.sequence, desired_height=a.height, desired_width=a.width, end=a.frames if a.frames > 0 else -1)
    n = len(src)
    W, H, K = src.W, src.H, src.K.astype(np.float64)
    poses = src.c2w.numpy().astype(np.float64)
    cfg = LoopConfig(track_iters=a.track_iters, map_iters=a.map_iters, baseframe_every=a.baseframe_every,
                     map_every=a.map_every, use_graph=not a.no_graph, track_sections=a.track_sections,
                     align_sections=a.align_sections)
    if a.align_sections > 0:
        cfg.map_lrs = dict(cfg.map_lrs, cam_unnorm_rots=a.align_lr_rot, cam_trans=a.align_lr_trans)
    slam = ViewTiedSLAM(W, H, K, cfg)
    t0 = time.perf_counter()
    gen = 0.0                                                       # decoding runs on the prefetch thread
    for fr in src.prefetch("cuda:0", ahead=2):
        slam.process(fr)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    est = np.stack([np.linalg.inv(m) for m in slam.w2c])
    still = np.tile(np.eye(4), (n, 1, 1))
    st = slam.stats
    print(json.dumps(dict(
        source=a.source, shape=a.shape if a.source == "synthetic" else a.sequence, W=W, H=H, frames=n, sections=len(slam.sections),
        gaussians_per_section=int(slam.sections[-1]["params"]["means3D"].shape[0]),
        ate_rmse_m=ate_rmse(est, poses), ate_rmse_if_not_tracking_m=ate_rmse(still, poses),
        ate_mean_after_alignment_m=ate_after_alignment(list(poses), list(est)),        # the reference's evaluate_ate
        track_iters=st["track_iters"], track_iters_per_s=st["track_iters"] / max(st["track_s"], 1e-9),
        map_keyframe_iters=st["map_iters"], map_keyframe_iters_per_s=st["map_iters"] / max(st["map_s"], 1e-9),
        align_sections=a.align_sections, align_share_of_map_s=st["align_s"] / max(st["map_s"], 1e-9),
        align_corrections=[dict(frame=i, frozen=f, shift_m=dt, angle_deg=da) for i, f, dt, da in st["align"]],
        frames_per_s=n / wall, wall_s=wall)))


if __name__ == "__main__":
    main()
