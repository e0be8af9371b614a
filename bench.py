#!/usr/bin/env python
"""bench.py -- fwd+bwd render iterations/s of the VTGaussian-SLAM hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched with torchrun)
    python bench.py --impl reference --steps K --warmup W    (CPU oracle port on the host cores)
    python bench.py --steps K --warmup W --dump-outputs DIR  (also writes the last timed step's outputs to DIR/*.npy)

A "step" is one tracking iteration of BASELINE.json configs[1] (Replica room0-shaped 1200x680,
~1.0 M view-tied Gaussians): fused six-plane render -> masked-L1 tracking loss -> backward to
the 7 pose numbers -> Adam (reference src/vtgaussian_slam.py:1794-1891).  At N>1 the image is
sharded by tile bands with one 16-float all-reduce per iteration ("strong" scaling).

Prints ONE JSON line (rank 0):
  value          iterations/s with everything resident in HBM (CUDA graph replay, CUDA-event timed, max over ranks)
  e2e            the same iteration through the reference-facing API (slam_ops.get_loss + backward + torch Adam) with
                 the frame copied H2D from pinned memory and the loss read back D2H every step
  roofline       the dominant kernel: algorithmic GB/s against the measured HBM peak, its issue-slot and FP32 view
                 (instruction / DRAM counters from this round's ncu capture, profiles/r02_counters.json; FP32 peak
                 measured here with an FFMA probe), and the iteration's T_min of SURVEY.md section 8(d)
  cpu_baseline   the oracle port on the host cores, plus parity_check: the GPU iteration against that CPU iteration
  mapping        BASELINE configs[2]: 8 keyframes per mapping iteration, keyframe-sharded over the ranks
  configs        short legs of configs[0] (c1), configs[3] (c4) and configs[4] (c5)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fwd+bwd render iters/s, Replica 1200x680 view-tied Gaussians"
UNIT = "iters/s"
LOSS_W = dict(im=0.5, depth=0.025)          # configs/replica/room0.py:74-77
SIL_THRES = 0.99
FP32_NOMINAL_TFLOPS = 74.4                  # 148 SM x 128 lanes x 2 x 1.965 GHz (BASELINE.md)
ITERATION = "fused 6-plane render + masked-L1 tracking loss + backward to pose + Adam"


def build_workload(kind="c2", seed=0):
    """c2 (configs[1]): one Replica-shaped frame, one Gaussian per pixel (816 000) + 200 000 edge-densified Gaussians of
    the 2x grid, a mapped ('trained') section, pose perturbed by ~1 cm / 0.5 deg.  c1 (configs[0]): the same frame with
    ~300 k Gaussians.  c5 (configs[4]): a ScanNet++-sized view of four overlapping view-tied sections (~8 M Gaussians).
    small: 300x170 debug workload."""
    from vtgaussian_slam_b200 import synthetic
    if kind == "c5":
        from vtgaussian_slam_b200.slam_loop import quat_from_matrix
        frames, poses, p = synthetic.multi_section_scene("scannetpp", sections=4, spacing_m=0.3, seed=seed)
        fr = frames[-1]
        w2c = np.linalg.inv(poses[-1])
        q = quat_from_matrix(w2c[:3, :3]).astype(np.float32)
        t = (w2c[:3, 3] + np.random.default_rng(1).normal(0, 0.01, 3)).astype(np.float32)
        s = synthetic.setup_camera(fr["W"], fr["H"], fr["K"], np.eye(4))
        name = "tracking_scannetpp_%dx%d_N%d_4sections" % (fr["W"], fr["H"], p["means3D"].shape[0])
        return dict(frame=fr, params=p, q=q, t=t, settings=s, name=name)
    if kind == "small":
        fr = synthetic.make_frame("replica", 300, 170, seed=seed)
        p = synthetic.view_tied_gaussians(fr, n_edge=12000, opacity="trained")
    elif kind == "c1":
        fr = synthetic.make_frame("replica", seed=seed)
        p = synthetic.view_tied_gaussians(fr, n_target=300000, opacity="trained")
    else:
        fr = synthetic.make_frame("replica", seed=seed)
        p = synthetic.view_tied_gaussians(fr, n_edge=200000, opacity="trained")
    q, t = synthetic.perturbed_pose(seed=1, trans_sigma=0.01, rot_deg=0.5)
    s = synthetic.setup_camera(fr["W"], fr["H"], fr["K"], np.eye(4))
    name = "tracking_replica_%dx%d_N%d" % (fr["W"], fr["H"], p["means3D"].shape[0])
    return dict(frame=fr, params=p, q=q, t=t, settings=s, name=name)


def config_of(wl, gpus):
    """The `config` both arms print (identical by construction)."""
    fr = wl["frame"]
    return {"workload": wl["name"], "gaussians": int(wl["params"]["means3D"].shape[0]), "resolution": "%dx%d" % (fr["W"], fr["H"]),
            "iteration": ITERATION, "gpus": int(gpus),
            "parallelism": f"tile-band x{gpus} + 16-float all-reduce" if gpus > 1 else "single GPU",
            "l2": "per-iteration working set (~250 MB) exceeds the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_threads():
    """Every core this process may use, whatever OMP_NUM_THREADS the launcher exported (torchrun sets it to 1)."""
    import oracle                                         # the checker; timed here only as the CPU baseline
    return oracle.set_threads(len(os.sched_getaffinity(0)))


def cpu_iteration(wl, tile_rows=(0, 0), want_grads=False):
    """One tracking iteration of the oracle port: front end + six-plane forward + tracking loss +
    backward (all host cores through OpenMP).  Returns (seconds, loss, forward outputs[, rasteriser-input gradients])."""
    import oracle                                         # the checker; timed here only as the CPU baseline
    fr, p, s = wl["frame"], wl["params"], wl["settings"]
    cam = oracle.make_camera(fr["W"], fr["H"], s["tanfovx"], s["tanfovy"], s["viewmatrix"], s["projmatrix"], tile_rows=tile_rows)
    t0 = time.perf_counter()
    m, sc, rot, op, c6 = oracle.frontend(p["means3D"], p["rgb_colors"], p["unnorm_rotations"], p["logit_opacities"],
                                         p["log_scales"], wl["q"], wl["t"])
    orc = oracle.Oracle()
    out = orc.forward(cam, m, sc, rot, op, c6)
    img = out["color"]
    gd = fr["depth"][0]
    mask = (gd > 0) & (img[4] > SIL_THRES) & ~np.isnan(img[3]) & ~np.isnan(img[5] - img[3] ** 2)
    if tile_rows[1] > tile_rows[0]:
        band = np.zeros_like(mask)
        band[tile_rows[0] * 16:tile_rows[1] * 16] = True
        mask &= band
    dL = np.zeros((6,) + gd.shape, np.float32)
    e_im = img[:3] - fr["im"]
    e_d = img[3] - gd
    dL[:3] = LOSS_W["im"] * np.sign(e_im) * mask
    dL[3] = LOSS_W["depth"] * np.sign(e_d) * mask
    loss = LOSS_W["im"] * np.abs(e_im)[:, mask].astype(np.float64).sum() + LOSS_W["depth"] * np.abs(e_d)[mask].astype(np.float64).sum()
    g = orc.backward(dL)
    dt = time.perf_counter() - t0
    return (dt, float(loss), out, g) if want_grads else (dt, float(loss), out)


def cpu_pose_gradient(wl, g):
    """dL/d(cam_unnorm_rot)[4], dL/d(cam_trans)[3] from the oracle's rasteriser-input gradients through the reference's
    own chain (get_depth_and_silhouette, transform_to_frame: the host mirrors of slam_ops, fp64, CPU)."""
    import torch
    from vtgaussian_slam_b200 import slam_ops
    p = wl["params"]
    P = {k: torch.tensor(v, dtype=torch.float64) for k, v in p.items()}
    P["cam_unnorm_rots"] = torch.tensor(wl["q"], dtype=torch.float64).reshape(1, 4, 1).requires_grad_(True)
    P["cam_trans"] = torch.tensor(wl["t"], dtype=torch.float64).reshape(1, 3, 1).requires_grad_(True)
    tg = slam_ops.transform_to_frame(P, 0, gaussians_grad=False, camera_grad=True)
    dsc = slam_ops.get_depth_and_silhouette(tg["means3D"], torch.eye(4, dtype=torch.float64))
    torch.autograd.backward([tg["means3D"], dsc], [torch.tensor(g["means3D"], dtype=torch.float64),
                                                   torch.tensor(g["colors"][:, 3:], dtype=torch.float64)])
    return P["cam_unnorm_rots"].grad.numpy().reshape(4), P["cam_trans"].grad.numpy().reshape(3)


def run_reference_arm(args, wl):
    cores = cpu_threads()
    gy = (wl["frame"]["H"] + 15) // 16
    # bounded sample: a centred band of tile rows sized so that W+K steps finish within a few minutes
    t_full, _, _ = cpu_iteration(wl)
    budget = 150.0
    frac = min(1.0, budget / max(t_full * (args.steps + args.warmup), 1e-9))
    rows = max(1, int(round(gy * frac)))
    r0 = (gy - rows) // 2
    band = (0, 0) if rows >= gy else (r0, r0 + rows)
    for _ in range(args.warmup):
        cpu_iteration(wl, band)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_iteration(wl, band)
    dt = (time.perf_counter() - t0) / args.steps
    work_frac = rows / gy
    value = work_frac / dt            # iterations/s, extrapolated by tile rows when a band was sampled
    sample = ("full iteration" if rows >= gy else f"{rows} of {gy} tile rows per step (value extrapolated by rows)") + \
             f"; first full iteration took {t_full:.2f} s on {cores} OpenMP threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3 / work_frac, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": config_of(wl, args.gpus),
        "what": "CPU oracle port of the splatting path on the host cores (the reference's rasteriser is an absent pip dependency)",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def balanced_bands(row_work, world, row_peak=None):
    """Contiguous tile-row bands of near-equal work: row_work[r] = cost proxy of tile row r (sum of n_contrib).
    Deterministic, covers [0, rows) exactly, every band non-empty (rows >= world)."""
    w = np.asarray(row_work, dtype=np.float64) + 1e-9
    rows = len(w)
    cum = np.concatenate([[0.0], np.cumsum(w)])
    cuts = [0]
    for k in range(1, world):
        target = cum[-1] * k / world
        c = int(np.searchsorted(cum, target))
        c = min(max(c, cuts[-1] + 1), rows - (world - k))
        cuts.append(c)
    cuts.append(rows)
    return [(cuts[k], cuts[k + 1]) for k in range(world)]


def make_settings(wl, dev):
    import torch
    from vtgaussian_slam_b200.rasterizer import GaussianRasterizationSettings
    fr, s = wl["frame"], wl["settings"]
    return GaussianRasterizationSettings(
        image_height=fr["H"], image_width=fr["W"], tanfovx=s["tanfovx"], tanfovy=s["tanfovy"], bg=torch.tensor(s["bg"], device=dev),
        scale_modifier=1.0, viewmatrix=torch.tensor(s["viewmatrix"], device=dev), projmatrix=torch.tensor(s["projmatrix"], device=dev),
        sh_degree=0, campos=torch.tensor(s["campos"], device=dev), prefiltered=False)


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def measure_fp32_peak(dev):
    """FP32 FMA throughput of this GPU in TFLOP/s (vtgs_ffma_probe: 8 independent FFMA chains per thread, 64 warps / SM)."""
    import torch
    from vtgaussian_slam_b200 import _lib
    L = _lib.lib()
    sink = torch.zeros(1, device=dev)
    n = ctypes.c_uint64(0)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.vtgs_ffma_probe(2000, ctypes.c_void_p(sink.data_ptr()), ctypes.byref(n), st))
    best = 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 100000
    for _ in range(3):
        e0.record()
        _lib.check(L.vtgs_ffma_probe(iters, ctypes.c_void_p(sink.data_ptr()), ctypes.byref(n), st))
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, 2.0 * 8 * iters * n.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def load_counters(name):
    """Per-launch instruction / DRAM counters of this round's ncu capture (profiles/r02_counters.json, written by
    tools/ncu_counters.py from the committed --set full capture of the SAME workload): {kernel: {warp_inst, dram_bytes}}."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_counters.json")))
        return d["kernels"] if d.get("workload") == name else {}
    except Exception:
        return {}


DUMP_BYTES = 64 << 20


def dump_outputs(path, solver, N):
    """Writes what the timed path's last step handed its caller as float32 <name>.npy files: the pose after the step's
    Adam update, the step's pose gradient and loss terms, the best (loss, pose) so far, and the step's six-plane render
    and radii.  Arrays of more than 4096 elements are replaced by a fixed seeded sample of their flattened elements
    (sorted indices) when the whole would exceed DUMP_BYTES, so two builds can be compared output for output."""
    outs = {"cam_unnorm_rot": solver.cam_q, "cam_trans": solver.cam_t, "pose_grad": solver.msg[0:7],
            "loss_terms": solver.loss_terms(), "best": solver.best, "image6": solver.r.image6, "radii": solver.r.radii[:N]}
    arrs = {k: t.detach().cpu().numpy().astype(np.float32) for k, t in outs.items()}
    big = sorted(k for k, a in arrs.items() if a.size > 4096)
    room = DUMP_BYTES - sum(a.nbytes for k, a in arrs.items() if k not in big)
    big_bytes = sum(arrs[k].nbytes for k in big)
    if big_bytes > room:
        for k in big:
            n = arrs[k].size
            idx = np.sort(np.random.default_rng(0).choice(n, n * room // big_bytes, replace=False))
            arrs[k] = arrs[k].reshape(-1)[idx]
    os.makedirs(path, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(path, k + ".npy"), a)


def run_tracking(args, wl, rank, world, dev, pg):
    """The headline leg.  -> dict of everything measured (rank 0 assembles the JSON line)."""
    import torch
    import torch.distributed as dist
    from vtgaussian_slam_b200 import _lib, slam_ops
    from vtgaussian_slam_b200.fused import FusedRenderer, TrackingSolver
    fr = wl["frame"]
    W, H = fr["W"], fr["H"]
    gy = (H + 15) // 16
    settings = make_settings(wl, dev)
    params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
    N = params["means3D"].shape[0]
    band = (0, 0)
    if world > 1:
        # one full-frame render per rank (identical on every rank, once per FRAME, outside the timed iterations)
        # measures the work of every tile row; bands are cut to equal work instead of equal rows
        probe = FusedRenderer(settings, N, device=dev)
        probe.forward(params, torch.tensor(wl["q"], device=dev), torch.tensor(wl["t"], device=dev))
        nc = probe.ws.n_contrib.to(torch.float64)
        pad = torch.zeros((gy * 16, nc.shape[1]), dtype=torch.float64, device=dev)
        pad[:H] = nc
        row_work = pad.reshape(gy, 16, -1).sum(dim=(1, 2)).cpu().numpy()
        band = balanced_bands(row_work, world)[rank]
        del probe, nc, pad
        torch.cuda.empty_cache()
    solver = TrackingSolver(settings, params, device=dev, w_im=LOSS_W["im"], w_depth=LOSS_W["depth"], sil_thres=SIL_THRES,
                            tile_rows=band, use_graph=True, process_group=pg, deterministic=True if args.deterministic else None)
    gt_rgb = torch.tensor(fr["im"]).pin_memory()
    gt_depth = torch.tensor(fr["depth"]).pin_memory()
    solver.set_frame(gt_rgb, gt_depth, wl["q"], wl["t"])

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- device-resident timed region: W warm-up + K timed graph replays ---------------------------
    warm = max(args.warmup, 3)
    for _ in range(warm):
        solver.step()
    overflow, R = solver.r.overflowed()
    if overflow:
        raise SystemExit(f"pair buffer overflow: R={R}")
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        solver.step()
    e1.record()
    sync_all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, solver, N)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms.item() / args.steps
    loss_now = solver.loss_terms()[0].item()

    # ---- per-kernel durations (eager, CUDA events around every launch of the library) --------------
    solver.use_graph = False
    _lib.profile_enable(True)
    torch.cuda.synchronize(dev)
    prof_steps = min(args.steps, 20)
    for _ in range(prof_steps):
        solver.step()
    torch.cuda.synchronize(dev)
    prof = _lib.profile_summary()
    _lib.profile_enable(False)
    launches_per_step = sum(n for n, _ in prof.values()) // prof_steps
    total_prof_ms = sum(t for _, t in prof.values())
    S = int(solver.r.ws.n_contrib.to(torch.int64).sum().item())
    _, R = solver.r.overflowed()
    P = W * H
    out = dict(ms_per_step=ms_per_step, clocks=clocks, loss_now=loss_now, prof=prof, launches_per_step=launches_per_step,
               total_prof_ms=total_prof_ms, S=S, R=R, P=P, N=N, warm=warm, band=band)
    if args.kernels_only:
        return out

    # ---- e2e (a): the repo's own tracking API with host buffers, at N GPUs ---------------------------
    # TrackingSolver.step() (graph replay; band-sharded + all-reduce at N > 1); every step uploads its frame from
    # pinned host memory on a copy stream (double-buffered staging, then a device copy into the solver's target
    # planes) and reads the step's loss back into pinned memory (asynchronously; consumed one step later).
    solver.use_graph = True
    stage = [dict(im=torch.empty((3, H, W), device=dev), depth=torch.empty((1, H, W), device=dev), ev=torch.cuda.Event())
             for _ in range(2)]
    cstream = torch.cuda.Stream(dev)
    loss_pin = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    sstate = {"k": 0, "last": None}
    y0 = band[0] * 16 if world > 1 else 0                    # a rank only needs the rows of its tile band
    y1 = min(H, band[1] * 16) if world > 1 else H
    h2d_bytes = 4 * 4 * W * (y1 - y0)

    def stage_upload(slot):
        b = stage[slot]
        with torch.cuda.stream(cstream):
            for ch in range(3):
                b["im"][ch, y0:y1].copy_(gt_rgb[ch, y0:y1], non_blocking=True)      # contiguous row blocks of pinned memory
            b["depth"][0, y0:y1].copy_(gt_depth[0, y0:y1], non_blocking=True)
            b["ev"].record(cstream)

    def solver_e2e_step():
        k = sstate["k"]
        cur = stage[k & 1]
        main = torch.cuda.current_stream(dev)
        main.wait_event(cur["ev"])
        solver.gt_rgb[:, y0:y1].copy_(cur["im"][:, y0:y1], non_blocking=True)
        solver.gt_depth[:, y0:y1].copy_(cur["depth"][:, y0:y1], non_blocking=True)
        cstream.wait_stream(main)
        stage_upload((k + 1) & 1)
        solver.step()
        if k >= 1:
            loss_ev[(k - 1) & 1].synchronize()                  # the previous step's loss is now on the host
            sstate["last"] = float(loss_pin[(k - 1) & 1][0])
        loss_pin[k & 1].copy_(solver.msg[8:9], non_blocking=True)
        loss_ev[k & 1].record(main)
        sstate["k"] = k + 1

    stage_upload(0)
    for _ in range(3):
        solver_e2e_step()
    sync_all()
    ks = max(3, min(args.steps, 200))
    e0.record()
    for _ in range(ks):
        solver_e2e_step()
    e1.record()
    sync_all()
    ms_s = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_s, op=dist.ReduceOp.MAX)
    solver_e2e_ms = ms_s.item() / ks
    h2d_t = torch.tensor([float(h2d_bytes)], device=dev)
    if world > 1:
        dist.all_reduce(h2d_t)
    e2e_solver = {"value": 1e3 / solver_e2e_ms, "unit": UNIT, "h2d_bytes_per_step": int(h2d_t.item()), "d2h_bytes_per_step": 4 * world,
                  "ms_per_step": solver_e2e_ms,
                  "api": "TrackingSolver.step() (graph replay" + (", tile bands + 16-float all-reduce" if world > 1 else "") +
                         "); per-step upload of the rank's rows of the frame from pinned memory on a copy stream, loss read back asynchronously"}
    out["e2e"] = e2e_solver

    # ---- e2e (b): the reference-facing API with host buffers (N = 1) -------------------------------
    if world == 1:
        del solver
        torch.cuda.empty_cache()
        P_ = {k: torch.nn.Parameter(v.clone()) for k, v in params.items()}
        P_["cam_unnorm_rots"] = torch.nn.Parameter(torch.tensor(wl["q"], device=dev).reshape(1, 4, 1).contiguous())
        P_["cam_trans"] = torch.nn.Parameter(torch.tensor(wl["t"], device=dev).reshape(1, 3, 1).contiguous())
        lrs = dict(means3D=0.0, rgb_colors=0.0, unnorm_rotations=0.0, logit_opacities=0.0, log_scales=0.0,
                   cam_unnorm_rots=0.0004, cam_trans=0.002)                  # configs/replica/room0.py:78-86
        opt = slam_ops.initialize_optimizer(P_, lrs, tracking=True)
        variables = dict(max_2D_radius=torch.zeros(N, device=dev))
        # double-buffered frame upload: the H2D copy of step k+1's inputs runs on a copy stream while step k computes
        # (every step's inputs are still copied from pinned host memory inside the timed region)
        bufs = [dict(im=torch.empty((3, H, W), device=dev), depth=torch.empty((1, H, W), device=dev), ev=torch.cuda.Event())
                for _ in range(2)]
        copy_stream = torch.cuda.Stream(dev)
        w2c_eye = torch.eye(4, device=dev)
        state = {"k": 0, "last": None}

        def upload(slot):
            b = bufs[slot]
            with torch.cuda.stream(copy_stream):
                b["im"].copy_(gt_rgb, non_blocking=True)           # H2D of a step's inputs (pinned)
                b["depth"].copy_(gt_depth, non_blocking=True)
                b["ev"].record(copy_stream)

        def e2e_step(backend="fused"):
            k = state["k"]
            cur = bufs[k & 1]
            torch.cuda.current_stream(dev).wait_event(cur["ev"])   # this step's inputs have landed
            copy_stream.wait_stream(torch.cuda.current_stream(dev))  # the other buffer's previous consumer is queued before the copy
            data = dict(cam=settings, im=cur["im"], depth=cur["depth"], w2c=w2c_eye)
            loss, _, _ = slam_ops.get_loss(P_, data, variables, 0, LOSS_W, True, SIL_THRES, True, False, tracking=True,
                                           tracking_iteration=k + 1, dataset_name="tum", backend=backend)
            upload((k + 1) & 1)                                    # prefetch the next step's inputs
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            # D2H of the step's result: asynchronous into pinned memory, consumed (event-synchronised) one step later, so
            # the host may run one step ahead of the device
            if k >= 1:
                loss_ev[(k - 1) & 1].synchronize()
                state["last"] = float(loss_pin[(k - 1) & 1][0])
            loss_pin[k & 1].copy_(loss.detach().reshape(1), non_blocking=True)
            loss_ev[k & 1].record(torch.cuda.current_stream(dev))
            state["k"] = k + 1

        upload(0)
        for _ in range(3):
            e2e_step()
        torch.cuda.synchronize(dev)
        k2 = max(3, min(args.steps, 100))
        e0.record()
        for _ in range(k2):
            e2e_step()
        e1.record()
        torch.cuda.synchronize(dev)
        e2e_ms = e0.elapsed_time(e1) / k2
        e2e = {"value": 1e3 / e2e_ms, "unit": UNIT, "h2d_bytes_per_step": int(4 * 4 * P), "d2h_bytes_per_step": 4,
               "ms_per_step": e2e_ms, "api": "slam_ops.get_loss(backend='fused') + loss.backward() + torch.optim.Adam.step(); frame upload double-buffered on a copy stream, loss read back asynchronously",
               "solver_api": e2e_solver}
        # the same step through the reference's literal structure: two three-channel rasteriser passes of the drop-in
        # module + torch loss / masks + autograd (backend='dropin'): what the fusion buys on identical kernels
        for _ in range(2):
            e2e_step("dropin")
        torch.cuda.synchronize(dev)
        k3 = max(3, min(args.steps, 10))
        e0.record()
        for _ in range(k3):
            e2e_step("dropin")
        e1.record()
        torch.cuda.synchronize(dev)
        e2e["two_pass_dropin_value"] = 1e3 / (e0.elapsed_time(e1) / k3)
        out["e2e"] = e2e
        del P_, opt, bufs
        slam_ops._RENDERERS.clear()
        torch.cuda.empty_cache()
    return out


def gpu_first_iteration(wl, dev):
    """One tracking iteration at the workload's start pose, everything read back: the GPU side of parity_check."""
    import torch
    from vtgaussian_slam_b200.fused import FusedRenderer
    fr = wl["frame"]
    settings = make_settings(wl, dev)
    params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
    N = params["means3D"].shape[0]
    r = FusedRenderer(settings, N, device=dev)
    q, t = torch.tensor(wl["q"], device=dev), torch.tensor(wl["t"], device=dev)
    img, radii = r.forward(params, q, t)
    terms = r.tracking_loss(torch.tensor(fr["im"], device=dev), torch.tensor(fr["depth"], device=dev), w_im=LOSS_W["im"],
                            w_depth=LOSS_W["depth"], use_sil_for_loss=True, sil_thres=SIL_THRES).clone()
    dq, dt = torch.zeros(4, device=dev), torch.zeros(3, device=dev)
    r.backward(params, q, t, pose_grads=(dq, dt))
    _, R = r.overflowed()
    res = dict(img=img.cpu().numpy(), radii=radii.cpu().numpy(), n_contrib=r.ws.n_contrib.cpu().numpy().astype(np.uint32),
               loss=float(terms[0].item()), dq=dq.cpu().numpy(), dt=dt.cpu().numpy(), R=R)
    del r
    torch.cuda.empty_cache()
    return res


def run_cpu_and_parity(wl, dev):
    """cpu_baseline (the oracle port timed on a bounded sample of the same workload) and parity_check (the GPU arm's
    iteration against that CPU iteration).  Rank 0, N = 1 only."""
    cores = cpu_threads()
    t_first, loss_cpu, out, g = cpu_iteration(wl, want_grads=True)        # doubles as the warm-up
    times = []
    while sum(times) < 12.0 and len(times) < 16:
        times.append(cpu_iteration(wl)[0])
    t_cpu = sum(times) / len(times)
    cpu = {"value": 1.0 / t_cpu, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{len(times)} full iterations of the same workload on the host cores after one warm-up "
                     f"({sum(times):.1f} s, {t_cpu:.2f} s each)"}
    gq, gt = cpu_pose_gradient(wl, g)
    gpu = gpu_first_iteration(wl, dev)
    rel = lambda a, b: float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-30))
    parity = {
        "against": "oracle port (CPU), same inputs, first iteration of the workload",
        "loss_gpu": gpu["loss"], "loss_cpu": loss_cpu, "loss_rel": abs(gpu["loss"] - loss_cpu) / max(abs(loss_cpu), 1e-30),
        "pose_grad_rel": max(rel(gpu["dq"], gq), rel(gpu["dt"], gt)),
        "R_equal": bool(gpu["R"] == out["R"]), "S_equal": bool(int(gpu["n_contrib"].sum()) == int(out["n_contrib"].sum())),
        "radii_equal": bool(np.array_equal(gpu["radii"], out["radii"])),
        "n_contrib_equal": bool(np.array_equal(gpu["n_contrib"], out["n_contrib"])),
        "planes_bit_exact": bool(np.array_equal(gpu["img"], out["color"])),
        "planes_max_abs": float(np.abs(gpu["img"] - out["color"]).max()),
    }
    counters = {"K_contributing_pairs": int(out["contributing"]), "S_pair_tests": int(out["n_contrib"].sum()), "R": int(out["R"])}
    return cpu, parity, counters


def run_mapping_leg(args, wl, rank, world, dev, pg, iters=None, keyframes=8, shape="replica"):
    """BASELINE configs[2]: one mapping iteration = a batch of `keyframes` posed keyframes of one section split over the
    ranks (keyframe k -> rank k mod world): fused six-plane render, SSIM mapping loss, backward to the Gaussian
    parameters; then ONE kernel over NVLink peer memory that reduce-scatters the gradients, steps Adam on the rank's slice
    and all-gathers the new parameters (NCCL all-reduce + replicated Adam where peer mapping is unavailable; the plain
    all-reduce of the same message is timed beside it).  Strong scaling (fixed batch).
    -> dict (identical on every rank)."""
    import torch
    import torch.distributed as dist
    from vtgaussian_slam_b200 import _lib, synthetic
    from vtgaussian_slam_b200.fused import MappingSolver
    from vtgaussian_slam_b200.slam_loop import quat_from_matrix
    fr = wl["frame"]
    W, H = fr["W"], fr["H"]
    settings = make_settings(wl, dev)
    params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
    N = params["means3D"].shape[0]
    ms = MappingSolver(settings, params, device=dev, process_group=pg)
    K_total = max(keyframes, world)
    poses = synthetic.trajectory(K_total, step_m=0.02, step_deg=1.0, seed=11)
    kf = []
    for k in range(rank, K_total, world):
        fk = synthetic.make_frame(shape, W, H, seed=50 + k, c2w=poses[k])
        w2c = np.linalg.inv(poses[k])
        kf.append(dict(cam_q=torch.tensor(quat_from_matrix(w2c[:3, :3]).astype(np.float32), device=dev),
                       cam_t=torch.tensor(w2c[:3, 3].astype(np.float32), device=dev),
                       gt_rgb=torch.tensor(fk["im"], device=dev), gt_depth=torch.tensor(fk["depth"], device=dev)))
    iters = iters or max(3, min(args.steps, 60))
    for _ in range(3):
        ms.iteration(kf)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        ms.iteration(kf)
    e1.record()
    torch.cuda.synchronize(dev)
    ms_t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    ar_us = step_us = None
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        # the collective alone (same message, same stream), max over ranks
        for _ in range(3):
            dist.all_reduce(ms.flat, group=pg)
        torch.cuda.synchronize(dev)
        dist.barrier()
        e0.record()
        for _ in range(10):
            dist.all_reduce(ms.flat, group=pg)
        e1.record()
        torch.cuda.synchronize(dev)
        at = torch.tensor([e0.elapsed_time(e1) / 10], device=dev)
        dist.all_reduce(at, op=dist.ReduceOp.MAX)
        ar_us = at.item() * 1e3
        ms.flat.zero_()
        if ms.sharded is not None:
            # the fused step alone: barrier + reduce-scatter / Adam / all-gather kernel + barrier (on zero gradients)
            for _ in range(3):
                ms._sharded_step()
            torch.cuda.synchronize(dev)
            dist.barrier()
            e0.record()
            for _ in range(10):
                ms._sharded_step()
            e1.record()
            torch.cuda.synchronize(dev)
            st = torch.tensor([e0.elapsed_time(e1) / 10], device=dev)
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
            step_us = st.item() * 1e3
    _lib.profile_enable(True)
    torch.cuda.synchronize(dev)
    for _ in range(2):
        ms.iteration(kf)
    torch.cuda.synchronize(dev)
    prof = _lib.profile_summary()
    _lib.profile_enable(False)
    msps = ms_t.item() / iters
    loss = float((ms.total_loss if ms.sharded is None else ms.sharded["loss"]).item())
    fused_step = ms.sharded is not None
    multicast = bool(fused_step and ms.sharded["mc"])
    sharded_error = ms.sharded_error
    del ms, kf
    torch.cuda.empty_cache()
    return {"workload": wl["name"].replace("tracking", "mapping"), "keyframes_per_step": K_total, "keyframes_per_rank": (K_total + world - 1) // world,
            "n_gpus": world, "steps": iters, "ms_per_step": msps, "value": K_total * 1e3 / msps, "unit": "keyframe fwd+bwd iters/s",
            "scaling": "strong", "loss_last": loss,
            "collective": ("ONE kernel over NVLink peer memory (vtgs_sharded_adam): reduce-scatter of dL/d{rgb, logit_opacity, "
                           "log_scale} (5 N fp32) in rank order + Adam on the rank's slice (sharded moments) + all-gather of the "
                           "new parameters, between two cross-device barriers") if fused_step else
                          ("NCCL all-reduce(SUM) of dL/d{rgb, logit_opacity, log_scale} = 5 N fp32 + loss, then a replicated Adam" if world > 1
                           else "none (single GPU): per-tensor Adam"),
            "fused_step": fused_step, "fused_step_nvls_multicast": multicast, "fused_step_us": step_us, "fused_step_unavailable": sharded_error,
            "allreduce_bytes": int(4 * (5 * N + 1)) if world > 1 else 0, "allreduce_us": ar_us,
            "per_kernel_us_per_step": {k: round(t * 1e3 / 2, 2) for k, (n, t) in prof.items()}}


def run_deterministic_leg(args, wl, dev, plain_ms):
    """VTGS_BUF_DETERMINISTIC: the same tracking iteration with the order-independent (exact fp32 hi / lo grid) gradient
    accumulation.  Reports its cost against the plain path and checks that two runs of the same 30 iterations end in
    bitwise identical poses and losses."""
    import torch
    from vtgaussian_slam_b200.fused import TrackingSolver
    fr = wl["frame"]
    params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
    solver = TrackingSolver(make_settings(wl, dev), params, device=dev, w_im=LOSS_W["im"], w_depth=LOSS_W["depth"],
                            sil_thres=SIL_THRES, use_graph=True, deterministic=True)
    gt_rgb, gt_depth = torch.tensor(fr["im"]), torch.tensor(fr["depth"])
    ends = []
    for _ in range(2):
        solver.set_frame(gt_rgb, gt_depth, wl["q"], wl["t"])
        for _ in range(30):
            solver.step()
        torch.cuda.synchronize(dev)
        ends.append(torch.cat([solver.cam_q, solver.cam_t, solver.msg]).cpu().numpy().tobytes())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = max(3, min(args.steps, 100))
    e0.record()
    for _ in range(k):
        solver.step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / k
    return {"value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "slowdown_vs_plain": ms / plain_ms - 1.0,
            "bitwise_repeatable_30_iterations": ends[0] == ends[1],
            "how": "TrackingSolver(deterministic=True): K6' partial sums split onto per-Gaussian power-of-two grids (exact, order-independent fp32 sums), K7' adds hi + lo"}


def run_c1_leg(dev, with_cpu):
    """configs[0]: one fwd+bwd of the ~300 k-Gaussian frame (tracking loss), GPU (CUDA events) and CPU oracle."""
    import torch
    from vtgaussian_slam_b200.fused import FusedRenderer
    wl = build_workload("c1")
    fr = wl["frame"]
    settings = make_settings(wl, dev)
    params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
    N = params["means3D"].shape[0]
    r = FusedRenderer(settings, N, device=dev)
    q, t = torch.tensor(wl["q"], device=dev), torch.tensor(wl["t"], device=dev)
    gt_rgb, gt_d = torch.tensor(fr["im"], device=dev), torch.tensor(fr["depth"], device=dev)
    dq, dt = torch.zeros(4, device=dev), torch.zeros(3, device=dev)

    def it():
        r.forward(params, q, t)
        r.tracking_loss(gt_rgb, gt_d, w_im=LOSS_W["im"], w_depth=LOSS_W["depth"], sil_thres=SIL_THRES)
        r.backward(params, q, t, pose_grads=(dq, dt))
    for _ in range(3):
        it()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(20):
        it()
    e1.record()
    torch.cuda.synchronize(dev)
    gpu_ms = e0.elapsed_time(e1) / 20
    res = {"workload": wl["name"], "gaussians": N, "gpu_ms_per_fwd_bwd": gpu_ms, "gpu_iters_per_s": 1e3 / gpu_ms,
           "loss": float(r.loss_terms[0].item())}
    if with_cpu:
        cpu_iteration(wl)
        tc, loss_cpu, _ = cpu_iteration(wl)
        res.update(cpu_s_per_fwd_bwd=tc, cpu_cores=len(os.sched_getaffinity(0)), loss_cpu=loss_cpu,
                   loss_rel=abs(res["loss"] - loss_cpu) / max(abs(loss_cpu), 1e-30))
    del r
    torch.cuda.empty_cache()
    return res


def run_c4_leg(dev, frames=24):
    """configs[3] shape (TUM fr1_desk 640x480, baseframe_every 30, tracking 200 / mapping 30 iterations): a short piece of
    the full tracking + mapping loop over synthetic posed frames (examples/synthetic_slam.py runs all 600)."""
    import torch
    from vtgaussian_slam_b200 import synthetic
    from vtgaussian_slam_b200.slam_loop import LoopConfig, ViewTiedSLAM, ate_rmse
    seq = synthetic.make_sequence("tum_fr1", num_frames=frames, step_m=0.004, step_deg=0.15, seed=0)
    cfg = LoopConfig(track_iters=200, map_iters=30, baseframe_every=30, map_every=5)
    slam = ViewTiedSLAM(seq[0]["W"], seq[0]["H"], seq[0]["K"], cfg, device=dev)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    est = slam.run(seq)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    gt = np.stack([f["c2w"] for f in seq])
    st = slam.stats
    res = {"workload": "tum_fr1_desk-shaped 640x480 loop, %d of 600 frames" % frames, "frames_per_s": frames / dt,
           "tracking_iters_per_s": st["track_iters"] / max(st["track_s"], 1e-9), "mapping_keyframe_iters_per_s": st["map_iters"] / max(st["map_s"], 1e-9),
           "ate_rmse_m": ate_rmse(est, gt), "path_extent_m": float(np.abs(gt[:, :3, 3]).max())}
    del slam
    torch.cuda.empty_cache()
    return res


def run_c5_leg(args, rank, world, dev, pg):
    """configs[4] shape: ScanNet++-sized 1752x1168 view of ~8 M Gaussians in four sections.  N = 1: tracking iterations/s
    (with the outlier-median mask of the ScanNet++ config); every N: keyframe-sharded mapping (4 keyframes)."""
    import torch
    from vtgaussian_slam_b200.fused import TrackingSolver
    wl = build_workload("c5")
    fr = wl["frame"]
    res = {"workload": wl["name"]}
    if world == 1:
        settings = make_settings(wl, dev)
        params = {k: torch.tensor(v, device=dev) for k, v in wl["params"].items()}
        solver = TrackingSolver(settings, params, device=dev, w_im=0.5, w_depth=1.0, sil_thres=SIL_THRES, use_graph=True,
                                ignore_outlier_depth_loss=True)
        solver.set_frame(torch.tensor(fr["im"]), torch.tensor(fr["depth"]), wl["q"], wl["t"])
        for _ in range(3):
            solver.step()
        if solver.check(grow=True, raise_on_overflow=False) is None:
            for _ in range(3):
                solver.step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(10):
            solver.step()
        e1.record()
        torch.cuda.synchronize(dev)
        res["tracking_ms_per_step"] = e0.elapsed_time(e1) / 10
        res["tracking_iters_per_s"] = 1e3 / res["tracking_ms_per_step"]
        res["tracking_options"] = "ignore_outlier_depth_loss (frame median by radix select), sil_thres 0.99"
        del solver, params
        torch.cuda.empty_cache()
    m = run_mapping_leg(args, wl, rank, world, dev, pg, iters=5, keyframes=max(4, world), shape="scannetpp")
    res["mapping"] = {k: m[k] for k in ("keyframes_per_step", "ms_per_step", "value", "unit", "fused_step", "fused_step_us", "allreduce_bytes",
                                        "allreduce_us")}
    return res


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    rank, world, local = dist_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    tr = run_tracking(args, wl, rank, world, dev, pg)
    prof, ms_per_step, S, R, P, N = tr["prof"], tr["ms_per_step"], tr["S"], tr["R"], tr["P"], tr["N"]
    per_kernel_us = {k: round(t * 1e3 / n, 2) for k, (n, t) in prof.items()}
    if args.kernels_only:
        if rank == 0:
            print(json.dumps({"value": 1e3 / ms_per_step, "ms_per_step": ms_per_step, "per_kernel_us": per_kernel_us,
                              "lib": os.environ.get("VTGS_LIB_PATH", "default")}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = parity = None
    exact = {}
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, parity, exact = run_cpu_and_parity(wl, dev)
    mapping = None if args.no_extra else run_mapping_leg(args, wl, rank, world, dev, pg)
    configs = None
    det = None
    if not args.no_extra and world == 1 and rank == 0:
        det = run_deterministic_leg(args, wl, dev, ms_per_step)
    if not args.no_extra and args.workload == "c2":
        configs = {}
        if world == 1:
            configs["c1"] = run_c1_leg(dev, with_cpu=not args.no_cpu)
            configs["c4"] = run_c4_leg(dev)
        configs["c5"] = run_c5_leg(args, rank, world, dev, pg)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
        fp32_peak = measure_fp32_peak(dev)
        kbytes = {       # ALGORITHMIC bytes per launch (DESIGN.md section 5)
            "preprocess_kernel": N * (12 + 4 + 16 + 4 + 12) + N * (64 + 4 + 4) + R * 4,
            "scatter_kernel": N * (4 + 16) + R * (8 + 4),
            "tile_sort_kernel": R * (8 + 8 + 4) + R * 32 + int(2.3 * R) * 8,
            "blend_forward_kernel": R * 52 + P * (6 * 4 + 4 + 4),
            "tracking_loss_kernel": P * (6 * 4 + 4 * 4 + 4 * 4),
            "blend_backward_kernel": R * 52 + P * (4 * 4 + 4 + 4) + N * 48,
            "fused_preprocess_backward_kernel": N * (48 + 12 + 4 + 16 + 4 + 64) + N * 48,
        }
        K = exact.get("K_contributing_pairs")
        kflops = {"blend_forward_kernel": 32.0 * S, "blend_backward_kernel": (76.0 * K) if K else None}    # SURVEY 8(d)
        dom_name, (dom_n, dom_ms) = max(prof.items(), key=lambda kv: kv[1][1])
        dom_s = dom_ms * 1e-3 / dom_n
        achieved = kbytes.get(dom_name, 0) / dom_s / 1e9
        counters = load_counters(wl["name"]) if world == 1 else {}
        dc = counters.get(dom_name, {})
        issue_peak = 148 * 4 * sm_mhz / 1e3                                   # G warp-instructions / s
        # iteration lower bound of SURVEY.md 8(d): sum over stages of max(bytes / measured HBM BW, flops / measured FP32)
        t_min = None
        if K:
            t_min = 0.0
            for k in prof:
                tb = kbytes.get(k, 0) / (hbm_peak * 1e9)
                tf = (kflops.get(k) or 0.0) / (fp32_peak * 1e12)
                t_min += max(tb, tf)
        blend = dom_name.startswith("blend_")
        roofline = {
            "bound": "issue" if blend else "hbm", "kernel": dom_name,
            "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": dc.get("dram_bytes"), "traffic_unit": "bytes/launch",
            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)",
            "kernel_us": dom_s * 1e6, "kernel_share_of_step": dom_ms / tr["total_prof_ms"],
            "note": "the blend kernels are issue / latency bound (no dense contraction, tensor cores unused); achieved / peak is "
                    "their algorithmic traffic against the HBM peak for the record, `issue` and `fp32` are the views that bind",
            "pair_tests_per_launch": S, "pair_tests_per_s": S / dom_s,
            "issue": ({"warp_inst_per_launch": dc["warp_inst"], "achieved_ginst_s": dc["warp_inst"] / dom_s / 1e9,
                       "peak_ginst_s": issue_peak, "frac": dc["warp_inst"] / dom_s / 1e9 / issue_peak,
                       "source": "profiles/r02_counters.json (ncu --set full of this workload, this round)"} if dc.get("warp_inst") else None),
            "fp32": {"peak_tflops_measured": fp32_peak, "peak_tflops_nominal": FP32_NOMINAL_TFLOPS,
                     "kernel_flops_per_launch": kflops.get(dom_name),
                     "frac_of_measured": (kflops[dom_name] / dom_s / 1e12 / fp32_peak) if kflops.get(dom_name) else None},
            "iteration": {"t_min_us": t_min * 1e6 if t_min else None, "frac_of_t_min": (t_min / (ms_per_step * 1e-3)) if t_min else None,
                          "hbm_floor_us": sum(kbytes.get(k, 0) for k in prof) / (hbm_peak * 1e9) * 1e6,
                          "formula": "sum over kernels of max(algorithmic bytes / measured HBM BW, (32 S | 76 K) flop / measured FP32 peak)"},
            "per_kernel_us": per_kernel_us,
        }
        line = {
            "metric": METRIC, "value": 1e3 / ms_per_step, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": tr["warm"], "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": config_of(wl, world),
            "counters": {"pairs_R": R, "pair_tests_S": S, "contributing_pairs_K": K, "pixels_P": P, "loss_after_run": tr["loss_now"]},
            "clocks": tr["clocks"], "e2e": tr["e2e"], "gpu_launches": tr["launches_per_step"] * args.steps,
            "launches_per_step": tr["launches_per_step"], "roofline": roofline, "cpu_baseline": cpu, "parity_check": parity,
            "mapping": mapping, "configs": configs, "deterministic": det,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--small", action="store_true", help="300x170 debug workload")
    ap.add_argument("--workload", choices=["c2", "c5", "c1"], default="c2",
                    help="c2 (default, the headline): Replica 1200x680, ~1 M Gaussians; c5 (side benchmark): ScanNet++-shaped 1752x1168, ~8 M Gaussians in 4 sections")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity_check leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the mapping block and the c1 / c4 / c5 legs")
    ap.add_argument("--kernels-only", action="store_true", help="kernel experiments: device-timed value + per-kernel durations only")
    ap.add_argument("--deterministic", action="store_true", help="kernel experiments: the headline leg with VTGS_BUF_DETERMINISTIC")
    ap.add_argument("--mode", default="tracking", choices=["tracking", "mapping"],
                    help="tracking = configs[1] (the driver's line, which also carries the mapping block); mapping = only the keyframe-sharded leg")
    ap.add_argument("--keyframes", type=int, default=8, help="--mode mapping: keyframes per mapping iteration (configs[2]: 8)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed tracking step computed as DIR/<name>.npy "
                         "(float32, at most 64 MB; rank 0's arrays when --gpus > 1, whose render covers its tile band only). "
                         "The order of the backward's float atomics moves them slightly from run to run; with --deterministic "
                         "they repeat bitwise")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.mode == "mapping"):
        ap.error("--dump-outputs writes the outputs of the GPU tracking path: not with --impl reference or --mode mapping")
    rank, world, local = dist_env()
    kind = "small" if args.small else args.workload
    if args.impl == "reference":
        if rank != 0:
            return
        run_reference_arm(args, build_workload(kind))
        return
    if args.mode == "mapping":
        import torch
        import torch.distributed as dist
        dev = torch.device("cuda", local)
        torch.cuda.set_device(dev)
        pg = None
        if world > 1:
            dist.init_process_group("nccl", device_id=dev)
            pg = dist.group.WORLD
        m = run_mapping_leg(args, build_workload(kind), rank, world, dev, pg, keyframes=args.keyframes)
        if rank == 0:
            print(json.dumps(dict(m, metric=METRIC + " (mapping, keyframe-sharded)", higher_is_better=True, dtype="fp32", data="synthetic")), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    run_ours(args, build_workload(kind))


if __name__ == "__main__":
    main()
