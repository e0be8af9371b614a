"""-m gpu: every caller that renders repeats its work with grown pair buffers when a render overflowed them, and ends with
the same bits as a run whose buffers were ample from the start (deterministic gradient accumulation wherever a backward
runs); a TrackingSolver whose buffers were regrown after its graphs were captured captures them again."""
import numpy as np
import pytest
import torch

from vtgaussian_slam_b200 import fused, rasterizer, synthetic
from vtgaussian_slam_b200.fused import MappingSolver, TrackingSolver

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TINY, AMPLE = 64, 4 << 20


def _settings(fr):
    from gpu_helpers import settings_from
    s = synthetic.setup_camera(fr["W"], fr["H"], fr["K"], np.eye(4))
    return settings_from(s, torch.device(DEV))


def _scene(W=200, H=120, seed=0):
    fr = synthetic.make_frame("replica", W, H, seed=seed)
    p = synthetic.view_tied_gaussians(fr, n_edge=1500, opacity="trained")
    q, t = synthetic.perturbed_pose(seed=1)
    return fr, p, q.astype(np.float32), t.astype(np.float32)


def _gp(p):
    return {k: torch.tensor(v, device=DEV) for k, v in p.items()}


@pytest.fixture
def regrowths(monkeypatch):
    """Counts the pair-buffer regrowths (every caller grows through Workspace.ensure_capacity)."""
    n = [0]
    grow = rasterizer.grown_pair_capacity

    def counting(R):
        n[0] += 1
        return grow(R)
    monkeypatch.setattr(rasterizer, "grown_pair_capacity", counting)
    return n


@pytest.fixture
def deterministic():
    rasterizer.set_deterministic(True)
    yield
    rasterizer.set_deterministic(False)


def _with_capacity(monkeypatch, cap):
    """New renderers and drop-in forwards start from `cap` pairs."""
    monkeypatch.setattr(fused, "initial_pair_capacity", lambda device, n: cap)
    monkeypatch.setattr(rasterizer, "initial_pair_capacity", lambda device, n: cap)


def test_mapping_iteration_regrows_before_the_update(regrowths):
    fr, p, q, t = _scene()
    settings = _settings(fr)
    kf = [dict(cam_q=torch.tensor(q, device=DEV), cam_t=torch.tensor(t, device=DEV),
               gt_rgb=torch.tensor(fr["im"], device=DEV), gt_depth=torch.tensor(fr["depth"], device=DEV))]

    def run(cap):
        ms = MappingSolver(settings, _gp(p), device=DEV, pair_capacity=cap, poll_every=1, deterministic=True)
        losses = [ms.iteration(kf).clone() for _ in range(3)]
        return torch.cat(losses), ms.params
    loss_a, par_a = run(AMPLE)
    assert regrowths[0] == 0
    loss_t, par_t = run(TINY)
    assert regrowths[0] == 1
    assert torch.equal(loss_t, loss_a)
    for k in par_a:
        assert torch.equal(par_t[k], par_a[k]), k


def test_frame_evaluator_render_regrows(monkeypatch, regrowths):
    from vtgaussian_slam_b200.evaluation import FrameEvaluator
    from vtgaussian_slam_b200.slam_loop import matrix_from_quat
    fr, p, q, t = _scene()
    w2c = matrix_from_quat(q, t)

    def run(cap):
        _with_capacity(monkeypatch, cap)
        return FrameEvaluator(_settings(fr), DEV).render(_gp(p), w2c).clone()
    ample = run(AMPLE)
    assert regrowths[0] == 0
    tiny = run(TINY)
    assert regrowths[0] >= 1 and torch.equal(tiny, ample)


def test_add_missing_gaussians_regrows(monkeypatch, regrowths, deterministic):
    from vtgaussian_slam_b200.slam_loop import LoopConfig, ViewTiedSLAM
    W, H, K = synthetic.intrinsics("tum_fr1", 160, 120)
    poses = synthetic.trajectory(2, step_m=0.25, step_deg=8.0, seed=7)
    f0 = synthetic.make_frame("tum_fr1", 160, 120, seed=0, c2w=poses[0])
    f1 = synthetic.make_frame("tum_fr1", 160, 120, seed=1, c2w=poses[1])
    rgb, depth = torch.as_tensor(f1["im"]).to(DEV), torch.as_tensor(f1["depth"]).to(DEV).reshape(1, H, W)

    def run(cap):
        _with_capacity(monkeypatch, cap)
        slam = ViewTiedSLAM(W, H, K, LoopConfig(track_iters=5, map_iters=2, baseframe_every=100), device=DEV)
        slam.process(f0)
        slam.w2c.append(np.linalg.inv(poses[1]))
        n = slam.add_missing_gaussians(1, rgb, depth)
        return n, {k: v.clone() for k, v in slam.sections[-1]["params"].items()}
    n_a, rows_a = run(AMPLE)
    assert regrowths[0] == 0
    n_t, rows_t = run(TINY)
    assert regrowths[0] >= 1 and n_a > 0 and n_t == n_a
    for k in rows_a:
        assert torch.equal(rows_t[k], rows_a[k]), k


def test_run_frame_with_metric_regrows(regrowths):
    fr, p, q, t = _scene()
    settings = _settings(fr)
    target = torch.tensor(t) + 0.01

    def run(cap):
        ts = TrackingSolver(settings, _gp(p), device=DEV, pair_capacity=cap, deterministic=True)
        ts.set_frame(torch.tensor(fr["im"]), torch.tensor(fr["depth"]), q, t)
        return ts.run_frame_with_metric(8, lambda q_, t_: float(((t_ - target) ** 2).sum()))
    ample = run(AMPLE)
    assert regrowths[0] == 0
    tiny = run(TINY)
    assert regrowths[0] == 1 and torch.equal(tiny, ample)


def test_drop_in_forward_and_backward_regrow(monkeypatch, regrowths, deterministic):
    from gpu_helpers import settings_from
    W, H = 160, 112
    K, sc = synthetic.random_scene(3000, W, H, seed=3)
    st = settings_from(synthetic.setup_camera(W, H, K, np.eye(4)), torch.device(DEV))

    def run(cap):
        _with_capacity(monkeypatch, cap)
        x = {k: torch.tensor(v, device=DEV, requires_grad=True) for k, v in sc.items()}
        m2d = torch.zeros_like(x["means3D"], requires_grad=True)
        color, radii, depth = rasterizer.GaussianRasterizer(raster_settings=st)(
            means3D=x["means3D"], means2D=m2d, opacities=x["opacities"], colors_precomp=x["colors"], scales=x["scales"],
            rotations=x["rotations"])
        w = torch.linspace(0.5, 1.5, color.numel(), device=DEV).reshape(color.shape)
        (color * w).sum().backward()
        return [color.detach(), radii, depth] + [x[k].grad for k in sorted(x)] + [m2d.grad]
    ample = run(AMPLE)
    assert regrowths[0] == 0
    tiny = run(TINY)
    assert regrowths[0] == 1
    for a, b in zip(tiny, ample):
        assert torch.equal(a, b)


def test_tracking_graphs_follow_regrown_buffers():
    fr, p, q, t = _scene()
    settings = _settings(fr)
    gt_rgb, gt_depth = torch.tensor(fr["im"]), torch.tensor(fr["depth"])

    def solver():
        ts = TrackingSolver(settings, _gp(p), device=DEV, use_graph=True, deterministic=True)
        ts.set_frame(gt_rgb, gt_depth, q, t)
        return ts
    ref = solver().run_frame(10)
    ts = solver()
    for _ in range(3):
        ts.step()                                   # the iteration graph is captured on the first pair buffers
    old_graph, gen = ts._graph, ts.r.ws.generation
    ts.r.ws.reserve_pairs(2 * ts.r.ws.pair_capacity)     # their memory goes back to the allocator
    assert ts.r.ws.generation == gen + 1
    ts.set_frame(gt_rgb, gt_depth, q, t)
    got = ts.run_frame(10)
    assert ts._graph is not old_graph and ts._graph_generation == ts.r.ws.generation
    assert torch.equal(got, ref)
