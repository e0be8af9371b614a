"""CPU tests of the oracle itself: closed-form golden cases (SURVEY.md 8(c) G1-G8),
structural invariants, and an independent fp64 PyTorch/autograd restatement that checks both
the forward values and the hand-derived backward.  No GPU."""
import math

import numpy as np
import pytest
import torch

import oracle
import torch_ref
from helpers import cam_dict, oracle_camera, rel_err
from vtgaussian_slam_b200 import synthetic


def _one(width=64, height=48, f=60.0):
    K = np.array([[f, 0, (width - 1) / 2.0], [0, f, (height - 1) / 2.0], [0, 0, 1.0]])
    return K


def _gauss_at_pixel(K, px, py, z, sigma_px, op=0.7, col=(0.2, 0.5, 0.9)):
    """Isotropic Gaussian whose centre projects exactly onto pixel centre (px, py)."""
    f = K[0, 0]
    # setup_camera's projection maps X to pixel fx*X/z + cx - 0.5 (hence get_pointcloud's +0.5)
    x = (px - K[0, 2] + 0.5) / f * z
    y = (py - K[1, 2] + 0.5) / f * z
    s = sigma_px * z / f
    return dict(means3D=np.array([[x, y, z]], np.float32), scales=np.full((1, 3), s, np.float32),
                rotations=np.array([[1, 0, 0, 0]], np.float32), opacities=np.array([op], np.float32),
                colors=np.array([col], np.float32))


def _cat(*gs):
    return {k: np.concatenate([g[k] for g in gs], 0) for k in gs[0]}


def _run(cam, g):
    o = oracle.Oracle()
    return o, o.forward(cam, g["means3D"], g["scales"], g["rotations"], g["opacities"], g["colors"])


def test_vexpf_accuracy():
    xs = np.concatenate([np.linspace(-87, 0, 20001), -np.logspace(-8, 1.9, 2000)]).astype(np.float32)
    got = np.array([oracle.vexpf(float(x)) for x in xs], np.float64)
    ref = np.exp(xs.astype(np.float64))
    ulp = np.spacing(ref.astype(np.float32)).astype(np.float64)
    assert np.max(np.abs(got - ref) / ulp) <= 1.5
    assert oracle.vexpf(0.0) == 1.0
    assert oracle.vexpf(-1000.0) > 0.0 and oracle.vexpf(-1000.0) < 1e-37


def test_g1_single_gaussian_closed_form():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    # on the optical axis (pixel 31, 23) the EWA Jacobian has no off-axis term: var = sigma^2 + 0.3
    g = _gauss_at_pixel(K, 31, 23, 2.0, sigma_px=1.0, op=0.7)
    _, out = _run(cam, g)
    var = 1.0 + 0.3
    assert out["radii"][0] == math.ceil(3 * math.sqrt(var))
    np.testing.assert_allclose(out["means2D"][0], [31, 23], atol=2e-4)
    alpha = 0.7
    np.testing.assert_allclose(out["color"][:, 23, 31], np.array([0.2, 0.5, 0.9]) * alpha, rtol=2e-5)
    np.testing.assert_allclose(out["final_T"][23, 31], 1 - alpha, rtol=2e-5)
    np.testing.assert_allclose(out["depth"][23, 31], 2.0 * alpha, rtol=2e-5)
    assert out["n_contrib"][23, 31] == 1
    # neighbouring pixel: alpha = o * exp(-0.5 / var)
    a1 = 0.7 * math.exp(-0.5 / var)
    np.testing.assert_allclose(out["final_T"][23, 32], 1 - a1, rtol=1e-4)
    np.testing.assert_allclose(out["final_T"][24, 31], 1 - a1, rtol=1e-4)
    # beyond the alpha >= 1/255 radius nothing contributes
    d = math.sqrt(2 * var * math.log(255 * 0.7)) + 0.6
    assert out["n_contrib"][23, 31 + int(math.ceil(d))] == 0
    # off-axis the variance grows by (1 + (tx/tz)^2): sigma_x^2 = s^2 (J00^2 + J02^2) + 0.3
    g = _gauss_at_pixel(K, 20, 23, 2.0, sigma_px=1.0, op=0.7)
    _, out = _run(cam, g)
    r = (20 - K[0, 2] + 0.5) / K[0, 0]
    a1 = 0.7 * math.exp(-0.5 / (1.0 + r * r + 0.3))
    np.testing.assert_allclose(out["final_T"][23, 21], 1 - a1, rtol=1e-4)


def test_g1_opacity_clamped_to_099():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    _, out = _run(cam, _gauss_at_pixel(K, 30, 30, 1.5, 2.0, op=1.0))
    np.testing.assert_allclose(out["final_T"][30, 30], 0.01, rtol=1e-4)


def test_g2_two_gaussians_depth_order():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    near = _gauss_at_pixel(K, 25, 20, 1.0, 1.5, op=0.6, col=(1, 0, 0))
    far = _gauss_at_pixel(K, 25, 20, 3.0, 1.5, op=0.5, col=(0, 1, 0))
    for g in (_cat(near, far), _cat(far, near)):       # input order must not matter
        _, out = _run(cam, g)
        np.testing.assert_allclose(out["color"][:, 20, 25], [0.6, 0.4 * 0.5, 0.0], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(out["final_T"][20, 25], 0.4 * 0.5, rtol=1e-4)
        np.testing.assert_allclose(out["depth"][20, 25], 1.0 * 0.6 + 3.0 * 0.5 * 0.4, rtol=1e-4)
        assert out["n_contrib"][20, 25] == 2


def test_g2_equal_depth_ties_keep_index_order():
    W, H = 32, 32
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    a = _gauss_at_pixel(K, 10, 10, 2.0, 1.0, op=0.5, col=(1, 0, 0))
    b = _gauss_at_pixel(K, 11, 10, 2.0, 1.0, op=0.5, col=(0, 1, 0))
    _, out = _run(cam, _cat(a, b))
    t = 0  # tile 0
    rb, re = out["ranges"][t]
    assert list(out["point_list"][rb:re]) == [0, 1]
    _, out2 = _run(cam, _cat(b, a))
    assert list(out2["point_list"][rb:re]) == [0, 1]
    # first in list is blended first: its colour weight is alpha, the second alpha*(1-alpha)
    assert out["color"][0, 10, 10] > out2["color"][0, 10, 10]


def test_g3_near_cull():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    _, out = _run(cam, _cat(_gauss_at_pixel(K, 30, 20, 0.2, 1.0), _gauss_at_pixel(K, 30, 20, np.float32(0.2) + 1e-4, 1.0)))
    assert out["radii"][0] == 0 and out["tiles_touched"][0] == 0
    assert out["radii"][1] > 0
    vis = oracle.mark_visible(cam, np.array([[0, 0, 0.2], [0, 0, 0.21], [0, 0, -1]], np.float32))
    assert list(vis) == [False, True, False]


def test_g4_straddles_four_tiles_and_keys():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    _, out = _run(cam, _gauss_at_pixel(K, 15.5, 15.5, 2.5, 1.0))
    assert out["tiles_touched"][0] == 4 and out["R"] == 4
    gx = out["grid"][0]
    tiles = sorted(int(k >> np.uint64(32)) for k in out["keys"])
    assert tiles == [0, 1, gx, gx + 1]
    depth_bits = np.array([2.5], np.float32).view(np.uint32)[0]
    assert all(int(k & np.uint64(0xFFFFFFFF)) == depth_bits for k in out["keys"])
    for t in (0, 1, gx, gx + 1):
        rb, re = out["ranges"][t]
        assert re - rb == 1


def test_g5_low_alpha_and_positive_power_skips():
    W, H = 64, 48
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    _, out = _run(cam, _gauss_at_pixel(K, 20, 20, 2.0, 1.0, op=0.003))     # o < 1/255: never contributes
    assert out["n_contrib"].max() == 0 and np.all(out["final_T"] == 1.0) and out["radii"][0] > 0


def test_g6_saturation_stops_early():
    W, H = 32, 32
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K)
    gs = [_gauss_at_pixel(K, 12, 12, 1.0 + 0.1 * i, 2.0, op=0.9) for i in range(12)]
    _, out = _run(cam, _cat(*gs))
    # T after k contributions = 0.1^k; the 4th keeps T=1e-4 (not < 1e-4 in exact math, fp32 decides), the 5th is refused
    n = out["n_contrib"][12, 12]
    assert n in (3, 4) and out["final_T"][12, 12] >= 1e-4 * 0.999
    assert n < 12


def test_g7_offscreen_clamped_jacobian():
    W, H = 64, 48
    K = _one(W, H)
    cam, s = oracle_camera(W, H, K)
    z = 1.0
    x = 2.0 * s["tanfovx"] * z        # beyond 1.3 * tanfov
    g = dict(means3D=np.array([[x, 0, z]], np.float32), scales=np.full((1, 3), 0.3, np.float32),
             rotations=np.array([[1, 0, 0, 0]], np.float32), opacities=np.array([0.5], np.float32),
             colors=np.array([[1, 1, 1]], np.float32))
    _, out = _run(cam, g)
    # cov2D xx with the clamped Jacobian: s^2 (J00^2 + J02^2) + 0.3, J02 = -fx * (1.3 tanfovx)
    fx = W / (2 * s["tanfovx"])
    a = 0.09 * (fx ** 2 + (fx * 1.3 * s["tanfovx"]) ** 2) + 0.3
    c = 0.09 * fx ** 2 + 0.3
    det = a * c
    np.testing.assert_allclose(out["conic_opacity"][0, :3], [c / det, 0.0, a / det], rtol=1e-4, atol=1e-9)


def test_radius_multiplier_is_a_parameter():
    W, H = 64, 48
    K = _one(W, H)
    g = _gauss_at_pixel(K, 20, 17, 2.0, sigma_px=2.0)
    r3 = _run(oracle_camera(W, H, K, sigma_mult=3.0)[0], g)[1]["radii"][0]
    r2 = _run(oracle_camera(W, H, K, sigma_mult=2.0)[0], g)[1]["radii"][0]
    assert r3 == math.ceil(3 * math.sqrt(4.3)) and r2 == math.ceil(2 * math.sqrt(4.3))


def test_empty_and_all_culled():
    W, H = 40, 24       # ragged: not multiples of 16
    K = _one(W, H)
    cam, _ = oracle_camera(W, H, K, bg=(0.1, 0.2, 0.3))
    e = dict(means3D=np.zeros((0, 3), np.float32), scales=np.zeros((0, 3), np.float32), rotations=np.zeros((0, 4), np.float32),
             opacities=np.zeros(0, np.float32), colors=np.zeros((0, 3), np.float32))
    _, out = _run(cam, e)
    assert out["R"] == 0 and np.all(out["final_T"] == 1)
    np.testing.assert_allclose(out["color"][:, 3, 3], [0.1, 0.2, 0.3])
    g = _gauss_at_pixel(K, 5, 5, -1.0, 1.0)
    _, out = _run(cam, g)
    assert out["R"] == 0 and out["radii"][0] == 0


@pytest.mark.parametrize("seed,aniso", [(0, True), (1, False), (2, True)])
def test_invariants_random_scene(seed, aniso):
    W, H = 100, 70          # ragged edge tiles
    K, sc = synthetic.random_scene(1500, W, H, seed=seed, anisotropic=aniso)
    cam, _ = oracle_camera(W, H, K)
    _, out = _run(cam, sc)
    gx, gy = out["grid"]
    assert (gx, gy) == (7, 5)
    R = out["R"]
    assert R == int(out["tiles_touched"].sum()) == int(out["offsets"][-1])
    assert np.all(np.diff(out["keys"].astype(np.uint64)) >= 0)
    # ranges partition [0, R) in tile order
    cur = 0
    for t in range(gx * gy):
        rb, re = out["ranges"][t]
        if re > rb:
            assert rb == cur
            cur = re
            assert np.all((out["keys"][rb:re] >> np.uint64(32)) == t)
        else:
            assert (rb, re) == (0, 0)
    assert cur == R
    # n_contrib never exceeds the tile list length
    lens = (out["ranges"][:, 1] - out["ranges"][:, 0]).reshape(gy, gx)
    per_px = np.kron(lens, np.ones((16, 16), dtype=lens.dtype))[:H, :W]
    assert np.all(out["n_contrib"] <= per_px)
    assert np.all((out["radii"] > 0) >= (out["tiles_touched"] > 0))
    # ties: equal keys keep Gaussian index order
    same = out["keys"][1:] == out["keys"][:-1]
    assert np.all(out["point_list"][1:][same] > out["point_list"][:-1][same])


def test_six_channel_pass_equals_two_three_channel_passes():
    """The reference renders [r,g,b] and [z,1,z^2] in two passes over identical geometry
    (src/vtgaussian_slam.py:461,466); one 6-channel pass must be bit-identical."""
    W, H = 96, 64
    K, sc = synthetic.random_scene(1200, W, H, seed=5)
    cam, _ = oracle_camera(W, H, K)
    z = sc["means3D"][:, 2:3]
    dsil = np.concatenate([z, np.ones_like(z), z * z], 1).astype(np.float32)
    o = oracle.Oracle()
    a = o.forward(cam, sc["means3D"], sc["scales"], sc["rotations"], sc["opacities"], sc["colors"])
    b = o.forward(cam, sc["means3D"], sc["scales"], sc["rotations"], sc["opacities"], dsil)
    c6 = o.forward(cam, sc["means3D"], sc["scales"], sc["rotations"], sc["opacities"], np.concatenate([sc["colors"], dsil], 1))
    assert np.array_equal(c6["color"][:3], a["color"]) and np.array_equal(c6["color"][3:], b["color"])
    assert np.array_equal(a["n_contrib"], b["n_contrib"]) and np.array_equal(a["point_list"], b["point_list"])
    # the rasteriser's own depth output equals the z channel when viewmatrix = I
    assert np.array_equal(b["color"][0], b["depth"])


def test_tile_band_is_a_restriction():
    W, H = 96, 80
    K, sc = synthetic.random_scene(1000, W, H, seed=9)
    full = _run(oracle_camera(W, H, K)[0], sc)[1]
    band = _run(oracle_camera(W, H, K, tile_rows=(1, 3))[0], sc)[1]
    assert np.array_equal(band["radii"], full["radii"])
    assert np.array_equal(band["color"][:, 16:48], full["color"][:, 16:48])
    assert np.array_equal(band["n_contrib"][16:48], full["n_contrib"][16:48])
    assert np.all(band["n_contrib"][:16] == 0) and np.all(band["n_contrib"][48:] == 0)


def _torch_inputs(sc, dtype=torch.float64):
    t = {k: torch.tensor(v, dtype=dtype, requires_grad=True) for k, v in sc.items()}
    t["means2D"] = torch.zeros(sc["means3D"].shape[0], 3, dtype=dtype, requires_grad=True)
    return t


@pytest.mark.parametrize("seed,aniso,bg,tiled", [pytest.param(3, True, (0, 0, 0), False, id="3-True-bg0"),
                                                 pytest.param(4, False, (0.3, 0.1, 0.6), False, id="4-False-bg1"),
                                                 pytest.param(11, True, (0, 0, 0), False, id="11-True-bg2"),
                                                 pytest.param(4, False, (0.3, 0.1, 0.6), True, id="4-False-bg1-tiled")])
def test_forward_and_backward_match_autograd(seed, aniso, bg, tiled):
    """tiled: torch_ref's tile-by-tile evaluation, which must also equal its dense form to fp64 rounding."""
    W, H = 48, 40
    K, sc = synthetic.random_scene(160, W, H, seed=seed, anisotropic=aniso, scale_px=(0.7, 5.0))
    cam, s = oracle_camera(W, H, K, bg=bg)
    o, out = _run(cam, sc)
    t = _torch_inputs(sc)
    ref = torch_ref.render(cam_dict(s), t["means3D"], t["scales"], t["rotations"], t["opacities"], t["colors"],
                           out["rects"], means2D=t["means2D"], tiled=tiled)
    assert np.array_equal(ref["n_contrib"].numpy(), out["n_contrib"])
    np.testing.assert_allclose(out["color"], ref["color"].detach().numpy(), atol=2e-5)
    np.testing.assert_allclose(out["depth"], ref["depth"].detach().numpy(), atol=5e-5)
    np.testing.assert_allclose(out["final_T"], ref["final_T"].detach().numpy(), atol=2e-5)
    vis = out["radii"] > 0
    np.testing.assert_allclose(out["means2D"][vis], ref["means2D"].detach().numpy()[vis], atol=2e-3)
    np.testing.assert_allclose(out["conic_opacity"][vis, :3], ref["conic"].detach().numpy()[vis], rtol=2e-4, atol=1e-7)

    rng = np.random.default_rng(seed)
    dL = rng.normal(size=(3, H, W)).astype(np.float32)
    (ref["color"] * torch.tensor(dL, dtype=torch.float64)).sum().backward()
    g = o.backward(dL)
    for name, key in [("means3D", "means3D"), ("scales", "scales"), ("rotations", "rotations"),
                      ("opacities", "opacities"), ("colors", "colors"), ("means2D", "means2D")]:
        want = t[key].grad.numpy()
        got = g[name]
        assert rel_err(got, want) < 1e-3, (name, rel_err(got, want))
    if tiled:
        td = _torch_inputs(sc)
        dense = torch_ref.render(cam_dict(s), td["means3D"], td["scales"], td["rotations"], td["opacities"], td["colors"],
                                 out["rects"], means2D=td["means2D"])
        assert torch.equal(dense["n_contrib"], ref["n_contrib"])
        for k in ("color", "depth", "final_T"):
            assert rel_err(ref[k].detach().numpy(), dense[k].detach().numpy()) <= 1e-12, k
        (dense["color"] * torch.tensor(dL, dtype=torch.float64)).sum().backward()
        for k in td:
            assert rel_err(t[k].grad.numpy(), td[k].grad.numpy(), floor=1e-300) <= 1e-12, k


def test_view_tied_frame_statistics():
    """A fresh one-Gaussian-per-pixel section: radius 4-5 px, 2-2.5 tiles per Gaussian,
    silhouette ~0.99 (SURVEY.md 8(d) analytic figures, which hold on the optical axis)."""
    fr = synthetic.make_frame("replica", 240, 136, seed=0)
    p = synthetic.view_tied_gaussians(fr)
    K = fr["K"]
    cam, _ = oracle_camera(fr["W"], fr["H"], K)
    m, sc, rot, op, col6 = oracle.frontend(p["means3D"], p["rgb_colors"], p["unnorm_rotations"], p["logit_opacities"],
                                           p["log_scales"], [1, 0, 0, 0], [0, 0, 0])
    assert np.array_equal(m, p["means3D"])
    np.testing.assert_allclose(op, 0.5)
    o = oracle.Oracle()
    out = o.forward(cam, m, sc, rot, op, col6)
    # radius = ceil(3 sqrt(1 + (tx/tz)^2 + 0.3)): 4 px on the axis, 5 towards the image corners
    assert set(np.unique(out["radii"][out["radii"] > 0])) <= {4, 5}
    cy, cx = fr["H"] // 2, fr["W"] // 2
    assert out["radii"][cy * fr["W"] + cx] == 4
    assert 1.9 < out["R"] / (out["radii"] > 0).sum() < 2.6
    sil = out["color"][4]
    assert 0.985 < np.median(sil) < 0.9995
    inner = (slice(8, -8), slice(8, -8))
    rel = np.abs(out["color"][3][inner] / sil[inner] / (fr["depth"][0][inner] * 1.005) - 1.0)
    assert np.median(rel) < 1e-2 and np.mean(rel < 0.03) > 0.9      # depth edges blend, flat areas agree
