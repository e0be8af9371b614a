"""-m gpu: section-start alignment in the SLAM loop (LoopConfig.align_sections): the base keyframe of every new section
but the first is mapped with bundle adjustment against frozen earlier sections, the new section re-tied to the stepped
pose after every step (reference src/vtgaussian_slam.py:2530-2552, :2706-2727)."""
import functools

import numpy as np
import pytest
import torch

from vtgaussian_slam_b200 import rasterizer, synthetic
from vtgaussian_slam_b200.fused import MappingSolver
from vtgaussian_slam_b200.slam_loop import LoopConfig, ViewTiedSLAM, ate_rmse, matrix_from_quat, section_from_frame

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W, H, K = synthetic.intrinsics("tum_fr1", 320, 240)
# explicit pose LRs (the tracking rates): the reference's own mapping pose LRs, 1e-8 / 1e-7, leave the pose in place
POSE_LRS = dict(LoopConfig().map_lrs, cam_unnorm_rots=4e-4, cam_trans=2e-3)
# a base-frame tracking error applied in the camera frame: 0.5 deg about y, then 1 cm (the camera centre moves by 1 cm)
E = matrix_from_quat([np.cos(np.radians(0.25)), 0.0, np.sin(np.radians(0.25)), 0.0], [0.006, -0.0048, 0.0064])
# Measured on a B200: at these LRs the section-start mapping moves the base pose AWAY from the ground truth (1 cm error
# -> about 35 mm after 20 steps; 13.8 -> 28.9 mm ATE on the two-section sequence).  The own term's pose gradient is not
# zero at the pose the section is tied to, and re-tying the section after every step keeps it so: Adam walks the pose
# about one LR per step in a fixed direction (the own term alone, re-tied, drifts ~40 mm in 20 steps; not re-tied, a few
# mm), and the frozen-section term does not hold it back.
# That gradient is a property of the method, not a kernel error: test_gpu_mapping_reference.py::
# test_own_term_pose_gradient_at_the_tied_pose_matches_fp64 finds the kernels' own-term pose gradient at the tied pose equal
# to fp64 autograd through the reference's chain (to 5e-5), and far from zero (|dL/dt| = 0.89 on a 100x70 section).
RUNAWAY = "section-start BA with re-tie drifts under the own term's pose gradient at the tracking LRs"


@functools.lru_cache(maxsize=None)
def _sequence(n):
    poses = synthetic.trajectory(n, step_m=0.01, step_deg=0.3)
    return poses, [synthetic.make_frame("tum_fr1", 320, 240, seed=i, c2w=poses[i]) for i in range(n)]


@pytest.fixture
def deterministic():
    was = rasterizer._DETERMINISTIC
    rasterizer.set_deterministic(True)
    yield
    rasterizer.set_deterministic(was)


def _run(cfg, n):
    slam = ViewTiedSLAM(W, H, K, cfg, device=DEV)
    for fr in _sequence(n)[1]:
        slam.process(fr)
    torch.cuda.synchronize()
    return slam


def _arena(slam):
    n = slam.store.num_gaussians
    return {k: v[:n].cpu() for k, v in slam.store.buf.items()}


def _assert_same_run(a, b):
    assert len(a.w2c) == len(b.w2c) and all(np.array_equal(x, y) for x, y in zip(a.w2c, b.w2c))
    assert a.store.offsets == b.store.offsets
    arena_b = _arena(b)
    for k, v in _arena(a).items():
        assert torch.equal(v, arena_b[k]), k


def _pose_error(w2c, c2w_gt):
    """-> (camera centre error in m, rotation error in degrees)."""
    c2w = np.linalg.inv(w2c)
    cos = (np.trace(c2w[:3, :3].T @ c2w_gt[:3, :3]) - 1.0) / 2.0
    return float(np.linalg.norm(c2w[:3, 3] - c2w_gt[:3, 3])), float(np.degrees(np.arccos(np.clip(cos, -1.0, 1.0))))


def _section(frame, c2w):
    return section_from_frame(torch.as_tensor(frame["im"]).to(DEV), torch.as_tensor(frame["depth"]).to(DEV), K, c2w, DEV)


def _record_mapping(monkeypatch):
    """-> list that collects (solver, keyframes, do_ba) of every MappingSolver.iteration call."""
    calls = []
    orig = MappingSolver.iteration

    def iteration(self, keyframes, *a, **kw):
        calls.append((self, keyframes, kw.get("do_ba", False)))
        return orig(self, keyframes, *a, **kw)
    monkeypatch.setattr(MappingSolver, "iteration", iteration)
    return calls


def _perturb(slam, b, wrong):
    """Frame b comes out of tracking at the pose `wrong`; tracking still runs and records its section choice."""
    for name in ("_track", "_track_base_frame"):
        orig = getattr(slam, name)

        def tracked(idx, rgb, depth, orig=orig):
            M = orig(idx, rgb, depth)
            return wrong.copy() if idx == b else M
        setattr(slam, name, tracked)


def test_off_leaves_the_loop_unchanged(deterministic):
    kw = dict(track_iters=30, map_iters=6, baseframe_every=4, map_every=2, track_sections=2)
    plain = _run(LoopConfig(**kw), 9)
    off = _run(LoopConfig(**kw, align_sections=0, map_lrs=POSE_LRS), 9)
    _assert_same_run(plain, off)
    assert off.stats["align"] == [] and off.stats["align_s"] == 0.0 and off.mapper.r_global is None


@pytest.mark.parametrize("mode", ["latest", "overlap"])
def test_section_start_alignment_steps_and_reties(mode, monkeypatch):
    # latest: frame 8 is tracked against (and aligned to) sections 0 and 1, row views of the arena.  overlap: frame 12 is
    # tracked against sections 0 and 2, a gathered copy whose trainable rows the mapper refreshes before every render.
    b, frozen = (8, [0, 1]) if mode == "latest" else (12, [0, 2])
    kw = dict(track_iters=40, map_iters=20, baseframe_every=4, map_every=2, align_sections=2, map_lrs=POSE_LRS)
    kw.update(track_sections=2) if mode == "latest" else kw.update(section_selection="overlap", overlap_every=2, topk_base=1)
    poses, frames = _sequence(b + 1)
    wrong = E @ np.linalg.inv(poses[b])
    slam = ViewTiedSLAM(W, H, K, LoopConfig(**kw), device=DEV)
    _perturb(slam, b, wrong)
    for fr in frames[:b]:
        slam.process(fr)
    before = [{k: v.clone() for k, v in s["params"].items()} for s in slam.sections]
    calls = _record_mapping(monkeypatch)
    slam.process(frames[b])
    torch.cuda.synchronize()
    k_new = len(slam.sections) - 1
    sec = slam.sections[-1]
    if mode == "overlap":
        assert slam.section_choices[-1] == (b, sec["tracked_against"])
    print(f"\n[{mode}] base frame {b} tracked against {sec['tracked_against']}, aligned to {sec['frozen']}")
    assert sec["base"] == b and sec["frozen"] == frozen and slam.stats["align"][-1][:2] == (b, frozen)
    assert slam.mapper._global_aliases == (mode == "latest")

    # (a) the base pose was stepped, and the stats record the step (whether it approaches the ground truth is
    # test_alignment_reduces_a_known_base_pose_error)
    e0, a0 = _pose_error(wrong, poses[b])
    e1, a1 = _pose_error(slam.w2c[b], poses[b])
    print(f"[{mode}] base frame {b}: centre error {e0 * 1e3:.3f} -> {e1 * 1e3:.3f} mm, rotation error {a0:.4f} -> {a1:.4f} deg;"
          f" stats {slam.stats['align'][-1]}")
    shift, _ = _pose_error(slam.w2c[b], np.linalg.inv(wrong))
    assert shift > 1e-4 and abs(slam.stats["align"][-1][2] - shift) < 1e-9

    # (b) the frozen sections -- every earlier section -- are bitwise unchanged
    for i, rows in enumerate(before):
        for k, v in rows.items():
            assert torch.equal(slam.store.rows(i)[k], v), (i, k)

    # (c) the tie: seen from the final base pose, the new section is the frame's back-projection (to fp32 re-tie
    # rounding), and it did move away from where the erroneous pose had put it
    X = slam.store.rows(k_new)["means3D"].cpu().double().numpy()
    M = slam.w2c[b]
    tie = np.abs(X @ M[:3, :3].T + M[:3, 3] - _section(frames[b], np.eye(4))["means3D"].cpu().double().numpy()).max()
    moved = np.abs(X - _section(frames[b], np.linalg.inv(wrong))["means3D"].cpu().double().numpy()).max()
    print(f"[{mode}] tie residual {tie:.2e} m, section moved by up to {moved * 1e3:.3f} mm")
    assert tie < 1e-4 and moved > 1e-3, (tie, moved)
    # the tracker aliases the arena, so it sees the re-tied rows without a copy
    first = k_new - 1 if mode == "latest" else k_new
    assert slam.tracker.params["means3D"].data_ptr() == slam.store.rows(first, k_new)["means3D"].data_ptr()

    # (d) the loop's estimate is the solver's stepped pose
    ba = [kfs for _, kfs, do_ba in calls if do_ba]
    assert len(ba) == kw["map_iters"] and all(len(kfs) == 1 for kfs in ba)
    kf = ba[-1][0]
    assert kf["global"] is True and kf["retie_last"] == X.shape[0] and kf["id"] == b
    stepped = matrix_from_quat(kf["cam_q"].cpu().numpy(), kf["cam_t"].cpu().numpy())
    assert np.array_equal(slam.w2c[b], stepped)
    if mode == "overlap":
        entry = next(e for e in slam.keyframe_list if e["id"] == b)
        assert torch.equal(entry["est_w2c"].cpu(), torch.as_tensor(stepped, dtype=torch.float32))


def test_only_the_base_keyframe_gets_the_global_term(monkeypatch):
    """The frozen-section render and the pose step run in the section-start mapping call alone; the section's later
    mapping calls render the trainable section only, as the reference's do away from section starts."""
    map_iters = 5
    cfg = LoopConfig(track_iters=20, map_iters=map_iters, baseframe_every=4, map_every=2, track_sections=2, align_sections=2,
                     map_lrs=POSE_LRS)
    global_renders = []
    orig = MappingSolver._render_backward

    def render_backward(self, r, *a, **kw):
        if r is self.r_global:
            global_renders.append(r)
        return orig(self, r, *a, **kw)
    monkeypatch.setattr(MappingSolver, "_render_backward", render_backward)
    calls = _record_mapping(monkeypatch)
    slam = ViewTiedSLAM(W, H, K, cfg, device=DEV)
    per_frame = []
    for i, fr in enumerate(_sequence(13)[1]):
        n_render, n_call = len(global_renders), len(calls)
        slam.process(fr)
        per_frame.append((i, len(global_renders) - n_render, sum(do_ba for _, _, do_ba in calls[n_call:]),
                          [kf["global"] for _, kfs, _ in calls[n_call:] for kf in kfs]))
    for i, renders, ba_calls, flags in per_frame:
        aligned = i in (4, 8, 12)
        assert renders == (map_iters if aligned else 0) and ba_calls == (map_iters if aligned else 0), (i, renders, ba_calls)
        assert all(flags) if aligned else not any(flags), (i, flags)
    assert [a[0] for a in slam.stats["align"]] == [4, 8, 12] and [a[1] for a in slam.stats["align"]] == [[0], [0, 1], [1, 2]]


def test_aligned_runs_are_repeatable(deterministic):
    cfg = dict(track_iters=30, map_iters=6, baseframe_every=4, map_every=2, track_sections=2, align_sections=2, map_lrs=POSE_LRS)
    a = _run(LoopConfig(**cfg), 9)
    b = _run(LoopConfig(**cfg), 9)
    assert len(a.stats["align"]) == 2
    _assert_same_run(a, b)


@pytest.mark.xfail(strict=True, reason=RUNAWAY)
def test_alignment_reduces_a_known_base_pose_error():
    b = 8
    poses, frames = _sequence(b + 1)
    wrong = E @ np.linalg.inv(poses[b])
    slam = ViewTiedSLAM(W, H, K, LoopConfig(track_iters=40, map_iters=20, baseframe_every=4, map_every=2, track_sections=2,
                                            align_sections=2, map_lrs=POSE_LRS), device=DEV)
    _perturb(slam, b, wrong)
    for fr in frames:
        slam.process(fr)
    (e0, a0), (e1, a1) = _pose_error(wrong, poses[b]), _pose_error(slam.w2c[b], poses[b])
    print(f"\nbase frame {b}: centre error {e0 * 1e3:.3f} -> {e1 * 1e3:.3f} mm, rotation error {a0:.4f} -> {a1:.4f} deg")
    assert e1 < 0.5 * e0 and a1 < a0, (e0, e1, a0, a1)


@pytest.mark.xfail(strict=True, reason=RUNAWAY)
def test_alignment_lowers_the_error_of_two_section_tracking():
    """The sequence of test_gpu_slam_loop.py::test_loop_tracks_against_two_consecutive_sections: two overlapping sections
    are displaced against each other by the pose error of the newer one's base frame, which the alignment reduces."""
    n = 11
    poses = _sequence(n)[0]
    kw = dict(track_iters=50, map_iters=8, baseframe_every=4, map_every=2, track_sections=2)
    err = {}
    for align in (0, 2):
        slam = _run(LoopConfig(**kw, align_sections=align, map_lrs=POSE_LRS), n)
        err[align] = ate_rmse(np.stack([np.linalg.inv(m) for m in slam.w2c]), poses)
        print(f"\nalign_sections={align}: ATE RMSE {err[align] * 1e3:.3f} mm, corrections {slam.stats['align']}")
    assert err[2] < err[0], err
