"""CPU: the parts of bench.py's contract that do not need a GPU -- the reference arm (CPU oracle port) prints one JSON
line with the agreed keys, the product arm refuses to run without CUDA (no CPU fallback), and --dump-outputs keeps
its size budget with a fixed sample.  -m gpu: the dumped outputs of the timed path themselves."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT, env=env)


def test_reference_arm_prints_the_contract_line():
    p = _run("--impl", "reference", "--small", "--steps", "1", "--warmup", "0")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "iters/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["config"]["workload"].startswith("tracking_replica_")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_uses_every_core_under_torchrun_env():
    """torchrun exports OMP_NUM_THREADS=1: the CPU arm must not inherit it (SCALE's vs_reference would be void), and its
    `config` is the product arm's config for the same --gpus."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--steps", "1", "--warmup", "0",
                        "--gpus", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.config_of(bench.build_workload("small"), 2)
    # ranks other than 0 exit without work
    env["RANK"] = "1"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--steps", "1", "--warmup", "0",
                        "--gpus", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_product_arm_fails_loudly_without_cuda():
    p = _run("--small", "--steps", "1", "--warmup", "0", "--no-cpu", timeout=300)
    assert p.returncode != 0
    assert "cuda" in (p.stderr + p.stdout).lower()


def test_steps_below_one_and_misplaced_dump_are_refused(tmp_path):
    p = _run("--small", "--steps", "0", timeout=300)
    assert p.returncode != 0 and "--steps" in p.stderr
    p = _run("--impl", "reference", "--small", "--steps", "1", "--dump-outputs", str(tmp_path), timeout=300)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr
    assert not any(tmp_path.iterdir())


def _fake_solver(W, H, N):
    g = torch.Generator().manual_seed(3)
    msg = torch.randn(16, generator=g)
    return SimpleNamespace(cam_q=torch.randn(4, generator=g), cam_t=torch.randn(3, generator=g), msg=msg,
                           loss_terms=lambda: msg[8:16], best=torch.randn(8, generator=g),
                           r=SimpleNamespace(image6=torch.rand(6, H, W, generator=g), radii=torch.arange(N + 5, dtype=torch.int32)))


def test_dump_outputs_writes_the_step_outputs_whole_within_the_budget(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    s = _fake_solver(40, 24, 1000)
    bench.dump_outputs(str(tmp_path), s, 1000)
    got = {f.stem: np.load(f) for f in tmp_path.iterdir()}
    assert set(got) == {"cam_unnorm_rot", "cam_trans", "pose_grad", "loss_terms", "best", "image6", "radii"}
    assert all(a.dtype == np.float32 for a in got.values())
    np.testing.assert_array_equal(got["image6"], s.r.image6.numpy())
    np.testing.assert_array_equal(got["radii"], np.arange(1000, dtype=np.float32))
    np.testing.assert_array_equal(got["pose_grad"], s.msg[:7].numpy())
    np.testing.assert_array_equal(got["loss_terms"], s.msg[8:].numpy())


def test_dump_outputs_samples_large_arrays_to_the_budget(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    s = _fake_solver(64, 48, 100_000)                        # 73 728 + 100 000 floats: 694 KB in full
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), s, 100_000)
    a = {f.stem: np.load(f) for f in (tmp_path / "a").iterdir()}
    b = {f.stem: np.load(f) for f in (tmp_path / "b").iterdir()}
    assert sum(x.nbytes for x in a.values()) <= 200_000
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])            # the sample is fixed
    np.testing.assert_array_equal(a["best"], s.best.numpy())  # small arrays stay whole
    r = a["radii"]
    assert r.ndim == 1 and 0 < r.size < 100_000 and np.all(np.diff(r) > 0) and r[-1] < 100_000
    assert a["image6"].ndim == 1 and np.isin(a["image6"], s.r.image6.numpy().reshape(-1)).all()


@pytest.mark.gpu
def test_dump_outputs_follow_steps_and_repeat_bitwise_in_deterministic_mode(tmp_path):
    """Two runs with the same arguments dump identical outputs (deterministic gradient accumulation); one more timed
    step moves the pose."""
    outs = {}
    for tag, steps in (("a", 3), ("b", 3), ("c", 4)):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--kernels-only", "--deterministic",
                            "--steps", str(steps), "--warmup", "0", "--dump-outputs", str(tmp_path / tag)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        outs[tag] = {f.stem: np.load(f) for f in (tmp_path / tag).iterdir()}
    assert outs["a"]["image6"].shape == (6, 170, 300) and np.isfinite(outs["a"]["image6"]).all()
    assert outs["a"]["loss_terms"][0] > 0
    for k in outs["a"]:
        np.testing.assert_array_equal(outs["a"][k], outs["b"][k], err_msg=k)
    assert not np.array_equal(outs["a"]["cam_trans"], outs["c"]["cam_trans"])
