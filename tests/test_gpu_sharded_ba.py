"""-m gpu: bundle adjustment with re-tie under keyframe-sharded mapping on one B200.

* `vtgs_retie_records` with 1, 2 and 3 ranks simulated by separate table tensors (the kernel reads every rank's table
  through `table_bases`, as it reads the peers' symmetric blocks): bitwise the sequence of `vtgs_retie_dev` calls in
  (rank, slot) order.
* `MappingSolver` under a one-rank process group (records, all-gather, re-tie) == the unsharded solver, bit for bit.
* the keyframe checks of a sharded do_ba iteration refuse before anything is updated.
(The multi-rank exchange is run by tools/check_multi_gpu.py on 2 or more GPUs.)"""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist

from vtgaussian_slam_b200 import _lib, synthetic
from vtgaussian_slam_b200.fused import BA_RECORDS_PER_RANK, MappingSolver, retie_dev

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W = _lib.BA_RECORD_WORDS


def _table(g, rpr, records):
    """A rank's table on the device: records = [(valid, id, n_last)] with random old / new poses."""
    t = torch.zeros((rpr, W), dtype=torch.int32)
    f = t.view(torch.float32)
    for s, (valid, k, n_last) in enumerate(records):
        t[s, 0], t[s, 1], t[s, 2] = valid, k, n_last
        f[s, 4:8] = torch.randn(4, generator=g) + torch.tensor([2.0, 0, 0, 0])
        f[s, 8:11] = torch.randn(3, generator=g)
        f[s, 11:15] = f[s, 4:8] + 0.05 * torch.randn(4, generator=g)
        f[s, 15:18] = f[s, 8:11] + 0.05 * torch.randn(3, generator=g)
    return t.to(DEV)


N = 100_003                     # > one grid of 296 x 256 threads: rows are strided
_RANKS = {
    # world 1: an empty slot, an invalid record with rows, overlapping ranges, nothing reaches the first rows
    1: (8, [[(1, 0, 0), (0, 1, 50_000), (1, 2, 700), (1, 3, 90_000), (1, 4, 1)]]),
    # world 2: + a record covering every row
    2: (8, [[(1, 0, 20_000)], [(1, 1, N), (0, 2, 0), (1, 3, 33)]]),
    # world 3, 30 records each: more records than one staged chunk (64), + n_last > n_rows
    3: (30, [[(1, 10 * r + s, (7919 * (r + 1) * (s + 1)) % 60_000 * (s % 3 != 1)) for s in range(25)] for r in range(2)]
        + [[(1, 20, N + 5), (1, 21, 3)]]),
}


@pytest.mark.parametrize("world", sorted(_RANKS))
def test_retie_records_equals_sequential_retie_dev(world):
    g = torch.Generator().manual_seed(world)
    rpr, recs = _RANKS[world]
    tables = [_table(g, rpr, r) for r in recs]
    means0 = torch.randn(N, 3, generator=g).to(DEV)
    got = means0.clone()
    out = torch.full((world * rpr * W,), -1, dtype=torch.int32, device=DEV)
    bases = (C.c_uint64 * world)(*[t.data_ptr() for t in tables])
    _lib.check(_lib.lib().vtgs_retie_records(world, bases, rpr, C.c_void_p(got.data_ptr()), N, C.c_void_p(out.data_ptr()),
                                             torch.cuda.current_stream().cuda_stream))
    ref, lo = means0.clone(), N
    for t in tables:                                      # (rank, slot) order
        f = t.view(torch.float32)
        for s in range(rpr):
            valid, n_last = int(t[s, 0]), int(t[s, 2])
            if valid and n_last > 0:
                m = min(n_last, N)
                retie_dev(ref[N - m:], f[s, 4:8], f[s, 8:11], f[s, 11:15], f[s, 15:18])
                lo = min(lo, N - m)
    torch.cuda.synchronize()
    assert torch.equal(got, ref)
    assert not torch.equal(got[lo:], means0[lo:])
    assert torch.equal(got[:lo], means0[:lo])             # rows outside every range are untouched
    assert torch.equal(out, torch.cat([t.reshape(-1) for t in tables]))
    if world == 1:
        assert lo > 0


@pytest.fixture(scope="module")
def pg(tmp_path_factory):
    path = os.path.join(tmp_path_factory.mktemp("pg"), "store")
    dist.init_process_group("nccl", store=dist.FileStore(path, 1), rank=0, world_size=1)
    yield dist.group.WORLD
    dist.destroy_process_group()


def _setup():
    from vtgaussian_slam_b200.slam_loop import quat_from_matrix
    from gpu_helpers import settings_from
    poses = synthetic.trajectory(3, step_m=0.05, step_deg=2.0, seed=5)
    frames = [synthetic.make_frame("replica", 160, 96, seed=k, c2w=poses[k]) for k in range(3)]
    train = synthetic.section_gaussians(frames[2], poses[2], seed=3)
    settings = settings_from(synthetic.setup_camera(160, 96, frames[2]["K"], np.eye(4)), torch.device(DEV))
    params = {k: torch.tensor(v, device=DEV) for k, v in train.items()}

    def keyframes():
        kfs = []
        for k, fr in enumerate(frames):
            w2c = np.linalg.inv(poses[k])
            kfs.append(dict(cam_q=torch.tensor(quat_from_matrix(w2c[:3, :3]).astype(np.float32), device=DEV),
                            cam_t=torch.tensor((w2c[:3, 3] + [0.01, -0.005, 0.0]).astype(np.float32), device=DEV),
                            gt_rgb=torch.tensor(fr["im"], device=DEV), gt_depth=torch.tensor(fr["depth"], device=DEV), id=100 + k))
        return kfs
    lrs = dict(rgb_colors=0.0025, logit_opacities=0.05, log_scales=0.005, cam_unnorm_rots=1e-4, cam_trans=1e-3)
    return settings, params, keyframes, lrs


def test_sharded_solver_ba_and_retie_equals_unsharded(pg):
    settings, params, keyframes, lrs = _setup()
    N = params["means3D"].shape[0]
    runs = []
    for group in (None, pg):
        ms = MappingSolver(settings, {k: v.clone() for k, v in params.items()}, device=DEV, lrs=lrs, process_group=group,
                           deterministic=True)
        kfs = keyframes()
        kfs[1]["retie_last"], kfs[2]["retie_last"] = N // 2, N          # overlapping re-ties
        for _ in range(4):
            loss = ms.iteration(kfs, do_ba=True)
        runs.append((ms, kfs, loss.clone()))
    (ref, ref_kfs, ref_loss), (got, got_kfs, got_loss) = runs
    assert got.sharded is None                            # (one rank: the all-gather path)
    assert torch.equal(got_loss, ref_loss)
    for k in ref.params:
        assert torch.equal(got.params[k], ref.params[k]), k
    assert not torch.equal(got.params["means3D"], params["means3D"])
    for a, b in zip(ref_kfs, got_kfs):
        assert torch.equal(a["cam_q"], b["cam_q"]) and torch.equal(a["cam_t"], b["cam_t"])
    poses = got.ba_poses()
    assert sorted(poses) == [kf["id"] for kf in got_kfs]
    for kf in got_kfs:
        q, t = poses[kf["id"]]
        assert torch.equal(q, kf["cam_q"].cpu()) and torch.equal(t, kf["cam_t"].cpu())


@pytest.mark.parametrize("case", ["no_id", "repeated_id", "too_many", "retie_past_n"])
def test_sharded_ba_refusals_change_nothing(pg, case):
    settings, params, keyframes, lrs = _setup()
    N = params["means3D"].shape[0]
    ms = MappingSolver(settings, {k: v.clone() for k, v in params.items()}, device=DEV, lrs=lrs, process_group=pg)
    kfs = keyframes()
    if case == "no_id":
        del kfs[1]["id"]
    elif case == "repeated_id":
        kfs[2]["id"] = kfs[0]["id"]
    elif case == "too_many":
        kfs = [dict(kfs[0], cam_q=kfs[0]["cam_q"].clone(), id=k) for k in range(BA_RECORDS_PER_RANK + 1)]
    else:
        kfs[0]["retie_last"] = N + 1
    before = ({k: v.clone() for k, v in ms.params.items()}, [(kf["cam_q"].clone(), kf["cam_t"].clone()) for kf in kfs])
    with pytest.raises(ValueError):
        ms.iteration(kfs, do_ba=True)
    torch.cuda.synchronize()
    for k in ms.params:
        assert torch.equal(ms.params[k], before[0][k]), k
    for kf, (q, t) in zip(kfs, before[1]):
        assert torch.equal(kf["cam_q"], q) and torch.equal(kf["cam_t"], t)
        assert "_ba" not in kf
