"""CPU tests of bundle adjustment under keyframe-sharded mapping: the argument checks of `vtgs_retie_records`, the host
packing of a rank's record table, and the exchange of the tables over a 2-rank gloo group (the NCCL fallback's all-gather)
with their decoding by `ba_poses`."""
import ctypes as C
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from vtgaussian_slam_b200 import _lib
from vtgaussian_slam_b200.fused import BA_RECORDS_PER_RANK, ba_record_table, decode_ba_poses

_D = 16                         # a device address: no check dereferences it
_INVALID = -1


@pytest.fixture(scope="module")
def L():
    _lib.build()
    return _lib.lib()


def _bases(*b):
    return (C.c_uint64 * 8)(*(b or [256] * 8))


_ARG_CASES = {
    "world_zero": (lambda L: L.vtgs_retie_records(0, _bases(), 8, _D, 10, None, None), "world must be 1..8"),
    "world_nine": (lambda L: L.vtgs_retie_records(9, _bases(), 8, _D, 10, None, None), "world must be 1..8"),
    "records_per_rank": (lambda L: L.vtgs_retie_records(2, _bases(), 0, _D, 10, None, None), "records_per_rank must be >= 1"),
    "negative_rows": (lambda L: L.vtgs_retie_records(2, _bases(), 8, _D, -1, None, None), "n_rows < 0"),
    "bases_null": (lambda L: L.vtgs_retie_records(2, None, 8, _D, 10, None, None), "pointer is NULL"),
    "means_null": (lambda L: L.vtgs_retie_records(2, _bases(), 8, None, 10, _D, None), "pointer is NULL"),
    "base_zero": (lambda L: L.vtgs_retie_records(2, _bases(256, 0), 8, _D, 10, None, None),
                  "table base must be a 16-byte aligned address"),
    "base_alignment": (lambda L: L.vtgs_retie_records(2, _bases(256, 264), 8, _D, 10, None, None),
                       "table base must be a 16-byte aligned address"),
}


@pytest.mark.parametrize("case", sorted(_ARG_CASES))
def test_retie_records_argument_checks(L, case):
    call, message = _ARG_CASES[case]
    assert call(L) == _INVALID
    assert message.encode() in L.vtgs_last_error()


def test_retie_records_without_rows_or_copy_launches_nothing(L):
    # no rows and no table_out: nothing to do, so no CUDA call (returns OK on a machine without a GPU)
    assert L.vtgs_retie_records(3, _bases(), 8, None, 0, None, None) == 0


def _kf(k, n_last=0):
    kf = dict(id=k)
    if n_last:
        kf["retie_last"] = n_last
    return kf


def test_record_table_packs_headers_in_list_order():
    t = ba_record_table([_kf(7, 5), _kf(-3), _kf(2 ** 31 - 1, 100)], 100)
    assert t.shape == (BA_RECORDS_PER_RANK, _lib.BA_RECORD_WORDS) and t.dtype == torch.int32
    assert t[:3, :4].tolist() == [[1, 7, 5, 0], [1, -3, 0, 0], [1, 2 ** 31 - 1, 100, 0]]
    assert not t[:, 4:].any() and not t[3:].any()
    assert not ba_record_table([], 10).any()


@pytest.mark.parametrize("kfs, match", [
    ([dict()], "integer 'id'"),
    ([dict(id=1.5)], "integer 'id'"),
    ([_kf(1), _kf(1)], "repeated"),
    ([_kf(2 ** 31)], "does not fit 32 bits"),
    ([_kf(k) for k in range(BA_RECORDS_PER_RANK + 1)], "at most 8 keyframes"),
    ([_kf(0, 11)], "not in 0..10"),
    ([dict(id=0, retie_last=-1)], "not in 0..10"),
])
def test_record_table_refuses_bad_keyframes(kfs, match):
    with pytest.raises(ValueError, match=match):
        ba_record_table(kfs, 10)


def test_decode_refuses_an_id_twice():
    a, b = ba_record_table([_kf(4)], 10), ba_record_table([_kf(4)], 10)
    with pytest.raises(ValueError, match="id 4 appears in two"):
        decode_ba_poses(torch.stack([a, b]))


def _pose(k):
    q = torch.tensor([1.0, 0.01 * k, -0.02 * k, 0.5], dtype=torch.float32)
    t = torch.tensor([0.1 * k, -0.3, 2.0 + k], dtype=torch.float32)
    return q, t


def _worker(rank, world, store_path, ret):
    dist.init_process_group("gloo", store=dist.FileStore(store_path, world), rank=rank, world_size=world)
    # rank-major keyframes: rank r steps ids 10 r, 10 r + 1, ... (one more keyframe on rank 1)
    kfs = [_kf(10 * rank + j, 3 * j) for j in range(2 + rank)]
    table = ba_record_table(kfs, 50)
    poses = table.view(torch.float32)                     # the solver writes the poses through the same float view
    for s, kf in enumerate(kfs):
        q, t = _pose(kf["id"])
        poses[s, 4:8], poses[s, 8:11] = q + 1, t - 1
        poses[s, 11:15], poses[s, 15:18] = q, t
    gathered = torch.empty((world,) + tuple(table.shape), dtype=torch.int32)
    dist.all_gather_into_tensor(gathered.view(-1, table.shape[1]), table)
    ret[rank] = (table.clone(), gathered.clone())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_gloo_exchange_gives_every_rank_every_table(tmp_path):
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, os.path.join(tmp_path, "store"), ret), nprocs=world, join=True)
    mine = [ret[r][0] for r in range(world)]
    for r in range(world):
        assert torch.equal(ret[r][1], torch.stack(mine))  # bit for bit, in rank order, on every rank
    poses = decode_ba_poses(ret[0][1])
    assert sorted(poses) == [0, 1, 10, 11, 12]
    for k, (q, t) in poses.items():
        assert torch.equal(q, _pose(k)[0]) and torch.equal(t, _pose(k)[1])
