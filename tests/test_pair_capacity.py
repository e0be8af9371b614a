"""CPU tests of the pair-buffer rule: a Workspace sizes every buffer from vtgs_workspace_query and counts its
reallocations, run_fitting repeats work until its renders fit, and the device's R / N estimate never decreases."""
import pytest
import torch

from vtgaussian_slam_b200 import _lib, rasterizer
from vtgaussian_slam_b200.rasterizer import Workspace, grown_pair_capacity, initial_pair_capacity, run_fitting

CPU = torch.device("cpu")
BUFFERS = ("geom", "tiles_touched", "tile_counts", "tile_ranges", "pair_keys", "point_list", "final_T", "n_contrib",
           "grad_geom", "counters", "region_pairs", "region_cnt", "region_masks", "region_done", "band_flags", "band_cand",
           "tile_order")


@pytest.fixture(scope="module", autouse=True)
def L():
    _lib.build()
    return _lib.lib()


def _query(ws):
    import ctypes as C
    sz = _lib.VtgsWorkspaceSizes()
    assert _lib.lib().vtgs_workspace_query(ws.W, ws.H, ws.N, ws.pair_capacity, C.byref(sz)) == 0
    return sz


def _assert_sized_from_query(ws):
    sz = _query(ws)
    for name in BUFFERS:
        assert getattr(ws, name).nbytes >= getattr(sz, name + "_bytes"), name
    assert ws.nbytes == sum(getattr(ws, name).nbytes for name in BUFFERS)


def test_workspace_buffers_follow_the_query():
    ws = Workspace(CPU, 200, 120, 5000, 3000)
    ws.ensure_grad_geom()
    _assert_sized_from_query(ws)
    gen = ws.generation
    ws.reserve_pairs(2000)                     # fits: nothing is reallocated
    assert ws.generation == gen and ws.pair_capacity == 3000
    keys = ws.pair_keys
    ws.reserve_pairs(70000)
    assert ws.generation == gen + 1 and ws.pair_capacity == 70000 and ws.pair_keys is not keys
    _assert_sized_from_query(ws)
    ws.reserve_pairs(70000)
    assert ws.generation == gen + 1


def _render(ws, R):
    """What a forward leaves in the counters: R pairs, overflow when they did not fit."""
    ws.counters[0], ws.counters[1] = R, int(R > ws.pair_capacity)


class CountingWorkspace(Workspace):
    def __init__(self, cap):
        super().__init__(CPU, 64, 48, 1000, cap)
        self.reads = 0

    def read_counters(self):
        self.reads += 1
        return super().read_counters()


def test_run_fitting_fits_the_first_time():
    ws, runs = CountingWorkspace(5000), []
    out = run_fitting(lambda: (runs.append(1), _render(ws, 4000), "out")[2], [ws])
    assert out == "out" and len(runs) == 1 and ws.reads == 1 and ws.generation == 1 and ws.pair_capacity == 5000


def test_run_fitting_regrows_once_and_returns_the_second_run():
    ws, runs, regrows = CountingWorkspace(5000), [], []

    def work():
        runs.append(ws.pair_capacity)
        _render(ws, 9000)
        return len(runs)
    assert run_fitting(work, [ws], on_regrow=lambda: regrows.append(1)) == 2
    assert runs == [5000, grown_pair_capacity(9000)] and len(regrows) == 1 and ws.generation == 2


def test_run_fitting_raises_when_the_overflow_persists():
    ws, runs = CountingWorkspace(10), []

    def work():
        runs.append(1)
        _render(ws, ws.pair_capacity + 1)
    with pytest.raises(_lib.VtgsError, match="persisted"):
        run_fitting(work, [ws], attempts=3)
    assert len(runs) == 3


def test_run_fitting_without_poll_reads_no_counters():
    ws = CountingWorkspace(10)
    run_fitting(lambda: _render(ws, 9000), [ws], poll=False)
    assert ws.reads == 0 and ws.pair_capacity == 10


def test_run_fitting_grows_only_the_renderer_that_overflowed():
    a, b = CountingWorkspace(5000), CountingWorkspace(5000)

    def work():
        _render(a, 100)
        _render(b, 8000)
    run_fitting(work, [a, b])
    assert (a.generation, a.pair_capacity) == (1, 5000)
    assert (b.generation, b.pair_capacity) == (2, grown_pair_capacity(8000))
    assert a.reads == b.reads == 2


def test_pair_estimate_never_decreases(monkeypatch):
    monkeypatch.setattr(rasterizer, "_PAIR_RATIO", {})
    ws = Workspace(CPU, 64, 48, 1000, 100)
    assert initial_pair_capacity(CPU, 1000) == 6000 + 65536          # no estimate yet: 6 pairs per Gaussian
    _render(ws, 10000)
    assert ws.read_counters()[0] == 10000 and ws.num_rendered == 10000
    high = initial_pair_capacity(CPU, 1000)
    assert high == 15000 + 65536
    _render(ws, 50)
    ws.read_counters()
    assert initial_pair_capacity(CPU, 1000) == high
