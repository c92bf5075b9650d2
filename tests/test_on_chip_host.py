"""CPU tests of what the two on-chip searches share on the host: the argument checks of the batched
BFS (K6 ts_bfs_local; K9's are in test_optimal_host.py) and the shared-memory plan both front-ends
in bfs.py size their launches with."""
import ctypes as C
import types

import pytest

OK = dict(size=6, n_tiles=4, goal_mode=0, n_puzzles=8, puzzle_capacity=128, max_depth=20, bitmap_words=16, queue_smem=64,
          n_levels=256, spill_per_cta=1024, d_walls=16, d_targets_packed=16, d_init=16, d_spill=16,
          d_states_per_puzzle=16, d_solve_depth=16, d_status=16, d_levels=16, d_counters=16)
PATHS = dict(d_lengths=16, d_moves=16, d_parent_scratch=16, max_moves=8)


def _local(lib, grid=1, **kw):
    from tiler_slider_b200 import _lib
    return lib.ts_bfs_local(C.byref(_lib.BfsLocalArgs(**{**OK, **kw})), grid, None)


@pytest.mark.parametrize("kw,code", [
    (dict(size=0), -7), (dict(size=9), -7), (dict(size=17), -7),
    (dict(n_tiles=0), -7), (dict(n_tiles=5), -7),
    (dict(goal_mode=2), -8),
    (dict(bitmap_words=2), -8), (dict(bitmap_words=18), -8),
    (dict(queue_smem=16), -8), (dict(queue_smem=96), -8), (dict(spill_per_cta=-1), -8),
    (dict(n_puzzles=-1), -8), (dict(puzzle_capacity=0), -8), (dict(puzzle_capacity=100), -8),
    (dict(max_depth=-1), -8), (dict(n_levels=0), -8),
    (dict(d_walls=None), -4), (dict(d_targets_packed=None), -4), (dict(d_init=None), -4),
    (dict(d_states_per_puzzle=None), -4), (dict(d_solve_depth=None), -4), (dict(d_status=None), -4),
    (dict(d_levels=None), -4), (dict(d_counters=None), -4), (dict(d_spill=None), -4),
    ({**PATHS, "d_moves": None}, -4), ({**PATHS, "d_parent_scratch": None}, -4), ({**PATHS, "max_moves": 0}, -4),
    (dict(grid=0), -8), (dict(grid=0, n_puzzles=0), 0), (dict(grid=0, n_puzzles=0, spill_per_cta=0, d_spill=None), 0),
])
def test_bfs_local_argument_checks_without_gpu(kw, code):
    """Every argument check of ts_bfs_local returns its TS_E_* code before any CUDA call, and an
    empty batch returns 0 before the grid is looked at (the pointers of OK are never dereferenced)."""
    from tiler_slider_b200 import _lib
    assert _local(_lib.lib(), **kw) == code


def test_bfs_local_queries_check_their_arguments_without_gpu():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    got, n_sm = C.c_int(0), C.c_int(0)
    for kw, code in ((dict(size=0), -7), (dict(size=17), -7), (dict(n_tiles=5), -7), (dict(goal_mode=2), -8),
                     (dict(bitmap_words=18), -8), (dict(queue_smem=48), -8), (dict(spill_per_cta=-1), -8)):
        a = _lib.BfsLocalArgs(**{**OK, **kw})
        assert lib.ts_bfs_local_smem_bytes(C.byref(a)) == code, kw
        assert lib.ts_bfs_local_ctas_per_sm(C.byref(a), C.byref(got), C.byref(n_sm)) == code, kw
    # the plan alone is checked: launch arguments are not
    a = _lib.BfsLocalArgs(**{**OK, "n_puzzles": -1, "d_walls": None, "n_levels": 0})
    assert lib.ts_bfs_local_smem_bytes(C.byref(a)) == 4 * (16 + 64)
    assert lib.ts_bfs_local_ctas_per_sm(C.byref(a), None, C.byref(n_sm)) == -4
    assert lib.ts_bfs_local_ctas_per_sm(C.byref(a), C.byref(got), None) == -4
    assert lib.ts_bfs_local_smem_bytes(None) == -4
    assert lib.ts_bfs_local_ctas_per_sm(None, C.byref(got), C.byref(n_sm)) == -4
    assert lib.ts_bfs_local(None, 1, None) == -4


class _SmemArithmetic:
    """Stand-in for the library's occupancy queries: CTAs per SM from the shared-memory arithmetic alone
    (the bitmap and ring plus the kernel's static part and the per-CTA reservation), 148 SMs."""

    def _ctas_per_sm(self, a_ref, got_ref, n_sm_ref):
        from tiler_slider_b200.bfs import OnChipSearch
        a = a_ref._obj
        got_ref._obj.value = OnChipSearch.SMEM_PER_SM // (4 * (a.bitmap_words + a.queue_smem) + OnChipSearch.STATIC_SMEM)
        n_sm_ref._obj.value = 148
        return 0

    ts_bfs_local_ctas_per_sm = ts_optimal_moves_ctas_per_sm = _ctas_per_sm


def _planners(monkeypatch, size, n_tiles):
    """Plan-for-F functions of both front-ends, planning with _SmemArithmetic (no device, no buffers
    read).  K6 plans a range of puzzles for their most free cells: puzzle f of its table has f."""
    import contextlib
    import torch
    from tiler_slider_b200 import bfs
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(bfs, "lib", _SmemArithmetic)
    z = torch.zeros(16, dtype=torch.uint8)
    blocked = torch.arange(size * size)[None, :] >= torch.arange(size * size + 1)[:, None]     # row f: f free cells
    table = types.SimpleNamespace(size=size, n_tiles=n_tiles, goal_mode=0, never_win=False, capacity=128, device=None,
                                  _walls=z, _targets=z, _pos=z, _init=z, blocked_cells=lambda: blocked)
    k6, k9 = bfs.CudaLocalKernels(table), bfs.CudaOptimalMoves(table)
    return {"k6": lambda f: k6.plan(f, f + 1), "k9": k9.plan}, k9


@pytest.mark.parametrize("front", ["k6", "k9"])
@pytest.mark.parametrize("n_tiles", [1, 2, 3, 4])
def test_on_chip_plans_for_the_most_free_cells_that_fit(monkeypatch, n_tiles, front):
    """Both searches plan a launch for envs of up to f_max free cells with one planner, and K9 plans
    for the largest F <= f_max whose bitmap fits one CTA, never a larger one.  With 4 tiles that is
    F = 38: 38*37*36*35 bits = 221,456 B of bitmap next to a 1,024-entry ring in one CTA per SM,
    while F = 39 needs 246,752 B.  With fewer tiles every 8x8 board fits."""
    planners, k9 = _planners(monkeypatch, 8, n_tiles)
    plan = planners[front]
    fits = [f for f in range(n_tiles, 65) if plan(f) is not None]
    f_star = fits[-1]
    assert fits == list(range(n_tiles, f_star + 1))              # a larger board never fits where a smaller one does not
    assert f_star == (38 if n_tiles == 4 else 64)
    assert all(plan(f)["f_max"] == f for f in fits)
    if front == "k9":
        for f_max in range(n_tiles, 65):
            assert k9.fitting_free_cells(f_max) == min(f_max, f_star), f_max
    else:
        assert all(plan(f)["smem_bytes"] == 4 * (plan(f)["bitmap_words"] + plan(f)["queue_smem"]) for f in fits)
    if n_tiles == 4:
        p = plan(38)
        assert (p["bitmap_words"], p["queue_smem"], p["ctas_per_sm"], p["grid"]) == (221456 // 4, 1024, 1, 148)
        assert p["spill_per_cta"] == 38 * 37 * 36 * 35 + 1
        assert plan(30)["ctas_per_sm"] == 2 and plan(39) is None and plan(64) is None
