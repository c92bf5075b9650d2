"""CPU tests of the device-memory-bitmap searches (ts_bfs_local_gmem, ts_optimal_moves_gmem,
ts_state_table_count_gmem / _fill_gmem and their occupancy queries): the prototypes against the C
header and the ctypes argtypes, every argument check of the shared entry points through the device
ones, the checks the device ones add, the gmem plan, and the ValueErrors device_bitmap=True still
raises before it needs a device."""
import contextlib
import ctypes as C
import os
import subprocess
import types

import pytest
import torch

from tests import test_on_chip_host as k6_host
from tests import test_optimal_host as k9_host
from tests import test_state_table_host as k10_host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROTOTYPES = {   # name -> (C signature, ctypes argument struct)
    "ts_bfs_local_gmem_ctas_per_sm": ("int (*)(const ts_bfs_local_args *, int *, int *)", "BfsLocalArgs"),
    "ts_bfs_local_gmem": ("int (*)(const ts_bfs_local_args *, uint32_t *, int, void *)", "BfsLocalArgs"),
    "ts_optimal_moves_gmem_ctas_per_sm": ("int (*)(const ts_optimal_moves_args *, int *, int *)", "OptimalMovesArgs"),
    "ts_optimal_moves_gmem": ("int (*)(const ts_optimal_moves_args *, uint32_t *, int, void *)", "OptimalMovesArgs"),
    "ts_state_table_gmem_ctas_per_sm": ("int (*)(const ts_state_table_args *, int *, int *)", "StateTableArgs"),
    "ts_state_table_count_gmem": ("int (*)(const ts_state_table_args *, uint32_t *, int, void *)", "StateTableArgs"),
    "ts_state_table_fill_gmem": ("int (*)(const ts_state_table_args *, uint32_t *, int, void *)", "StateTableArgs"),
}


def test_prototypes_match_the_header_and_the_argtypes(tmp_path):
    """A C file assigns each entry point to a pointer of the documented type (gcc -Werror rejects any
    mismatch), and the ctypes argtypes are those types."""
    from tiler_slider_b200 import _lib
    lines = ['#include <stdint.h>', '#include "tiler_slider.h"']
    for k, (name, (sig, _)) in enumerate(PROTOTYPES.items()):
        lines.append(f"{sig.replace('(*)', f'(*p{k})')} = {name};")
    lines.append("int main(void) { return " + " + ".join(f"(p{k} != 0)" for k in range(len(PROTOTYPES))) + "; }")
    src = tmp_path / "proto.c"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                    "-o", str(tmp_path / "proto.o")], check=True)
    P = C.POINTER
    for name, (sig, struct) in PROTOTYPES.items():
        res, args = _lib.SYMBOLS[name]
        arg = P(getattr(_lib, struct))
        want = [arg, P(C.c_int), P(C.c_int)] if name.endswith("ctas_per_sm") else [arg, C.c_void_p, C.c_int, C.c_void_p]
        assert res is C.c_int and args == want, name


def _cases(test):
    """The (kwargs, code) table an existing host test is parametrized with."""
    mark = next(m for m in test.pytestmark if m.name == "parametrize" and m.args[0] == "kw,code")
    return mark.args[1]


# (shared entry, device entry, ctypes struct, arguments every check below starts from, cases)
ENTRIES = [
    ("ts_bfs_local", "ts_bfs_local_gmem", "BfsLocalArgs", k6_host.OK,
     _cases(k6_host.test_bfs_local_argument_checks_without_gpu)),
    ("ts_optimal_moves", "ts_optimal_moves_gmem", "OptimalMovesArgs", k9_host.OK,
     _cases(k9_host.test_optimal_moves_argument_checks_without_gpu)),
    ("ts_state_table_count", "ts_state_table_count_gmem", "StateTableArgs", k10_host.OK,
     _cases(k10_host.test_count_argument_checks_without_gpu)),
    ("ts_state_table_fill", "ts_state_table_fill_gmem", "StateTableArgs", k10_host.OK,
     _cases(k10_host.test_fill_argument_checks_without_gpu)),
]


def _call(entry, struct, base, kw, d_bitmap=16):
    """entry(args, [d_bitmap,] grid, NULL) with base + kw (grid from kw, default 1)."""
    from tiler_slider_b200 import _lib
    kw = dict(kw)
    grid = kw.pop("grid", 1)
    a = getattr(_lib, struct)(**{**base, **kw})
    fn = getattr(_lib.lib(), entry)
    return fn(C.byref(a), d_bitmap, grid, None) if entry.endswith("_gmem") else fn(C.byref(a), grid, None)


@pytest.mark.parametrize("shared,gmem,struct,ok,cases", ENTRIES, ids=[e[1] for e in ENTRIES])
def test_every_shared_check_returns_the_same_code_through_the_device_entry(shared, gmem, struct, ok, cases):
    """Each case of the shared entry point's own table that fails a check fails the same one, with
    the same code, through the device entry point (on an 8x8 four-tile shape, which it covers)."""
    checked = 0
    for kw, code in cases:
        if code == 0:
            continue                                   # passes every check: nothing to compare without a device
        base = {**ok, "size": 8, "n_tiles": 4}
        assert _call(shared, struct, base, kw) == code, kw
        assert _call(gmem, struct, base, kw) == code, kw
        checked += 1
    assert checked >= 12


@pytest.mark.parametrize("shared,gmem,struct,ok,cases", ENTRIES, ids=[e[1] for e in ENTRIES])
def test_added_checks_shape_then_buffer_then_empty_query(shared, gmem, struct, ok, cases):
    n_key = "n_puzzles" if struct == "BfsLocalArgs" else "n_items"
    for size, n_tiles in ((6, 4), (8, 3), (7, 1)):
        assert _call(gmem, struct, {**ok, "size": size, "n_tiles": n_tiles}, {}) == -7, (size, n_tiles)
    for size in (7, 8):
        base = {**ok, "size": size, "n_tiles": 4}
        assert _call(gmem, struct, base, {}, d_bitmap=None) == -4
        assert _call(gmem, struct, base, {}, d_bitmap=8) == -5
        # every added check comes before the empty-query return
        assert _call(gmem, struct, base, {n_key: 0}, d_bitmap=None) == -4
        assert _call(gmem, struct, base, {n_key: 0}, d_bitmap=8) == -5
        assert _call(gmem, struct, {**ok, "size": 6}, {n_key: 0}) == -7
        assert _call(gmem, struct, base, {n_key: 0}) == 0          # nothing to launch
    from tiler_slider_b200 import _lib
    assert getattr(_lib.lib(), gmem)(None, 16, 1, None) == -4


@pytest.mark.parametrize("query,struct,ok", [
    ("ts_bfs_local_gmem_ctas_per_sm", "BfsLocalArgs", k6_host.OK),
    ("ts_optimal_moves_gmem_ctas_per_sm", "OptimalMovesArgs", k9_host.OK),
    ("ts_state_table_gmem_ctas_per_sm", "StateTableArgs", k10_host.OK),
])
def test_occupancy_queries_check_their_arguments_without_gpu(query, struct, ok):
    from tiler_slider_b200 import _lib
    fn = getattr(_lib.lib(), query)
    got, n_sm = C.c_int(0), C.c_int(0)
    shared = query.replace("_gmem", "")
    for kw in (dict(size=0), dict(size=17), dict(n_tiles=5), dict(goal_mode=2), dict(queue_smem=48), dict(bitmap_words=18)):
        a = getattr(_lib, struct)(**{**ok, "size": 8, **kw})
        want = getattr(_lib.lib(), shared)(C.byref(a), C.byref(got), C.byref(n_sm))
        assert want < 0 and fn(C.byref(a), C.byref(got), C.byref(n_sm)) == want, kw
    a = getattr(_lib, struct)(**{**ok, "size": 8})
    assert fn(C.byref(a), None, C.byref(n_sm)) == -4
    assert fn(C.byref(a), C.byref(got), None) == -4
    assert fn(None, C.byref(got), C.byref(n_sm)) == -4
    for size, n_tiles in ((6, 4), (8, 3), (7, 1)):
        a = getattr(_lib, struct)(**{**ok, "size": size, "n_tiles": n_tiles})
        assert fn(C.byref(a), C.byref(got), C.byref(n_sm)) == -7, (size, n_tiles)


# ---- the gmem plan, with occupancy from the shared-memory arithmetic alone ---------------------------

class _Arithmetic(k6_host._SmemArithmetic):
    """The shared queries as in test_on_chip_host; the device instances' queries count the ring only
    and allow at most 5 CTAs per SM (their registers)."""

    def _gmem(self, a_ref, got_ref, n_sm_ref):
        from tiler_slider_b200.bfs import OnChipSearch
        a = a_ref._obj
        got_ref._obj.value = min(5, OnChipSearch.SMEM_PER_SM // (4 * a.queue_smem + OnChipSearch.STATIC_SMEM))
        n_sm_ref._obj.value = 148
        return 0

    ts_bfs_local_gmem_ctas_per_sm = ts_optimal_moves_gmem_ctas_per_sm = _gmem


def _planner(monkeypatch, size, n_tiles, device_bitmap):
    from tiler_slider_b200 import bfs
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(bfs, "lib", _Arithmetic)
    z = torch.zeros(16, dtype=torch.uint8)
    blocked = torch.arange(size * size)[None, :] >= torch.arange(size * size + 1)[:, None]     # row f: f free cells
    table = types.SimpleNamespace(size=size, n_tiles=n_tiles, goal_mode=0, never_win=False, capacity=128, device=None,
                                  _walls=z, _targets=z, _pos=z, _init=z, blocked_cells=lambda: blocked)
    return bfs.CudaOptimalMoves(table), bfs.CudaLocalKernels(table, device_bitmap=device_bitmap)


@pytest.mark.parametrize("size", [7, 8])
def test_gmem_plans_take_over_where_the_shared_bitmap_ends(monkeypatch, size):
    """With four tiles the shared plan ends at F* = 38; the gmem plan exists for F*+1 .. S*S, keeps its
    bitmaps within MAX_SCRATCH_BYTES, has a power-of-two ring, and is only chosen with device_bitmap."""
    from tiler_slider_b200.bfs import OnChipSearch
    k9, k6 = _planner(monkeypatch, size, 4, True)
    f_star = max(f for f in range(4, size * size + 1) if k9.plan(f) is not None)
    assert f_star == 38
    for f in range(f_star + 1, size * size + 1):
        p = k9._plan_gmem(f)
        bits = f * (f - 1) * (f - 2) * (f - 3)
        assert p["gmem"] and p["f_max"] == f and p["bitmap_words"] * 32 >= bits and p["bitmap_words"] % 4 == 0
        assert p["grid"] * p["bitmap_words"] * 4 <= OnChipSearch.MAX_SCRATCH_BYTES
        assert p["queue_smem"] >= 32 and p["queue_smem"] & (p["queue_smem"] - 1) == 0
        assert p["spill_per_cta"] == min(bits + 1, OnChipSearch.MAX_SCRATCH_BYTES // 4 // p["grid"])
        assert k9.search_plan(f, device_bitmap=True) is p
        assert k9.search_plan(f) is k9.plan(f_star)                 # default: the fitting shared plan
        q = k6.plan(f, f + 1)
        assert q["gmem"] and q["smem_bytes"] == 4 * q["queue_smem"]
    for f in range(4, f_star + 1):                                  # fits: the shared plan, keyword or not
        assert k9.search_plan(f, device_bitmap=True) is k9.plan(f) and not k9.plan(f).get("gmem")
        assert not k6.plan(f, f + 1).get("gmem")
    _, k6_default = _planner(monkeypatch, size, 4, False)
    assert k6_default.plan(f_star + 1, f_star + 2) is None


@pytest.mark.parametrize("size,n_tiles", [(6, 4), (8, 3), (5, 2)])
def test_no_gmem_plan_for_shapes_without_device_instances(monkeypatch, size, n_tiles):
    k9, k6 = _planner(monkeypatch, size, n_tiles, True)
    F = size * size
    assert k9._plan_gmem(F) is None
    assert k9.search_plan(F, device_bitmap=True) is k9.plan(k9.fitting_free_cells(F))


# ---- ValueErrors before any device use -------------------------------------------------------------

@pytest.mark.parametrize("size,n_tiles,host_io", [(9, 4, False), (8, 5, False), (8, 4, True), (7, 4, True)])
def test_device_bitmap_still_rejects_before_touching_a_device(size, n_tiles, host_io):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io)   # no buffers: nothing past the checks may run
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, device_bitmap=True)
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, [0], torch.zeros(1, 4, dtype=torch.uint8), paths=True, device_bitmap=True)
    with pytest.raises(ValueError, match="state_table"):
        BatchedTilerSliderEnv.state_table(k10_host._stub(size, n_tiles, host_io), device_bitmap=True)


@pytest.mark.parametrize("size,n_tiles", [(9, 4), (8, 5)])
def test_solvable_and_local_bfs_reject_unsupported_shapes_with_device_bitmap(size, n_tiles):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    from tiler_slider_b200.bfs import CudaLocalKernels
    with pytest.raises(ValueError, match="sizes up to 8 with 1 to 4 tiles"):
        BatchedTilerSliderEnv.solvable(8, size, n_tiles, 8, device_bitmap=True)
    with pytest.raises(ValueError, match="up to 8 with 1 to 4 tiles"):
        CudaLocalKernels(types.SimpleNamespace(size=size, n_tiles=n_tiles), device_bitmap=True)
