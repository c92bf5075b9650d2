"""CPU tests of the hash-table state tables for 5 to 8 tiles (K12 ts_state_table_count_table /
ts_state_table_fill_table and their occupancy query): the prototypes against the C header and the
ctypes argtypes, every argument check in order with its code before the empty-query return, the
table plan for a max_states bound with a stubbed occupancy query, and the ValueErrors
state_table(hash_table=True) raises before it needs a device."""
import contextlib
import ctypes as C
import functools
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROTOTYPES = {   # name -> (C signature, ctypes argtypes as names)
    "ts_state_table_table_ctas_per_sm": ("int (*)(const ts_state_table_args *, int *, int *)",
                                         ["StateTableArgs*", "int*", "int*"]),
    "ts_state_table_count_table": ("int (*)(const ts_state_table_args *, uint64_t *, int64_t, int, void *)",
                                   ["StateTableArgs*", "void*", "int64", "int", "void*"]),
    "ts_state_table_fill_table": ("int (*)(const ts_state_table_args *, uint64_t *, int64_t, int, void *)",
                                  ["StateTableArgs*", "void*", "int64", "int", "void*"]),
}


def test_prototypes_match_the_header_and_the_argtypes(tmp_path):
    """A C file assigns each entry point to a pointer of the documented type (gcc -Werror rejects any
    mismatch), and the ctypes argtypes are those types."""
    from tiler_slider_b200 import _lib
    lines = ['#include <stdint.h>', '#include "tiler_slider.h"']
    for k, (name, (sig, _)) in enumerate(PROTOTYPES.items()):
        lines.append(f"{sig.replace('(*)', f'(*p{k})')} = {name};")
    src = tmp_path / "proto.c"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                    "-o", str(tmp_path / "proto.o")], check=True)
    types_ = {"int*": C.POINTER(C.c_int), "void*": C.c_void_p, "int64": C.c_int64, "int": C.c_int}
    for name, (_, args) in PROTOTYPES.items():
        res, got = _lib.SYMBOLS[name]
        want = [C.POINTER(getattr(_lib, a[:-1])) if a[0].isupper() else types_[a] for a in args]
        assert res is C.c_int and got == want, name


# ---- K12 argument checks ----------------------------------------------------------------------------

# pointers that are never dereferenced: every case below fails a check before any CUDA call
OK = dict(size=6, n_tiles=5, goal_mode=0, n_items=8, capacity=128, bitmap_words=0, queue_smem=64, spill_per_cta=1024,
          d_walls=16, d_targets_packed=16, d_pos=16, d_spill=16, d_counters=16, d_count=16, d_status=16,
          d_offsets=16, d_rows=16, d_distance=16, d_mask=16)

# in the order the entry points check them: each case passes every check before its own
PLAN_AND_TABLE = [
    (dict(size=0), -1), (dict(size=17), -1), (dict(size=9), -7),
    (dict(n_tiles=4), -7), (dict(n_tiles=1), -7), (dict(n_tiles=9), -7),
    (dict(goal_mode=2), -8),
    (dict(bitmap_words=4), -8), (dict(bitmap_words=-4), -8), (dict(queue_smem=16), -8), (dict(queue_smem=96), -8),
    (dict(capacity=0), -3), (dict(capacity=100), -3),
    (dict(n_items=-1), -6), (dict(n_items=129), -6),
    (dict(d_walls=None), -4), (dict(d_targets_packed=None), -4), (dict(d_pos=None), -4),
    (dict(d_counters=None), -4), (dict(d_status=None), -4), (dict(grid=0), -8),
]
COUNT = PLAN_AND_TABLE + [
    (dict(spill_per_cta=0), -8), (dict(spill_per_cta=1 << 32), -8), (dict(d_spill=None), -4), (dict(d_count=None), -4),
]
FILL = PLAN_AND_TABLE + [
    (dict(d_offsets=None), -4), (dict(d_rows=None), -4), (dict(d_distance=None), -4), (dict(d_mask=None), -4),
    (dict(spill_per_cta=0), -8), (dict(spill_per_cta=1 << 32), -8), (dict(d_spill=None), -4),
]
BUFFER = [   # (struct fields, d_table, table_slots), code
    (({}, 16, 1536), -8), (({}, 16, 1024), -8), (({}, 16, 0), -8), (({}, 16, -2048), -8),
    (({}, None, 1024), -8),                              # the size before the buffer
    (({}, None, 2048), -4),
    (({}, 12, 2048), -5), ((dict(d_spill=20), 16, 2048), -5),
]


def _call(entry, kw, d_table=16, table_slots=2048):
    from tiler_slider_b200 import _lib
    kw = dict(kw)
    grid = kw.pop("grid", 1)
    a = _lib.StateTableArgs(**{**OK, **kw})
    return getattr(_lib.lib(), entry)(C.byref(a), d_table, table_slots, grid, None)


def _empty(kw):
    """The same case with no items (a case about n_items keeps its own)."""
    return kw if "n_items" in kw else {**kw, "n_items": 0}


@pytest.mark.parametrize("kw,code", COUNT)
def test_count_argument_checks_without_gpu(kw, code):
    assert _call("ts_state_table_count_table", kw) == code
    if "grid" not in kw:                                  # grid < 1 is an error with items only (K10's rule)
        assert _call("ts_state_table_count_table", _empty(kw)) == code      # before the empty-query return


@pytest.mark.parametrize("kw,code", FILL)
def test_fill_argument_checks_without_gpu(kw, code):
    assert _call("ts_state_table_fill_table", kw) == code
    if "grid" not in kw:
        assert _call("ts_state_table_fill_table", _empty(kw)) == code


@pytest.mark.parametrize("entry", ["ts_state_table_count_table", "ts_state_table_fill_table"])
@pytest.mark.parametrize("case,code", BUFFER)
def test_table_buffer_checks_without_gpu(entry, case, code):
    kw, d_table, slots = case
    assert _call(entry, kw, d_table, slots) == code
    assert _call(entry, _empty(kw), d_table, slots) == code


def test_fill_checks_the_rows_alignment_last():
    assert _call("ts_state_table_fill_table", dict(d_rows=20)) == -5
    assert _call("ts_state_table_fill_table", dict(d_rows=20, n_items=0)) == -5
    assert _call("ts_state_table_fill_table", dict(d_rows=20), d_table=None) == -4      # the table before the rows
    assert _call("ts_state_table_count_table", dict(d_rows=20, n_items=0)) == 0         # the count pass has no rows


@pytest.mark.parametrize("entry", ["ts_state_table_count_table", "ts_state_table_fill_table"])
def test_grid_and_empty_queries(entry):
    from tiler_slider_b200 import _lib
    assert _call(entry, dict(grid=0)) == -8
    assert _call(entry, dict(grid=0, n_items=0)) == 0                 # nothing to launch
    assert _call(entry, dict(n_items=0)) == 0
    assert getattr(_lib.lib(), entry)(None, 16, 2048, 1, None) == -4


def test_occupancy_query_checks_its_arguments_without_gpu():
    from tiler_slider_b200 import _lib
    fn = _lib.lib().ts_state_table_table_ctas_per_sm
    got, n_sm = C.c_int(0), C.c_int(0)
    for kw, code in ((dict(size=0), -1), (dict(size=9), -7), (dict(n_tiles=4), -7), (dict(n_tiles=9), -7),
                     (dict(goal_mode=2), -8), (dict(bitmap_words=4), -8), (dict(queue_smem=48), -8)):
        a = _lib.StateTableArgs(**{**OK, **kw})
        assert fn(C.byref(a), C.byref(got), C.byref(n_sm)) == code, kw
    a = _lib.StateTableArgs(**OK)
    assert fn(C.byref(a), None, C.byref(n_sm)) == -4
    assert fn(C.byref(a), C.byref(got), None) == -4
    assert fn(None, C.byref(got), C.byref(n_sm)) == -4


# ---- the table plan for a bound, with a stubbed occupancy query -------------------------------------

class _Occupancy:
    """ts_state_table_table_ctas_per_sm from shared memory alone (the ring), at most 5 CTAs per SM."""

    @staticmethod
    def ts_state_table_table_ctas_per_sm(a_ref, got_ref, n_sm_ref):
        from tiler_slider_b200.bfs import OnChipSearch
        a = a_ref._obj
        assert a.bitmap_words == 0 and 5 <= a.n_tiles <= 8
        got_ref._obj.value = min(5, OnChipSearch.SMEM_PER_SM // (8 * a.queue_smem + OnChipSearch.STATIC_SMEM))
        n_sm_ref._obj.value = 148
        return 0


def _planner(monkeypatch, n_tiles, **kw):
    from tiler_slider_b200 import bfs
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(bfs, "lib", lambda: _Occupancy)
    z = torch.zeros(16, dtype=torch.uint8)
    table = types.SimpleNamespace(size=6, n_tiles=n_tiles, goal_mode=0, never_win=False, capacity=128, device=None,
                                  _walls=z, _targets=z, _pos=z, _init=z)
    return bfs.CudaStateTable(table, **kw)


@pytest.mark.parametrize("max_states", [1, 2, 3, 32, 1000, 4096, 131072, 250_000, 1 << 22, 100_000_000])
@pytest.mark.parametrize("kw", [{}, dict(ctas_per_sm=1), dict(queue_smem=32)])
@pytest.mark.parametrize("n_tiles", [5, 8])
def test_plan_for_a_bound(monkeypatch, n_tiles, kw, max_states):
    from tiler_slider_b200.bfs import OnChipSearch
    p = _planner(monkeypatch, n_tiles, **kw)
    base = p._plan_table()
    got = p._plan_table(max_states)
    slots, spill, grid = got["table_slots"], got["spill_per_cta"], got["grid"]
    assert spill == max_states
    assert slots & (slots - 1) == 0 and slots >= 2 * spill and slots < 4 * spill
    assert 1 <= grid <= base["ctas_per_sm"] * 148
    assert grid * (8 * slots + 8 * spill) <= OnChipSearch.MAX_SCRATCH_BYTES            # tables and slabs within 4 GiB
    assert grid == min(base["ctas_per_sm"] * 148, OnChipSearch.MAX_SCRATCH_BYTES // (8 * slots + 8 * spill))
    assert got["table"] and got["bitmap_words"] == 0
    assert got["queue_smem"] == base["queue_smem"] and got["ctas_per_sm"] == base["ctas_per_sm"]
    assert p._plan_table(max_states) is got                                           # cached per bound
    assert p._plans[("table", max_states)] is got
    assert p._plan_table(None) is base and p._plan_table() == base                    # None: the default plan


@pytest.mark.parametrize("n_tiles", [5, 8])
def test_none_is_the_default_plan(monkeypatch, n_tiles):
    """None is _plan_table()'s own plan (the largest table within 4 GiB, half of it the bound),
    whichever bounds were planned before."""
    from tiler_slider_b200.bfs import OnChipSearch
    fresh = _planner(monkeypatch, n_tiles)._plan_table()
    p = _planner(monkeypatch, n_tiles)
    p._plan_table(4096)
    p._plan_table(1 << 20)
    got = p._plan_table(None)
    assert got == fresh and got["spill_per_cta"] * 2 == got["table_slots"]
    assert got["grid"] * 12 * (2 * got["table_slots"]) > OnChipSearch.MAX_SCRATCH_BYTES >= got["grid"] * 12 * got["table_slots"]


def test_a_bound_no_cta_can_hold_is_a_value_error(monkeypatch):
    from tiler_slider_b200.bfs import OnChipSearch
    p = _planner(monkeypatch, 5)
    big = OnChipSearch.MAX_SCRATCH_BYTES // 16             # slots 2^29 + slab: 6 GiB for one CTA
    with pytest.raises(ValueError, match="max_states"):
        p._plan_table(big)
    assert p._plan_table(big // 2)["grid"] == 1            # 2^28 slots and 2^27 entries: 3 GiB


# ---- ValueErrors before any device use -------------------------------------------------------------

def _stub(size=6, n_tiles=5, host_io=False, n_envs=8):
    """A batch with no buffers: nothing past the checks may run."""
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io, n_envs=n_envs,
                                 pos_bytes=8 if n_tiles > 4 else 4, device=torch.device("cuda", 0),
                                 _require_loaded=lambda: None)
    stub._search_items = functools.partial(BatchedTilerSliderEnv._search_items, stub)
    return stub


@pytest.mark.parametrize("stub,kw,msg", [
    (dict(n_tiles=5), {}, "1 to 4 tiles"),                                   # 5..8 tiles without hash_table
    (dict(n_tiles=8), dict(device_bitmap=True), "1 to 4 tiles"),
    (dict(n_tiles=5), dict(max_states=1000), "1 to 4 tiles"),                # max_states without hash_table
    (dict(n_tiles=4), dict(max_states=1000), "max_states"),                  # ... on a 1..4-tile batch
    (dict(n_tiles=4), dict(max_states=1000, hash_table=True), "max_states"),
    (dict(n_tiles=2), dict(max_states=1, hash_table=True), "max_states"),
    (dict(n_tiles=5), dict(max_states=0, hash_table=True), ">= 1"),
    (dict(n_tiles=8), dict(max_states=-5, hash_table=True), ">= 1"),
    (dict(size=9, n_tiles=5), dict(hash_table=True), "sizes up to 8"),
    (dict(size=16, n_tiles=8), dict(hash_table=True, max_states=64), "sizes up to 8"),
    (dict(n_tiles=9), dict(hash_table=True), "1 to 8 tiles"),
    (dict(n_tiles=5, host_io=True), dict(hash_table=True), "host_io"),
    (dict(n_tiles=8, host_io=True), dict(hash_table=True, max_states=64), "host_io"),
])
def test_state_table_rejects_before_touching_a_device(stub, kw, msg):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    with pytest.raises(ValueError, match=msg):
        BatchedTilerSliderEnv.state_table(_stub(**stub), **kw)
    with pytest.raises(ValueError, match=msg):
        BatchedTilerSliderEnv.state_table(_stub(**stub), [0, 1], torch.zeros(2, 8, dtype=torch.uint8), **kw)


@pytest.mark.parametrize("ids", [[0, 8], [-1, 3], [100]])
def test_ids_are_range_checked(ids):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = _stub()
    stub.device = torch.device("cpu")
    with pytest.raises(IndexError, match=r"\[0, 8\)"):
        BatchedTilerSliderEnv.state_table(stub, ids, hash_table=True, max_states=64)
