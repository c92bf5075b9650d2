"""CPU tests of the hash-table search for 5 to 8 tiles (K11 ts_optimal_moves_table and its occupancy
query) and of K7 for those tile counts (ts_synth_candidates_t8): the prototypes against the C header
and the ctypes argtypes, every argument check in order with its code before any CUDA call, the table
plan with a stubbed occupancy query, and the ValueErrors hash_table=True still raises before it needs
a device."""
import contextlib
import ctypes as C
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROTOTYPES = {   # name -> (C signature, ctypes argtypes as names)
    "ts_optimal_moves_table_ctas_per_sm": ("int (*)(const ts_optimal_moves_args *, int *, int *)",
                                           ["OptimalMovesArgs*", "int*", "int*"]),
    "ts_optimal_moves_table": ("int (*)(const ts_optimal_moves_args *, uint64_t *, int64_t, int, void *)",
                               ["OptimalMovesArgs*", "void*", "int64", "int", "void*"]),
    "ts_synth_candidates_t8": ("int (*)(const ts_synth_candidates_args *, void *)", ["SynthCandidatesArgs*", "void*"]),
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


# ---- K11 argument checks ----------------------------------------------------------------------------

OK = dict(size=6, n_tiles=5, goal_mode=0, n_items=8, capacity=128, max_depth=20, bitmap_words=0, queue_smem=64,
          spill_per_cta=1024, d_walls=16, d_targets_packed=16, d_pos=16, d_spill=16, d_counters=16, d_distance=16, d_mask=16)


def _table(kw, d_table=16, table_slots=2048):
    from tiler_slider_b200 import _lib
    kw = dict(kw)
    grid = kw.pop("grid", 1)
    a = _lib.OptimalMovesArgs(**{**OK, **kw})
    return _lib.lib().ts_optimal_moves_table(C.byref(a), d_table, table_slots, grid, None)


# in the order the entry point checks them: each case passes every check before its own
@pytest.mark.parametrize("kw,code", [
    (dict(size=0), -1), (dict(size=17), -1), (dict(size=9), -7),
    (dict(n_tiles=4), -7), (dict(n_tiles=1), -7), (dict(n_tiles=9), -7),
    (dict(goal_mode=2), -8),
    (dict(bitmap_words=4), -8), (dict(bitmap_words=-4), -8), (dict(queue_smem=16), -8), (dict(queue_smem=96), -8),
    (dict(capacity=0), -3), (dict(capacity=100), -3),
    (dict(n_items=-1), -6), (dict(n_items=129), -6),
    (dict(max_depth=0), -8), (dict(max_depth=255), -8), (dict(spill_per_cta=0), -8),
    (dict(d_walls=None), -4), (dict(d_targets_packed=None), -4), (dict(d_pos=None), -4),
    (dict(d_spill=None), -4), (dict(d_counters=None), -4), (dict(d_distance=None), -4), (dict(d_mask=None), -4),
])
def test_table_argument_checks_without_gpu(kw, code):
    """Every check of ts_optimal_moves, with its code, through the table entry point (the pointers of
    OK are never dereferenced: each case fails a check first)."""
    assert _table(kw) == code
    assert _table({**kw, "n_items": 0} if "n_items" not in kw else kw) == code     # before the empty-query return


def test_table_added_checks_size_then_buffer_then_empty_query():
    for slots in (1536, 1024, 0, -2048):                  # not a power of two, or below 2 * spill_per_cta
        assert _table({}, table_slots=slots) == -8, slots
    assert _table({}, d_table=None) == -4
    assert _table({}, d_table=8 + 4) == -5
    assert _table({"d_spill": 16 + 4}) == -5
    assert _table({}, table_slots=1024, d_table=None) == -8   # the size before the buffer
    for kw, extra in ((dict(n_items=0), dict(table_slots=1024)), (dict(n_items=0), dict(d_table=None)),
                      (dict(n_items=0), dict(d_table=12)), (dict(n_items=0, d_spill=20), {})):
        assert _table(kw, **extra) != 0, (kw, extra)      # every added check comes before the empty-query return
    assert _table(dict(n_items=0)) == 0                   # nothing to launch
    assert _table(dict(grid=0)) == -8
    from tiler_slider_b200 import _lib
    assert _lib.lib().ts_optimal_moves_table(None, 16, 2048, 1, None) == -4


def test_table_occupancy_query_checks_its_arguments_without_gpu():
    from tiler_slider_b200 import _lib
    fn = _lib.lib().ts_optimal_moves_table_ctas_per_sm
    got, n_sm = C.c_int(0), C.c_int(0)
    for kw, code in ((dict(size=0), -1), (dict(size=9), -7), (dict(n_tiles=4), -7), (dict(goal_mode=2), -8),
                     (dict(bitmap_words=4), -8), (dict(queue_smem=48), -8)):
        a = _lib.OptimalMovesArgs(**{**OK, **kw})
        assert fn(C.byref(a), C.byref(got), C.byref(n_sm)) == code, kw
    a = _lib.OptimalMovesArgs(**OK)
    assert fn(C.byref(a), None, C.byref(n_sm)) == -4
    assert fn(C.byref(a), C.byref(got), None) == -4
    assert fn(None, C.byref(got), C.byref(n_sm)) == -4


def test_synth_candidates_t8_checks_without_gpu():
    """K7 for 5..8 tiles: K7's checks with its codes, in its order, before any CUDA call; the tile
    counts each entry point covers."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    ok = dict(size=6, n_tiles=5, n_walls=8, goal_mode=0, recipe=1, walk_len=20, n_items=8, capacity=128)

    def cand(entry="ts_synth_candidates_t8", **kw):
        return getattr(lib, entry)(C.byref(_lib.SynthCandidatesArgs(**{**ok, **kw})), None)
    assert cand() == -4                                   # every shape argument fine: the buffers are missing
    assert cand(n_tiles=8) == -4 and cand(n_tiles=4) == -7 and cand(n_tiles=9) == -7 and cand(size=9) == -7
    assert cand("ts_synth_candidates") == -7 and cand("ts_synth_candidates", n_tiles=8) == -7
    assert cand(size=0) == -1 and cand(n_tiles=33) == -2 and cand(capacity=100) == -3
    assert cand(goal_mode=2) == -8 and cand(recipe=2) == -8 and cand(walk_len=-1) == -8 and cand(attempt=-1) == -8
    assert cand(n_walls=32) == -8 and cand(n_walls=31) == -4    # walk: walls + 5 tiles on 36 cells
    assert cand(n_walls=25, recipe=0, n_tiles=6) == -8 and cand(n_walls=24, recipe=0, n_tiles=6) == -4
    assert cand(size=2, n_walls=0) == -8                 # no board below 3x3 holds five tiles
    assert cand(n_items=129) == -6 and cand(env_index_base=-1) == -6
    assert lib.ts_synth_candidates_t8(None, None) == -4


# ---- the table plan, with a stubbed occupancy query --------------------------------------------------

class _Occupancy:
    """ts_optimal_moves_table_ctas_per_sm from shared memory alone (the ring), at most 5 CTAs per SM."""

    @staticmethod
    def ts_optimal_moves_table_ctas_per_sm(a_ref, got_ref, n_sm_ref):
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
    return bfs.CudaOptimalMoves(table, **kw)


@pytest.mark.parametrize("kw", [{}, dict(ctas_per_sm=1), dict(ctas_per_sm=3), dict(queue_smem=32),
                                dict(table_slots=64), dict(table_slots=1 << 12, ctas_per_sm=2)])
@pytest.mark.parametrize("n_tiles", [5, 8])
def test_table_plan_invariants(monkeypatch, n_tiles, kw):
    from tiler_slider_b200.bfs import OnChipSearch
    p = _planner(monkeypatch, n_tiles, **kw)._plan_table()
    slots, spill, grid = p["table_slots"], p["spill_per_cta"], p["grid"]
    assert p["table"] and p["bitmap_words"] == 0
    assert slots & (slots - 1) == 0 and slots >= 2 * spill and spill >= 1
    assert grid * (8 * slots + 8 * spill) <= OnChipSearch.MAX_SCRATCH_BYTES     # tables and slabs within 4 GiB
    assert grid == p["ctas_per_sm"] * 148
    assert p["queue_smem"] >= 32 and p["queue_smem"] & (p["queue_smem"] - 1) == 0
    assert (8 * p["queue_smem"] + OnChipSearch.STATIC_SMEM) * p["ctas_per_sm"] <= OnChipSearch.SMEM_PER_SM
    if "table_slots" in kw:
        assert slots == kw["table_slots"]
    else:                                                 # the largest such power of two
        assert grid * 12 * (2 * slots) > OnChipSearch.MAX_SCRATCH_BYTES
    if "ctas_per_sm" in kw:                               # the ring planned for that many CTAs; more may fit
        assert p["ctas_per_sm"] >= kw["ctas_per_sm"]
        assert p["queue_smem"] == 1 << (min(OnChipSearch.SMEM_PER_SM // kw["ctas_per_sm"] - OnChipSearch.STATIC_SMEM,
                                            64 * 1024) // 8).bit_length() - 1
    if "queue_smem" in kw:
        assert p["queue_smem"] == kw["queue_smem"]


# ---- ValueErrors before any device use -------------------------------------------------------------

@pytest.mark.parametrize("size,n_tiles,host_io,max_depth", [
    (9, 5, False, 20), (9, 4, False, 20), (6, 9, False, 20), (6, 0, False, 20),
    (6, 5, True, 20), (8, 8, True, 20), (6, 5, False, 255), (6, 5, False, 0),
])
def test_optimal_moves_hash_table_rejects_before_touching_a_device(size, n_tiles, host_io, max_depth):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io)   # no buffers: nothing past the checks may run
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, max_depth=max_depth, hash_table=True)
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, [0], torch.zeros(1, 8, dtype=torch.uint8), max_depth=max_depth,
                                            paths=True, hash_table=True)


@pytest.mark.parametrize("kw", [
    dict(size=9, n_tiles=5, n_walls=8), dict(size=6, n_tiles=9, n_walls=8), dict(size=2, n_tiles=5, n_walls=0),
    dict(size=6, n_tiles=5, n_walls=8, min_depth=4, max_depth=255, max_steps=300),
    dict(size=6, n_tiles=5, n_walls=8, min_depth=9, max_depth=8),
    dict(size=6, n_tiles=5, n_walls=8, max_depth=40, max_steps=30),
    dict(size=6, n_tiles=5, n_walls=32),
])
def test_solvable_hash_table_rejects_before_touching_a_device(kw):
    import tiler_slider_b200 as ts
    a = dict(kw)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.solvable(64, a.pop("size"), a.pop("n_tiles"), a.pop("n_walls"), True, hash_table=True, **a)


def test_without_hash_table_five_tiles_are_still_rejected():
    import tiler_slider_b200 as ts
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    with pytest.raises(ValueError, match="1 to 4 tiles"):
        BatchedTilerSliderEnv.optimal_moves(types.SimpleNamespace(size=6, n_tiles=5, host_io=False))
    with pytest.raises(ValueError, match="sizes up to 8 with 1 to 4 tiles"):
        ts.BatchedTilerSliderEnv.solvable(64, 6, 5, 8, True)
