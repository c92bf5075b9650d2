"""CPU tests of the optimal-move query (K9 ts_optimal_moves): the C-ABI struct against its ctypes
mirror, the argument checks of the new entry points, the free-cell count a launch is planned for,
and the ValueErrors BatchedTilerSliderEnv.optimal_moves raises before it needs a device."""
import ctypes as C
import os
import subprocess
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_optimal_moves_ctypes_mirror_matches_the_c_header(tmp_path):
    """ts_optimal_moves_args compiled as plain C by gcc has the size and the field offsets of its
    ctypes mirror in _lib.py, and the result codes agree."""
    from tiler_slider_b200 import _lib
    mirror, cname = _lib.OptimalMovesArgs, "ts_optimal_moves_args"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
             f'printf("SIZEOF {cname} - %zu\\n", sizeof({cname}));']
    for field, _ in mirror._fields_:
        lines.append(f'printf("OFFSET {cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines.append('printf("CODES %d %d %d %d\\n", TS_OPT_UNSOLVABLE, TS_OPT_CUTOFF, TS_OPT_NOT_SEARCHED, TS_OPT_MAX_DEPTH);')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 2 + len(mirror._fields_)
    for line in out[:-1]:
        kind, _, field, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == C.sizeof(mirror)
        else:
            assert int(value) == getattr(mirror, field).offset, field
    assert [int(x) for x in out[-1].split()[1:]] == [_lib.OPT_UNSOLVABLE, _lib.OPT_CUTOFF, _lib.OPT_NOT_SEARCHED, _lib.OPT_MAX_DEPTH]


OK = dict(size=6, n_tiles=4, goal_mode=0, n_items=8, capacity=128, max_depth=20, bitmap_words=16, queue_smem=64,
          spill_per_cta=1024, d_walls=16, d_targets_packed=16, d_pos=16, d_spill=16, d_counters=16, d_distance=16, d_mask=16)


def _opt(lib, **kw):
    from tiler_slider_b200 import _lib
    return lib.ts_optimal_moves(C.byref(_lib.OptimalMovesArgs(**{**OK, **kw})), 1, None)


@pytest.mark.parametrize("kw,code", [
    (dict(size=0), -1), (dict(size=17), -1), (dict(size=9), -7), (dict(size=16), -7),
    (dict(n_tiles=0), -7), (dict(n_tiles=5), -7),
    (dict(goal_mode=2), -8),
    (dict(bitmap_words=2), -8), (dict(bitmap_words=18), -8),
    (dict(queue_smem=16), -8), (dict(queue_smem=96), -8),
    (dict(capacity=0), -3), (dict(capacity=100), -3),
    (dict(n_items=-1), -6), (dict(n_items=129), -6),
    (dict(max_depth=0), -8), (dict(max_depth=255), -8), (dict(spill_per_cta=0), -8),
    (dict(d_walls=None), -4), (dict(d_targets_packed=None), -4), (dict(d_pos=None), -4),
    (dict(d_spill=None), -4), (dict(d_counters=None), -4), (dict(d_distance=None), -4), (dict(d_mask=None), -4),
])
def test_optimal_moves_argument_checks_without_gpu(kw, code):
    """Every argument check returns its TS_E_* code before any CUDA call (the pointers of OK are
    never dereferenced: each case fails a check first)."""
    from tiler_slider_b200 import _lib
    assert _opt(_lib.lib(), **kw) == code


def test_optimal_moves_queries_check_their_arguments_without_gpu():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    a = _lib.OptimalMovesArgs(**{**OK, "queue_smem": 48})
    got, n_sm = C.c_int(0), C.c_int(0)
    assert lib.ts_optimal_moves_smem_bytes(C.byref(a)) == -8
    assert lib.ts_optimal_moves_ctas_per_sm(C.byref(a), C.byref(got), C.byref(n_sm)) == -8
    a = _lib.OptimalMovesArgs(**OK)
    assert lib.ts_optimal_moves_smem_bytes(C.byref(a)) == 4 * (16 + 64)
    assert lib.ts_optimal_moves_ctas_per_sm(C.byref(a), None, C.byref(n_sm)) == -4
    assert lib.ts_optimal_moves_smem_bytes(None) == -4
    for kw, code in ((dict(size=9), -7), (dict(capacity=100), -3), (dict(d_walls=None), -4), (dict(n_items=-1), -6)):
        b = _lib.OptimalMovesArgs(**{**OK, **kw})
        assert lib.ts_optimal_max_free_cells(C.byref(b), 16, None) == code, kw
    assert lib.ts_optimal_max_free_cells(C.byref(a), None, None) == -4
    assert lib.ts_optimal_max_free_cells(None, 16, None) == -4


class _SmemArithmetic:
    """Stand-in for the library's occupancy query: CTAs per SM from the shared-memory arithmetic alone
    (the bitmap and ring plus the kernel's static part and the per-CTA reservation), 148 SMs."""

    def ts_optimal_moves_ctas_per_sm(self, a_ref, got_ref, n_sm_ref):
        from tiler_slider_b200.bfs import CudaOptimalMoves
        a = a_ref._obj
        got_ref._obj.value = CudaOptimalMoves.SMEM_PER_SM // (4 * (a.bitmap_words + a.queue_smem) + CudaOptimalMoves.STATIC_SMEM)
        n_sm_ref._obj.value = 148
        return 0


def _planner(monkeypatch, size, n_tiles):
    """A CudaOptimalMoves whose plans come from _SmemArithmetic (no device, no buffers read)."""
    import contextlib
    import torch
    from tiler_slider_b200.bfs import CudaOptimalMoves
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    p = object.__new__(CudaOptimalMoves)
    z = torch.zeros(16, dtype=torch.uint8)
    p.t = types.SimpleNamespace(size=size, n_tiles=n_tiles, goal_mode=0, never_win=False, capacity=128, _walls=z, _targets=z, _pos=z)
    p.lib, p.device, p.want_ctas, p.want_queue, p._plans = _SmemArithmetic(), None, None, None, {}
    return p


@pytest.mark.parametrize("n_tiles", [1, 2, 3, 4])
def test_optimal_moves_plans_for_the_most_free_cells_that_fit(monkeypatch, n_tiles):
    """A launch for envs of up to f_max free cells is planned for the largest F <= f_max whose bitmap
    fits one CTA, never a larger one.  With 4 tiles that is F = 38: 38*37*36*35 bits = 221,456 B of
    bitmap next to a 1,024-entry ring in one CTA per SM, while F = 39 needs 246,752 B.  With fewer
    tiles every 8x8 board fits."""
    p = _planner(monkeypatch, 8, n_tiles)
    fits = [f for f in range(n_tiles, 65) if p.plan(f) is not None]
    f_star = fits[-1]
    assert fits == list(range(n_tiles, f_star + 1))              # a larger board never fits where a smaller one does not
    assert f_star == (38 if n_tiles == 4 else 64)
    for f_max in range(n_tiles, 65):
        assert p.fitting_free_cells(f_max) == min(f_max, f_star), f_max
    if n_tiles == 4:
        plan = p.plan(38)
        assert (plan["bitmap_words"], plan["queue_smem"], plan["ctas_per_sm"], plan["grid"]) == (221456 // 4, 1024, 1, 148)
        assert plan["spill_per_cta"] == 38 * 37 * 36 * 35 + 1
        assert p.plan(30)["ctas_per_sm"] == 2 and p.plan(39) is None and p.plan(64) is None


@pytest.mark.parametrize("size,n_tiles,host_io,max_depth", [
    (9, 2, False, 20), (16, 4, False, 20), (6, 0, False, 20), (6, 5, False, 20), (6, 8, False, 20),
    (6, 4, True, 20), (6, 4, False, 0), (6, 4, False, 255),
])
def test_optimal_moves_rejects_before_touching_a_device(size, n_tiles, host_io, max_depth):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io)   # no buffers: nothing past the checks may run
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, max_depth=max_depth)
