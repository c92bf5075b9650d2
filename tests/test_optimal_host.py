"""CPU tests of the optimal-move query (K9 ts_optimal_moves): the C-ABI struct against its ctypes
mirror, the argument checks of the new entry points, and the ValueErrors
BatchedTilerSliderEnv.optimal_moves raises before it needs a device (the shared-memory plan: test_on_chip_host.py)."""
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


@pytest.mark.parametrize("size,n_tiles,host_io,max_depth", [
    (9, 2, False, 20), (16, 4, False, 20), (6, 0, False, 20), (6, 5, False, 20), (6, 8, False, 20),
    (6, 4, True, 20), (6, 4, False, 0), (6, 4, False, 255),
])
def test_optimal_moves_rejects_before_touching_a_device(size, n_tiles, host_io, max_depth):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io)   # no buffers: nothing past the checks may run
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, max_depth=max_depth)
