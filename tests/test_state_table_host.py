"""CPU tests of the state tables (K10 ts_state_table_count / ts_state_table_fill): the C-ABI struct
against its ctypes mirror, every argument check of the new entry points, and the ValueErrors and
IndexErrors BatchedTilerSliderEnv.state_table raises before it needs a device."""
import ctypes as C
import functools
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_table_ctypes_mirror_matches_the_c_header(tmp_path):
    from tiler_slider_b200 import _lib
    mirror, cname = _lib.StateTableArgs, "ts_state_table_args"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
             f'printf("SIZEOF {cname} - %zu\\n", sizeof({cname}));']
    for field, _ in mirror._fields_:
        lines.append(f'printf("OFFSET {cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 1 + len(mirror._fields_)
    for line in out:
        kind, _, field, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == C.sizeof(mirror)
        else:
            assert int(value) == getattr(mirror, field).offset, field


# pointers that are never dereferenced: every case below fails a check before any CUDA call
OK = dict(size=6, n_tiles=4, goal_mode=0, n_items=8, capacity=128, bitmap_words=16, queue_smem=64, spill_per_cta=1024,
          d_walls=16, d_targets_packed=16, d_pos=16, d_spill=16, d_counters=16, d_count=16, d_status=16,
          d_offsets=16, d_rows=16, d_distance=16, d_mask=16)

COMMON = [
    (dict(size=0), -1), (dict(size=17), -1), (dict(size=9), -7), (dict(size=16), -7),
    (dict(n_tiles=0), -7), (dict(n_tiles=5), -7), (dict(goal_mode=2), -8),
    (dict(bitmap_words=2), -8), (dict(bitmap_words=18), -8), (dict(queue_smem=16), -8), (dict(queue_smem=96), -8),
    (dict(capacity=0), -3), (dict(capacity=100), -3),
    (dict(n_items=-1), -6), (dict(n_items=129), -6),
    (dict(d_walls=None), -4), (dict(d_targets_packed=None), -4), (dict(d_pos=None), -4),
    (dict(d_counters=None), -4), (dict(d_status=None), -4),
]


def _call(entry, grid=1, **kw):
    from tiler_slider_b200 import _lib
    return getattr(_lib.lib(), entry)(C.byref(_lib.StateTableArgs(**{**OK, **kw})), grid, None)


@pytest.mark.parametrize("kw,code", COMMON + [
    (dict(spill_per_cta=0), -8), (dict(spill_per_cta=1 << 32), -8), (dict(d_spill=None), -4), (dict(d_count=None), -4),
])
def test_count_argument_checks_without_gpu(kw, code):
    assert _call("ts_state_table_count", **kw) == code


@pytest.mark.parametrize("kw,code", COMMON + [
    (dict(d_offsets=None), -4), (dict(d_rows=None), -4), (dict(d_distance=None), -4), (dict(d_mask=None), -4),
])
def test_fill_argument_checks_without_gpu(kw, code):
    assert _call("ts_state_table_fill", **kw) == code


@pytest.mark.parametrize("entry", ["ts_state_table_count", "ts_state_table_fill"])
def test_grid_and_empty_queries(entry):
    from tiler_slider_b200 import _lib
    assert _call(entry, grid=0) == -8
    assert _call(entry, grid=0, n_items=0) == 0                     # nothing to launch
    assert getattr(_lib.lib(), entry)(None, 1, None) == -4


def test_occupancy_query_checks_its_arguments_without_gpu():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    got, n_sm = C.c_int(0), C.c_int(0)
    for kw, code in ((dict(size=9), -7), (dict(size=0), -1), (dict(n_tiles=5), -7), (dict(queue_smem=48), -8)):
        a = _lib.StateTableArgs(**{**OK, **kw})
        assert lib.ts_state_table_ctas_per_sm(C.byref(a), C.byref(got), C.byref(n_sm)) == code, kw
    a = _lib.StateTableArgs(**OK)
    assert lib.ts_state_table_ctas_per_sm(C.byref(a), None, C.byref(n_sm)) == -4
    assert lib.ts_state_table_ctas_per_sm(C.byref(a), C.byref(got), None) == -4
    assert lib.ts_state_table_ctas_per_sm(None, C.byref(got), C.byref(n_sm)) == -4


def _stub(size=6, n_tiles=4, host_io=False, n_envs=8, device=torch.device("cuda", 0)):
    """A batch with no buffers: nothing past the checks may run."""
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io, n_envs=n_envs, pos_bytes=4, device=device,
                                 _require_loaded=lambda: None)
    stub._search_items = functools.partial(BatchedTilerSliderEnv._search_items, stub)
    return stub


@pytest.mark.parametrize("size,n_tiles,host_io", [(9, 2, False), (16, 4, False), (6, 0, False), (6, 5, False), (6, 4, True)])
def test_shapes_rejected_before_touching_a_device(size, n_tiles, host_io):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    with pytest.raises(ValueError, match="state_table"):
        BatchedTilerSliderEnv.state_table(_stub(size, n_tiles, host_io))


@pytest.mark.parametrize("pos,msg", [
    ([[0, 1, 2, 3]] * 8, "uint8 tensor"),                                              # not a tensor
    (torch.zeros(8, 4, dtype=torch.int32), "uint8 tensor"),
    (torch.zeros(8, 3, dtype=torch.uint8), "uint8 tensor"),
    (torch.zeros(8, 4, 1, dtype=torch.uint8), "uint8 tensor"),
    (torch.zeros(7, 4, dtype=torch.uint8), "rows"),
    (torch.zeros(8, 4, dtype=torch.uint8), "is on cpu"),                               # not on the batch's device
    (torch.zeros(16, 4, dtype=torch.uint8)[::2], "contiguous"),
])
def test_positions_are_validated(pos, msg):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = _stub()
    if msg == "contiguous":
        stub.device = torch.device("cpu")
    with pytest.raises(ValueError, match=msg):
        BatchedTilerSliderEnv.state_table(stub, None, pos)


@pytest.mark.parametrize("ids", [[0, 8], [-1, 3], [100]])
def test_ids_are_range_checked(ids):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    with pytest.raises(IndexError, match=r"\[0, 8\)"):
        BatchedTilerSliderEnv.state_table(_stub(device=torch.device("cpu")), ids)
