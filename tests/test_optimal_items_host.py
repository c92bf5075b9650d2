"""CPU tests of optimal-move queries on items (K9 ts_optimal_moves with d_item_pos / d_plan): the
result code TS_OPT_BAD_STATE against its Python mirror, the new fields at the end of the argument
struct, the argument checks with and without them, and the ValueErrors optimal_moves(pos=) raises
before it needs a device."""
import ctypes as C
import os
import subprocess
import types

import pytest
import torch

from tests.test_optimal_host import OK, _opt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bad_state_code_and_new_fields_match_the_c_header(tmp_path):
    from tiler_slider_b200 import _lib
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join([
        '#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
        'printf("%d %zu %zu %zu %zu\\n", TS_OPT_BAD_STATE, offsetof(ts_optimal_moves_args, d_mask),',
        '       offsetof(ts_optimal_moves_args, d_item_pos), offsetof(ts_optimal_moves_args, d_plan),',
        '       sizeof(ts_optimal_moves_args));',
        'return 0;', '}']))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    code, d_mask, d_item_pos, d_plan, size = map(int, subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert code == _lib.OPT_BAD_STATE == -4
    m = _lib.OptimalMovesArgs
    # appended after d_mask: every earlier offset is what it was
    assert d_mask == m.d_mask.offset and d_item_pos == m.d_item_pos.offset == d_mask + 8
    assert d_plan == m.d_plan.offset == d_item_pos + 8 and size == C.sizeof(m) == d_plan + 8
    assert [f for f, _ in m._fields_][-3:] == ["d_mask", "d_item_pos", "d_plan"]


@pytest.mark.parametrize("kw,code", [
    (dict(size=9), -7), (dict(n_tiles=5), -7), (dict(goal_mode=2), -8), (dict(queue_smem=96), -8),
    (dict(capacity=100), -3), (dict(n_items=129), -6), (dict(max_depth=0), -8), (dict(max_depth=255), -8),
    (dict(d_pos=None), -4), (dict(d_spill=None), -4), (dict(d_distance=None), -4), (dict(d_mask=None), -4),
])
@pytest.mark.parametrize("items", [dict(d_item_pos=None, d_plan=None), dict(d_item_pos=16, d_plan=16)])
def test_argument_checks_with_and_without_items(kw, code, items):
    """The checks of ts_optimal_moves return their codes whether the new fields are NULL or set (no
    pointer is dereferenced: each case fails a check first)."""
    from tiler_slider_b200 import _lib
    assert _opt(_lib.lib(), **kw, **items) == code


def test_empty_query_with_items_returns_before_any_launch():
    from tiler_slider_b200 import _lib
    assert _opt(_lib.lib(), n_items=0, d_item_pos=16, d_plan=16) == 0


@pytest.mark.parametrize("pos,n,msg", [
    ([[0, 1, 2, 3]] * 8, 8, "uint8 tensor"),                                          # not a tensor
    (torch.zeros(8, 4, dtype=torch.int32), 8, "uint8 tensor"),
    (torch.zeros(8, 3, dtype=torch.uint8), 8, "uint8 tensor"),
    (torch.zeros(8, 4, 1, dtype=torch.uint8), 8, "uint8 tensor"),
    (torch.zeros(7, 4, dtype=torch.uint8), 8, "rows"),
    (torch.zeros(8, 4, dtype=torch.uint8), 8, "is on cpu"),                           # not on the batch's device
])
def test_item_positions_are_validated(pos, n, msg):
    from tiler_slider_b200.batch_env import check_item_pos
    with pytest.raises(ValueError, match=msg):
        check_item_pos("optimal_moves", pos, n, False, 4, torch.device("cuda", 0))


@pytest.mark.parametrize("size,n_tiles,host_io,max_depth", [(9, 2, False, 20), (6, 5, False, 20), (6, 4, True, 20),
                                                             (6, 4, False, 0), (6, 4, False, 255)])
def test_items_and_paths_reject_before_touching_a_device(size, n_tiles, host_io, max_depth):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    stub = types.SimpleNamespace(size=size, n_tiles=n_tiles, host_io=host_io)   # no buffers: nothing past the checks may run
    with pytest.raises(ValueError):
        BatchedTilerSliderEnv.optimal_moves(stub, [0], torch.zeros(1, 4, dtype=torch.uint8), max_depth=max_depth, paths=True)
