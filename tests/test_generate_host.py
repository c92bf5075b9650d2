"""CPU tests of the puzzle generator and the reset pool: the C-ABI structs against their ctypes
mirrors, argument checks of the new entry points, the ValueErrors BatchedTilerSliderEnv.solvable
raises before it needs a device, and the Python restatement of the generator's streams."""
import ctypes as C
import os
import subprocess

import pytest

from tests import gen_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_generator_ctypes_mirrors_match_the_c_header(tmp_path):
    """ts_synth_candidates_args / ts_pool_reset_args compiled as plain C by gcc have the size and
    the field offsets of their ctypes mirrors in _lib.py."""
    from tiler_slider_b200 import _lib
    pairs = {"ts_synth_candidates_args": _lib.SynthCandidatesArgs, "ts_pool_reset_args": _lib.PoolResetArgs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {']
    for cname, mirror in pairs.items():
        lines.append(f'printf("SIZEOF {cname} - %zu\\n", sizeof({cname}));')
        for field, _ in mirror._fields_:
            lines.append(f'printf("OFFSET {cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 2 + len(_lib.SynthCandidatesArgs._fields_) + len(_lib.PoolResetArgs._fields_)
    for line in out:
        kind, cname, field, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == C.sizeof(pairs[cname]), f"sizeof({cname})"
        else:
            assert int(value) == getattr(pairs[cname], field).offset, f"{cname}.{field}"


def test_generator_argument_validation_without_gpu():
    """Shape, capacity, ranges, recipe, walk length, pool size and null pointers are checked before
    any CUDA call."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    ok = dict(size=6, n_tiles=4, n_walls=8, goal_mode=0, recipe=1, walk_len=20, n_items=8, capacity=128)

    def cand(**kw):
        return lib.ts_synth_candidates(C.byref(_lib.SynthCandidatesArgs(**{**ok, **kw})), None)
    assert cand() == -4                                   # every shape argument fine: the buffers are missing
    assert cand(size=9) == -7 and cand(n_tiles=5) == -7 and cand(n_tiles=0) == -7
    assert cand(capacity=100) == -3
    assert cand(recipe=2) == -8 and cand(walk_len=-1) == -8 and cand(walk_len=_lib.MAX_WALK + 1) == -8
    assert cand(attempt=-1) == -8 and cand(goal_mode=2) == -8
    assert cand(n_walls=33) == -8 and cand(n_walls=32) == -4   # walk: walls + 4 tiles on 36 cells
    assert cand(n_walls=29, recipe=0) == -8 and cand(n_walls=28, recipe=0) == -4
    assert cand(n_items=129) == -6 and cand(env_index_base=-1) == -6
    okp = dict(size=6, n_tiles=4, goal_mode=0, count_bytes=1, n_envs=8, capacity=128, n_pool=5, pool_capacity=128)

    def pool(**kw):
        return lib.ts_pool_reset(C.byref(_lib.PoolResetArgs(**{**okp, **kw})), None)
    assert pool() == -4
    assert pool(n_pool=0) == -8 and pool(count_bytes=2) == -8
    assert pool(pool_capacity=100) == -3 and pool(n_pool=129) == -3
    assert pool(first_env=2) == -6 and pool(n_envs=129) == -6
    assert pool(size=17) == -1 and pool(n_tiles=33) == -2


@pytest.mark.parametrize("kw", [
    dict(size=9, n_tiles=2, n_walls=4), dict(size=6, n_tiles=5, n_walls=8), dict(size=6, n_tiles=0, n_walls=8),
    dict(size=6, n_tiles=4, n_walls=8, min_depth=9, max_depth=8),
    dict(size=6, n_tiles=4, n_walls=8, max_depth=40, max_steps=30),
    dict(size=6, n_tiles=4, n_walls=8, recipe="maze"),
    dict(size=6, n_tiles=4, n_walls=8, walk_len=1 << 20),
    dict(size=4, n_tiles=4, n_walls=9, recipe="uniform"),
])
def test_solvable_rejects_before_touching_a_device(kw):
    import tiler_slider_b200 as ts
    a = dict(kw)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.solvable(64, a.pop("size"), a.pop("n_tiles"), a.pop("n_walls"), True, **a)


def test_walk_port_makes_solvable_puzzles():
    """The restated walk recipe (oracle moves) yields puzzles the oracle BFS solves."""
    from oracle import oracle as orc
    S, T, W = 6, 4, 8
    for g in range(40):
        b, tiles, targets = gen_port.candidate(orc, S, T, W, True, "walk", 20, 11, g % 3, g)
        st = orc.OracleState(S, [divmod(c, S) for c in b], tiles, targets, True)
        assert st.bfs(max_depth=64, max_states=1 << 20)[2] >= 1
        assert len(set(b) | {r * S + c for r, c in tiles}) == W + T


def test_pool_draw_is_uniform_enough():
    n_pool = 7
    counts = [0] * n_pool
    for g in range(2000):
        counts[gen_port.pool_draw(3, g, 0, n_pool)] += 1
    assert min(counts) > 200 and max(counts) < 380
