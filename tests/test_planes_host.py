"""CPU-only tests of ts_observe_planes' C-ABI: the ctypes mirror of its argument struct against the
header compiled by gcc, the channel count of every goal mode and n_targets convention, and the
argument checks it makes before any CUDA call.  The pointers are fake (non-null, 16-byte aligned)
and never dereferenced: every call here has n_envs = 0 or is refused on the host."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x10000       # a non-null, 16-byte-aligned address no kernel is ever handed


def _planes_args(_lib, **kw):
    a = _lib.ObservePlanesArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, n_targets=0, first_env=0, n_envs=0,
                               capacity=128, d_walls=FAKE, d_targets_packed=FAKE, d_pos=FAKE, dtype=_lib.OBS_F32,
                               d_out=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_planes_ctypes_mirror_matches_the_c_header(tmp_path):
    """ts_observe_planes_args compiled as plain C by gcc has the size and field offsets of
    _lib.ObservePlanesArgs, and the dtype codes the values of _lib.OBS_*."""
    from tiler_slider_b200 import _lib
    mirror = _lib.ObservePlanesArgs
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
             'printf("SIZEOF - %zu\\n", sizeof(ts_observe_planes_args));']
    for field, _ in mirror._fields_:
        lines.append(f'printf("OFFSET {field} %zu\\n", offsetof(ts_observe_planes_args, {field}));')
    for name in ("U8", "BF16", "F16", "F32"):
        lines.append(f'printf("CODE OBS_{name} %d\\n", TS_OBS_{name});')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 1 + len(mirror._fields_) + 4
    for line in out:
        kind, name, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == ctypes.sizeof(mirror)
        elif kind == "OFFSET":
            assert int(value) == getattr(mirror, name).offset, name
        else:
            assert int(value) == getattr(_lib, name), name


@pytest.mark.parametrize("T,nt,want", [
    (4, 0, 9), (1, 0, 3), (0, 0, 1), (32, 0, 65),         # as many targets as tiles
    (3, 5, 9), (2, 32, 35), (0, 2, 3),                     # k targets of their own (never-win batches)
    (2, -1, 3), (32, -1, 33),                              # no targets
])
def test_planes_channels_ordered(T, nt, want):
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for dtype in (_lib.OBS_U8, _lib.OBS_BF16, _lib.OBS_F16, _lib.OBS_F32):
        assert lib.ts_observe_planes_channels(ctypes.byref(_planes_args(_lib, n_tiles=T, n_targets=nt, dtype=dtype))) == want


def test_planes_channels_set_goal_is_three():
    """Single colour: walls, tile cells, target cells, whatever the tile count; n_targets is unused
    (the targets are a bitboard)."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for T in (0, 1, 4, 32):
        for nt in (0, -1, 7, 40):
            assert lib.ts_observe_planes_channels(ctypes.byref(_planes_args(_lib, n_tiles=T, n_targets=nt, goal_mode=_lib.GOAL_SET))) == 3


def test_planes_channels_refuses_what_observe_planes_refuses():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    cases = [(dict(n_targets=33), -2, b"n_targets 33"), (dict(n_targets=-2), -2, b"n_targets -2"),
             (dict(n_tiles=33), -2, b"n_tiles 33"), (dict(goal_mode=2), -8, b"goal_mode 2"),
             (dict(dtype=4), -8, b"dtype 4"), (dict(dtype=-1), -8, b"dtype -1")]
    for kw, code, msg in cases:
        assert lib.ts_observe_planes_channels(ctypes.byref(_planes_args(_lib, **kw))) == code, kw
        assert msg in lib.ts_last_error_string(), kw
    assert lib.ts_observe_planes_channels(None) == -4


def test_planes_argument_errors_before_the_empty_range_return():
    """Every check but the alignment of d_out runs before the n_envs = 0 return, as in ts_observe."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    cases = [
        (dict(size=0), -1, b"size 0"), (dict(size=17), -1, b"size 17"),
        (dict(n_tiles=-1), -2, b"n_tiles -1"), (dict(n_tiles=33), -2, b"n_tiles 33"),
        (dict(capacity=100), -3, b"capacity 100"), (dict(capacity=1 << 33), -3, b"too large"),
        (dict(first_env=2), -6, b"env range"), (dict(first_env=4, n_envs=128), -6, b"env range"), (dict(n_envs=-4), -6, b"env range"),
        (dict(goal_mode=2), -8, b"goal_mode 2"), (dict(goal_mode=-1), -8, b"goal_mode -1"),
        (dict(n_targets=33), -2, b"n_targets 33"), (dict(n_targets=-2), -2, b"n_targets -2"),
        (dict(dtype=4), -8, b"dtype 4"), (dict(dtype=-1), -8, b"dtype -1"),
        (dict(d_walls=None), -4, b"null device pointer"), (dict(d_targets_packed=None), -4, b"null device pointer"),
        (dict(d_pos=None), -4, b"null device pointer"), (dict(d_out=None), -4, b"null device pointer"),
    ]
    for kw, code, msg in cases:
        a = _planes_args(_lib, **kw)
        assert lib.ts_observe_planes(ctypes.byref(a), None) == code, kw
        assert msg in lib.ts_last_error_string(), kw
    assert lib.ts_observe_planes(None, None) == -4
    # accepted with nothing to do: the documented n_targets range, any n_targets with a set goal,
    # every dtype, and a misaligned d_out (alignment is checked only when there is something to write)
    for kw in [dict(n_targets=-1), dict(n_targets=32), dict(goal_mode=_lib.GOAL_SET, n_targets=40),
               dict(dtype=_lib.OBS_U8), dict(dtype=_lib.OBS_BF16), dict(dtype=_lib.OBS_F16), dict(d_out=FAKE + 4)]:
        assert lib.ts_observe_planes(ctypes.byref(_planes_args(_lib, **kw)), None) == 0, kw


def test_planes_misaligned_out_is_refused_before_a_launch():
    """With envs to write, a d_out off 16-byte alignment is TS_E_MISALIGNED; the check comes before
    the launch, so the fake pointers are never touched."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for off in (1, 4, 8):
        a = _planes_args(_lib, n_envs=4, d_out=FAKE + off)
        assert lib.ts_observe_planes(ctypes.byref(a), None) == -5
        assert b"not 16-byte aligned" in lib.ts_last_error_string()
