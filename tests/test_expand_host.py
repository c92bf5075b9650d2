"""CPU-only tests of ts_expand and ts_observe_planes_items: the ctypes mirror of ts_expand_args against
the header compiled by gcc, every argument check of both entry points with its code and message
(before the n_items = 0 return), the alignment checks made before a launch, and the ValueError /
IndexError checks of BatchedTilerSliderEnv.expand and of observe_planes with items.  The pointers are
fake (non-null, 16-byte aligned) and never dereferenced: every call here has n_items = 0 or is refused
on the host."""
import ctypes
import functools
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x10000       # a non-null, 16-byte-aligned address no kernel is ever handed


def _expand_args(_lib, **kw):
    a = _lib.ExpandArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, never_win=0, n_items=0, capacity=128,
                        d_env_ids=None, d_walls=FAKE, d_targets_packed=FAKE, d_pos=FAKE, d_item_pos=None,
                        d_succ=FAKE, d_moved=FAKE, d_won=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _planes_args(_lib, **kw):
    a = _lib.ObservePlanesArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, n_targets=0, first_env=0, n_envs=0,
                               capacity=128, d_walls=FAKE, d_targets_packed=FAKE, d_pos=FAKE, dtype=_lib.OBS_F32,
                               d_out=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_expand_ctypes_mirror_matches_the_c_header(tmp_path):
    """ts_expand_args compiled as plain C by gcc has the size and field offsets of _lib.ExpandArgs, and
    the library exports both new entry points."""
    from tiler_slider_b200 import _lib
    mirror = _lib.ExpandArgs
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
             'printf("SIZEOF - %zu\\n", sizeof(ts_expand_args));']
    for field, _ in mirror._fields_:
        lines.append(f'printf("OFFSET {field} %zu\\n", offsetof(ts_expand_args, {field}));')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    # the prototypes the ctypes SYMBOLS entries mirror (compiled only: nothing is called)
    proto = tmp_path / "proto.c"
    proto.write_text('#include "tiler_slider.h"\n'
                     'int (*f)(const ts_expand_args *, void *) = ts_expand;\n'
                     'int (*g)(const ts_observe_planes_args *, const int32_t *, const uint8_t *, int64_t, void *) = ts_observe_planes_items;\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(proto), "-o", str(tmp_path / "proto.o")],
                   check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 1 + len(mirror._fields_)
    for line in out:
        kind, name, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == ctypes.sizeof(mirror)
        else:
            assert int(value) == getattr(mirror, name).offset, name
    assert _lib.SYMBOLS["ts_expand"][1][0]._type_ is mirror
    lib = _lib.lib()
    assert hasattr(lib, "ts_expand") and hasattr(lib, "ts_observe_planes_items")


def test_expand_argument_errors_before_the_empty_return():
    """Every check but alignment runs before the n_items = 0 return."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    cases = [
        (dict(size=0), -1, b"size 0"), (dict(size=17), -1, b"size 17"),
        (dict(n_tiles=-1), -2, b"n_tiles -1"), (dict(n_tiles=33), -2, b"n_tiles 33"),
        (dict(capacity=100), -3, b"capacity 100"), (dict(capacity=0), -3, b"capacity 0"), (dict(capacity=1 << 33), -3, b"too large"),
        (dict(goal_mode=2), -8, b"goal_mode 2"), (dict(goal_mode=-1), -8, b"goal_mode -1"),
        (dict(never_win=2), -8, b"never_win 2"), (dict(never_win=-1), -8, b"never_win -1"),
        (dict(n_items=-1), -6, b"n_items -1"), (dict(n_items=129), -6, b"n_items 129"),
        (dict(d_walls=None), -4, b"null device pointer"), (dict(d_targets_packed=None), -4, b"null device pointer"),
        (dict(d_succ=None), -4, b"null device pointer"), (dict(d_pos=None), -4, b"null device pointer"),
    ]
    for kw, code, msg in cases:
        assert lib.ts_expand(ctypes.byref(_expand_args(_lib, **kw)), None) == code, kw
        assert msg in lib.ts_last_error_string(), kw
    assert lib.ts_expand(None, None) == -4
    # accepted with nothing to do: any item count with ids, no d_pos when item positions are given, the
    # optional masks left out, every board class, and misaligned buffers (alignment matters only with items)
    for kw in [dict(d_env_ids=FAKE, n_items=0), dict(d_pos=None, d_item_pos=FAKE), dict(d_moved=None, d_won=None),
               dict(n_tiles=0), dict(n_tiles=32), dict(size=16, n_tiles=8), dict(goal_mode=_lib.GOAL_SET, never_win=1),
               dict(d_succ=FAKE + 4), dict(d_item_pos=FAKE + 1)]:
        assert lib.ts_expand(ctypes.byref(_expand_args(_lib, **kw)), None) == 0, kw


@pytest.mark.parametrize("field", ["d_succ", "d_item_pos"])
def test_expand_misaligned_buffers_are_refused_before_a_launch(field):
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for off in (1, 4, 8):
        a = _expand_args(_lib, n_items=4, **{"d_item_pos": FAKE, field: FAKE + off})
        assert lib.ts_expand(ctypes.byref(a), None) == -5
        assert f"{field} ".encode() in lib.ts_last_error_string() and b"not 16-byte aligned" in lib.ts_last_error_string()


def test_planes_items_argument_errors_before_the_empty_return():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    ids, ipos = None, None
    cases = [
        (dict(size=0), {}, -1, b"size 0"), (dict(size=17), {}, -1, b"size 17"),
        (dict(n_tiles=-1), {}, -2, b"n_tiles -1"), (dict(n_tiles=33), {}, -2, b"n_tiles 33"),
        (dict(capacity=100), {}, -3, b"capacity 100"), (dict(capacity=1 << 33), {}, -3, b"too large"),
        (dict(goal_mode=2), {}, -8, b"goal_mode 2"), (dict(n_targets=33), {}, -2, b"n_targets 33"),
        (dict(n_targets=-2), {}, -2, b"n_targets -2"), (dict(dtype=4), {}, -8, b"dtype 4"), (dict(dtype=-1), {}, -8, b"dtype -1"),
        ({}, dict(n=-1), -6, b"n_items -1"), ({}, dict(n=129), -6, b"n_items 129"),
        (dict(d_walls=None), {}, -4, b"null device pointer"), (dict(d_targets_packed=None), {}, -4, b"null device pointer"),
        (dict(d_pos=None), {}, -4, b"null device pointer"), (dict(d_out=None), {}, -4, b"null device pointer"),
    ]
    for kw, it, code, msg in cases:
        a = _planes_args(_lib, **kw)
        assert lib.ts_observe_planes_items(ctypes.byref(a), it.get("ids", ids), it.get("pos", ipos), it.get("n", 0), None) == code, (kw, it)
        assert msg in lib.ts_last_error_string(), (kw, it)
    assert lib.ts_observe_planes_items(None, None, None, 0, None) == -4
    # first_env / n_envs are not read; ids lift the item bound; item positions replace d_pos
    for kw, it in [(dict(first_env=2, n_envs=-7), {}), ({}, dict(ids=FAKE, n=0)), (dict(d_pos=None), dict(pos=FAKE)),
                   (dict(d_out=FAKE + 4), {}), (dict(goal_mode=_lib.GOAL_SET, n_targets=40), {})]:
        a = _planes_args(_lib, **kw)
        assert lib.ts_observe_planes_items(ctypes.byref(a), it.get("ids"), it.get("pos"), it.get("n", 0), None) == 0, (kw, it)


def test_planes_items_misaligned_buffers_are_refused_before_a_launch():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for off in (1, 4, 8):
        assert lib.ts_observe_planes_items(ctypes.byref(_planes_args(_lib, d_out=FAKE + off)), None, None, 4, None) == -5
        assert b"d_out" in lib.ts_last_error_string()
        assert lib.ts_observe_planes_items(ctypes.byref(_planes_args(_lib)), None, FAKE + off, 4, None) == -5
        assert b"d_item_pos" in lib.ts_last_error_string()


def _stub(host_io=False):
    """What expand() / observe_planes() read of a batch before their first launch (no buffers: a call
    that got past the checks would fail on the missing attributes instead of raising the tested error)."""
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    s = types.SimpleNamespace(host_io=host_io, n_envs=10, capacity=128, pos_bytes=4, size=6, plane_count=9,
                              device=torch.device("cuda", 0), _require_loaded=lambda: None)
    s._items = functools.partial(BatchedTilerSliderEnv._items, s)
    return s


@pytest.mark.parametrize("call", ["expand", "observe_planes"])
def test_item_calls_refuse_bad_ids_and_pos_before_a_launch(call):
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    f = functools.partial(getattr(BatchedTilerSliderEnv, call), _stub())
    with pytest.raises(IndexError, match=r"\[0, 10\)"):
        f(ids=[0, 10])
    with pytest.raises(IndexError):
        f(ids=torch.tensor([-1, 3]))
    with pytest.raises(IndexError):
        f(ids=range(11))
    with pytest.raises(ValueError, match="integers"):
        f(ids=[0.5, 1.0])
    with pytest.raises(ValueError, match="integers"):
        f(ids=torch.tensor([True]))
    ok = torch.zeros(10, 4, dtype=torch.uint8)
    for pos in (torch.zeros(10, 4, dtype=torch.int32), torch.zeros(10, 8, dtype=torch.uint8), torch.zeros(40, dtype=torch.uint8),
                torch.zeros(9, 4, dtype=torch.uint8), ok.numpy(), ok):     # the last two: not a tensor / not on the device
        with pytest.raises(ValueError):
            f(pos=pos)
    with pytest.raises(ValueError, match="rows"):
        f(ids=[1, 2, 3], pos=torch.zeros(2, 4, dtype=torch.uint8))
    with pytest.raises(ValueError, match="host_io"):
        getattr(BatchedTilerSliderEnv, call)(_stub(host_io=True), ids=[0])


def test_expand_refuses_bad_out_before_a_launch():
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    s = _stub()
    u8 = torch.uint8
    good = (torch.zeros(10, 4, 4, dtype=u8), torch.zeros(10, dtype=u8), torch.zeros(10, dtype=u8))
    bad = [good[:2], [good[0]], torch.zeros(10, 4, 4, dtype=u8),
           (torch.zeros(10, 4, 2, dtype=u8), good[1], good[2]), (good[0], torch.zeros(10, dtype=torch.int32), good[2]),
           (good[0], good[1], torch.zeros(11, dtype=u8)), (good[0].transpose(0, 1).contiguous().transpose(0, 1), good[1], good[2]),
           good]   # the last: right shapes, but host tensors
    for out in bad:
        with pytest.raises(ValueError):
            BatchedTilerSliderEnv.expand(s, out=out)
