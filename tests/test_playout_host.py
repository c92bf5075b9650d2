"""CPU-only tests of ts_playout: the ctypes mirror of ts_playout_args against the header compiled by gcc,
every argument check with its code and message (before the n_items = 0 return), the alignment checks
made before a launch, and the ValueError / IndexError checks of BatchedTilerSliderEnv.playout.  The
pointers are fake (non-null, 16-byte aligned) and never dereferenced: every call here has n_items = 0
or is refused on the host."""
import ctypes
import functools
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x10000       # a non-null, 16-byte-aligned address no kernel is ever handed


def _args(_lib, **kw):
    a = _lib.PlayoutArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, never_win=0, policy=_lib.PLAYOUT_PLAN, n_steps=8,
                         n_items=0, capacity=128, seed=0, d_env_ids=None, d_walls=FAKE, d_targets_packed=FAKE, d_pos=FAKE,
                         d_item_pos=None, d_plan=FAKE, d_final=FAKE, d_steps=FAKE, d_won=FAKE, d_moves=FAKE, d_traj=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_playout_ctypes_mirror_matches_the_c_header(tmp_path):
    """ts_playout_args compiled as plain C by gcc has the size and field offsets of _lib.PlayoutArgs, the
    policy codes agree, the prototype is the one SYMBOLS declares, and the library exports it."""
    from tiler_slider_b200 import _lib
    mirror = _lib.PlayoutArgs
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tiler_slider.h"', 'int main(void) {',
             'printf("SIZEOF - %zu\\n", sizeof(ts_playout_args));',
             'printf("CONST PLAN %d\\n", TS_PLAYOUT_PLAN);', 'printf("CONST RANDOM %d\\n", TS_PLAYOUT_RANDOM);']
    for field, _ in mirror._fields_:
        lines.append(f'printf("OFFSET {field} %zu\\n", offsetof(ts_playout_args, {field}));')
    lines += ['return 0;', '}']
    src, exe = tmp_path / "abi.c", tmp_path / "abi"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    proto = tmp_path / "proto.c"
    proto.write_text('#include "tiler_slider.h"\nint (*f)(const ts_playout_args *, void *) = ts_playout;\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(proto), "-o", str(tmp_path / "proto.o")],
                   check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == 3 + len(mirror._fields_)
    for line in out:
        kind, name, value = line.split()
        if kind == "SIZEOF":
            assert int(value) == ctypes.sizeof(mirror)
        elif kind == "CONST":
            assert int(value) == {"PLAN": _lib.PLAYOUT_PLAN, "RANDOM": _lib.PLAYOUT_RANDOM}[name]
        else:
            assert int(value) == getattr(mirror, name).offset, name
    assert _lib.SYMBOLS["ts_playout"][1][0]._type_ is mirror
    assert hasattr(_lib.lib(), "ts_playout")


def test_playout_argument_errors_before_the_empty_return():
    """Every check but alignment runs before the n_items = 0 return."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    cases = [
        (dict(size=0), -1, b"size 0"), (dict(size=17), -1, b"size 17"),
        (dict(n_tiles=-1), -2, b"n_tiles -1"), (dict(n_tiles=33), -2, b"n_tiles 33"),
        (dict(capacity=100), -3, b"capacity 100"), (dict(capacity=0), -3, b"capacity 0"), (dict(capacity=1 << 33), -3, b"too large"),
        (dict(goal_mode=2), -8, b"goal_mode 2"), (dict(goal_mode=-1), -8, b"goal_mode -1"),
        (dict(never_win=2), -8, b"never_win 2"), (dict(never_win=-1), -8, b"never_win -1"),
        (dict(policy=2), -8, b"policy 2"), (dict(policy=-1), -8, b"policy -1"),
        (dict(n_steps=-1), -8, b"n_steps -1"),
        (dict(n_items=-1), -6, b"n_items -1"), (dict(n_items=129), -6, b"n_items 129"),
        (dict(d_walls=None), -4, b"null device pointer"), (dict(d_targets_packed=None), -4, b"null device pointer"),
        (dict(d_pos=None), -4, b"null device pointer"), (dict(d_final=None), -4, b"null device pointer"),
        (dict(d_steps=None), -4, b"null device pointer"), (dict(d_won=None), -4, b"null device pointer"),
        (dict(d_plan=None), -4, b"null device pointer"),
        # n_steps * n_items * pos_bytes past int64 (only reachable with listed ids)
        (dict(d_env_ids=FAKE, n_items=1 << 62, n_steps=1), -6, b"overflows"),
        (dict(d_env_ids=FAKE, n_items=(1 << 63) // 32 + 1, n_steps=8), -6, b"overflows"),
        # more items than one launch of 128-thread blocks covers
        (dict(d_env_ids=FAKE, n_items=(2 ** 31 - 1) * 128 + 1, n_steps=0), -6, b"items of one launch"),
    ]
    for kw, code, msg in cases:
        assert lib.ts_playout(ctypes.byref(_args(_lib, **kw)), None) == code, kw
        assert msg in lib.ts_last_error_string(), kw
    assert lib.ts_playout(None, None) == -4
    # accepted with nothing to do: the random policy without a plan, no d_pos when item positions are
    # given, the records left out, n_steps = 0, every board class, a large item count that does not
    # overflow, and misaligned buffers (alignment matters only with items)
    for kw in [dict(policy=_lib.PLAYOUT_RANDOM, d_plan=None), dict(d_pos=None, d_item_pos=FAKE), dict(d_moves=None, d_traj=None),
               dict(n_steps=0), dict(n_tiles=0), dict(n_tiles=32), dict(size=16, n_tiles=8), dict(goal_mode=_lib.GOAL_SET, never_win=1),
               dict(d_env_ids=FAKE, n_items=0, n_steps=2 ** 31 - 1), dict(d_final=FAKE + 4), dict(d_traj=FAKE + 1),
               dict(d_item_pos=FAKE + 1), dict(seed=2 ** 64 - 1)]:
        assert lib.ts_playout(ctypes.byref(_args(_lib, **kw)), None) == 0, kw


@pytest.mark.parametrize("field", ["d_final", "d_item_pos", "d_traj"])
def test_playout_misaligned_buffers_are_refused_before_a_launch(field):
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for off in (1, 4, 8):
        a = _args(_lib, n_items=4, **{"d_item_pos": FAKE, field: FAKE + off})
        assert lib.ts_playout(ctypes.byref(a), None) == -5
        assert f"{field} ".encode() in lib.ts_last_error_string() and b"not 16-byte aligned" in lib.ts_last_error_string()


def _stub(host_io=False):
    """What playout() reads of a batch before its first launch (no buffers: a call that got past the
    checks would fail on the missing attributes instead of raising the tested error)."""
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    s = types.SimpleNamespace(host_io=host_io, n_envs=10, capacity=128, pos_bytes=4, size=6,
                              device=torch.device("cuda", 0), _require_loaded=lambda: None)
    s._items = functools.partial(BatchedTilerSliderEnv._items, s)
    return s


def test_playout_refuses_bad_ids_and_pos_before_a_launch():
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    f = functools.partial(BatchedTilerSliderEnv.playout, _stub(), n_steps=4)
    with pytest.raises(IndexError, match=r"\[0, 10\)"):
        f(ids=[0, 10])
    with pytest.raises(IndexError):
        f(ids=torch.tensor([-1, 3]))
    with pytest.raises(ValueError, match="integers"):
        f(ids=[0.5, 1.0])
    ok = torch.zeros(10, 4, dtype=torch.uint8)
    for pos in (torch.zeros(10, 4, dtype=torch.int32), torch.zeros(10, 8, dtype=torch.uint8), torch.zeros(9, 4, dtype=torch.uint8),
                ok.numpy(), ok):     # the last two: not a tensor / not on the device
        with pytest.raises(ValueError):
            f(pos=pos)
    with pytest.raises(ValueError, match="host_io"):
        BatchedTilerSliderEnv.playout(_stub(host_io=True), ids=[0], n_steps=4)


def test_playout_refuses_bad_policies_before_a_launch():
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    f = functools.partial(BatchedTilerSliderEnv.playout, _stub())
    with pytest.raises(ValueError, match="n_steps"):
        f()                                                          # random without n_steps
    with pytest.raises(ValueError, match="outside"):
        f(n_steps=-1)
    with pytest.raises(ValueError, match="outside"):
        f(n_steps=2 ** 31)
    plan = torch.zeros(5, 10, dtype=torch.uint8)
    with pytest.raises(ValueError, match="not both"):
        f(actions=plan, n_steps=5)
    for bad in (plan.to(torch.int32), plan[0], torch.zeros(5, 11, dtype=torch.uint8), plan.numpy(),
                torch.zeros(10, 5, dtype=torch.uint8).t()):
        with pytest.raises(ValueError):
            f(actions=bad)                     # dtype, dimensions, item count, not a tensor, host / not contiguous
    with pytest.raises(ValueError, match="on cpu"):
        f(actions=plan)                        # right shape and dtype, but a host tensor


def test_playout_refuses_bad_out_before_a_launch():
    from tiler_slider_b200.batch_env import BatchedTilerSliderEnv
    s = _stub()
    u8, i32 = torch.uint8, torch.int32
    good = (torch.zeros(10, 4, dtype=u8), torch.zeros(10, dtype=i32), torch.zeros(10, dtype=u8))
    rec = good + (torch.zeros(6, 10, dtype=u8), torch.zeros(6, 10, 4, dtype=u8))
    bad = [good[:2], [good[0]], torch.zeros(10, 4, dtype=u8), rec,
           (torch.zeros(10, 2, dtype=u8), good[1], good[2]), (good[0], torch.zeros(10, dtype=u8), good[2]),
           (good[0], good[1], torch.zeros(11, dtype=u8)), (good[0].t().contiguous().t(), good[1], good[2]),
           good]   # the last: right shapes, but host tensors
    for out in bad:
        with pytest.raises(ValueError):
            BatchedTilerSliderEnv.playout(s, n_steps=6, out=out)
    bad_rec = [good, rec[:4], rec[:3] + (torch.zeros(5, 10, dtype=u8), rec[4]), rec[:4] + (torch.zeros(6, 10, 2, dtype=u8),),
               rec]   # the last: host tensors
    for out in bad_rec:
        with pytest.raises(ValueError):
            BatchedTilerSliderEnv.playout(s, n_steps=6, record=True, out=out)
