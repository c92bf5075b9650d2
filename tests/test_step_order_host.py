"""CPU-only tests of ts_step_args.order, the traversal order of a step launch: the header field and its
ctypes mirror, and the argument check ts_step makes before any CUDA call.  The pointers are fake
(non-null, 16-byte aligned) and never dereferenced: every call here is refused on the host or names
an empty range."""
import ctypes
import os
import re

FAKE = 0x10000       # a non-null, 16-byte-aligned address no kernel is ever handed
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _step_args(_lib, **kw):
    a = _lib.StepArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, first_env=0, n_envs=0, capacity=128,
                      d_walls=FAKE, d_targets_packed=FAKE, d_init=FAKE, d_pos=FAKE, d_step_count=FAKE,
                      count_bytes=1, max_steps=100, auto_reset=1, d_actions=FAKE, d_reward=FAKE, d_done=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_order_takes_the_place_of_reserved0():
    """The field sits where reserved0 was, so the struct keeps its size and every other offset."""
    from tiler_slider_b200 import _lib
    with open(os.path.join(ROOT, "include", "tiler_slider.h")) as f:
        body = re.search(r"typedef struct ts_step_args \{(.*?)\} ts_step_args;", f.read(), re.S).group(1)
    assert "int32_t count_bytes, max_steps, auto_reset, order;" in body
    assert "reserved0" not in body
    S = _lib.StepArgs
    assert [n for n, _ in S._fields_].count("order") == 1
    assert S.order.offset == S.auto_reset.offset + 4 and S.d_actions.offset == S.order.offset + 4
    assert ctypes.sizeof(S) == 152
    assert _step_args(_lib).order == 0          # existing callers that never set it walk ascending


def test_step_rejects_an_unknown_order():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for order in (2, -1, 255):
        a = _step_args(_lib, order=order)
        assert lib.ts_step(ctypes.byref(a), None) == -8          # TS_E_BAD_ARGUMENT
        assert f"order {order}".encode() in lib.ts_last_error_string()
    for order in (0, 1):                                         # an empty range is accepted either way
        assert lib.ts_step(ctypes.byref(_step_args(_lib, order=order)), None) == 0
