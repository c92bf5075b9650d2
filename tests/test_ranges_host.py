"""CPU-only tests of the range and argument checks that ts_observe and ts_step make before any
CUDA call.  The pointers are fake (non-null, 16-byte aligned) and never dereferenced: every call
here is refused on the host -- the observe calls have n_envs = 0, and the step call names a range
that is refused before dispatch."""
import ctypes

FAKE = 0x10000       # a non-null, 16-byte-aligned address no kernel is ever handed


def _observe_args(_lib, **kw):
    a = _lib.ObserveArgs(size=6, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, n_targets=0, first_env=0, n_envs=0,
                         capacity=128, d_walls=FAKE, d_targets_packed=FAKE, d_pos=FAKE, d_obs=FAKE)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_observe_rejects_more_than_32_ordered_targets():
    """Ordered targets are read as a position word of ts_pos_bytes(n_targets) bytes (at most 32):
    33 would read past the env's word and place targets from the next env's bytes."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    a = _observe_args(_lib, n_targets=33)
    assert lib.ts_observe(ctypes.byref(a), None) == -2            # TS_E_BAD_TILES
    assert b"n_targets 33" in lib.ts_last_error_string()
    a = _observe_args(_lib, n_targets=-2)
    assert lib.ts_observe(ctypes.byref(a), None) == -2
    for nt in (-1, 0, 32):                                        # the documented range
        a = _observe_args(_lib, n_targets=nt)
        assert lib.ts_observe(ctypes.byref(a), None) == 0
    a = _observe_args(_lib, n_targets=40, goal_mode=_lib.GOAL_SET)   # set goal: targets are a bitboard, n_targets unused
    assert lib.ts_observe(ctypes.byref(a), None) == 0


def test_observe_rejects_an_unknown_goal_mode():
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    for mode in (2, -1):
        a = _observe_args(_lib, goal_mode=mode)
        assert lib.ts_observe(ctypes.byref(a), None) == -8        # TS_E_BAD_ARGUMENT
        assert f"goal_mode {mode}".encode() in lib.ts_last_error_string()


def test_wide_step_refuses_ranges_past_2_to_the_32():
    """The wide step kernel (size 9..16, 1..8 tiles) indexes envs with 32 bits: a range that reaches
    2^32 is a range error (TS_E_BAD_RANGE), although the capacity itself is valid (< 2^33)."""
    from tiler_slider_b200 import _lib
    lib = _lib.lib()
    cap = (1 << 33) - 128
    a = _lib.StepArgs(size=12, n_tiles=4, goal_mode=_lib.GOAL_ORDERED, first_env=(1 << 32) - 128, n_envs=256,
                      capacity=cap, d_walls=FAKE, d_targets_packed=FAKE, d_init=FAKE, d_pos=FAKE, d_step_count=FAKE,
                      count_bytes=1, max_steps=100, auto_reset=1, d_actions=FAKE, d_reward=FAKE, d_done=FAKE)
    assert lib.ts_step(ctypes.byref(a), None) == -6                # TS_E_BAD_RANGE
    assert b"2^32" in lib.ts_last_error_string()
    a.goal_mode, a.first_env, a.n_envs = _lib.GOAL_SET, cap - 4096, 4096     # the far end of the capacity, set goal
    assert lib.ts_step(ctypes.byref(a), None) == -6
