"""ctypes front-end of the CPU oracle (oracle/ts_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module; the product package tiler_slider_b200 never does.

Every entry point names the reference code whose results it reproduces (paths relative to
the reference checkout): see the header of ts_oracle.c for the full map.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libts_oracle.so")

F_DONE, F_WON, F_INVALID, F_TIMEOUT, F_STALE = 1, 2, 4, 8, 16
DEFAULT_REWARDS = (1.0, -0.01, -0.05)  # r_win, r_step, r_invalid (repo-defined, not in the reference)


def build(force: bool = False) -> str:
    """Compile libts_oracle.so with gcc if it is missing or older than its source."""
    src = os.path.join(_HERE, "ts_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libts_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        vp, ci, cl = ctypes.c_void_p, ctypes.c_int, ctypes.c_long
        L.tso_new.restype = vp
        L.tso_new.argtypes = [ci, ci, vp, ci, vp, ci, vp, ci]
        L.tso_free.argtypes = [vp]
        L.tso_move.argtypes = [vp, ci]
        L.tso_is_won.argtypes = [vp]
        L.tso_get_locations.argtypes = [vp, vp]
        L.tso_set_locations.argtypes = [vp, vp]
        L.tso_get_move_to.argtypes = [vp, vp]
        L.tso_observe.argtypes = [vp, vp]
        L.tso_valid_moves.argtypes = [vp]
        L.tso_rollout.argtypes = [ci, ci, ci, ci, cl, ci, vp, vp, vp, vp, ci, ci,
                                  ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                  vp, vp, vp, vp, vp, vp]
        L.tso_bfs.restype = cl
        L.tso_bfs.argtypes = [vp, ci, cl, vp, vp, vp, vp]
        _lib = L
    return _lib


def _rc_array(locs: Sequence[Sequence[int]]) -> np.ndarray:
    a = np.asarray(list(locs), dtype=np.int32).reshape(-1, 2)
    return np.ascontiguousarray(a)


class OracleState:
    """One board, mirroring GameState (state.py:18-222): move / is_won / get_state_array /
    move_to / current_locations, all computed by ts_oracle.c."""

    def __init__(self, size, blocked_locations, initial_locations, target_locations, multi_color=False):
        self.size = int(size)
        self.multi_color = bool(multi_color)
        self._b = _rc_array(blocked_locations)
        self._i = _rc_array(initial_locations)
        self._t = _rc_array(target_locations)
        self.n_tiles = len(self._i)
        self.n_targets = len(self._t)
        self._h = lib().tso_new(self.size, len(self._b), self._b.ctypes.data, self.n_tiles,
                                self._i.ctypes.data, self.n_targets, self._t.ctypes.data,
                                int(self.multi_color))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.tso_free(h)

    def move(self, move: int) -> bool:
        return bool(lib().tso_move(self._h, int(move)))

    def is_won(self) -> bool:
        return bool(lib().tso_is_won(self._h))

    @property
    def current_locations(self) -> list[tuple[int, int]]:
        out = np.zeros((max(self.n_tiles, 1), 2), dtype=np.int32)
        lib().tso_get_locations(self._h, out.ctypes.data)
        return [(int(r), int(c)) for r, c in out[: self.n_tiles]]

    def set_locations(self, locs) -> None:
        a = _rc_array(locs)
        assert len(a) == self.n_tiles
        lib().tso_set_locations(self._h, a.ctypes.data)

    @property
    def move_to(self) -> np.ndarray:
        out = np.zeros((self.size, self.size, 4, 2), dtype=np.int32)
        lib().tso_get_move_to(self._h, out.ctypes.data)
        return out

    def get_state_array(self) -> np.ndarray:
        out = np.zeros((self.size, self.size, 3), dtype=np.float32)
        lib().tso_observe(self._h, out.ctypes.data)
        return out

    def valid_moves(self) -> list[int]:
        mask = lib().tso_valid_moves(self._h)
        return [d for d in range(4) if mask >> d & 1]

    def bfs(self, max_depth: int = 256, max_states: int = 1 << 22, by_level: bool = False):
        """CPU BFS over tso_move.  Returns (n_states, level_counts, solve_depth, sorted keys);
        by_level: the keys in the order their levels were reached instead (depth 0 first, each
        level sorted), so that level d is the level_counts[d] keys after those of depths < d."""
        levels = np.zeros(max_depth + 2, dtype=np.int64)
        depth = ctypes.c_int(-1)
        states = np.zeros(max_states + 4, dtype=np.uint64)
        ordered = np.zeros(max_states + 4, dtype=np.uint64) if by_level else None
        saved = self.current_locations
        n = lib().tso_bfs(self._h, max_depth, max_states, levels.ctypes.data, ctypes.byref(depth),
                          states.ctypes.data, None if ordered is None else ordered.ctypes.data)
        self.set_locations(saved)
        if n < 0:
            raise RuntimeError("oracle BFS overflow (raise max_states)")
        lv = levels.tolist()
        while lv and lv[-1] == 0:
            lv.pop()
        return int(n), lv, int(depth.value), (states if ordered is None else ordered)[:n].copy()


def rollout(S: int, multi_color: bool, blocked: np.ndarray, tiles: np.ndarray, targets: np.ndarray,
            actions: np.ndarray, max_steps: int = 100, auto_reset: bool = False,
            rewards=DEFAULT_REWARDS) -> dict:
    """Scripted batch rollout (environment.py:82-143 driven as `step; if done: reset`).

    blocked u8[N,S*S]; tiles u8[N,T,2]; targets u8[N,NT,2]; actions u8[K,N].
    Returns pos i16[K,N,T,2] (after the move, before any auto-reset), flags u8[K,N],
    count i32[K,N] (info['step_count'], pre-increment), reward f32[K,N],
    final_pos i16[N,T,2], final_count i32[N].
    """
    blocked = np.ascontiguousarray(blocked, dtype=np.uint8)
    tiles = np.ascontiguousarray(tiles, dtype=np.uint8)
    targets = np.ascontiguousarray(targets, dtype=np.uint8)
    actions = np.ascontiguousarray(actions, dtype=np.uint8)
    N = blocked.shape[0]
    assert blocked.shape == (N, S * S)
    T, NT = tiles.shape[1], targets.shape[1]
    K = actions.shape[0]
    assert actions.shape == (K, N) and tiles.shape == (N, T, 2) and targets.shape == (N, NT, 2)
    pos = np.zeros((K, N, max(T, 1), 2), dtype=np.int16)[:, :, :T]
    pos = np.ascontiguousarray(pos)
    flags = np.zeros((K, N), dtype=np.uint8)
    count = np.zeros((K, N), dtype=np.int32)
    reward = np.zeros((K, N), dtype=np.float32)
    fpos = np.ascontiguousarray(np.zeros((N, max(T, 1), 2), dtype=np.int16)[:, :T])
    fcount = np.zeros(N, dtype=np.int32)
    rc = lib().tso_rollout(S, T, NT, int(bool(multi_color)), N, K, blocked.ctypes.data,
                           tiles.ctypes.data, targets.ctypes.data, actions.ctypes.data,
                           int(max_steps), int(bool(auto_reset)), rewards[0], rewards[1], rewards[2],
                           pos.ctypes.data, flags.ctypes.data, count.ctypes.data, reward.ctypes.data,
                           fpos.ctypes.data, fcount.ctypes.data)
    assert rc == 0
    return dict(pos=pos, flags=flags, count=count, reward=reward, final_pos=fpos, final_count=fcount)
