"""ctypes binding of libtiler_slider.so (C-ABI declared in include/tiler_slider.h).

The library is the product: if it is missing, import of anything that computes fails
loudly -- there is no CPU or PyTorch fallback.  `build()` compiles it in-tree with nvcc for
sm_100a (tiler_slider_b200/csrc/Makefile).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# TS_LIB_PATH: load another build of the same library (kernel experiments only)
LIB_PATH = os.environ.get("TS_LIB_PATH") or os.path.join(_HERE, "libtiler_slider.so")
CSRC = os.path.join(_HERE, "csrc")

CAP_ALIGN = 128
MAX_SIZE = 16
MAX_TILES = 32        # 0..8: register kernels; 9..32: per-env generic kernels
F_DONE, F_WON, F_INVALID, F_TIMEOUT, F_STALE = 1, 2, 4, 8, 16
GOAL_ORDERED, GOAL_SET = 0, 1
RECIPE_UNIFORM, RECIPE_WALK = 0, 1
MAX_WALK = 65535
OPT_UNSOLVABLE, OPT_CUTOFF, OPT_NOT_SEARCHED, OPT_BAD_STATE = -1, -2, -3, -4
OPT_MAX_DEPTH = 254
OBS_U8, OBS_BF16, OBS_F16, OBS_F32 = 0, 1, 2, 3
PLAYOUT_PLAN, PLAYOUT_RANDOM = 0, 1

_vp, _i32, _i64, _f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class EncodeArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("n_targets", _i32), ("goal_mode", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_blocked", _vp), ("d_tiles", _vp), ("d_targets", _vp),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_pos", _vp)]


class SynthArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("n_walls", _i32), ("goal_mode", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64), ("env_index_base", _i64),
                ("seed", C.c_uint64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_pos", _vp)]


class StepArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_pos", _vp),
                ("d_step_count", _vp),
                ("count_bytes", _i32), ("max_steps", _i32), ("auto_reset", _i32), ("order", _i32),
                ("d_actions", _vp),
                ("r_win", _f32), ("r_step", _f32), ("r_invalid", _f32), ("reserved1", _f32),
                ("d_reward", _vp), ("d_done", _vp), ("d_flags", _vp), ("d_terminal_pos", _vp)]


class ObserveArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("n_targets", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp), ("d_obs", _vp)]


class ObservePlanesArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("n_targets", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp),
                ("dtype", _i32), ("reserved0", _i32), ("d_out", _vp)]


class ExpandArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("n_items", _i64), ("capacity", _i64),
                ("d_env_ids", _vp), ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp), ("d_item_pos", _vp),
                ("d_succ", _vp), ("d_moved", _vp), ("d_won", _vp)]


class PlayoutArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("policy", _i32), ("n_steps", _i32), ("n_items", _i64), ("capacity", _i64), ("seed", C.c_uint64),
                ("d_env_ids", _vp), ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp), ("d_item_pos", _vp),
                ("d_plan", _vp), ("d_final", _vp), ("d_steps", _vp), ("d_won", _vp), ("d_moves", _vp), ("d_traj", _vp)]


class ValidArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_walls", _vp), ("d_pos", _vp), ("d_mask", _vp)]


class GoalArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64),
                ("d_targets_packed", _vp), ("d_pos", _vp), ("d_won", _vp)]


class BfsArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32), ("n_ranks", _i32),
                ("rank", _i32),
                ("n_items", _i64), ("puzzle_capacity", _i64), ("table_capacity", _i64), ("out_capacity", _i64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_in_keys", _vp),
                ("d_out_keys", _vp), ("d_table", _vp), ("d_counts", _vp),
                ("d_parent_keys", _vp), ("d_table_parent", _vp), ("d_moves", _vp), ("d_lengths", _vp),
                ("max_moves", _i64), ("d_won_keys", _vp), ("won_capacity", _i64),
                ("d_states_per_puzzle", _vp), ("d_solve_depth", _vp), ("d_goal_keys", _vp),
                ("depth", _i32), ("reserved2", _i32),
                ("d_peer_bufs", _vp), ("inbox_capacity", _i64), ("parity", _i32), ("parent_per_item", _i32),
                ("d_n_items", _vp), ("n_items_scale", _i64), ("d_out_parents", _vp), ("d_goal_parents", _vp)]


class BfsLocalArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("n_puzzles", _i64), ("puzzle_capacity", _i64),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_puzzle_ids", _vp),
                ("max_depth", _i32), ("bitmap_words", _i32), ("queue_smem", _i32), ("n_levels", _i32),
                ("d_spill", _vp), ("spill_per_cta", _i64), ("d_parent_scratch", _vp),
                ("d_states_per_puzzle", _vp), ("d_solve_depth", _vp), ("d_status", _vp),
                ("d_levels", _vp), ("d_counters", _vp), ("d_moves", _vp), ("d_lengths", _vp), ("max_moves", _i64)]


class SynthCandidatesArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("n_walls", _i32), ("goal_mode", _i32),
                ("recipe", _i32), ("walk_len", _i32), ("attempt", _i32), ("reserved0", _i32),
                ("n_items", _i64), ("capacity", _i64), ("env_index_base", _i64), ("seed", C.c_uint64),
                ("d_env_ids", _vp), ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_pos", _vp)]


class PoolResetArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("count_bytes", _i32),
                ("first_env", _i64), ("n_envs", _i64), ("capacity", _i64), ("env_index_base", _i64),
                ("seed", C.c_uint64), ("d_done", _vp), ("d_episode", _vp),
                ("d_walls", _vp), ("d_targets_packed", _vp), ("d_init", _vp), ("d_pos", _vp),
                ("d_step_count", _vp), ("d_solve_depth", _vp), ("n_pool", _i64), ("pool_capacity", _i64),
                ("d_pool_walls", _vp), ("d_pool_targets", _vp), ("d_pool_init", _vp), ("d_pool_depth", _vp)]


class OptimalMovesArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("n_items", _i64), ("capacity", _i64),
                ("d_env_ids", _vp), ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp),
                ("max_depth", _i32), ("bitmap_words", _i32), ("queue_smem", _i32), ("reserved0", _i32),
                ("d_spill", _vp), ("spill_per_cta", _i64), ("d_counters", _vp), ("d_distance", _vp), ("d_mask", _vp),
                ("d_item_pos", _vp), ("d_plan", _vp)]


class StateTableArgs(C.Structure):
    _fields_ = [("size", _i32), ("n_tiles", _i32), ("goal_mode", _i32), ("never_win", _i32),
                ("n_items", _i64), ("capacity", _i64),
                ("d_env_ids", _vp), ("d_walls", _vp), ("d_targets_packed", _vp), ("d_pos", _vp), ("d_item_pos", _vp),
                ("bitmap_words", _i32), ("queue_smem", _i32), ("d_spill", _vp), ("spill_per_cta", _i64),
                ("d_counters", _vp), ("d_count", _vp), ("d_status", _vp), ("d_offsets", _vp),
                ("d_rows", _vp), ("d_distance", _vp), ("d_mask", _vp)]


# every symbol include/tiler_slider.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "ts_version": (C.c_int, []),
    "ts_last_error_string": (C.c_char_p, []),
    "ts_pos_bytes": (C.c_int, [C.c_int]),
    "ts_board_bytes": (C.c_int, [C.c_int]),
    "ts_board_stride": (C.c_int, [C.c_int]),
    "ts_pos_stride": (C.c_int, [C.c_int]),
    "ts_walls_bytes": (C.c_int, [C.c_int]),
    "ts_target_board_bytes": (C.c_int, [C.c_int]),
    "ts_plane_count": (C.c_int, [C.c_int]),
    "ts_plane_width": (C.c_int, [C.c_int, C.c_int]),
    "ts_plane_offset": (C.c_int, [C.c_int, C.c_int]),
    "ts_supported": (C.c_int, [C.c_int, C.c_int]),
    "ts_encode": (C.c_int, [C.POINTER(EncodeArgs), _vp]),
    "ts_synth": (C.c_int, [C.POINTER(SynthArgs), _vp]),
    "ts_step": (C.c_int, [C.POINTER(StepArgs), _vp]),
    "ts_observe": (C.c_int, [C.POINTER(ObserveArgs), _vp]),
    "ts_observe_planes_channels": (C.c_int, [C.POINTER(ObservePlanesArgs)]),
    "ts_observe_planes": (C.c_int, [C.POINTER(ObservePlanesArgs), _vp]),
    "ts_observe_planes_items": (C.c_int, [C.POINTER(ObservePlanesArgs), _vp, _vp, _i64, _vp]),
    "ts_expand": (C.c_int, [C.POINTER(ExpandArgs), _vp]),
    "ts_playout": (C.c_int, [C.POINTER(PlayoutArgs), _vp]),
    "ts_valid_moves": (C.c_int, [C.POINTER(ValidArgs), _vp]),
    "ts_goal_check": (C.c_int, [C.POINTER(GoalArgs), _vp]),
    "ts_bfs_seed": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_expand": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_expand_exchange": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_levels": (C.c_int, [C.POINTER(BfsArgs), C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, C.c_int64, C.c_int64, _vp]),
    "ts_bfs_partition_count": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_partition_scatter": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_hash_insert": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_traceback": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_trace_step": (C.c_int, [C.POINTER(BfsArgs), _vp]),
    "ts_bfs_local_smem_bytes": (C.c_int, [C.POINTER(BfsLocalArgs)]),
    "ts_bfs_local_ctas_per_sm": (C.c_int, [C.POINTER(BfsLocalArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_bfs_local": (C.c_int, [C.POINTER(BfsLocalArgs), C.c_int, _vp]),
    "ts_bfs_local_gmem_ctas_per_sm": (C.c_int, [C.POINTER(BfsLocalArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_bfs_local_gmem": (C.c_int, [C.POINTER(BfsLocalArgs), _vp, C.c_int, _vp]),
    "ts_synth_candidates": (C.c_int, [C.POINTER(SynthCandidatesArgs), _vp]),
    "ts_synth_candidates_t8": (C.c_int, [C.POINTER(SynthCandidatesArgs), _vp]),
    "ts_pool_reset": (C.c_int, [C.POINTER(PoolResetArgs), _vp]),
    "ts_optimal_moves_smem_bytes": (C.c_int, [C.POINTER(OptimalMovesArgs)]),
    "ts_optimal_moves_ctas_per_sm": (C.c_int, [C.POINTER(OptimalMovesArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_optimal_max_free_cells": (C.c_int, [C.POINTER(OptimalMovesArgs), _vp, _vp]),
    "ts_optimal_moves": (C.c_int, [C.POINTER(OptimalMovesArgs), C.c_int, _vp]),
    "ts_optimal_moves_gmem_ctas_per_sm": (C.c_int, [C.POINTER(OptimalMovesArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_optimal_moves_gmem": (C.c_int, [C.POINTER(OptimalMovesArgs), _vp, C.c_int, _vp]),
    "ts_optimal_moves_table_ctas_per_sm": (C.c_int, [C.POINTER(OptimalMovesArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_optimal_moves_table": (C.c_int, [C.POINTER(OptimalMovesArgs), _vp, C.c_int64, C.c_int, _vp]),
    "ts_state_table_ctas_per_sm": (C.c_int, [C.POINTER(StateTableArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_state_table_count": (C.c_int, [C.POINTER(StateTableArgs), C.c_int, _vp]),
    "ts_state_table_fill": (C.c_int, [C.POINTER(StateTableArgs), C.c_int, _vp]),
    "ts_state_table_gmem_ctas_per_sm": (C.c_int, [C.POINTER(StateTableArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_state_table_count_gmem": (C.c_int, [C.POINTER(StateTableArgs), _vp, C.c_int, _vp]),
    "ts_state_table_fill_gmem": (C.c_int, [C.POINTER(StateTableArgs), _vp, C.c_int, _vp]),
    "ts_state_table_table_ctas_per_sm": (C.c_int, [C.POINTER(StateTableArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ts_state_table_count_table": (C.c_int, [C.POINTER(StateTableArgs), _vp, C.c_int64, C.c_int, _vp]),
    "ts_state_table_fill_table": (C.c_int, [C.POINTER(StateTableArgs), _vp, C.c_int64, C.c_int, _vp]),
    "ts_host_ctx_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "ts_host_ctx_destroy": (C.c_int, [_vp]),
    "ts_step_host": (C.c_int, [_vp, C.POINTER(StepArgs), _vp, _vp, _vp, _vp, _i64]),
}


class TilerSliderError(RuntimeError):
    """A C-ABI call failed (negative: argument error, positive: cudaError_t)."""


def build(force: bool = False, jobs: int | None = None) -> str:
    """Compile libtiler_slider.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, f"-j{jobs or os.cpu_count() or 4}"]
    if force:
        cmd.append("-B")
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TilerSliderError(
                f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
                "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
                f"`make -C {CSRC}`.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().ts_last_error_string().decode(errors="replace")
        raise TilerSliderError(f"{what} failed with code {rc}: {msg}")
