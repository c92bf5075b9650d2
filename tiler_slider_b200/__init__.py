"""tiler_slider_b200 -- B200-native batched Tiler-Slider environment.

Public surface (reference names kept; see DESIGN.md):
  GameState, TilerSliderEnv, TilerSliderEnvFactory   single-env drop-ins (batch size 1 on CUDA)
  Move                                               action enum (state.py:29-45)
  BatchedTilerSliderEnv                              N boards per GPU, one kernel launch per step
  Puzzle, parse_board_text, load_puzzle_file         text grammar + `-input_file` loader
  levels.load_level / load_level_image               screenshot ingest (host-side, cv2)
  bfs.LocalBfs                                       batched breadth-first search, one CTA per puzzle, on chip
  bfs.BfsSolver                                      hash-partitioned search (HBM table, NVLink / NCCL exchange)
Every computation runs in libtiler_slider.so (hand-written sm_100a CUDA, C-ABI in
include/tiler_slider.h); there is no CPU fallback.
"""
from ._lib import (F_DONE, F_INVALID, F_STALE, F_TIMEOUT, F_WON, GOAL_ORDERED, GOAL_SET, TilerSliderError, build, lib)
from .moves import Move
from .puzzle import Puzzle, load_puzzle_file, parse_board_text, parse_puzzle_file_text, puzzle_to_text
from .batch_env import DEFAULT_REWARDS, BatchedTilerSliderEnv, StateTable, shard_range
from .env import GameState, TilerSliderEnv, TilerSliderEnvFactory

__version__ = "0.2.0"
__all__ = ["GameState", "TilerSliderEnv", "TilerSliderEnvFactory", "Move", "BatchedTilerSliderEnv", "StateTable", "Puzzle",
           "parse_board_text", "parse_puzzle_file_text", "load_puzzle_file", "puzzle_to_text", "shard_range",
           "DEFAULT_REWARDS", "TilerSliderError", "build", "lib",
           "F_DONE", "F_WON", "F_INVALID", "F_TIMEOUT", "F_STALE", "GOAL_ORDERED", "GOAL_SET"]
