"""BatchedTilerSliderEnv: N independent Tiler-Slider boards advanced in lock-step on one B200.

Host-side mirror of the reference's TilerSliderEnv (explainrl/environment/environment.py:
14-194) for a batch: same vocabulary (reset / step / done / is_won / invalid_move / timeout /
max_steps), PyTorch tensors as containers, every computation done by the sm_100a kernels of
libtiler_slider.so through the C-ABI (include/tiler_slider.h).  No CPU fallback.

Packed state (see include/tiler_slider.h): `pos` is uint8[N, pos_bytes(T)], byte i of a row
= row*pos_stride + col of tile i.  `positions()` decodes to uint8[N, T, 2].
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Sequence

import numpy as np
import torch

from . import _lib
from ._lib import (CAP_ALIGN, F_WON, GOAL_ORDERED, GOAL_SET, MAX_SIZE, MAX_TILES, OBS_BF16, OBS_F16, OBS_F32, OBS_U8, OPT_MAX_DEPTH,
                   PLAYOUT_PLAN, PLAYOUT_RANDOM, EncodeArgs, ExpandArgs, GoalArgs, ObserveArgs, ObservePlanesArgs, PlayoutArgs,
                   PoolResetArgs, StepArgs, SynthArgs, ValidArgs, check, lib)
from .puzzle import Puzzle, as_puzzle, uniform_shape

DEFAULT_REWARDS = (1.0, -0.01, -0.05)   # r_win, r_step, r_invalid -- repo-defined (the reference has no reward)
# element types observe_planes() writes, and their codes in include/tiler_slider.h
PLANE_DTYPES = {torch.uint8: OBS_U8, torch.bfloat16: OBS_BF16, torch.float16: OBS_F16, torch.float32: OBS_F32}


def _round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


class BatchedTilerSliderEnv:
    """A batch of boards of one shape (size S, T tiles, one colour mode) on one CUDA device."""

    def __init__(self, size: int, n_tiles: int, n_envs: int, multi_color: bool = False, *,
                 max_steps: int = 100, auto_reset: bool = False, device: str | torch.device = "cuda",
                 rewards: Sequence[float] = DEFAULT_REWARDS, track_terminal: bool = False,
                 n_targets: int | None = None, track_flags: bool = True, host_io: bool = False):
        if not torch.cuda.is_available():
            raise _lib.TilerSliderError("BatchedTilerSliderEnv needs a CUDA device (no CPU fallback)")
        self._lib = lib()
        if not 1 <= size <= MAX_SIZE:
            raise ValueError(f"board size {size} outside 1..{MAX_SIZE}")
        if not 0 <= n_tiles <= MAX_TILES:
            raise ValueError(f"tile count {n_tiles} outside 0..{MAX_TILES}")
        if n_envs < 1:
            raise ValueError("n_envs must be positive")
        if not self._lib.ts_supported(size, n_tiles):
            raise ValueError(f"no step kernel for size {size} with {n_tiles} tiles")
        self.size, self.n_tiles, self.n_envs = int(size), int(n_tiles), int(n_envs)
        self.multi_color = bool(multi_color)
        self.n_targets = self.n_tiles if n_targets is None else int(n_targets)
        # T == 1 with one target: ordered and set equality coincide; use the cheaper compare
        self.goal_mode = GOAL_ORDERED if (self.multi_color or (self.n_tiles == 1 and self.n_targets == 1)) else GOAL_SET
        # ordered list equality with a length mismatch is never true (state.py:183-184): such a
        # batch plays normally and never reports a win (never_win); its targets do not fit the
        # packed word the step kernel compares, so the observation kernel gets them separately
        self.never_win = self.multi_color and self.n_targets != self.n_tiles
        if self.never_win and self.n_targets > MAX_TILES:
            raise ValueError(f"multi-colour boards with {self.n_targets} targets exceed the supported maximum of {MAX_TILES}")
        self.max_steps = int(max_steps)
        self.auto_reset = bool(auto_reset)
        # the status byte (is_won / invalid_move / timeout / stale) is optional with auto-reset:
        # reward and done are always written, and without it the step moves 26 instead of 27 bytes
        # per env (6x6 / 4 tiles); without auto-reset the done state of an env lives in that byte
        self.track_flags = bool(track_flags) or not self.auto_reset
        self.rewards = tuple(float(x) for x in rewards)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.capacity = _round_up(self.n_envs, CAP_ALIGN)
        self.pos_bytes = self._lib.ts_pos_bytes(self.n_tiles)
        self.board_bytes = self._lib.ts_board_bytes(self.size)
        self.board_stride = self._lib.ts_board_stride(self.size)
        self.pos_stride = self._lib.ts_pos_stride(self.size)
        self.count_bytes = 1 if self.max_steps <= (255 if self.auto_reset else 254) else 4
        cap, dev = self.capacity, self.device
        u8 = torch.uint8
        self.wide = self.size > 8
        self._walls = torch.zeros(cap * self._lib.ts_walls_bytes(self.size), dtype=u8, device=dev)
        tbytes = self.pos_bytes if self.goal_mode == GOAL_ORDERED else self._lib.ts_target_board_bytes(self.size)
        self._targets = torch.zeros(cap * tbytes, dtype=u8, device=dev)
        self._init = torch.zeros(cap, self.pos_bytes, dtype=u8, device=dev)
        # host_io (the single-env adapter): positions, actions and the step's outputs live in pinned HOST
        # memory that the kernels address directly (unified addressing), so a step is launches + one
        # stream synchronisation, with no copy calls; meant for tiny batches, where latency is all
        self.host_io = bool(host_io)

        def io(*shape, dtype=u8):
            return torch.zeros(*shape, dtype=dtype, pin_memory=True) if self.host_io else torch.zeros(*shape, dtype=dtype, device=dev)
        self._pos = io(cap, self.pos_bytes)
        self._count = torch.zeros(cap, dtype=u8 if self.count_bytes == 1 else torch.int32, device=dev)
        self._actions = io(cap)
        self._reward = io(cap, dtype=torch.float32)
        self._done = io(cap)
        self._flags = io(cap)
        self._terminal = torch.zeros(cap, self.pos_bytes, dtype=u8, device=dev) if track_terminal else None
        self._obs_targets = None      # ordered targets of a never_win batch, for observe() / target_positions()
        self._scratch_count = None
        self._scratch_flags = None
        self._scratch_reward = None
        self._host_ctx = None
        self._cached_args = None
        self._cached_out = None
        self._cached_obs_args = None
        self._io_np = None
        self._loaded = False
        self._pool = None             # set_reset_pool: the batch finished envs draw their next puzzle from
        self._pool_args = None
        self._episodes = None         # uint32 per env: puzzles drawn from a pool so far
        self._solve_depth = None      # int32 per env: shortest solution of the current puzzle (-1: not known)
        self._optimal = None          # optimal_moves(): the K9 driver (plans and scratch)
        self._state_table = None      # state_table(): the K10 driver

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_puzzles(cls, puzzles: Sequence, **kw) -> "BatchedTilerSliderEnv":
        """Batch from Puzzle objects (or anything with the ImageProcessed fields,
        dataloader.py:21-27) of one shape; boards are validated then encoded by K1."""
        ps = [as_puzzle(p).validate() for p in puzzles]
        S, T, NT, multi = uniform_shape(ps)
        n = len(ps)
        blocked = np.zeros((n, S * S), np.uint8)
        tiles = np.zeros((n, T, 2), np.uint8)
        targets = np.zeros((n, NT, 2), np.uint8)
        for i, p in enumerate(ps):
            for r, c in p.blocked_locations:
                blocked[i, int(r) * S + int(c)] = 1
            tiles[i] = np.asarray(p.initial_locations, np.uint8).reshape(T, 2)
            targets[i] = np.asarray(p.target_locations, np.uint8).reshape(NT, 2)
        return cls.from_arrays(S, blocked, tiles, targets, multi, **kw)

    @classmethod
    def from_arrays(cls, size: int, blocked, tiles, targets, multi_color: bool = False, **kw) -> "BatchedTilerSliderEnv":
        """blocked u8[N,S*S] (nonzero = wall), tiles u8[N,T,2], targets u8[N,NT,2] (row, col);
        numpy arrays or tensors on any device."""
        blocked = torch.as_tensor(blocked, dtype=torch.uint8)
        tiles = torch.as_tensor(tiles, dtype=torch.uint8)
        targets = torch.as_tensor(targets, dtype=torch.uint8)
        n, T, NT = blocked.shape[0], tiles.shape[1], targets.shape[1]
        if blocked.shape != (n, size * size) or tiles.shape != (n, T, 2) or targets.shape != (n, NT, 2):
            raise ValueError("expected blocked[N,S*S], tiles[N,T,2], targets[N,NT,2]")
        env = cls(size, T, n, multi_color, n_targets=NT, **kw)
        env.encode(blocked, tiles, targets)
        return env

    @classmethod
    def synthetic(cls, n_envs: int, size: int, n_tiles: int, n_walls: int, multi_color: bool = False, *,
                  seed: int = 0, env_index_base: int = 0, **kw) -> "BatchedTilerSliderEnv":
        """Random well-formed puzzles generated on the device by K0 (the create_simple_env
        recipe, environment.py:221-226).  `env_index_base` = global index of env 0, so a
        shard of a larger job draws the same puzzles whatever the GPU count."""
        env = cls(size, n_tiles, n_envs, multi_color, **kw)
        a = SynthArgs(size=size, n_tiles=n_tiles, n_walls=n_walls, goal_mode=env.goal_mode,
                      first_env=0, n_envs=n_envs, capacity=env.capacity, env_index_base=env_index_base,
                      seed=seed & (2 ** 64 - 1), d_walls=_ptr(env._walls), d_targets_packed=_ptr(env._targets),
                      d_init=_ptr(env._init), d_pos=_ptr(env._pos))
        with torch.cuda.device(env.device):
            check(env._lib.ts_synth(C.byref(a), env._stream()), "ts_synth")
        env._loaded = True
        env.reset()
        return env

    @classmethod
    def solvable(cls, n_envs: int, size: int, n_tiles: int, n_walls: int, multi_color: bool = False, *,
                 min_depth: int = 1, max_depth: int = 30, recipe: str = "walk", walk_len: int | None = None,
                 seed: int = 0, env_index_base: int = 0, max_attempts: int | None = None, device_bitmap: bool = False,
                 hash_table: bool = False, **kw) -> "BatchedTilerSliderEnv":
        """Solvable puzzles whose shortest solution takes between `min_depth` and `max_depth` steps,
        generated and graded on the device (K7 candidates, K6 search; tiler_slider_b200/generate.py).
        `solve_depth` holds each env's shortest-solution length.  recipe "walk": targets where a
        random walk of `walk_len` (default max(8, 2 * max_depth)) state-changing moves leaves the
        tiles; "uniform": synthetic()'s draw, redrawn until it lands in the band.  Env i's puzzle
        depends on (seed, recipe, walk_len, band, env_index_base + i) only.  Sizes up to 8, 1..4 tiles.
        A 7x7 board with four tiles and fewer than 11 walls, or an 8x8 one with fewer than 26, has a
        state space too large for the shared-memory bitmap of the grading search: ValueError, unless
        device_bitmap=True, which grades such boards with the bitmap in device memory.
        hash_table=True also takes 5..8 tiles (sizes 3..8): K7 candidates graded by K11's distance of
        their initial positions (optimal_moves(hash_table=True), bounded at max_depth <= 254); a
        candidate whose search outgrows the plan's bound (-3) is rejected like one outside the band."""
        from .generate import DEFAULT_MAX_ATTEMPTS, solvable
        return solvable(cls, n_envs, size, n_tiles, n_walls, multi_color, min_depth=min_depth, max_depth=max_depth,
                        recipe=recipe, walk_len=walk_len, seed=seed, env_index_base=env_index_base,
                        max_attempts=DEFAULT_MAX_ATTEMPTS if max_attempts is None else max_attempts,
                        device_bitmap=device_bitmap, hash_table=hash_table, **kw)

    def encode(self, blocked: torch.Tensor, tiles: torch.Tensor, targets: torch.Tensor) -> None:
        """K1: dense description -> packed planes (GameState.__init__, state.py:61-73)."""
        dev = self.device
        b = blocked.to(dev, torch.uint8).contiguous()
        t = tiles.to(dev, torch.uint8).contiguous()
        g = targets.to(dev, torch.uint8).contiguous()
        nt = g.shape[1]
        a = EncodeArgs(size=self.size, n_tiles=self.n_tiles, n_targets=nt, goal_mode=self.goal_mode,
                       first_env=0, n_envs=self.n_envs, capacity=self.capacity,
                       d_blocked=_ptr(b), d_tiles=_ptr(t), d_targets=_ptr(g) if nt else None,
                       d_walls=_ptr(self._walls), d_targets_packed=_ptr(self._targets),
                       d_init=_ptr(self._init), d_pos=_ptr(self._pos))
        with torch.cuda.device(dev):
            check(self._lib.ts_encode(C.byref(a), self._stream()), "ts_encode")
            torch.cuda.current_stream().synchronize()   # b, t, g are temporaries
        if self.never_win:
            pw = self._lib.ts_pos_bytes(nt)
            self._obs_targets = torch.zeros(self.capacity, pw, dtype=torch.uint8, device=dev)
            self._obs_targets[: self.n_envs, :nt] = g[..., 0] * self.pos_stride + g[..., 1]
        self._loaded = True
        self.reset()

    # ------------------------------------------------------------------ episode API
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def reset(self) -> torch.Tensor:
        """TilerSliderEnv.reset (environment.py:89-97) for every env: positions <- initial,
        step_count <- 0, done <- False.  Returns the packed positions uint8[N, pos_bytes]."""
        self._require_loaded()
        self._pos.copy_(self._init)
        self._count.zero_()
        self._flags.zero_()
        self._done.zero_()
        return self._pos[: self.n_envs]

    def _step_args(self, actions_ptr: int, *, count=None, flags=None, max_steps=None, count_bytes=None,
                   auto_reset=None, raw: bool = False) -> StepArgs:
        return StepArgs(size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, never_win=int(self.never_win),
                        first_env=0, n_envs=self.n_envs, capacity=self.capacity,
                        d_walls=_ptr(self._walls), d_targets_packed=_ptr(self._targets), d_init=_ptr(self._init),
                        d_pos=_ptr(self._pos), d_step_count=_ptr(self._count if count is None else count),
                        count_bytes=self.count_bytes if count_bytes is None else count_bytes,
                        max_steps=self.max_steps if max_steps is None else max_steps,
                        auto_reset=int(self.auto_reset if auto_reset is None else auto_reset),
                        d_actions=actions_ptr, r_win=self.rewards[0], r_step=self.rewards[1], r_invalid=self.rewards[2],
                        d_reward=_ptr(self._reward), d_done=None if raw else _ptr(self._done),
                        d_flags=_ptr(self._flags if flags is None else flags) if (self.track_flags or flags is not None) else None,
                        d_terminal_pos=None if raw else _ptr(self._terminal))

    def _stage_actions(self, actions) -> int:
        n = self.n_envs
        if isinstance(actions, torch.Tensor) and actions.dtype == torch.uint8 and actions.is_cuda \
                and actions.device == self.device and actions.is_contiguous() and actions.numel() >= self.capacity \
                and actions.data_ptr() % 16 == 0:   # kernels may read (and ignore) the padding envs up to capacity
            return actions.data_ptr()
        a = torch.as_tensor(actions)
        if a.numel() != n:
            raise ValueError(f"expected {n} actions, got {a.numel()}")
        self._actions[:n].copy_(a.reshape(n), non_blocking=True)
        return self._actions.data_ptr()

    def step(self, actions) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """One step for every env: K2 (slide + goal check + bookkeeping + reward [+ reset]).

        actions: uint8[N] (0 UP, 1 DOWN, 2 LEFT, 3 RIGHT; state.py:31-34), ideally already on
        the device.  Returns (state, reward, done): the packed positions uint8[N,pos_bytes],
        float32[N], bool[N] -- views of buffers that the next step overwrites.  `flags`
        holds is_won / invalid_move / timeout; with auto_reset the state of a finished env is
        already its reset state (its last positions are in `terminal_pos` if tracked).
        Successive calls walk the envs in alternating order (ts_step_args.order), which changes no
        result and lets each step start on what the previous one left in L2."""
        self._require_loaded()
        ptr = self._stage_actions(actions)
        a = self._cached_args
        if a is None:
            a = self._cached_args = self._step_args(ptr)
            n = self.n_envs
            self._cached_out = (self._pos[:n], self._reward[:n], self._done[:n].view(torch.bool))
        a.d_actions = ptr
        pool = self._pool_args
        if torch.cuda.current_device() == self.device.index:      # skip the device-guard round trip (host-bound small batches)
            stream = torch.cuda.current_stream().cuda_stream
            rc = self._lib.ts_step(C.byref(a), stream)
            if pool is not None and not rc:   # finished envs draw their next puzzle (K8 reads the done bytes K2 just wrote)
                rc_pool = self._lib.ts_pool_reset(C.byref(pool), stream)
        else:
            with torch.cuda.device(self.device):
                rc = self._lib.ts_step(C.byref(a), self._stream())
                if pool is not None and not rc:
                    rc_pool = self._lib.ts_pool_reset(C.byref(pool), self._stream())
        a.order ^= 1              # the next step walks the envs the other way and starts on what this one left in L2
        if rc:
            check(rc, "ts_step")
        if pool is not None and rc_pool:
            check(rc_pool, "ts_pool_reset")
        if self.host_io:          # the outputs are host memory: they are valid once the stream has drained
            torch.cuda.current_stream(self.device).synchronize()
        return self._cached_out

    def step_host_io(self, action: int, obs_out: torch.Tensor | None = None) -> None:
        """host_io batches: every env takes `action`; K2 (and K3 into the pinned `obs_out`) are launched
        and the stream is synchronised -- afterwards pos / reward / done / flags (and obs_out) can be
        read on the host as they are.  No tensor is created on this path."""
        if not self.host_io:
            raise RuntimeError("step_host_io needs a batch built with host_io=True")
        self._require_loaded()
        if self._io_np is None:
            self._io_np = self._actions.numpy()
        self._io_np[: self.n_envs] = action
        a = self._cached_args
        if a is None:
            a = self._cached_args = self._step_args(self._actions.data_ptr())
            n = self.n_envs
            self._cached_out = (self._pos[:n], self._reward[:n], self._done[:n].view(torch.bool))
        a.d_actions = self._actions.data_ptr()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream()
            rc = self._lib.ts_step(C.byref(a), stream.cuda_stream)
            if rc:
                check(rc, "ts_step")
            if obs_out is not None:
                o = self._cached_obs_args
                if o is None or o.d_obs != obs_out.data_ptr():
                    self._check_obs_out(obs_out)
                    o = self._cached_obs_args = self._observe_args(obs_out)
                rc = self._lib.ts_observe(C.byref(o), stream.cuda_stream)
                if rc:
                    check(rc, "ts_observe")
            stream.synchronize()

    def capture_steps(self, action_rows: torch.Tensor) -> "torch.cuda.CUDAGraph":
        """Capture `len(action_rows)` consecutive steps (row k = the actions of step k, uint8
        [R, capacity] on this device) into one CUDA graph; `graph.replay()` then advances the
        batch R steps with a single host call.  For launch-bound batches (about 1M envs and
        below) the per-step host cost of Python + ctypes otherwise exceeds the kernel time."""
        self._require_loaded()
        if action_rows.dtype != torch.uint8 or action_rows.device != self.device or action_rows.dim() != 2 \
                or action_rows.shape[1] < self.capacity or not action_rows.is_contiguous():
            raise ValueError("action_rows must be a contiguous uint8 [R, >= capacity] tensor on the env's device")
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.device(self.device):
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            pool_args, self._pool_args = self._pool_args, None   # the warm-up must not draw puzzles: reset() cannot undo that
            try:
                with torch.cuda.stream(side):
                    self.step(action_rows[0])                  # warm-up outside capture (lazy init)
            finally:
                self._pool_args = pool_args
            torch.cuda.current_stream(self.device).wait_stream(side)
            self.reset()
            with torch.cuda.graph(graph):
                for k in range(action_rows.shape[0]):
                    self.step(action_rows[k])
        return graph

    def raw_move(self, actions) -> torch.Tensor:
        """GameState.move (state.py:120-170) without episode bookkeeping: slides the tiles and
        returns the flags (WON / INVALID bits); step_count, done state and `flags` of the
        episode are untouched."""
        self._require_loaded()
        if self._scratch_count is None:
            self._scratch_count = torch.zeros(self.capacity, dtype=torch.int32, device=self.device)
            self._scratch_flags = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        self._scratch_count.zero_()
        self._scratch_flags.zero_()
        a = self._step_args(self._stage_actions(actions), count=self._scratch_count, flags=self._scratch_flags,
                            max_steps=2 ** 31 - 1, count_bytes=4, auto_reset=False, raw=True)
        if self._scratch_reward is None:
            self._scratch_reward = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        a.d_reward = self._scratch_reward.data_ptr()          # the episode's reward buffer stays untouched
        with torch.cuda.device(self.device):
            check(self._lib.ts_step(C.byref(a), self._stream()), "ts_step")
        return self._scratch_flags[: self.n_envs]

    # ------------------------------------------------------------------ host-buffer path
    def step_host(self, h_actions: torch.Tensor, h_reward: torch.Tensor | None = None, h_done: torch.Tensor | None = None,
                  h_flags: torch.Tensor | None = None, chunk_envs: int | None = None, n_streams: int = 4) -> None:
        """The same step driven from pinned HOST buffers (ts_step_host): uploads the actions,
        runs K2 and downloads reward + done (and / or the status byte `flags`), pipelined in
        chunks; returns when everything has landed.  With only `h_flags` given, 1 byte per env
        comes back instead of 5: bit 0 is done, and the reward follows from the WON / INVALID
        bits (`rewards`)."""
        self._require_loaded()
        if self._pool is not None:
            raise ValueError("step_host does not draw from a reset pool: use step() or detach the pool")
        if h_flags is None and (h_reward is None or h_done is None):
            raise ValueError("step_host needs h_reward and h_done, or h_flags")
        if h_flags is not None and not self.track_flags:
            raise ValueError("this batch was built with track_flags=False: there is no status byte to download")
        for t, dt in ((h_actions, torch.uint8), (h_reward, torch.float32), (h_done, torch.uint8), (h_flags, torch.uint8)):
            if t is not None and (t.is_cuda or t.dtype != dt or t.numel() < self.n_envs or not t.is_contiguous()):
                raise ValueError("step_host needs contiguous host tensors: uint8 actions, float32 reward, uint8 done / flags")
        if chunk_envs is None:      # 2M-env chunks keep PCIe busy (profiles/r1_pcie_e2e.json); small batches: one chunk per stream
            chunk_envs = min(1 << 21, max(1 << 16, -(-self.n_envs // n_streams)))
        if self._host_ctx is None:
            h = C.c_void_p()
            with torch.cuda.device(self.device):
                check(self._lib.ts_host_ctx_create(C.byref(h), n_streams), "ts_host_ctx_create")
            self._host_ctx = h
        a = self._step_args(self._actions.data_ptr())
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().synchronize()
            check(self._lib.ts_step_host(self._host_ctx, C.byref(a), h_actions.data_ptr(), _ptr(h_reward), _ptr(h_done),
                                         _ptr(h_flags), _round_up(chunk_envs, CAP_ALIGN)), "ts_step_host")

    # ------------------------------------------------------------------ reset pool
    def set_reset_pool(self, pool: "BatchedTilerSliderEnv | None", *, seed: int = 0, draw_now: bool = False) -> None:
        """Auto-reset into a pool of puzzles: from now on every step() is followed by K8 (ts_pool_reset),
        which gives each env that finished in that step pool puzzle H(seed, global env index, episode)
        (include/tiler_slider.h), so the returned state already shows the new puzzle (`terminal_pos`
        keeps the positions before the reset); inside capture_steps too.  `pool`: a batch of the same
        size, tile count, goal mode and target count on the same device (e.g. from solvable() or
        from_puzzles()); None detaches it.  draw_now: every env draws a pool puzzle now and starts a new
        episode.  `episodes` counts the draws per env; `solve_depth` follows the pool's depths (None
        when the pool has none).  Needs auto_reset; not available for host_io batches or step_host."""
        self._require_loaded()
        if pool is None:
            self._pool, self._pool_args = None, None
            return
        if not isinstance(pool, BatchedTilerSliderEnv):
            raise ValueError("the reset pool must be a BatchedTilerSliderEnv")
        if not self.auto_reset:
            raise ValueError("a reset pool needs auto_reset=True")
        if self.host_io:
            raise ValueError("host_io batches do not support a reset pool")
        if (pool.size, pool.n_tiles, pool.goal_mode, pool.n_targets) != (self.size, self.n_tiles, self.goal_mode, self.n_targets):
            raise ValueError(f"the pool holds size {pool.size} / {pool.n_tiles} tiles / goal mode {pool.goal_mode} / {pool.n_targets} "
                             f"targets, this batch size {self.size} / {self.n_tiles} / {self.goal_mode} / {self.n_targets}")
        if pool.never_win:
            raise ValueError("a never_win pool (target count != tile count, ordered goal) cannot be won")
        if pool.device != self.device:
            raise ValueError(f"the pool is on {pool.device}, this batch on {self.device}")
        pool._require_loaded()
        cap = self.capacity
        if self._episodes is None:
            self._episodes = torch.zeros(cap, dtype=torch.int32, device=self.device)
        if pool._solve_depth is None:
            self._solve_depth = None
        elif self._solve_depth is None:
            self._solve_depth = torch.full((cap,), -1, dtype=torch.int32, device=self.device)
        self._pool = pool
        self._pool_args = PoolResetArgs(
            size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, count_bytes=self.count_bytes,
            first_env=0, n_envs=self.n_envs, capacity=cap, env_index_base=0, seed=seed & (2 ** 64 - 1),
            d_done=_ptr(self._done), d_episode=_ptr(self._episodes), d_walls=_ptr(self._walls),
            d_targets_packed=_ptr(self._targets), d_init=_ptr(self._init), d_pos=_ptr(self._pos),
            d_step_count=_ptr(self._count), d_solve_depth=_ptr(self._solve_depth), n_pool=pool.n_envs,
            pool_capacity=pool.capacity, d_pool_walls=_ptr(pool._walls), d_pool_targets=_ptr(pool._targets),
            d_pool_init=_ptr(pool._init), d_pool_depth=_ptr(pool._solve_depth))
        if draw_now:
            a = PoolResetArgs.from_buffer_copy(self._pool_args)
            a.d_done = None
            with torch.cuda.device(self.device):
                check(self._lib.ts_pool_reset(C.byref(a), self._stream()), "ts_pool_reset")
            self._flags.zero_()
            self._done.zero_()

    @property
    def episodes(self) -> torch.Tensor:
        """uint32[N]: puzzles each env has drawn from a reset pool (one per finished episode while a
        pool is attached, plus one for set_reset_pool(draw_now=True))."""
        if self._episodes is None:
            self._episodes = torch.zeros(self.capacity, dtype=torch.int32, device=self.device)
        return self._episodes[: self.n_envs].view(torch.uint32)

    @property
    def solve_depth(self) -> torch.Tensor | None:
        """int32[N]: the fewest steps that win the current puzzle from its reset state (K6's solve
        depth; the goal is checked after every move), -1 where not known; None when the puzzles
        were not graded (synthetic / from_puzzles batches, or a reset pool without depths)."""
        return None if self._solve_depth is None else self._solve_depth[: self.n_envs]

    def __del__(self):
        h, self._host_ctx = getattr(self, "_host_ctx", None), None
        if h is not None:
            try:
                self._lib.ts_host_ctx_destroy(h)
            except Exception:
                pass

    # ------------------------------------------------------------------ views and queries
    def _require_loaded(self):
        if not self._loaded:
            raise RuntimeError("no puzzles loaded: use from_puzzles / from_arrays / synthetic / encode")

    @property
    def pos(self) -> torch.Tensor:
        return self._pos[: self.n_envs]

    @property
    def flags(self) -> torch.Tensor:
        """uint8[N]: F_DONE | F_WON | F_INVALID | F_TIMEOUT | F_STALE of the last step."""
        if not self.track_flags:
            raise RuntimeError("this batch was built with track_flags=False: the step stores reward and done only")
        return self._flags[: self.n_envs]

    @property
    def done(self) -> torch.Tensor:
        return self._done[: self.n_envs].view(torch.bool)

    @property
    def reward(self) -> torch.Tensor:
        return self._reward[: self.n_envs]

    @property
    def step_count(self) -> torch.Tensor:
        return self._count[: self.n_envs]

    @property
    def terminal_pos(self) -> torch.Tensor | None:
        return None if self._terminal is None else self._terminal[: self.n_envs]

    def is_won(self) -> torch.Tensor:
        """bool[N]: WON bit of the last step (the reference evaluates the goal only after a
        move, environment.py:123; nothing is won straight after reset)."""
        if not self.track_flags:      # reward = r_win exactly when the step won
            if self.rewards[0] in self.rewards[1:]:
                raise RuntimeError("track_flags=False and r_win equals another reward: is_won() cannot be told from the reward")
            return self.reward == self.rewards[0]
        return (self.flags & F_WON) != 0

    def goal_check(self) -> torch.Tensor:
        """bool[N]: GameState.is_won (state.py:172-186) of the CURRENT positions, without moving."""
        self._require_loaded()
        won = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        a = GoalArgs(size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, never_win=int(self.never_win),
                     first_env=0, n_envs=self.n_envs, capacity=self.capacity,
                     d_targets_packed=_ptr(self._targets), d_pos=_ptr(self._pos), d_won=_ptr(won))
        with torch.cuda.device(self.device):
            check(self._lib.ts_goal_check(C.byref(a), self._stream()), "ts_goal_check")
        return won[: self.n_envs].view(torch.bool)

    def positions(self, packed: torch.Tensor | None = None) -> torch.Tensor:
        """Decode packed position words to uint8[N, T, 2] (row, col)."""
        p = self.pos if packed is None else packed
        p = p[:, : self.n_tiles]
        ps = self.pos_stride
        return torch.stack((p // ps, p % ps), dim=-1)

    def _board_cells(self, buf: torch.Tensor, walls: bool = False) -> torch.Tensor:
        """Unpack a plane-layout bitboard buffer to bool[N, S*S] (load-time / debugging aid)."""
        nb, cap, n = self.board_bytes, self.capacity, self.n_envs
        if self.wide:   # u16 lines: walls [axis][capacity][S rounded up to even] (last plane = rows), targets [capacity][16]
            per_env = (self.size + 1) // 2 * 2 if walls else 17    # targets: 16 rows + the distinct-target count
            lines = buf.view(torch.int16).view(-1, cap, per_env)[-1, :n, :16 if not walls else per_env].to(torch.int32) & 0xFFFF
            lead = 1 if walls and self.size <= 14 else 0     # wall lines of S <= 14 start with an edge sentinel
            bits = (lines.unsqueeze(-1) >> (torch.arange(16, device=buf.device) + lead)) & 1
            return bits[:, : self.size, : self.size].reshape(n, self.size * self.size).bool()
        cols = []
        for k in range(self._lib.ts_plane_count(nb)):
            w, off = self._lib.ts_plane_width(nb, k), self._lib.ts_plane_offset(nb, k)
            cols.append(buf[off * cap: (off + w) * cap].view(cap, w)[:n])
        by = torch.cat(cols, dim=1)                                          # [N, nb] bytes, little endian
        bits = (by.unsqueeze(-1) >> torch.arange(8, device=by.device, dtype=torch.uint8)) & 1
        S, bs = self.size, self.board_stride
        return bits.reshape(n, nb * 8)[:, : S * bs].reshape(n, S, bs)[:, :, :S].reshape(n, S * S).bool()

    def blocked_cells(self) -> torch.Tensor:
        return self._board_cells(self._walls, walls=True)

    def target_positions(self) -> torch.Tensor:
        """Ordered mode: uint8[N,T,2].  Set mode: bool[N,S*S] target cells."""
        if self.goal_mode == GOAL_ORDERED:
            if self._obs_targets is not None:       # target count != tile count (never_win)
                t = self._obs_targets[: self.n_envs, : self.n_targets]
            else:
                t = self._targets.view(self.capacity, self.pos_bytes)[: self.n_envs, : self.n_tiles]
            return torch.stack((t // self.pos_stride, t % self.pos_stride), dim=-1)
        return self._board_cells(self._targets)

    def observe(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """K3: float32[N,S,S,3] observation, GameState.get_state_array (state.py:188-211).  `out`:
        a contiguous float32[N,S,S,3] tensor on the batch's device or in pinned host memory, 16-byte
        aligned; anything else raises ValueError (misalignment: TilerSliderError) before a launch."""
        self._require_loaded()
        S, n = self.size, self.n_envs
        if out is None:
            out = torch.empty(n, S, S, 3, dtype=torch.float32, device=self.device)
        else:
            self._check_obs_out(out)
        # single colour with one tile is stored as an ordered batch: index+1 == 1, same values
        a = self._observe_args(out)
        with torch.cuda.device(self.device):
            check(self._lib.ts_observe(C.byref(a), self._stream()), "ts_observe")
        return out

    def _check_obs_out(self, out: torch.Tensor) -> None:
        # the kernel writes n*S*S*3 floats from out.data_ptr() on and cannot check a size: a wrong
        # tensor would be written past its end (16-byte alignment is checked by ts_observe)
        S, n = self.size, self.n_envs
        if not isinstance(out, torch.Tensor) or tuple(out.shape) != (n, S, S, 3) or out.dtype != torch.float32:
            raise ValueError(f"observe(out): out must be a float32 tensor of shape ({n}, {S}, {S}, 3)")
        if not out.is_contiguous():
            raise ValueError("observe(out): out must be contiguous")
        if out.device != self.device and not (out.device.type == "cpu" and out.is_pinned()):
            raise ValueError(f"observe(out): out must live on {self.device} (or in pinned host memory), not on {out.device}")

    def _observe_args(self, out: torch.Tensor | None) -> ObserveArgs:
        # a never_win batch draws its ordered targets from their own buffer (count != tile count)
        nt = 0 if self._obs_targets is None else (self.n_targets or -1)
        tg = self._targets if self._obs_targets is None else self._obs_targets
        return ObserveArgs(size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, n_targets=nt,
                           first_env=0, n_envs=self.n_envs, capacity=self.capacity, d_walls=_ptr(self._walls),
                           d_targets_packed=_ptr(tg), d_pos=_ptr(self._pos), d_obs=_ptr(out))

    @property
    def plane_count(self) -> int:
        """C of observe_planes(): 1 + T + NT with multi colour (the walls, one plane per tile and one
        per target), 3 with single colour (walls, tile cells, target cells)."""
        c = self._lib.ts_observe_planes_channels(C.byref(self._observe_planes_args(None, torch.float32)))
        if c < 0:
            check(c, "ts_observe_planes_channels")
        return c

    def observe_planes(self, out: torch.Tensor | None = None, *, dtype: torch.dtype = torch.float32, ids=None,
                       pos: torch.Tensor | None = None) -> torch.Tensor:
        """Network input [N, C, S, S] (C = plane_count), channel first, every element 0 or 1 in
        `dtype` (uint8, bfloat16, float16 or float32), written by one kernel (ts_observe_planes).
        Plane 0: blocked cells; multi colour: plane 1+i tile i, plane 1+T+j target j; single
        colour: plane 1 the tile cells, plane 2 the target cells.  No host synchronisation, and
        with `out` no allocation, so it can be captured in a CUDA graph beside step().  `out`: a
        contiguous `dtype` tensor of that shape on the batch's device or in pinned host memory,
        16-byte aligned; anything else raises ValueError (misalignment: TilerSliderError) before a
        launch.

        With `ids` and / or `pos` the images are of ITEMS, as expand() takes them
        (ts_observe_planes_items): image i shows env ids[i]'s walls and targets with the tiles of
        pos[i], so [n, C, S, S] for n items -- e.g. the successors expand() returned, with
        ids.repeat_interleave(4) and pos = succ.reshape(-1, pos_bytes)."""
        self._require_loaded()
        if dtype not in PLANE_DTYPES:
            raise ValueError(f"observe_planes: dtype {dtype} is not one of uint8, bfloat16, float16, float32")
        items = ids is not None or pos is not None
        n = self.n_envs
        if items:
            n, ids, pos = self._items("observe_planes", ids, pos)
        shape = (n, self.plane_count, self.size, self.size)
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=self.device)
        elif not isinstance(out, torch.Tensor) or tuple(out.shape) != shape or out.dtype != dtype:
            raise ValueError(f"observe_planes(out): out must be a {dtype} tensor of shape {shape}")
        elif not out.is_contiguous():
            raise ValueError("observe_planes(out): out must be contiguous")
        elif out.device != self.device and not (out.device.type == "cpu" and out.is_pinned()):
            raise ValueError(f"observe_planes(out): out must live on {self.device} (or in pinned host memory), not on {out.device}")
        a = self._observe_planes_args(out, dtype)
        with torch.cuda.device(self.device):
            if not items:
                check(self._lib.ts_observe_planes(C.byref(a), self._stream()), "ts_observe_planes")
            elif n:
                check(self._lib.ts_observe_planes_items(C.byref(a), _ptr(ids), _ptr(pos), n, self._stream()),
                      "ts_observe_planes_items")
        return out

    def _items(self, what: str, ids, pos: torch.Tensor | None) -> tuple[int, torch.Tensor | None, torch.Tensor | None]:
        """(n, int32 ids on the device or None, pos or None) of an item call; raises ValueError /
        IndexError before any launch.  Host ids are range-checked against [0, n_envs); device ids
        are not (that would cost a synchronisation): the kernels give an id outside [0, capacity)
        an all-zero result and read nothing of it."""
        if self.host_io:
            raise ValueError(f"{what}: not available for host_io batches (their positions live in host memory)")
        n = self.n_envs
        if ids is not None:
            if isinstance(ids, torch.Tensor) and ids.is_cuda:
                if ids.device != self.device:
                    raise ValueError(f"{what}: ids are on {ids.device}, the batch on {self.device}")
                if ids.is_floating_point() or ids.is_complex() or ids.dtype == torch.bool:
                    raise ValueError(f"{what}: ids must be integers, not {ids.dtype}")
                if ids.dtype != torch.int32 or not ids.is_contiguous():
                    ids = ids.to(torch.int32).contiguous()
                ids = ids.reshape(-1)
            else:
                t = torch.as_tensor(ids).reshape(-1)
                if t.numel() and (t.is_floating_point() or t.is_complex() or t.dtype == torch.bool):
                    raise ValueError(f"{what}: ids must be integers, not {t.dtype}")
                if t.numel():
                    lo, hi = int(t.min()), int(t.max())
                    if lo < 0 or hi >= self.n_envs:
                        raise IndexError(f"{what}: env ids must lie in [0, {self.n_envs}), got [{lo}, {hi}]")
                ids = t.to(torch.int32)          # copied to the device once pos has passed its checks too
            n = ids.numel()
        if pos is not None:
            check_item_pos(what, pos, n, ids is not None, self.pos_bytes, self.device)
        if ids is not None and not ids.is_cuda:
            ids = ids.to(self.device)
        return n, ids, pos

    def expand(self, ids=None, pos: torch.Tensor | None = None, *,
               out: tuple[torch.Tensor, torch.Tensor, torch.Tensor] | None = None) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """The four successors of many states, for search (beam search, A* with a learned heuristic,
        MCTS expansion, value-iteration targets), in one kernel (ts_expand).  An item is (env id,
        positions): the env gives the puzzle (walls and targets), the position word the tiles.
        ids: any integer sequence or tensor of env ids (default: every env); pos: uint8 [n, pos_bytes]
        on the device (default: each listed env's current positions; without ids it needs n_envs
        rows).  Returns (succ uint8[n, 4, pos_bytes], moved uint8[n], won uint8[n]):
          succ[i, a]  the positions after move a (0 UP, 1 DOWN, 2 LEFT, 3 RIGHT) -- what step()
                      would leave, before any reset, with the tile order kept (no sorting with a
                      single colour); succ.reshape(-1, pos_bytes) with ids.repeat_interleave(4) is
                      the next level's item list;
          moved[i]    bit a set iff move a changes the positions (valid_moves() of the item);
          won[i]      bit a set iff the positions after move a meet the goal (the step's is_won).
        `out`: preallocated (succ, moved, won) of those shapes, contiguous uint8 on the device; with it
        and device ids (int32, contiguous, passed as they are) or none, the call neither allocates nor
        synchronises, so it can be captured in a CUDA graph beside step().  Host ids outside
        [0, n_envs) raise IndexError; device ids are not checked: one outside [0, capacity) gets
        zero successors and masks.  Runs on the current stream and changes no env state.  Not
        available for host_io batches."""
        self._require_loaded()
        n, ids, pos = self._items("expand", ids, pos)
        shapes = ((n, 4, self.pos_bytes), (n,), (n,))
        if out is None:
            out = tuple(torch.empty(s, dtype=torch.uint8, device=self.device) for s in shapes)
        else:
            if not isinstance(out, (tuple, list)) or len(out) != 3:
                raise ValueError("expand(out): out must be a tuple (succ, moved, won)")
            for t, s in zip(out, shapes):
                if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or tuple(t.shape) != s:
                    raise ValueError(f"expand(out): expected uint8 tensors of shapes {shapes}")
                if t.device != self.device:
                    raise ValueError(f"expand(out): out must live on {self.device}, not on {t.device}")
                if not t.is_contiguous():
                    raise ValueError("expand(out): out must be contiguous")
            out = tuple(out)
        if n:
            a = ExpandArgs(size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, never_win=int(self.never_win),
                           n_items=n, capacity=self.capacity, d_env_ids=_ptr(ids), d_walls=_ptr(self._walls),
                           d_targets_packed=_ptr(self._targets), d_pos=_ptr(self._pos), d_item_pos=_ptr(pos),
                           d_succ=_ptr(out[0]), d_moved=_ptr(out[1]), d_won=_ptr(out[2]))
            with torch.cuda.device(self.device):
                check(self._lib.ts_expand(C.byref(a), self._stream()), "ts_expand")
        return out

    def playout(self, ids=None, pos: torch.Tensor | None = None, *, actions: torch.Tensor | None = None,
                n_steps: int | None = None, seed: int = 0, record: bool = False, out=None) -> tuple[torch.Tensor, ...]:
        """Up to L moves from many states in one kernel (ts_playout), for MCTS simulation, replaying
        plans and recording trajectories.  Items as expand() takes them: ids (default every env) give
        the puzzles, pos (default each listed env's current positions) the start positions.
          actions   a plan: contiguous uint8 [L, n] on the batch's device, step-major (row k = move k
                    of every item; 0 UP, 1 DOWN, 2 LEFT, 3 RIGHT); a byte >= 4 ends the item's plan
                    (pad ragged move strings with 255).  L = actions.shape[0]; `n_steps` must not be
                    given.  A move that changes nothing is played and counted, as step() counts it.
          otherwise random moves: `n_steps` (required) moves, each drawn uniformly among the moves
                    that change the positions (valid_moves()); item i's draws depend on (seed, i) only
                    (K7's walk rule, include/tiler_slider.h); a state where nothing can move ends it.
        The goal is checked after every move and a win ends the item's playout.  Returns (final uint8
        [n, pos_bytes], steps int32 [n], won uint8 [n]): the positions after the last move played, the
        moves played and 1 iff the last one won; with record=True also (moves uint8 [L, n], traj uint8
        [L, n, pos_bytes]): the move played as move k (255 for k >= steps) and the positions after it
        (zero for k >= steps).  `out`: preallocated tensors of those shapes and dtypes, contiguous on
        the device (3 of them, 5 with record); with it and device ids (int32, contiguous) or none,
        the call neither allocates nor synchronises, so it can be captured in a CUDA graph beside
        step() -- the seed is then fixed at capture.  Host ids outside [0, n_envs) raise IndexError;
        a device id outside [0, capacity) gets zero positions, 0 steps, not won.  Runs on the current
        stream and changes no env state.  Not available for host_io batches."""
        self._require_loaded()
        n, ids, pos = self._items("playout", ids, pos)
        if actions is not None:
            if n_steps is not None:
                raise ValueError("playout: give either actions (a plan) or n_steps (random moves), not both")
            if not isinstance(actions, torch.Tensor) or actions.dtype != torch.uint8 or actions.dim() != 2 or actions.shape[1] != n:
                raise ValueError(f"playout: actions must be a uint8 tensor [L, {n}] (step-major: row k = move k of every item)")
            if actions.device != self.device:
                raise ValueError(f"playout: actions are on {actions.device}, the batch on {self.device}")
            if not actions.is_contiguous():
                raise ValueError("playout: actions must be contiguous")
            # an empty plan plays no move: the random policy with no moves gives the same result and
            # needs no plan buffer (an empty tensor has no data pointer)
            L, policy = actions.shape[0], PLAYOUT_PLAN if actions.shape[0] else PLAYOUT_RANDOM
        else:
            if n_steps is None:
                raise ValueError("playout: random playouts need n_steps (or pass actions, a plan)")
            L, policy = int(n_steps), PLAYOUT_RANDOM
        if not 0 <= L < 2 ** 31:
            raise ValueError(f"playout: {L} moves outside 0 .. 2^31 - 1")
        PW = self.pos_bytes
        specs = [((n, PW), torch.uint8), ((n,), torch.int32), ((n,), torch.uint8)]
        if record:
            specs += [((L, n), torch.uint8), ((L, n, PW), torch.uint8)]
        if out is None:
            out = tuple(torch.empty(s, dtype=dt, device=self.device) for s, dt in specs)
        else:
            if not isinstance(out, (tuple, list)) or len(out) != len(specs):
                raise ValueError(f"playout(out): out must be a tuple of {len(specs)} tensors "
                                 f"({'final, steps, won, moves, traj' if record else 'final, steps, won'})")
            for t, (s, dt) in zip(out, specs):
                if not isinstance(t, torch.Tensor) or t.dtype != dt or tuple(t.shape) != s:
                    raise ValueError(f"playout(out): expected tensors of shapes and dtypes {[(s, str(dt)) for s, dt in specs]}")
                if t.device != self.device:
                    raise ValueError(f"playout(out): out must live on {self.device}, not on {t.device}")
                if not t.is_contiguous():
                    raise ValueError("playout(out): out must be contiguous")
            out = tuple(out)
        if n:
            a = PlayoutArgs(size=self.size, n_tiles=self.n_tiles, goal_mode=self.goal_mode, never_win=int(self.never_win),
                            policy=policy, n_steps=L, n_items=n, capacity=self.capacity, seed=int(seed) & (2 ** 64 - 1),
                            d_env_ids=_ptr(ids), d_walls=_ptr(self._walls), d_targets_packed=_ptr(self._targets),
                            d_pos=_ptr(self._pos), d_item_pos=_ptr(pos), d_plan=_ptr(actions), d_final=_ptr(out[0]),
                            d_steps=_ptr(out[1]), d_won=_ptr(out[2]), d_moves=_ptr(out[3]) if record else None,
                            d_traj=_ptr(out[4]) if record else None)
            with torch.cuda.device(self.device):
                check(self._lib.ts_playout(C.byref(a), self._stream()), "ts_playout")
        return out

    def _observe_planes_args(self, out: torch.Tensor | None, dtype: torch.dtype) -> ObservePlanesArgs:
        o = self._observe_args(None)      # the same targets and n_targets convention as observe()
        return ObservePlanesArgs(size=o.size, n_tiles=o.n_tiles, goal_mode=o.goal_mode, n_targets=o.n_targets,
                                 first_env=o.first_env, n_envs=o.n_envs, capacity=o.capacity, d_walls=o.d_walls,
                                 d_targets_packed=o.d_targets_packed, d_pos=o.d_pos, dtype=PLANE_DTYPES[dtype],
                                 d_out=_ptr(out))

    def valid_moves(self) -> torch.Tensor:
        """uint8[N]: bit d set when move d changes the state (get_valid_moves,
        environment.py:149-171)."""
        self._require_loaded()
        mask = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        a = ValidArgs(size=self.size, n_tiles=self.n_tiles, first_env=0, n_envs=self.n_envs, capacity=self.capacity,
                      d_walls=_ptr(self._walls), d_pos=_ptr(self._pos), d_mask=_ptr(mask))
        with torch.cuda.device(self.device):
            check(self._lib.ts_valid_moves(C.byref(a), self._stream()), "ts_valid_moves")
        return mask[: self.n_envs]

    def optimal_moves(self, ids=None, pos: torch.Tensor | None = None, *, max_depth: int = 254,
                      paths: bool = False, device_bitmap: bool = False, hash_table: bool = False) -> tuple[torch.Tensor, ...]:
        """Exact solver answers for items (K9, ts_optimal_moves), as supervision for imitation
        learning, value targets, optimality gaps, reward shaping or an exact expert policy.  Items as
        expand() takes them: ids (default every env) give the puzzles, pos (default each listed
        env's CURRENT positions) the states to solve from; pos is a contiguous uint8 [n, pos_bytes]
        on the batch's device (n_envs rows without ids).  Returns (distance int32[n], mask uint8[n])
        in item order, and with paths=True also plan:
          distance: the fewest steps that win from the item's state (>= 1; the goal is checked after
                    every move, as solve_depth; max_steps and the step counter play no part), or
                    -1 no win reachable (also every env of a never_win batch), -2 none within
                    max_depth steps, -3 this env's state space is larger than the largest bitmap
                    one CTA can hold in shared memory (4 tiles on a 7x7 board with fewer than 11
                    walls or an 8x8 one with fewer than 26; with device_bitmap=True such boards
                    are searched with the bitmap in device memory instead), or than the slab of
                    the launch (it does not depend on the other items of the query; with
                    hash_table=True and 5 to 8 tiles: the item discovered more states than the
                    plan's bound, see below), -4 the
                    position word is not a well-formed state of
                    its env (a tile on a wall or off the board, two tiles on one cell; e.g. the
                    zero rows playout(record=True) writes past an item's end);
          mask:     bit a (valid_moves() order) set iff move a starts a shortest solution; 0 when
                    distance < 0;
          plan:     uint8 [max_depth, n], step-major as playout(actions=) takes it: rows
                    0 .. distance[i]-1 of column i hold the lexicographically smallest shortest
                    solution of item i (UP < DOWN < LEFT < RIGHT: each move the lowest bit of the
                    mask of the state it is played from), every other entry is 255.  So
                    playout(ids, pos, actions=plan) wins every item with distance >= 1 in exactly
                    distance moves.  distance and mask are the same with and without paths.
        Ids are range-checked against [0, n_envs) (IndexError), host and device ids alike.  Runs on
        the current stream after the steps queued before it, reads one scalar back, and changes no
        env state.  Sizes up to 8, 1..4 tiles, device-memory batches (not host_io).
        hash_table=True also takes 5..8 tiles (K11, ts_optimal_moves_table): the same answers from a
        search whose visited set is a per-CTA hash table in device memory, bounded by the plan's
        spill_per_cta discovered states per item (-3 beyond); it reads nothing back.  With 1..4 tiles
        it changes nothing."""
        from .bfs import CudaOptimalMoves, check_optimal_moves
        check_optimal_moves(self.size, self.n_tiles, self.host_io, int(max_depth), hash_table=bool(hash_table))
        self._require_loaded()
        ids = self._search_items("optimal_moves", ids, pos)
        if self._optimal is None:
            self._optimal = CudaOptimalMoves(self)
        if not paths:
            return self._optimal.query(ids, int(max_depth), pos, device_bitmap=bool(device_bitmap), hash_table=bool(hash_table))
        n = self.n_envs if ids is None else ids.numel()
        plan = torch.empty((int(max_depth), n), dtype=torch.uint8, device=self.device)
        return (*self._optimal.query(ids, int(max_depth), pos, plan, bool(device_bitmap), bool(hash_table)), plan)

    def state_table(self, ids=None, pos: torch.Tensor | None = None, *, device_bitmap: bool = False,
                    hash_table: bool = False, max_states: int | None = None) -> StateTable:
        """Every state reachable from items, each with its exact distance to a win and its optimal
        moves (K10, ts_state_table), for value / policy datasets over whole state spaces, reverse
        curricula (states a chosen distance from the goal) and puzzle statistics (dead states, the
        distance histogram).  Items as optimal_moves() takes them: ids (default every env) give the
        walls and the goal, row i of pos (default each listed env's CURRENT positions) the root.
        Returns a StateTable: item i owns rows offsets[i] .. offsets[i+1]-1, which hold every state
        reachable from its root, the root included, each once, in ascending order of the perfect
        hash the search keys states by (so the table is the same from call to call); set-goal
        batches store the canonical word (bytes ascending).  distance and mask of a row are what
        optimal_moves(ids=..., pos=row) answers for it (max_depth plays no part: every finite
        distance is found), -1 and 0 where no win is reachable (every row of a never_win batch).
        status[i] is 0, or -3 (the item's state space is larger than the largest bitmap one CTA can
        hold in shared memory, unless device_bitmap=True: as in optimal_moves()) or -4 (a malformed
        root, as optimal_moves() reports it); such items own no rows.
        Ids are range-checked as in optimal_moves() (IndexError).  Runs on the current stream,
        changes no env state and reads back two scalars (the free-cell maximum and the row count,
        to allocate), so it cannot be captured in a CUDA graph.  Sizes up to 8, 1..4 tiles,
        device-memory batches (not host_io).
        hash_table=True also takes 5..8 tiles (K12, ts_state_table_count_table / _fill_table): the
        same table from a search whose visited set is a per-CTA hash table in device memory (as
        optimal_moves(hash_table=True)), pos uint8 [M, 8].  Each item's rows are in ascending order
        of their 8 bytes read as a little-endian 64-bit word (table.pos.view(torch.int64) ascends
        per item), the same from call to call and whatever the launch plan.  status -3 means the
        item reaches more than max_states states, the root included: a bound that depends on
        max_states alone (None: the bound of optimal_moves(hash_table=True)'s plan).  A larger
        max_states runs on fewer CTAs, as their tables and slabs share 4 GiB (ValueError when not
        even one fits).  Reads back the row count only.  With 1..4 tiles hash_table changes nothing,
        and max_states is taken with hash_table=True and 5..8 tiles only (ValueError)."""
        from .bfs import CudaStateTable, check_optimal_moves
        check_optimal_moves(self.size, self.n_tiles, self.host_io, OPT_MAX_DEPTH, "state_table", hash_table=bool(hash_table))
        if max_states is not None:
            if not (hash_table and self.n_tiles >= 5):
                raise ValueError("state_table: max_states bounds the hash-table tables (hash_table=True, 5 to 8 tiles)")
            if int(max_states) < 1:
                raise ValueError(f"state_table: max_states must be >= 1 (got {max_states})")
        self._require_loaded()
        ids = self._search_items("state_table", ids, pos)
        if self._state_table is None:
            self._state_table = CudaStateTable(self)
        return StateTable(*self._state_table.build(ids, pos, bool(device_bitmap), bool(hash_table),
                                                   None if max_states is None else int(max_states)))

    def _search_items(self, what: str, ids, pos: torch.Tensor | None) -> torch.Tensor | None:
        """The ids of a solver query as int32 on the device (None: every env), range-checked against
        [0, n_envs) (IndexError), and its pos validated (ValueError)."""
        if ids is not None:
            ids = torch.as_tensor(ids).to(device=self.device, dtype=torch.int32).reshape(-1).contiguous()
        if pos is not None:
            check_item_pos(what, pos, self.n_envs if ids is None else ids.numel(), ids is not None,
                           self.pos_bytes, self.device)
        if ids is not None and ids.numel():
            lo, hi = torch.aminmax(ids)
            lo, hi = int(lo), int(hi)
            if lo < 0 or hi >= self.n_envs:
                raise IndexError(f"env ids must lie in [0, {self.n_envs}), got [{lo}, {hi}]")
        return ids

    def set_positions(self, tiles) -> None:
        """Overwrite current positions from uint8[N,T,2] (row, col) -- e.g. to expand a search
        frontier; validity is the caller's responsibility."""
        t = torch.as_tensor(tiles, dtype=torch.uint8).to(self.device)
        packed = t[..., 0] * self.pos_stride + t[..., 1]
        self._pos[: self.n_envs, : self.n_tiles] = packed

    def puzzle(self, i: int) -> Puzzle:
        """Decode env i back to a Puzzle (host copy)."""
        S = self.size
        blocked = [(int(c) // S, int(c) % S) for c in torch.nonzero(self.blocked_cells()[i]).flatten().tolist()]
        init = self._init[i, : self.n_tiles].cpu()
        tiles = [divmod(int(b), self.pos_stride) for b in init.tolist()]
        if self.goal_mode == GOAL_ORDERED:
            tg = [(int(r), int(c)) for r, c in self.target_positions()[i].cpu().tolist()]
        else:
            tg = [(int(c) // S, int(c) % S) for c in torch.nonzero(self.target_positions()[i]).flatten().tolist()]
        return Puzzle(S, blocked, tiles, tg, self.multi_color)


@dataclass(frozen=True)
class StateTable:
    """The states reachable from items with their exact labels (BatchedTilerSliderEnv.state_table):
    item i owns rows offsets[i] .. offsets[i+1]-1 of pos / distance / mask.
      offsets   int64 [n+1]
      status    int32 [n]: 0 enumerated, -3 the state space does not fit one CTA (hash_table=True:
                more than max_states states), -4 malformed root
      pos       uint8 [M, pos_bytes]: the states, per item ascending by the search's perfect hash (1
                to 4 tiles) or as little-endian 64-bit words (5 to 8 tiles, hash_table=True)
      distance  int32 [M]: fewest moves that win (>= 1), -1 if no win is reachable
      mask      uint8 [M]: bit a set iff move a starts a shortest solution (0 where distance < 0)"""
    offsets: torch.Tensor
    status: torch.Tensor
    pos: torch.Tensor
    distance: torch.Tensor
    mask: torch.Tensor


def check_item_pos(what: str, pos, n: int, with_ids: bool, pos_bytes: int, device: torch.device) -> None:
    """The position words of n items: a contiguous uint8 [n, pos_bytes] tensor on `device`, else
    ValueError."""
    if not isinstance(pos, torch.Tensor) or pos.dtype != torch.uint8 or pos.dim() != 2 or pos.shape[1] != pos_bytes:
        raise ValueError(f"{what}: pos must be a uint8 tensor [n, {pos_bytes}]")
    if pos.shape[0] != n:
        raise ValueError(f"{what}: pos has {pos.shape[0]} rows, expected {n} "
                         f"({'one per id' if with_ids else 'one per env without ids'})")
    if pos.device != device:
        raise ValueError(f"{what}: pos is on {pos.device}, the batch on {device}")
    if not pos.is_contiguous():
        raise ValueError(f"{what}: pos must be contiguous")


def shard_range(n_total: int, rank: int, world_size: int) -> tuple[int, int]:
    """Contiguous env-index shard [lo, hi) of rank `rank` (SURVEY 8(e)): envs never interact,
    so the step path needs no collective; the remainder goes to the first ranks."""
    base, rem = divmod(n_total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)
