"""Breadth-first state-space search over many puzzles at once (BASELINE config 5).

The reference has no solver; the closest primitive is TilerSliderEnv.get_valid_moves
(explainrl/environment/environment.py:149-171), which tries the four moves on copies.  Here
the successor function is GameState.move (explainrl/environment/state.py:120-170) run by the
sm_100a kernels of csrc/ts_bfs.cu, the goal test is is_won (state.py:172-186), and the visited
set is an open-addressing hash table in HBM.  BFS itself is defined by this repo (parity
unpinned); level histograms are pinned to a plain BFS over the reference's move
(tests/golden/misc.json).

Two searches, same results (states per puzzle, level histogram, solve depths, shortest move strings):

* `LocalBfs` (K6, csrc/ts_bfs_local.cu): a batch of small puzzles (size <= 8, up to 4 tiles), one CTA
  per puzzle, visited set and frontier in shared memory; puzzles sharded over the ranks by index,
  nothing exchanged.  Puzzles that outgrow the chip fall back to the search below.
* `BfsSolver`: one visited table in HBM, hash-partitioned over the ranks -- every rank holds the
  (small, static) puzzle table and the slice of the visited set whose keys hash to it; key = puzzle
  id || canonical positions.  One exchange per depth, either fused into the expansion (K4x: the
  successors go straight into the owners' inboxes through NVLink peer memory, levels separated by
  an 8-byte all-reduce) or as
      expand local frontier (K4)  ->  bucket successors by owner rank  ->  all_gather of the
      bucket sizes, all_to_all_single of the u64 keys (NCCL)  ->  insert into the local table (K5);
      the keys that were new form the next local frontier; a level in which nobody sent anything
      ends the search.
  Single-rank and peer-memory searches keep the frontier sizes on the device and launch 16 levels
  between host read-backs.  with_paths records parents (over several ranks they travel with the
  keys) and walks the chains back from the recorded last link of every solution.
`solve_batch` picks the search that fits a batch.  `CudaOptimalMoves` (K9, csrc/ts_optimal.cu) is
K6's sibling for the envs of a batch as they stand: the distance of their current positions to a win
and the moves that start a shortest solution (BatchedTilerSliderEnv.optimal_moves).  `CudaStateTable`
(K10, csrc/ts_state_table.cu) enumerates every state reachable from items and labels each with K9's
answer (BatchedTilerSliderEnv.state_table).

The device kernels sit behind `CudaBfsKernels`; tests run the same driver logic on CPU
tensors over gloo with a CPU stand-in for the kernels (tests/test_bfs_gloo.py).
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass, field
from typing import Sequence

import torch
import torch.distributed as dist

from ._lib import OPT_MAX_DEPTH, OPT_NOT_SEARCHED, BfsArgs, BfsLocalArgs, OptimalMovesArgs, StateTableArgs, check, lib
from .batch_env import BatchedTilerSliderEnv, shard_range
from .puzzle import Puzzle

NONE = -1                       # TS_BFS_NONE as int64
WON_BIT = -(1 << 63)            # bit 63 as int64


@dataclass
class BfsResult:
    n_states: int                              # reachable states, all puzzles, all ranks
    levels: list[int]                          # new states per depth (depth 0 = the initial states)
    solve_depth: int                           # first depth at which some successor met the goal (-1: none)
    states_per_puzzle: torch.Tensor | None = None   # int64[P] reachable states per puzzle (this rank's share summed over ranks)
    solve_depth_per_puzzle: torch.Tensor | None = None   # int32[P], -1 where unsolved within max_depth
    generated: int = 0                         # successors generated (state x move), all ranks
    per_level_seconds: list[float] = field(default_factory=list)
    solutions: list[str | None] | None = None  # with_paths: a shortest move string per puzzle ('UDLR'), None if unsolved
    fallback_puzzles: int = 0                  # LocalBfs: puzzles that did not fit on chip and went through the hash-partitioned search
    exchanged_keys: int = 0                    # hash-partitioned search over several ranks: keys sent to their owners (all ranks, all levels)


@dataclass
class BfsStats:
    """Per-puzzle tallies ts_bfs_hash_insert keeps on the device (CudaBfsKernels.insert(stats=...))."""
    states: torch.Tensor                       # int64[P]  += 1 per new key
    solve_depth: torch.Tensor                  # int32[P]  min over goal successors of `depth`
    goal_keys: torch.Tensor | None             # int64[2, P]  with_paths: a goal successor at that depth, and the state it was generated from
    depth: int = 0                             # depth of the keys being inserted


class CudaBfsKernels:
    """ctypes front-end of the ts_bfs_* entry points for one puzzle table."""

    WON_CAPACITY = 1 << 16

    def __init__(self, table: BatchedTilerSliderEnv):
        if table.size > 8 or not 1 <= table.n_tiles <= 8:
            raise ValueError("BFS supports board sizes up to 8 with 1 to 8 tiles")
        if table.n_tiles > 4 and table.n_envs > 1:
            raise ValueError("more than 4 tiles: the key has no room for a puzzle id, solve one puzzle at a time")
        self.t, self.lib, self.device = table, lib(), table.device
        self._won_buf = None
        self.last_won = None
        self._bufs: dict[str, torch.Tensor] = {}
        self._flip = 0

    # Level buffers live in a workspace that only ever grows, geometrically: a search whose frontier
    # swells level after level would otherwise send the caching allocator to cudaMalloc at every
    # level (measured: 50 cudaMallocs = 0.31 of 0.45 s for a 2.2e8-state search).
    def workspace(self, name: str, n: int) -> torch.Tensor:
        buf = self._bufs.get(name)
        if buf is None or buf.numel() < n:
            buf = torch.empty(max(n, 2 * (0 if buf is None else buf.numel())), dtype=torch.int64, device=self.device)
            self._bufs[name] = buf
        return buf[:n]

    def reserve(self, frontier_states: int) -> None:
        """Size the workspace for frontiers of up to `frontier_states` keys ahead of a search."""
        for name, n in (("out0", frontier_states), ("out1", frontier_states), ("succ", 4 * frontier_states)):
            self.workspace(name, n)

    def _args(self, **kw) -> BfsArgs:
        t = self.t
        base = dict(size=t.size, n_tiles=t.n_tiles, goal_mode=t.goal_mode, never_win=int(t.never_win), n_ranks=1,
                    puzzle_capacity=t.capacity, d_walls=t._walls.data_ptr(), d_targets_packed=t._targets.data_ptr(),
                    d_init=t._init.data_ptr())
        base.update(kw)
        return BfsArgs(**base)

    def _call(self, fn, a: BfsArgs, what: str):
        with torch.cuda.device(self.device):
            check(fn(C.byref(a), torch.cuda.current_stream(self.device).cuda_stream), what)

    def seed(self) -> torch.Tensor:
        out = torch.empty(self.t.n_envs, dtype=torch.int64, device=self.device)
        self._call(self.lib.ts_bfs_seed, self._args(n_items=self.t.n_envs, d_out_keys=out.data_ptr()), "ts_bfs_seed")
        return out

    def expand(self, frontier: torch.Tensor) -> torch.Tensor:
        """Successor keys, 4 per frontier key (bit 63 of the input keys is ignored).  The result
        lives in the workspace: it is valid until the next expand."""
        out = self.workspace("succ", 4 * frontier.numel())
        self._call(self.lib.ts_bfs_expand, self._args(n_items=frontier.numel(), d_in_keys=frontier.data_ptr(),
                                                      d_out_keys=out.data_ptr()), "ts_bfs_expand")
        return out

    def partition(self, keys: torch.Tensor, n_ranks: int, parents: torch.Tensor | None = None):
        """Bucket keys by owner rank (NONE dropped).  Returns (bucketed keys, bucket sizes, bucketed
        parents or None): with `parents` = the frontier `keys` was expanded from, the parent of
        every key is written next to it, in the same order."""
        counts = torch.zeros(n_ranks, dtype=torch.int64, device=self.device)
        a = self._args(n_items=keys.numel(), n_ranks=n_ranks, d_in_keys=keys.data_ptr(), d_counts=counts.data_ptr())
        self._call(self.lib.ts_bfs_partition_count, a, "ts_bfs_partition_count")
        sizes = counts.tolist()                                    # host copy: the all-to-all needs split sizes
        cursor = torch.cumsum(counts, 0) - counts
        out = self.workspace("send", sum(sizes))
        out_par = self.workspace("send_par", sum(sizes)) if parents is not None else None
        a = self._args(n_items=keys.numel(), n_ranks=n_ranks, d_in_keys=keys.data_ptr(), d_counts=cursor.data_ptr(),
                       d_out_keys=out.data_ptr(),
                       d_parent_keys=None if parents is None else parents.data_ptr(),
                       d_out_parents=None if parents is None else out_par.data_ptr())
        self._call(self.lib.ts_bfs_partition_scatter, a, "ts_bfs_partition_scatter")
        return out, sizes, out_par

    def new_table(self, capacity: int) -> torch.Tensor:
        return torch.full((capacity,), NONE, dtype=torch.int64, device=self.device)

    # ---- device-driven levels: frontier sizes stay on the device ------------------------------
    def levels_on_device(self, table: torch.Tensor, front: list, succ: torch.Tensor, lvl: torch.Tensor,
                         first_depth: int, n_levels: int, parent_table: torch.Tensor | None,
                         stats: "BfsStats | None", known_frontier: int = -1) -> None:
        """ts_bfs_levels: expand level d and insert its successors as level d+1, for n_levels
        consecutive levels, without the host knowing any frontier size: lvl is int64[levels, 4] =
        (new keys, goal successors, overflow, -) per level; front[d & 1] holds lvl[d, 0] keys."""
        kw = {}
        if stats is not None:
            kw = dict(d_states_per_puzzle=stats.states.data_ptr(), d_solve_depth=stats.solve_depth.data_ptr(),
                      d_goal_keys=None if stats.goal_keys is None else stats.goal_keys[0].data_ptr(),
                      d_goal_parents=None if stats.goal_keys is None else stats.goal_keys[1].data_ptr())
        a = self._args(table_capacity=table.numel(), d_table=table.data_ptr(),
                       d_table_parent=None if parent_table is None else parent_table.data_ptr(), **kw)
        with torch.cuda.device(self.device):
            check(self.lib.ts_bfs_levels(C.byref(a), first_depth, n_levels, front[0].data_ptr(), front[1].data_ptr(),
                                         succ.data_ptr(), lvl.data_ptr(), front[0].numel(), known_frontier,
                                         torch.cuda.current_stream(self.device).cuda_stream), "ts_bfs_levels")

    # ---- exchange through NVLink peer memory (ts_bfs_expand_exchange) ----------------------
    XHDR = 16                                   # TS_BFS_XHDR: header words ahead of the two inboxes

    def setup_peer_exchange(self, group, inbox_capacity: int) -> bool:
        """Allocate this rank's exchange buffer (two inboxes + cursors) in symmetric memory and
        map every peer's buffer (torch.distributed._symmetric_memory: CUDA VMM handles over
        NVLink).  Returns False when peer mapping is not available; the caller then keeps the
        NCCL all-to-all path."""
        try:
            import torch.distributed._symmetric_memory as symm
            group = group if group is not None else dist.group.WORLD
            buf = symm.empty(self.XHDR + 2 * inbox_capacity, dtype=torch.int64, device=self.device)
            hdl = symm.rendezvous(buf, group)
        except Exception as e:                  # no peer access / no fabric handles
            self.peer_exchange_error = repr(e)
            return False
        buf[: self.XHDR].zero_()
        self._xbuf, self._xhdl, self._xcap = buf, hdl, int(inbox_capacity)
        self._xpeers = torch.tensor(list(hdl.buffer_ptrs), dtype=torch.int64, device=self.device)
        self._xworld = len(hdl.buffer_ptrs)
        self._xcounts = torch.zeros(4, dtype=torch.int64, device=self.device)
        torch.cuda.synchronize(self.device)
        hdl.barrier()                           # every header is zero before anyone sends
        return True

    def expand_exchange(self, frontier: torch.Tensor, parity: int) -> None:
        """K4x: successors of `frontier` go straight into inbox `parity` of their owner ranks;
        self._xcounts[3] accumulates the number of keys this rank sent."""
        a = self._args(n_items=frontier.numel(), n_ranks=self._xworld, d_in_keys=frontier.data_ptr(),
                       d_counts=self._xcounts.data_ptr(), d_peer_bufs=self._xpeers.data_ptr(),
                       inbox_capacity=self._xcap, parity=parity)
        self._call(self.lib.ts_bfs_expand_exchange, a, "ts_bfs_expand_exchange")

    def expand_exchange_on_device(self, front: torch.Tensor, n_ptr: int, parity: int, xcounts: torch.Tensor) -> None:
        """K4x on a frontier whose size sits in device memory (*n_ptr); xcounts = int64[4] of this
        level: [2] overflow, [3] keys sent."""
        a = self._args(n_items=front.numel(), n_ranks=self._xworld, d_in_keys=front.data_ptr(),
                       d_counts=xcounts.data_ptr(), d_peer_bufs=self._xpeers.data_ptr(),
                       inbox_capacity=self._xcap, parity=parity, d_n_items=n_ptr, n_items_scale=1)
        self._call(self.lib.ts_bfs_expand_exchange, a, "ts_bfs_expand_exchange")

    def insert_inbox_on_device(self, table: torch.Tensor, parity: int, out: torch.Tensor, counts: torch.Tensor,
                               stats: "BfsStats | None", depth: int) -> None:
        """K5 over what arrived in inbox `parity` (its arrival cursor is the item count, read on
        the device); new keys -> out, counters -> counts = int64[4] of the new level."""
        kw = {}
        if stats is not None:
            kw = dict(d_states_per_puzzle=stats.states.data_ptr(), d_solve_depth=stats.solve_depth.data_ptr(),
                      d_goal_keys=None, depth=depth)
        o = self.XHDR + parity * self._xcap
        a = self._args(n_items=self._xcap, table_capacity=table.numel(), out_capacity=out.numel(),
                       d_in_keys=self._xbuf[o:].data_ptr(), d_out_keys=out.data_ptr(), d_table=table.data_ptr(),
                       d_counts=counts.data_ptr(), d_n_items=self._xbuf[parity:].data_ptr(), n_items_scale=1, **kw)
        self._call(self.lib.ts_bfs_hash_insert, a, "ts_bfs_hash_insert")

    def inbox(self, parity: int, n: int) -> torch.Tensor:
        o = self.XHDR + parity * self._xcap
        return self._xbuf[o: o + n]

    def insert(self, table: torch.Tensor, keys: torch.Tensor, parents: torch.Tensor | None = None,
               parent_table: torch.Tensor | None = None, stats: "BfsStats | None" = None,
               parent_per_item: bool = False) -> tuple[torch.Tensor, int]:
        """Insert keys; returns (keys that were new, with their goal bit; #goal successors seen).
        With `parent_table` (same capacity as `table`) every new key also records its parent:
        `parents` must be the frontier `keys` was expanded from (None for roots), or, with
        `parent_per_item`, one parent per key (what `partition` wrote and the exchange delivered).
        The new keys live in one of two alternating workspace buffers: valid until the insert after next."""
        out = self.workspace(f"out{self._flip}", keys.numel())
        self._flip ^= 1
        counts = torch.zeros(4, dtype=torch.int64, device=self.device)
        kw = {}
        if stats is not None:       # per-puzzle tallies kept by the kernel itself
            kw = dict(d_states_per_puzzle=stats.states.data_ptr(), d_solve_depth=stats.solve_depth.data_ptr(),
                      d_goal_keys=None if stats.goal_keys is None else stats.goal_keys[0].data_ptr(),
                      d_goal_parents=None if stats.goal_keys is None else stats.goal_keys[1].data_ptr(), depth=stats.depth)
        else:                       # hand the goal successors back to the caller instead
            if self._won_buf is None:
                self._won_buf = torch.empty(self.WON_CAPACITY, dtype=torch.int64, device=self.device)
            kw = dict(d_won_keys=self._won_buf.data_ptr(), won_capacity=self.WON_CAPACITY)
        a = self._args(n_items=keys.numel(), table_capacity=table.numel(), out_capacity=out.numel(),
                       d_in_keys=keys.data_ptr(), d_out_keys=out.data_ptr(), d_table=table.data_ptr(),
                       d_counts=counts.data_ptr(),
                       d_parent_keys=None if parents is None else parents.data_ptr(),
                       d_table_parent=None if parent_table is None else parent_table.data_ptr(),
                       parent_per_item=int(parent_per_item), **kw)
        self._call(self.lib.ts_bfs_hash_insert, a, "ts_bfs_hash_insert")
        n_new, n_won, overflow, _ = counts.tolist()              # the one host sync of a BFS level
        if overflow:
            raise RuntimeError("BFS visited table is full: raise table_capacity")
        # goal successors of this call (duplicates included); None if there were too many to buffer
        self.last_won = None
        if stats is None and n_won <= self.WON_CAPACITY:
            self.last_won = self._won_buf[:n_won].clone()
        return out[:n_new], n_won


    def traceback(self, table: torch.Tensor, parent_table: torch.Tensor, goals: torch.Tensor, max_moves: int):
        """Shortest move strings: goals = int64[2, n], the goal successor of every puzzle (NONE = no
        goal) and the state it was generated from.  Returns (moves uint8[n, max_moves], lengths int32[n])."""
        n = goals.shape[1]
        moves = torch.zeros(n, max_moves, dtype=torch.uint8, device=self.device)
        lengths = torch.full((n,), -1, dtype=torch.int32, device=self.device)
        a = self._args(n_items=n, table_capacity=table.numel(), d_in_keys=goals[0].data_ptr(), d_parent_keys=goals[1].data_ptr(),
                       d_table=table.data_ptr(), d_table_parent=parent_table.data_ptr(), d_moves=moves.data_ptr(),
                       d_lengths=lengths.data_ptr(), max_moves=max_moves)
        self._call(self.lib.ts_bfs_traceback, a, "ts_bfs_traceback")
        return moves, lengths

    def trace_step(self, table: torch.Tensor, parent_table: torch.Tensor, keys: torch.Tensor, rank: int, n_ranks: int,
                   given_parents: torch.Tensor | None = None) -> torch.Tensor:
        """One traceback step for the keys this rank owns: int64[2, n] = (parent, move) per key;
        parent is INT64_MIN for NONE items and for keys of other ranks, -1 for a root, -2 for a broken
        chain -- a MAX all-reduce over the ranks assembles the step for every key.  given_parents
        (the last link of a solution): nothing is looked up, every rank answers for every key."""
        n = keys.numel()
        out = torch.zeros(2, n, dtype=torch.int64, device=self.device)
        mv = torch.zeros(n, dtype=torch.uint8, device=self.device)
        a = self._args(n_items=n, n_ranks=n_ranks, rank=rank, table_capacity=table.numel(), d_in_keys=keys.data_ptr(),
                       d_out_keys=out[0].data_ptr(), d_table=table.data_ptr(), d_table_parent=parent_table.data_ptr(),
                       d_moves=mv.data_ptr(), d_parent_keys=None if given_parents is None else given_parents.data_ptr())
        self._call(self.lib.ts_bfs_trace_step, a, "ts_bfs_trace_step")
        out[1] = mv
        return out


class BfsSolver:
    """Level-synchronous BFS over a batch of puzzles, hash-partitioned over the ranks of `group`."""

    def __init__(self, puzzles: Sequence[Puzzle] | BatchedTilerSliderEnv | None = None, *, table_capacity: int = 1 << 22,
                 device="cuda", group=None, kernels=None, n_puzzles: int | None = None, profile: bool = False,
                 exchange: str = "auto"):
        if kernels is None:
            table = puzzles if isinstance(puzzles, BatchedTilerSliderEnv) else \
                BatchedTilerSliderEnv.from_puzzles(list(puzzles), device=device)
            kernels = CudaBfsKernels(table)
            n_puzzles = table.n_envs
        self.k = kernels
        self.n_puzzles = int(n_puzzles)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        if table_capacity & (table_capacity - 1):
            raise ValueError("table_capacity must be a power of two")
        self.table_capacity = table_capacity
        # how successors reach their owner rank: "nccl" = bucket + all_to_all_single; "p2p" = the
        # expand kernel writes them into the owners' inboxes through NVLink peer memory; "auto" =
        # p2p when the peer mapping can be set up
        if exchange not in ("auto", "nccl", "p2p"):
            raise ValueError("exchange must be 'auto', 'nccl' or 'p2p'")
        self.exchange = "nccl"
        if self.world > 1 and exchange != "nccl" and isinstance(self.k, CudaBfsKernels):
            ok = self.k.setup_peer_exchange(group, max(1 << 20, table_capacity // 2))
            flag = torch.tensor([int(ok)], device=self.k.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)          # all ranks or none
            if int(flag.item()):
                self.exchange = "p2p"
            elif exchange == "p2p":
                raise RuntimeError(f"peer-memory exchange unavailable: {getattr(self.k, 'peer_exchange_error', 'a peer failed')}")
        self.profile = profile          # synchronise after every phase and sum wall time per phase into self.phase_seconds
        self.phase_seconds: dict[str, float] = {}

    def _timed(self, name, fn, *a):
        if not self.profile:
            return fn(*a)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn(*a)
        torch.cuda.synchronize()
        self.phase_seconds[name] = self.phase_seconds.get(name, 0.0) + time.perf_counter() - t0
        return r

    # ---- one exchange: every key travels to the rank that owns it -------------------------
    def _exchange(self, keys: torch.Tensor, parents: torch.Tensor | None = None):
        """Returns (keys this rank owns, anything_sent_anywhere, their parents or None).  Two
        collectives: an all_gather of the per-owner bucket sizes of every rank -- it doubles as the
        termination test, a search is over when no rank has anything to send -- and the all-to-all
        of the keys themselves (a second one for the parents, when a search records them: `parents`
        is the frontier `keys` was expanded from)."""
        if self.world == 1:
            return keys, bool(keys.numel()), None
        send, sizes, send_par = self._timed("partition", self.k.partition, keys, self.world, parents)

        def gather_sizes():
            mine = torch.tensor(sizes, dtype=torch.int64, device=send.device)
            allsz = torch.empty(self.world * self.world, dtype=torch.int64, device=send.device)
            dist.all_gather_into_tensor(allsz, mine, group=self.group)
            return allsz.view(self.world, self.world).tolist()       # m[src][dst]
        m = self._timed("all_gather_sizes", gather_sizes)
        rs = [m[src][self.rank] for src in range(self.world)]
        if not any(any(row) for row in m):
            return send[:0], False, None
        ws = getattr(self.k, "workspace", None)

        def deliver(name, what):
            recv = ws(name, sum(rs)) if ws else torch.empty(sum(rs), dtype=torch.int64, device=send.device)
            self._timed("all_to_all", lambda: dist.all_to_all_single(recv, what, rs, sizes, group=self.group))
            return recv
        return deliver("recv", send), True, None if send_par is None else deliver("recv_par", send_par)

    def _peer_level(self, parents: torch.Tensor, parity: int) -> tuple[torch.Tensor, bool]:
        """One level of the peer-memory exchange: K4x, then one all-reduce of the sent counts --
        it orders the ranks (every rank's K4x is complete, so every inbox is) and tells whether
        anything is left anywhere -- then this rank's arrivals are read from its own inbox."""
        k = self.k
        k._xcounts.zero_()
        k.expand_exchange(parents, parity)
        sent = k._xcounts[3:4].clone()
        dist.all_reduce(sent, group=self.group)
        n_sent, n_in, overflow = torch.cat([sent, k._xbuf[parity: parity + 1], k._xbuf[2:3] + k._xcounts[2:3]]).tolist()
        if overflow:
            raise RuntimeError("BFS exchange inbox is full: raise table_capacity")
        k._xbuf[parity: parity + 1].zero_()        # nobody writes this inbox again before the level after next
        return k.inbox(parity, n_in), bool(n_sent)

    def _solve_p2p_on_device(self, max_depth: int, per_puzzle: bool) -> BfsResult:
        """Several ranks, peer-memory exchange, frontier sizes on the device.  Per level and rank:
        K4x (frontier -> the owners' inboxes), an all-reduce of the sent counts (orders the ranks,
        and its result is what the termination test reads later), K5 over the own inbox (item
        count = its arrival cursor, read on the device), cursor reset -- LEVELS_PER_SYNC levels in
        a row without a host read-back.  Every rank takes the same decisions because it decides
        on all-reduced numbers only."""
        k, P, dev = self.k, self.n_puzzles, self.k.device
        table = k.new_table(self.table_capacity)
        states_pp = torch.zeros(P, dtype=torch.int64, device=dev) if per_puzzle else None
        depth_pp = torch.full((P,), 1 << 30, dtype=torch.int32, device=dev) if per_puzzle else None
        stats = BfsStats(states_pp, depth_pp, None) if per_puzzle else None
        cap = max(1 << 16, P, min(self.table_capacity // 4, 1 << 28))
        front = [k.workspace("front0", cap), k.workspace("front1", cap)]
        n_lvl = 256
        lvl = torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)       # per level: new keys, goal successors, overflow, -
        xlvl = torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)      # per level: -, -, inbox overflow, keys sent (all-reduced)
        # depth 0: seeds to their owners through the NCCL path, ordinary insert
        mine, _, _ = self._exchange(k.seed())
        seeds, _ = k.insert(table, mine, None, None, stats) if stats is not None else k.insert(table, mine)
        front[0][: seeds.numel()].copy_(seeds)
        lvl[0, 0] = seeds.numel()
        depth, rows, xrows = 0, None, None
        while depth < max_depth:
            batch = min(self.LEVELS_PER_SYNC, max_depth - depth)
            if depth + batch + 1 > n_lvl:
                lvl = torch.cat([lvl, torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)])
                xlvl = torch.cat([xlvl, torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)])
                n_lvl *= 2
            for d in range(depth, depth + batch):
                parity = d & 1
                k.expand_exchange_on_device(front[parity], lvl[d].data_ptr(), parity, xlvl[d])
                dist.all_reduce(xlvl[d, 3:4], group=self.group)
                k.insert_inbox_on_device(table, parity, front[parity ^ 1], lvl[d + 1], stats, d + 1)
                k._xbuf[parity: parity + 1].zero_()    # nobody writes this inbox again before the level after next
            depth += batch
            both = torch.cat([lvl[: depth + 1], xlvl[: depth + 1]], dim=1).tolist()      # the host sync of the batch
            rows, xrows = [r[:4] for r in both], [r[4:] for r in both]
            if any(r[2] for r in rows) or any(x[2] for x in xrows) or int(k._xbuf[2].item()):
                raise RuntimeError("BFS visited table is full (or an inbox / frontier outgrew its buffer): raise table_capacity")
            if any(x[3] == 0 for x in xrows[:depth]):      # a level in which no rank sent anything: the search is over
                break
        # tallies over all ranks; counter rows past the end of the search are zero
        tally = lvl[: depth + 1, :2].t().contiguous()       # [new keys per level, goal successors per level]
        dist.all_reduce(tally, group=self.group)
        levels, won_per_level = tally[0].tolist(), tally[1].tolist()
        while len(levels) > 1 and levels[-1] == 0:
            levels.pop()
        generated = 4 * sum(levels[:max_depth] if len(levels) > max_depth else levels)   # 4 per key of every expanded level
        solve_depth = next((d for d, w in enumerate(won_per_level) if w), -1)
        if per_puzzle:
            dist.all_reduce(states_pp, group=self.group)
            dist.all_reduce(depth_pp, op=dist.ReduceOp.MIN, group=self.group)
            depth_pp = torch.where(depth_pp >= (1 << 30), torch.full_like(depth_pp, -1), depth_pp)
        return BfsResult(n_states=sum(levels), levels=levels, solve_depth=solve_depth, states_per_puzzle=states_pp,
                         solve_depth_per_puzzle=depth_pp, generated=generated,
                         exchanged_keys=int(sum(x[3] for x in (xrows or []))))

    LEVELS_PER_SYNC = 16        # device-driven search: levels launched between two host read-backs
    BIG_LEVEL = 1 << 19         # frontiers from this size on get their own launch geometry and read-back

    def _solve_on_device(self, max_depth: int, per_puzzle: bool, with_paths: bool) -> BfsResult:
        """Single rank: the frontier sizes never leave the device.  The kernels read their item
        counts from the per-level counter blocks the previous insert filled, so LEVELS_PER_SYNC
        levels are launched back to back and the host only looks every so often whether the
        frontier has run dry (levels launched past that point find a zero count and do nothing).
        A host-driven level costs a round trip of 0.1-0.2 ms, and most levels of a search are
        far smaller than that."""
        k, P, dev = self.k, self.n_puzzles, self.k.device
        table = k.new_table(self.table_capacity)
        parent_table = k.new_table(self.table_capacity) if with_paths else None
        goal_keys = torch.full((2, P), NONE, dtype=torch.int64, device=dev) if with_paths else None
        states_pp = torch.zeros(P, dtype=torch.int64, device=dev) if per_puzzle else None
        depth_pp = torch.full((P,), 1 << 30, dtype=torch.int32, device=dev) if per_puzzle else None
        stats = BfsStats(states_pp, depth_pp, goal_keys) if per_puzzle else None
        cap = max(1 << 16, P, min(self.table_capacity // 4, 1 << 28))          # frontier capacity
        front = [k.workspace("front0", cap), k.workspace("front1", cap)]
        succ = k.workspace("succ", 4 * cap)
        n_lvl = 256
        lvl = torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)
        # depth 0 through the ordinary insert (host knows P); its new keys land in the workspace
        # buffer out{flip}: copy them to front0 and seed the counters
        seeds, _ = k.insert(table, k.seed(), None, parent_table, stats) if stats is not None else \
            k.insert(table, k.seed(), None, parent_table)
        front[0][: seeds.numel()].copy_(seeds)
        lvl[0, 0] = seeds.numel()
        depth, rows, known = 0, None, seeds.numel()
        while depth < max_depth:
            # a big level is worth a grid of its own size and a read-back of its own; small ones are
            # launched LEVELS_PER_SYNC at a time as single persistent waves that find their size on the device
            big = known >= self.BIG_LEVEL
            batch = 1 if big else min(self.LEVELS_PER_SYNC, max_depth - depth)
            if depth + batch + 1 > n_lvl:                                     # more counter blocks
                lvl = torch.cat([lvl, torch.zeros(n_lvl, 4, dtype=torch.int64, device=dev)])
                n_lvl *= 2
            k.levels_on_device(table, front, succ, lvl, depth, batch, parent_table, stats, known if big else -1)
            depth += batch
            rows = lvl[: depth + 1].tolist()                                  # the only host sync of the batch
            if any(r[2] for r in rows):
                raise RuntimeError("BFS visited table is full (or a frontier outgrew its buffer): raise table_capacity")
            if any(r[0] == 0 for r in rows):
                break
            known = rows[-1][0]
        rows = rows if rows is not None else lvl[:1].tolist()
        levels = [r[0] for r in rows]
        won_per_level = [r[1] for r in rows]
        if 0 in levels:
            cut = levels.index(0)
            levels, won_per_level = levels[:cut], won_per_level[: cut + 1]
        generated = 4 * sum(levels[:max_depth] if len(levels) > max_depth else levels)
        solve_depth = next((d for d, w in enumerate(won_per_level) if w), -1)
        if per_puzzle:
            depth_pp = torch.where(depth_pp >= (1 << 30), torch.full_like(depth_pp, -1), depth_pp)
        solutions = None
        if with_paths:
            max_moves = max(1, int(depth_pp.max()))
            moves, lengths = k.traceback(table, parent_table, goal_keys, max_moves)
            mv, ln = moves.cpu().tolist(), lengths.cpu().tolist()
            solutions = ["".join("UDLR"[m] for m in mv[i][:ln[i]]) if ln[i] >= 0 else None for i in range(P)]
        return BfsResult(n_states=sum(levels), levels=levels, solve_depth=solve_depth, states_per_puzzle=states_pp,
                         solve_depth_per_puzzle=depth_pp, generated=generated, solutions=solutions)

    def _trace_over_ranks(self, table, parent_table, goal_keys: torch.Tensor, max_moves: int):
        """Shortest move strings when the visited set (and its parent links) is spread over the
        ranks.  A puzzle has ONE goal state (the targets, canonical), so exactly one rank holds its
        goal key; after a MAX all-reduce every rank knows all of them.  Then one collective per
        move: each rank looks up the keys it owns (ts_bfs_trace_step), the MAX all-reduce of the
        (parent, move) pairs gives every rank the whole step.  Returns what `traceback` returns."""
        k, dev, P = self.k, goal_keys.device, goal_keys.shape[1]
        goals = torch.where(goal_keys == NONE, goal_keys, goal_keys & 0x7FFFFFFFFFFFFFFF)     # [2, P]: goal successor, its parent
        dist.all_reduce(goals, op=dist.ReduceOp.MAX, group=self.group)
        cur, last_from = goals[0].contiguous(), goals[1].contiguous()
        has_goal = cur != NONE
        moves = torch.zeros(P, max_moves, dtype=torch.uint8, device=dev)
        lengths = torch.zeros(P, dtype=torch.int64, device=dev)
        broken = torch.zeros(P, dtype=torch.bool, device=dev)
        for step in range(max_moves + 1):
            if step == 0:     # the last link is the recorded one (a puzzle that starts on its goal: the root has no parent)
                pm = k.trace_step(table, parent_table, cur, self.rank, self.world, given_parents=last_from)
            else:
                pm = k.trace_step(table, parent_table, cur, self.rank, self.world)
                dist.all_reduce(pm, op=dist.ReduceOp.MAX, group=self.group)
            parent, move = pm[0], pm[1]
            active = parent >= 0
            broken |= (parent < -1) & (cur != NONE)          # -2: broken chain; INT64_MIN: no rank knew the key
            if step == 0:
                broken |= (parent == -1) & (cur != NONE)     # a goal successor always has a parent
            if step == max_moves:
                broken |= active                             # longer than the depth the search reported
                break
            if not bool(active.any()):
                break
            moves[:, step] = torch.where(active, move, torch.zeros_like(move)).to(torch.uint8)
            lengths += active
            cur = torch.where(active, parent, torch.full_like(parent, NONE))
        # the chain was walked goal -> root: reverse each string over its own length
        idx = (lengths[:, None] - 1 - torch.arange(max_moves, device=dev)[None, :]).clamp_(min=0)
        moves = moves.gather(1, idx)
        lengths = torch.where(has_goal & ~broken, lengths, torch.full_like(lengths, -1)).to(torch.int32)
        return moves, lengths

    def solve(self, max_depth: int = 1 << 20, per_puzzle: bool = True, with_paths: bool = False,
              device_driven: bool | None = None) -> BfsResult:
        """Search every puzzle to exhaustion (or max_depth).  with_paths: also record parents and
        return a shortest solution string per puzzle (SURVEY 8(f) N4); over several ranks the
        parents travel with the keys (host-driven levels, all-to-all exchange) and the chains are
        walked one step per collective, every rank answering for the keys it owns.
        device_driven (default: on for a single rank on the CUDA kernels): see _solve_on_device."""
        k, P = self.k, self.n_puzzles
        if with_paths and not per_puzzle:
            raise ValueError("with_paths needs per_puzzle statistics")
        dist_paths = with_paths and self.world > 1
        can = self.world == 1 and isinstance(k, CudaBfsKernels) and not self.profile
        can_p2p = self.world > 1 and self.exchange == "p2p" and not self.profile and not with_paths
        if device_driven is None:
            device_driven = can or can_p2p
        if device_driven:
            if can_p2p:
                return self._solve_p2p_on_device(max_depth, per_puzzle)
            if not can:
                raise ValueError("device-driven search needs the CUDA kernels on one rank, or the peer-memory "
                                 "exchange on several (and no phase profiling)")
            return self._solve_on_device(max_depth, per_puzzle, with_paths)
        table = k.new_table(self.table_capacity)
        parent_table = k.new_table(self.table_capacity) if with_paths else None
        dev = k.device
        if hasattr(k, "reserve"):
            k.reserve(max(1 << 16, min(self.table_capacity // 8, 1 << 27)))
        goal_keys = torch.full((2, P), NONE, dtype=torch.int64, device=dev) if with_paths else None
        states_pp = torch.zeros(P, dtype=torch.int64, device=dev) if per_puzzle else None
        depth_pp = torch.full((P,), 1 << 30, dtype=torch.int32, device=dev) if per_puzzle else None
        single_puzzle_keys = getattr(k, "t", None) is not None and k.t.n_tiles > 4   # no id bits in the key

        def pid_of(keys):
            return torch.zeros_like(keys) if single_puzzle_keys else (keys >> 32) & 0x7FFFFFFF

        # depth 0: every rank seeds all puzzles and keeps the keys it owns (the owner receives one
        # copy per rank; dedup keeps one)
        # per-puzzle tallies: inside the insert kernel when the kernels offer it, else with torch ops
        stats = BfsStats(states_pp, depth_pp, goal_keys) if per_puzzle and isinstance(k, CudaBfsKernels) else None

        def insert(keys, parents, depth):
            if stats is not None:
                stats.depth = depth
            if with_paths:                                    # several ranks: one parent per key, as delivered
                return k.insert(table, keys, parents, parent_table, stats, parent_per_item=dist_paths and parents is not None)
            return k.insert(table, keys, None, None, stats) if stats is not None else k.insert(table, keys)

        mine, _, _ = self._exchange(k.seed())
        frontier, _ = insert(mine, None, 0)
        # per-rank tallies; summed over the ranks once, after the search
        local_levels, local_won, generated = [frontier.numel()], [0], 0

        def tally_states(keys):                               # frontier buffers are recycled: count per level
            if per_puzzle and stats is None and keys.numel():
                states_pp.add_(torch.bincount(pid_of(keys), minlength=P)[:P])

        tally_states(frontier)
        depth = 0
        while depth < max_depth:
            parents = frontier                                # expand / insert ignore the goal bit of their inputs
            recv_parents = parents
            if self.exchange == "p2p" and not dist_paths:
                recv, alive = self._timed("expand_exchange", self._peer_level, parents, depth & 1)
            else:
                succ = self._timed("expand", k.expand, parents)
                # single rank: successors go straight to the table (it skips NONE) and successor i stays
                # next to its parent i // 4; several ranks: bucket by owner and exchange (the fused
                # peer-memory kernel moves keys only, so a search that records parents takes this path)
                recv, alive, got = self._exchange(succ, parents if dist_paths else None)
                recv_parents = got if dist_paths else parents
            if not alive:
                break
            depth += 1
            generated += 4 * parents.numel()
            frontier, n_won = self._timed("insert", insert, recv, recv_parents, depth)
            if per_puzzle and n_won and stats is None:
                won = getattr(k, "last_won", None)
                if won is None:                              # stand-in kernels / overflowed buffer: scan
                    won = recv[(recv < 0) & (recv != NONE)]
                if with_paths:                               # first goal successor seen for a puzzle = a shortest solution
                    at = torch.nonzero((recv < 0) & (recv != NONE)).flatten()
                    won = recv[at]
                    won_from = recv_parents[at if dist_paths else at // 4]
                    fresh = depth_pp[pid_of(won)] >= (1 << 30)
                    goal_keys[0, pid_of(won[fresh])] = won[fresh]
                    goal_keys[1, pid_of(won[fresh])] = won_from[fresh] & 0x7FFFFFFFFFFFFFFF
                d = torch.full((won.numel(),), depth, dtype=torch.int32, device=dev)
                depth_pp.scatter_reduce_(0, pid_of(won), d, reduce="amin")
            local_levels.append(frontier.numel())
            local_won.append(n_won)
            self._timed("tally", tally_states, frontier)
        # ---- tallies over all ranks (every rank ran the same number of levels) ---------------
        tally = torch.tensor([local_levels, local_won], dtype=torch.int64, device=dev)
        gen = torch.tensor([generated], dtype=torch.int64, device=dev)
        if self.world > 1:
            dist.all_reduce(tally, group=self.group)
            dist.all_reduce(gen, group=self.group)
        levels, won_per_level = tally[0].tolist(), tally[1].tolist()
        while len(levels) > 1 and levels[-1] == 0:
            levels.pop()
        solve_depth = next((d for d, w in enumerate(won_per_level) if w), -1)
        generated = int(gen.item())
        if per_puzzle and self.world > 1:
            dist.all_reduce(states_pp, group=self.group)
            dist.all_reduce(depth_pp, op=dist.ReduceOp.MIN, group=self.group)
        if per_puzzle:
            depth_pp = torch.where(depth_pp >= (1 << 30), torch.full_like(depth_pp, -1), depth_pp)
        solutions = None
        if with_paths:
            max_moves = max(1, int(depth_pp.max()))
            if dist_paths:
                moves, lengths = self._trace_over_ranks(table, parent_table, goal_keys, max_moves)
            else:
                moves, lengths = k.traceback(table, parent_table, goal_keys, max_moves)
            mv, ln = moves.cpu().tolist(), lengths.cpu().tolist()
            solutions = ["".join("UDLR"[m] for m in mv[i][:ln[i]]) if ln[i] >= 0 else None for i in range(P)]
        return BfsResult(n_states=sum(levels), levels=levels, solve_depth=solve_depth, states_per_puzzle=states_pp,
                         solve_depth_per_puzzle=depth_pp, generated=generated, solutions=solutions)


class OnChipSearch:
    """What the front-ends of the on-chip searches (K6 `CudaLocalKernels`, K9 `CudaOptimalMoves`, K10
    `CudaStateTable`) share: the plan of a launch, the rule that picks it, the launch on the shared
    or the device-memory-bitmap instance and the per-CTA scratch slabs.  `want_ctas` fixes the CTAs per SM; `want_queue` caps the ring entries kept in shared
    memory (tests: force the slab)."""

    N_LEVELS = 256                  # levels a search may have on chip (the kernels' level buffers)
    SMEM_PER_SM = 228 * 1024
    STATIC_SMEM = 4 * 1024          # the kernel's static shared memory + the per-CTA reservation
    MAX_SCRATCH_BYTES = 4 << 30
    CTAS_PER_SM = ""                # the library's occupancy query of the front-end's kernel
    GMEM_CTAS_PER_SM = ""           # ... of its device-memory-bitmap instance
    TABLE_CTAS_PER_SM = ""          # ... of its hash-table instance (5 to 8 tiles)
    GMEM_SHAPES = ((7, 4), (8, 4))  # (size, tiles) with device instances: boards a shared bitmap may not hold
    ARGS = None                     # the argument struct of the front-end's entry points (K9, K10: _args)

    def __init__(self, table: BatchedTilerSliderEnv, ctas_per_sm: int | None = None, queue_smem: int | None = None,
                 table_slots: int | None = None):
        self.t, self.lib, self.device = table, lib(), table.device
        self.want_ctas = ctas_per_sm
        self.want_queue = queue_smem
        self.want_slots = table_slots   # tests: force a small hash table (and so a small bound)
        self._plans: dict = {}
        self._scratch: dict[str, torch.Tensor] = {}
        self.counters = torch.zeros(4, dtype=torch.int64, device=self.device)   # K9, K10: of the last call, see include/tiler_slider.h

    def _args(self, **kw):
        """The front-end's argument struct for its table (K9 and K10's fields), with kw set."""
        t = self.t
        base = dict(size=t.size, n_tiles=t.n_tiles, goal_mode=t.goal_mode, never_win=int(t.never_win), capacity=t.capacity,
                    d_walls=t._walls.data_ptr(), d_targets_packed=t._targets.data_ptr(), d_pos=t._pos.data_ptr())
        base.update(kw)
        return self.ARGS(**base)

    def plan(self, f_max: int) -> dict | None:
        """The plan for states on up to f_max free cells."""
        return self._plan(f_max, f_max)

    def _plan(self, key, f_max: int) -> dict | None:
        """Shared-memory split and grid for states of T tiles on up to f_max free cells, cached under
        `key` (None: the bitmap does not fit one CTA per SM).  The bitmap must hold F!/(F-T)! bits;
        the more CTAs fit an SM next to it, the better the level-synchronisation latency of one
        puzzle hides behind the others, so the ring gets what is left of the CTA's share."""
        if key not in self._plans:
            self._plans[key] = self._fit(f_max, gmem=False) or {}
        return self._plans[key] or None

    def _plan_gmem(self, f_max: int) -> dict | None:
        """The plan of the device-memory-bitmap instance for up to f_max free cells (None: no such
        instance for this shape), marked gmem=True: the same CTA-per-SM loop as _plan with the ring
        alone in shared memory, and the grid capped so that its bitmaps (grid x F!/(F-T)! bits, 1.9 MB
        per CTA at F = 64) stay within MAX_SCRATCH_BYTES."""
        key = ("gmem", f_max)
        if key not in self._plans:
            ok = (self.t.size, self.t.n_tiles) in self.GMEM_SHAPES
            self._plans[key] = (self._fit(f_max, gmem=True) if ok else None) or {}
        return self._plans[key] or None

    def _fit(self, f_max: int, gmem: bool) -> dict | None:
        bits = 1
        for i in range(self.t.n_tiles):                          # arrangements of T distinct tiles on f_max cells
            bits *= max(f_max - i, 1)
        bitmap_bytes = max(16, -(-bits // 128) * 16)
        smem_bitmap = 0 if gmem else bitmap_bytes
        query = getattr(self.lib, self.GMEM_CTAS_PER_SM if gmem else self.CTAS_PER_SM)
        for k in ([self.want_ctas] if self.want_ctas else [8, 6, 5, 4, 3, 2, 1]):
            budget = self.SMEM_PER_SM // k - self.STATIC_SMEM
            if smem_bitmap + 1024 > budget:
                continue
            queue = 1 << (min(budget - smem_bitmap, 64 * 1024) // 4).bit_length() - 1     # ring entries: a power of two
            if self.want_queue is not None:
                queue = max(32, 1 << (min(queue, self.want_queue).bit_length() - 1))
            a = self._args(bitmap_words=bitmap_bytes // 4, queue_smem=queue)
            got, n_sm = C.c_int(0), C.c_int(0)
            with torch.cuda.device(self.device):
                rc = query(C.byref(a), C.byref(got), C.byref(n_sm))
            if rc == 0 and got.value >= (k if self.want_ctas is None else 1):
                grid = got.value * n_sm.value
                if gmem:
                    grid = min(grid, self.MAX_SCRATCH_BYTES // bitmap_bytes)
                plan = dict(bitmap_words=bitmap_bytes // 4, queue_smem=queue, grid=grid, ctas_per_sm=got.value,
                            spill_per_cta=int(min(bits + 1, self.MAX_SCRATCH_BYTES // 4 // grid)), f_max=f_max)
                return {**plan, "gmem": True} if gmem else plan
        return None

    def _plan_table(self, max_states: int | None = None) -> dict | None:
        """The plan of the hash-table instance (5 to 8 tiles, marked table=True): the same CTA-per-SM
        loop as _plan with a ring of 8-byte entries alone in shared memory; per CTA a table of
        table_slots 8-byte slots (the largest power of two with grid x 12 x table_slots <=
        MAX_SCRATCH_BYTES, or the constructor's table_slots) and a slab of spill_per_cta =
        table_slots / 2 entries, the states an item may discover.  It does not depend on the envs'
        walls, so it needs no free-cell read-back.  max_states (state tables): that bound instead,
        spill_per_cta = max_states and table_slots the smallest power of two >= 2 x max_states, on
        that plan's ring and as many of its CTAs as fit MAX_SCRATCH_BYTES (ValueError: not one)."""
        if max_states is not None:
            key = ("table", int(max_states))
            if key not in self._plans:
                base = self._plan_table()
                if base is None:
                    return None
                spill = int(max_states)
                slots = 1 << (2 * spill - 1).bit_length()
                grid = min(base["grid"], self.MAX_SCRATCH_BYTES // (8 * slots + 8 * spill))
                if grid < 1:
                    raise ValueError(f"max_states={spill}: the table and slab of one CTA "
                                     f"({8 * slots + 8 * spill} bytes) exceed {self.MAX_SCRATCH_BYTES} bytes")
                self._plans[key] = dict(base, grid=grid, table_slots=slots, spill_per_cta=spill)
            return self._plans[key]
        if "table" not in self._plans:
            self._plans["table"] = {}
            query = getattr(self.lib, self.TABLE_CTAS_PER_SM)
            for k in ([self.want_ctas] if self.want_ctas else [8, 6, 5, 4, 3, 2, 1]):
                budget = self.SMEM_PER_SM // k - self.STATIC_SMEM
                queue = 1 << (min(budget, 64 * 1024) // 8).bit_length() - 1                    # ring entries: a power of two
                if self.want_queue is not None:
                    queue = max(32, 1 << (min(queue, self.want_queue).bit_length() - 1))
                a = self._args(bitmap_words=0, queue_smem=queue)
                got, n_sm = C.c_int(0), C.c_int(0)
                with torch.cuda.device(self.device):
                    rc = query(C.byref(a), C.byref(got), C.byref(n_sm))
                if rc == 0 and got.value >= (k if self.want_ctas is None else 1):
                    grid = got.value * n_sm.value
                    slots = self.want_slots or 1 << (self.MAX_SCRATCH_BYTES // (12 * grid)).bit_length() - 1
                    self._plans["table"] = dict(bitmap_words=0, queue_smem=queue, grid=grid, ctas_per_sm=got.value,
                                                table_slots=slots, spill_per_cta=slots // 2, table=True)
                    break
        return self._plans["table"] or None

    def search_plan(self, f_max: int, device_bitmap: bool = False) -> dict | None:
        """The plan of a query whose envs have up to f_max free cells, one rule for K9 and K10: the
        shared plan for f_max when it exists; else, with device_bitmap on a shape that has device
        instances, the gmem plan for f_max (every item of the call then runs on the device instance);
        else the plan of the most free cells that fit (fitting_free_cells), the larger envs getting
        -3.  Both instances give the same answers, so an env's answer never depends on the others."""
        if device_bitmap and self.plan(f_max) is None:
            gp = self._plan_gmem(f_max)
            if gp is not None:
                return gp
        return self.plan(self.fitting_free_cells(f_max))

    def _bitmap(self, plan: dict) -> int:
        """The device-memory bitmaps of a gmem plan (grid x bitmap_words words, contents undefined)."""
        return self._buf("bitmap", plan["grid"] * plan["bitmap_words"], torch.int32).data_ptr()

    def _launch(self, entry: str, a, plan: dict, stream) -> None:
        """Launch the library's `entry` with arguments a on plan's grid; with a gmem plan its device
        counterpart `entry`_gmem, on the bitmaps of _bitmap; with a table plan `entry`_table, on
        grid x table_slots cached 8-byte slots (contents undefined)."""
        if plan.get("table"):
            entry += "_table"
            tab = self._buf("table", plan["grid"] * plan["table_slots"], torch.int64).data_ptr()
            rc = getattr(self.lib, entry)(C.byref(a), tab, plan["table_slots"], plan["grid"], stream)
        elif plan.get("gmem"):
            entry += "_gmem"
            rc = getattr(self.lib, entry)(C.byref(a), self._bitmap(plan), plan["grid"], stream)
        else:
            rc = getattr(self.lib, entry)(C.byref(a), plan["grid"], stream)
        check(rc, entry)

    def fitting_free_cells(self, f_max: int) -> int:
        """The largest F <= f_max whose plan fits (down to F = n_tiles): the free-cell count a launch
        for envs of up to f_max free cells is planned for (K9, K10: plans keyed by free cells).  The
        kernel reports -3 for each env whose own state space exceeds that bitmap, so an env's answer
        never depends on the other envs."""
        f = f_max
        while f > self.t.n_tiles and self._plan(f, f) is None:
            f -= 1
        return f

    def _max_free_cells(self, ids: torch.Tensor | None, n: int) -> int:
        """The most free cells among the envs of n items (ts_optimal_max_free_cells; one read-back)."""
        t, dev = self.t, self.device
        f_max = torch.zeros(1, dtype=torch.int32, device=dev)
        a = OptimalMovesArgs(size=t.size, n_tiles=t.n_tiles, goal_mode=t.goal_mode, never_win=int(t.never_win), n_items=n,
                             capacity=t.capacity, d_env_ids=None if ids is None else ids.data_ptr(),
                             d_walls=t._walls.data_ptr(), d_targets_packed=t._targets.data_ptr(), d_pos=t._pos.data_ptr())
        with torch.cuda.device(dev):
            check(self.lib.ts_optimal_max_free_cells(C.byref(a), f_max.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                  "ts_optimal_max_free_cells")
        return int(f_max.item())

    def _buf(self, name: str, n: int, dtype) -> torch.Tensor:
        b = self._scratch.get(name)
        if b is None or b.numel() < n or b.dtype != dtype:
            b = torch.empty(n, dtype=dtype, device=self.device)
            self._scratch[name] = b
        return b[:n]


class CudaLocalKernels(OnChipSearch):
    """ctypes front-end of ts_bfs_local for one puzzle table: the shared-memory plan and the launch
    that searches a contiguous range of puzzles into caller-provided result tensors."""

    MAX_MOVES = 255
    CTAS_PER_SM = "ts_bfs_local_ctas_per_sm"
    GMEM_CTAS_PER_SM = "ts_bfs_local_gmem_ctas_per_sm"

    def __init__(self, table: BatchedTilerSliderEnv, ctas_per_sm: int | None = None, queue_smem: int | None = None,
                 device_bitmap: bool = False):
        if table.size > 8 or not 1 <= table.n_tiles <= 4:
            raise ValueError("the on-chip BFS covers board sizes up to 8 with 1 to 4 tiles")
        super().__init__(table, ctas_per_sm, queue_smem)
        self.device_bitmap = bool(device_bitmap)   # plan(): fall back to the device-memory bitmap (7x7 / 8x8, 4 tiles)

    def _args(self, **kw) -> BfsLocalArgs:
        t = self.t
        base = dict(size=t.size, n_tiles=t.n_tiles, goal_mode=t.goal_mode, never_win=int(t.never_win),
                    puzzle_capacity=t.capacity, d_walls=t._walls.data_ptr(), d_targets_packed=t._targets.data_ptr(),
                    d_init=t._init.data_ptr(), n_levels=self.N_LEVELS)
        base.update(kw)
        return BfsLocalArgs(**base)

    def plan(self, lo: int, hi: int) -> dict | None:
        """The plan for puzzles [lo, hi): F = the most free cells of any of them.  With device_bitmap,
        a range whose bitmap does not fit shared memory gets the gmem plan of its shape, if any."""
        t = self.t
        if (lo, hi) not in self._plans:
            blocked = t.blocked_cells()[lo:hi]
            f_max = int(t.size * t.size - blocked.sum(1).min()) if hi > lo else 1
            plan = self._plan((lo, hi), f_max)
            if plan is None and self.device_bitmap:
                plan = self._plan_gmem(f_max)
                self._plans[(lo, hi)] = plan or {}
            if plan:
                plan["smem_bytes"] = 4 * (plan["queue_smem"] + (0 if plan.get("gmem") else plan["bitmap_words"]))
        return self._plans[(lo, hi)] or None

    def puzzle(self, i: int) -> Puzzle:
        return self.t.puzzle(i)

    def search(self, lo: int, hi: int, max_depth: int, out: dict, ids: torch.Tensor | None = None) -> None:
        """Search puzzles [lo, hi) into out = {states, depth, status, levels, counters[, moves, lengths]}
        (tensors over ALL puzzles of the table); puzzles that do not fit get status != 0.  ids: search
        only these puzzles (int32 on the device, each in [lo, hi); the plan is that of the range)."""
        plan = self.plan(lo, hi)
        if plan is None:
            if ids is None:
                out["status"][lo:hi] = 1                       # nothing fits on chip
            else:
                out["status"][ids.long()] = 1
            return
        if hi <= lo or (ids is not None and ids.numel() == 0):
            return
        dev = self.device
        if ids is None:
            ids = torch.arange(lo, hi, dtype=torch.int32, device=dev) if lo else None
            n_puzzles = hi - lo
        else:
            if ids.dtype != torch.int32 or ids.device != dev or not ids.is_contiguous():
                raise ValueError("ids must be a contiguous int32 tensor on the table's device")
            n_puzzles = ids.numel()
        with_paths = out.get("lengths") is not None
        a = self._args(n_puzzles=n_puzzles, d_puzzle_ids=None if ids is None else ids.data_ptr(),
                       max_depth=min(int(max_depth), (1 << 31) - 1), bitmap_words=plan["bitmap_words"],
                       queue_smem=plan["queue_smem"], spill_per_cta=plan["spill_per_cta"],
                       d_spill=self._buf("spill", plan["grid"] * max(plan["spill_per_cta"], 1), torch.int32).data_ptr(),
                       d_parent_scratch=self._buf("parents", plan["grid"] * plan["spill_per_cta"], torch.int32).data_ptr() if with_paths else None,
                       d_states_per_puzzle=out["states"].data_ptr(), d_solve_depth=out["depth"].data_ptr(),
                       d_status=out["status"].data_ptr(), d_levels=out["levels"].data_ptr(), d_counters=out["counters"].data_ptr(),
                       d_moves=out["moves"].data_ptr() if with_paths else None,
                       d_lengths=out["lengths"].data_ptr() if with_paths else None, max_moves=self.MAX_MOVES)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            self._launch("ts_bfs_local", a, plan, stream)


def check_optimal_moves(size: int, n_tiles: int, host_io: bool, max_depth: int, what: str = "optimal_moves",
                        hash_table: bool = False) -> None:
    """The shapes ts_optimal_moves (and ts_state_table, `what`) covers, with hash_table also those
    of ts_optimal_moves_table (and ts_state_table_*_table: 5 to 8 tiles); raised before anything
    touches the device."""
    if size > 8:
        raise ValueError(f"{what} covers board sizes up to 8 (got {size})")
    if not 1 <= n_tiles <= (8 if hash_table else 4):
        raise ValueError(f"{what} covers 1 to {8 if hash_table else 4} tiles (got {n_tiles})")
    if host_io:
        raise ValueError(f"{what} is not available for host_io batches")
    if not 1 <= max_depth <= OPT_MAX_DEPTH:
        raise ValueError(f"max_depth {max_depth} outside 1..{OPT_MAX_DEPTH}")


class CudaOptimalMoves(OnChipSearch):
    """ctypes front-end of ts_optimal_moves (K9, csrc/ts_optimal.cu) for one batch: the distance to
    the goal, the optimal first moves and optionally a shortest solution of items (env id, positions:
    the env's current ones or given words).  The bitmap is sized per
    call from the most free cells among the queried envs, counted on the device (a reset pool changes
    the walls of a batch between calls), or from the most free cells one CTA can hold when that is
    fewer; the plan is cached per free-cell count."""

    CTAS_PER_SM = "ts_optimal_moves_ctas_per_sm"
    GMEM_CTAS_PER_SM = "ts_optimal_moves_gmem_ctas_per_sm"
    TABLE_CTAS_PER_SM = "ts_optimal_moves_table_ctas_per_sm"
    ARGS = OptimalMovesArgs

    def query(self, ids: torch.Tensor | None, max_depth: int, pos: torch.Tensor | None = None,
              plan: torch.Tensor | None = None, device_bitmap: bool = False,
              hash_table: bool = False) -> tuple[torch.Tensor, torch.Tensor]:
        """(distance int32[n], mask uint8[n]) of items (env `ids[i]`, positions `pos[i]`) on the
        current stream.  ids: int32 on the device, each in [0, n_envs) (None: every env); pos:
        contiguous uint8 [n, pos_bytes] on the device (None: the envs' current positions); plan:
        uint8 [max_depth, n] on the device that receives a shortest solution per item (every entry
        is written); device_bitmap: envs too large for a shared-memory bitmap are searched with one
        in device memory (search_plan); hash_table: 5 to 8 tiles are searched by K11
        (ts_optimal_moves_table, _plan_table); it changes nothing for 1 to 4 tiles."""
        t, dev = self.t, self.device
        n = t.n_envs if ids is None else ids.numel()
        distance = torch.full((n,), OPT_NOT_SEARCHED, dtype=torch.int32, device=dev)
        mask = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.counters.zero_()
        if n == 0:
            return distance, mask
        ids_ptr = None if ids is None else ids.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            # one plan with and without paths: the same grid and slab, so the same answers (the plan
            # kernel instance may fit fewer CTAs per SM; the surplus CTAs find no ticket left)
            table = hash_table and t.n_tiles >= 5
            sp = self._plan_table() if table else self.search_plan(self._max_free_cells(ids, n), device_bitmap)
            if sp is None:                       # not even T free cells fit on chip
                if plan is not None:
                    plan.fill_(255)
                return distance, mask
            a = self._args(n_items=n, d_env_ids=ids_ptr, max_depth=int(max_depth), bitmap_words=sp["bitmap_words"],
                           queue_smem=sp["queue_smem"], spill_per_cta=sp["spill_per_cta"],
                           d_spill=self._buf("spill", sp["grid"] * sp["spill_per_cta"], torch.int64 if table else torch.int32).data_ptr(),
                           d_counters=self.counters.data_ptr(), d_distance=distance.data_ptr(), d_mask=mask.data_ptr(),
                           d_item_pos=None if pos is None else pos.data_ptr(),
                           d_plan=None if plan is None else plan.data_ptr())
            self._launch("ts_optimal_moves", a, sp, stream)
        return distance, mask


class CudaStateTable(OnChipSearch):
    """ctypes front-end of ts_state_table_count / ts_state_table_fill (K10, csrc/ts_state_table.cu)
    and, for 5 to 8 tiles, of their hash-table counterparts (K12, csrc/ts_table_state_table.cu) for
    one batch: every state reachable from items (env id, positions), each with K9's distance and
    mask.  Planned per call as CudaOptimalMoves.query plans (the most free cells among the queried
    envs; K12: the table plan); both launches share the plan, so they agree on the items that fit."""

    CTAS_PER_SM = "ts_state_table_ctas_per_sm"
    GMEM_CTAS_PER_SM = "ts_state_table_gmem_ctas_per_sm"
    TABLE_CTAS_PER_SM = "ts_state_table_table_ctas_per_sm"
    ARGS = StateTableArgs

    def build(self, ids: torch.Tensor | None, pos: torch.Tensor | None = None, device_bitmap: bool = False,
              hash_table: bool = False, max_states: int | None = None) -> tuple[torch.Tensor, ...]:
        """(offsets int64[n+1], status int32[n], pos uint8[M, pos_bytes], distance int32[M], mask
        uint8[M]) of items (env `ids[i]`, root `pos[i]`) on the current stream; ids: int32 on the
        device, each in [0, n_envs) (None: every env); pos: contiguous uint8 [n, pos_bytes] on the
        device (None: the envs' current positions); device_bitmap as in CudaOptimalMoves.query;
        hash_table: 5 to 8 tiles are enumerated by K12 (ts_state_table_*_table) on
        _plan_table(max_states), whose slab both passes share (the fill sorts through it); it changes
        nothing for 1 to 4 tiles.  Reads back the row count and, without the hash table, the
        free-cell maximum."""
        t, dev = self.t, self.device
        n = t.n_envs if ids is None else ids.numel()
        offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        status = torch.full((n,), OPT_NOT_SEARCHED, dtype=torch.int32, device=dev)
        self.counters.zero_()
        table = hash_table and t.n_tiles >= 5
        if not n:
            sp = None
        elif table:
            sp = self._plan_table(max_states)
        else:
            sp = self.search_plan(self._max_free_cells(ids, n), device_bitmap)
        if sp is None:                           # no items, or not even T free cells fit on chip
            return (offsets, status, torch.empty((0, t.pos_bytes), dtype=torch.uint8, device=dev),
                    torch.empty(0, dtype=torch.int32, device=dev), torch.empty(0, dtype=torch.uint8, device=dev))
        count = torch.empty(n, dtype=torch.int64, device=dev)
        # the count pass's slab (grid x spill_per_cta words, ~0.9 GB at the benchmark shape) lives for
        # this call only: it goes back to the allocator's cache on return, for the rows or K9's slab
        spill = torch.empty(sp["grid"] * sp["spill_per_cta"], dtype=torch.int64 if table else torch.int32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        a = self._args(n_items=n, d_env_ids=None if ids is None else ids.data_ptr(),
                       d_item_pos=None if pos is None else pos.data_ptr(), bitmap_words=sp["bitmap_words"],
                       queue_smem=sp["queue_smem"], spill_per_cta=sp["spill_per_cta"],
                       d_spill=spill.data_ptr(), d_counters=self.counters.data_ptr(), d_count=count.data_ptr(),
                       d_status=status.data_ptr())
        with torch.cuda.device(dev):
            self._launch("ts_state_table_count", a, sp, stream)
            torch.cumsum(count, 0, out=offsets[1:])
            total = int(offsets[-1].item())
            rows = torch.empty((total, t.pos_bytes), dtype=torch.uint8, device=dev)
            distance = torch.empty(total, dtype=torch.int32, device=dev)
            mask = torch.empty(total, dtype=torch.uint8, device=dev)
            if total:
                a.d_offsets, a.d_rows, a.d_distance, a.d_mask = offsets.data_ptr(), rows.data_ptr(), distance.data_ptr(), mask.data_ptr()
                self._launch("ts_state_table_fill", a, sp, stream)
        return offsets, status, rows, distance, mask


class LocalBfs:
    """Batched BFS with one CTA per puzzle and the visited set in shared memory (K6,
    csrc/ts_bfs_local.cu): for batches of small puzzles, which is what the domain offers (a 6x6
    board with 4 tiles and 8 walls has 3,300 reachable states on average, the reference's real
    levels 51-950).  Several ranks: the puzzles are sharded by index (`shard_range`), every rank
    searches its shard with no exchange at all, and the per-puzzle results are combined once at
    the end.  A puzzle that does not fit on chip (state space above the shared-memory bitmap,
    more than 255 levels) is searched by the hash-partitioned `BfsSolver` instead.  Same result
    definitions as BfsSolver; boards of size <= 8 with 1..4 tiles.  device_bitmap=True: 7x7 and 8x8
    boards with four tiles whose bitmap outgrows shared memory are searched on chip all the same,
    with the bitmap in device memory (same results, and per-puzzle levels rather than a fallback).

    The device work sits behind `CudaLocalKernels`; tests run this driver on CPU tensors over
    gloo with a stand-in (tests/test_bfs_gloo.py)."""

    def __init__(self, puzzles: Sequence[Puzzle] | BatchedTilerSliderEnv | None = None, *, device="cuda", group=None,
                 ctas_per_sm: int | None = None, queue_smem: int | None = None, fallback_table_capacity: int = 1 << 24,
                 kernels=None, n_puzzles: int | None = None, fallback=None, device_bitmap: bool = False):
        if kernels is None:
            table = puzzles if isinstance(puzzles, BatchedTilerSliderEnv) else \
                BatchedTilerSliderEnv.from_puzzles(list(puzzles), device=device)
            kernels = CudaLocalKernels(table, ctas_per_sm, queue_smem, device_bitmap)
            n_puzzles = table.n_envs
        self.k, self.device, self.group = kernels, kernels.device, group
        self.n_puzzles = int(n_puzzles)
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.fallback_table_capacity = fallback_table_capacity
        self._fallback = fallback          # (puzzle ids, max_depth, with_paths) -> BfsResult; default: BfsSolver on the CUDA kernels

    def plan(self) -> dict | None:
        """The launch plan of this rank's shard (None: nothing fits on chip)."""
        return self.k.plan(*shard_range(self.n_puzzles, self.rank, self.world))

    def _search_rest(self, rest: list[int], max_depth: int, with_paths: bool) -> BfsResult:
        if self._fallback is not None:
            return self._fallback(rest, max_depth, with_paths)
        sub = BatchedTilerSliderEnv.from_puzzles([self.k.puzzle(i) for i in rest], device=self.device)
        cap = self.fallback_table_capacity
        while True:
            try:
                return BfsSolver(sub, table_capacity=cap, group=self.group).solve(max_depth=max_depth, with_paths=with_paths)
            except RuntimeError as e:                     # visited table full: double it
                if "table" not in str(e) or cap >= 1 << 32:
                    raise
                cap *= 2

    def solve(self, max_depth: int = 1 << 20, per_puzzle: bool = True, with_paths: bool = False) -> BfsResult:
        dev, P = self.device, self.n_puzzles
        n_levels, max_moves = getattr(self.k, "N_LEVELS", 256), getattr(self.k, "MAX_MOVES", 255)
        out = dict(states=torch.zeros(P, dtype=torch.int64, device=dev),
                   depth=torch.full((P,), -(1 << 30), dtype=torch.int32, device=dev),
                   status=torch.zeros(P, dtype=torch.int32, device=dev),
                   levels=torch.zeros(n_levels, dtype=torch.int64, device=dev),
                   counters=torch.zeros(8, dtype=torch.int64, device=dev),
                   moves=torch.zeros(P, max_moves, dtype=torch.uint8, device=dev) if with_paths else None,
                   lengths=torch.full((P,), -(1 << 30), dtype=torch.int32, device=dev) if with_paths else None)
        lo, hi = shard_range(P, self.rank, self.world)
        self.k.search(lo, hi, max_depth, out)
        states_pp, depth_pp, status, levels, counters = out["states"], out["depth"], out["status"], out["levels"], out["counters"]
        if self.world > 1:              # every puzzle has exactly one owner: sums / maxima over the ranks put the pieces together
            dist.all_reduce(states_pp, group=self.group)
            dist.all_reduce(depth_pp, op=dist.ReduceOp.MAX, group=self.group)
            dist.all_reduce(status, op=dist.ReduceOp.MAX, group=self.group)
            dist.all_reduce(levels, group=self.group)
            gen = counters[1:2].clone()
            dist.all_reduce(gen, group=self.group)
            counters[1:2] = gen
            if with_paths:
                dist.all_reduce(out["lengths"], op=dist.ReduceOp.MAX, group=self.group)
                mv32 = out["moves"].to(torch.int32)       # (uint8 reductions are not available on every backend)
                dist.all_reduce(mv32, op=dist.ReduceOp.MAX, group=self.group)
                out["moves"] = mv32.to(torch.uint8)
        generated = int(counters[1].item())
        lv = levels.tolist()
        solutions = None
        if with_paths:
            mv, ln = out["moves"].cpu().tolist(), out["lengths"].cpu().tolist()
            solutions = ["".join("UDLR"[m] for m in mv[i][:ln[i]]) if ln[i] >= 0 else None for i in range(P)]
        # ---- puzzles that did not fit on chip: the hash-partitioned search (collective over the same ranks)
        rest = torch.nonzero(status).flatten().tolist()
        if rest:
            r = self._search_rest(rest, max_depth, with_paths)
            idx = torch.tensor(rest, dtype=torch.int64, device=dev)
            states_pp[idx] = r.states_per_puzzle.to(dev)
            depth_pp[idx] = r.solve_depth_per_puzzle.to(device=dev, dtype=torch.int32)
            generated += r.generated
            n = max(len(lv), len(r.levels))
            lv = [(lv[i] if i < len(lv) else 0) + (r.levels[i] if i < len(r.levels) else 0) for i in range(n)]
            if solutions is not None and r.solutions is not None:
                for j, i in enumerate(rest):
                    solutions[i] = r.solutions[j]
        while len(lv) > 1 and lv[-1] == 0:
            lv.pop()
        solved = depth_pp[depth_pp >= 0]
        return BfsResult(n_states=int(sum(lv)), levels=lv, solve_depth=int(solved.min()) if solved.numel() else -1,
                         states_per_puzzle=states_pp if per_puzzle else None,
                         solve_depth_per_puzzle=depth_pp if per_puzzle else None,
                         generated=generated, solutions=solutions, fallback_puzzles=len(rest))


def solve_batch(puzzles: Sequence[Puzzle] | BatchedTilerSliderEnv, *, max_depth: int = 1 << 20, with_paths: bool = False,
                device="cuda", group=None) -> BfsResult:
    """BFS of a batch of puzzles of one shape with whichever search fits: the on-chip search (K6,
    `LocalBfs`) for up to 4 tiles -- puzzles that outgrow it fall back by themselves -- and the
    hash-partitioned search (`BfsSolver`) for 5 to 8 tiles, where the key has no room for a puzzle id
    and the puzzles are searched one after the other."""
    table = puzzles if isinstance(puzzles, BatchedTilerSliderEnv) else BatchedTilerSliderEnv.from_puzzles(list(puzzles), device=device)
    if table.size > 8:
        raise ValueError("BFS supports board sizes up to 8")
    if 1 <= table.n_tiles <= 4:
        return LocalBfs(table, group=group).solve(max_depth=max_depth, with_paths=with_paths)
    if table.n_envs == 1:
        return BfsSolver(table, group=group).solve(max_depth=max_depth, with_paths=with_paths)
    parts = [BfsSolver([table.puzzle(i)], device=table.device, group=group).solve(max_depth=max_depth, with_paths=with_paths)
             for i in range(table.n_envs)]
    n = max(len(r.levels) for r in parts)
    solved = [r.solve_depth for r in parts if r.solve_depth >= 0]
    return BfsResult(n_states=sum(r.n_states for r in parts),
                     levels=[sum(r.levels[d] for r in parts if d < len(r.levels)) for d in range(n)],
                     solve_depth=min(solved) if solved else -1,
                     states_per_puzzle=torch.cat([r.states_per_puzzle for r in parts]),
                     solve_depth_per_puzzle=torch.cat([r.solve_depth_per_puzzle for r in parts]),
                     generated=sum(r.generated for r in parts),
                     solutions=[r.solutions[0] for r in parts] if with_paths else None)


def solve_puzzle(puzzle: Puzzle, **kw) -> BfsResult:
    """BFS of one puzzle on the current CUDA device."""
    return BfsSolver([puzzle], **kw).solve()
