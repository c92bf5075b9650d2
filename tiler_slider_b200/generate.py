"""Puzzles worth playing: solvable puzzles graded by their shortest-solution length.

`BatchedTilerSliderEnv.synthetic` draws the create_simple_env recipe (environment.py:221-226), and
for the benchmark shape (6x6, 4 coloured tiles, 8 walls) fewer than 1 % of those puzzles can be won
at all.  `solvable` fills every env with a puzzle whose shortest solution lies in a band
[min_depth, max_depth], all on the device, in rounds:

  round a:  K7 (ts_synth_candidates) writes attempt-a candidates into the env slots not yet accepted;
            K6 (ts_bfs_local, bounded at max_depth) grades exactly those slots;
            a slot is accepted when its search completed and its solve depth is in the band.

A slot's candidate of attempt a depends on (seed, recipe, walk_len, global env index) only, and so
does the first attempt that lands in the band: env i's puzzle depends on (seed, recipe, walk_len,
band, env_index_base + i) and not on the batch size or the GPU count.  With recipe "uniform" an env
whose synthetic() puzzle is in the band keeps exactly that puzzle.  The solve depth (K6's: the fewest
steps that reach the goal, the goal being checked after every move, as the step does) lands in
`env.solve_depth`.  No reference counterpart (parity unpinned).

With 5 to 8 tiles (hash_table=True) K7's ts_synth_candidates_t8 writes the candidates and K11
(ts_optimal_moves_table, bounded at max_depth) grades each pending slot by the distance of its
initial positions, which is its solve depth.  A candidate whose search discovers more states than
the plan's bound gets -3 and is rejected like one outside the band, so the accepted puzzles are
drawn conditioned on fitting that bound.
"""
from __future__ import annotations

import ctypes as C

import torch

from ._lib import MAX_WALK, OPT_MAX_DEPTH, OPT_NOT_SEARCHED, RECIPE_UNIFORM, RECIPE_WALK, SynthCandidatesArgs, check
from .batch_env import BatchedTilerSliderEnv
from .bfs import CudaLocalKernels, CudaOptimalMoves

RECIPES = {"uniform": RECIPE_UNIFORM, "walk": RECIPE_WALK}
# enough rounds for the uniform recipe on the benchmark shape (0.7 % of its candidates are solvable:
# 65,536 slots need about 1,700 rounds); a walk fills a wide band in a handful
DEFAULT_MAX_ATTEMPTS = 4096


def default_walk_len(max_depth: int) -> int:
    return max(8, 2 * int(max_depth))


def write_candidates(env: BatchedTilerSliderEnv, ids: torch.Tensor | None, n_walls: int, recipe: str, walk_len: int,
                     attempt: int, seed: int, env_index_base: int = 0) -> None:
    """K7: attempt-`attempt` candidates into env slots `ids` (int32 on the device; None: every env)."""
    n = env.n_envs if ids is None else ids.numel()
    a = SynthCandidatesArgs(size=env.size, n_tiles=env.n_tiles, n_walls=n_walls, goal_mode=env.goal_mode,
                            recipe=RECIPES[recipe], walk_len=walk_len, attempt=attempt, n_items=n, capacity=env.capacity,
                            env_index_base=env_index_base, seed=seed & (2 ** 64 - 1),
                            d_env_ids=None if ids is None else ids.data_ptr(), d_walls=env._walls.data_ptr(),
                            d_targets_packed=env._targets.data_ptr(), d_init=env._init.data_ptr(), d_pos=env._pos.data_ptr())
    entry = "ts_synth_candidates_t8" if env.n_tiles >= 5 else "ts_synth_candidates"
    with torch.cuda.device(env.device):
        check(getattr(env._lib, entry)(C.byref(a), env._stream()), entry)


def fill(env: BatchedTilerSliderEnv, n_walls: int, *, min_depth: int, max_depth: int, recipe: str, walk_len: int,
         seed: int, env_index_base: int, max_attempts: int, device_bitmap: bool = False) -> dict:
    """Run up to `max_attempts` rounds over the envs of `env`; accepted envs get their solve depth in
    env._solve_depth.  device_bitmap: grade boards whose bitmap outgrows shared memory with one in
    device memory (7x7 / 8x8, 4 tiles).  Returns {rounds, candidates, accepted, unfilled}; 5 to 8
    tiles: fill_table."""
    if env.n_tiles >= 5:
        return fill_table(env, n_walls, min_depth=min_depth, max_depth=max_depth, recipe=recipe, walk_len=walk_len,
                          seed=seed, env_index_base=env_index_base, max_attempts=max_attempts)
    dev, n = env.device, env.n_envs
    k = CudaLocalKernels(env, device_bitmap=device_bitmap)
    depth = torch.full((env.capacity,), -1, dtype=torch.int32, device=dev)
    out = dict(states=torch.zeros(n, dtype=torch.int64, device=dev), depth=torch.zeros(n, dtype=torch.int32, device=dev),
               status=torch.zeros(n, dtype=torch.int32, device=dev),
               levels=torch.zeros(k.N_LEVELS, dtype=torch.int64, device=dev),
               counters=torch.zeros(8, dtype=torch.int64, device=dev))
    pending = torch.arange(n, dtype=torch.int32, device=dev)
    rounds = candidates = 0
    while pending.numel() and rounds < max_attempts:
        write_candidates(env, pending, n_walls, recipe, walk_len, rounds, seed, env_index_base)
        if rounds == 0 and k.plan(0, n) is None:      # every candidate has n_walls walls: one plan fits all
            raise ValueError(f"size {env.size} with {env.n_tiles} tiles and {n_walls} walls: the state bitmap does not fit "
                             "the on-chip search that grades the puzzles"
                             + ("" if device_bitmap or (env.size, env.n_tiles) not in k.GMEM_SHAPES else
                                " (device_bitmap=True keeps it in device memory)"))
        out["counters"].zero_()                       # [0] is K6's ticket counter
        k.search(0, n, max_depth, out, ids=pending)
        idx = pending.long()
        d = out["depth"][idx]
        ok = (out["status"][idx] == 0) & (d >= min_depth) & (d <= max_depth)
        depth[idx[ok]] = d[ok]
        candidates += pending.numel()
        rounds += 1
        pending = pending[~ok]
    env._solve_depth = depth
    return dict(rounds=rounds, candidates=candidates, accepted=n - pending.numel(), unfilled=pending.numel())


def fill_table(env: BatchedTilerSliderEnv, n_walls: int, *, min_depth: int, max_depth: int, recipe: str, walk_len: int,
               seed: int, env_index_base: int, max_attempts: int) -> dict:
    """fill for 5 to 8 tiles: each round grades the pending slots by K11's distance of their initial
    positions (bounded at max_depth).  Also returns over_bound, the rejections that were -3, and
    bound, the states K11's plan lets an item discover."""
    dev, n = env.device, env.n_envs
    search = CudaOptimalMoves(env)
    depth = torch.full((env.capacity,), -1, dtype=torch.int32, device=dev)
    pending = torch.arange(n, dtype=torch.int32, device=dev)
    rounds = candidates = 0
    over = torch.zeros((), dtype=torch.int64, device=dev)
    while pending.numel() and rounds < max_attempts:
        write_candidates(env, pending, n_walls, recipe, walk_len, rounds, seed, env_index_base)
        d, _ = search.query(pending, max_depth, hash_table=True)      # pos = the candidates' initial positions
        ok = (d >= min_depth) & (d <= max_depth)
        over += (d == OPT_NOT_SEARCHED).sum()
        depth[pending.long()[ok]] = d[ok]
        candidates += pending.numel()
        rounds += 1
        pending = pending[~ok]
    env._solve_depth = depth
    return dict(rounds=rounds, candidates=candidates, accepted=n - pending.numel(), unfilled=pending.numel(),
                over_bound=int(over), bound=search._plan_table()["spill_per_cta"])


def solvable(cls, n_envs: int, size: int, n_tiles: int, n_walls: int, multi_color: bool = False, *, min_depth: int = 1,
             max_depth: int = 30, recipe: str = "walk", walk_len: int | None = None, seed: int = 0,
             env_index_base: int = 0, max_attempts: int = DEFAULT_MAX_ATTEMPTS, device_bitmap: bool = False,
             hash_table: bool = False, **kw) -> BatchedTilerSliderEnv:
    """BatchedTilerSliderEnv.solvable (see there)."""
    table = hash_table and 5 <= n_tiles <= 8
    if table and not 3 <= size <= 8:
        raise ValueError(f"graded generation with 5 to 8 tiles covers sizes 3 to 8 (got size {size})")
    if not table and not (1 <= size <= 8 and 1 <= n_tiles <= 4):
        raise ValueError(f"graded generation covers sizes up to 8 with 1 to 4 tiles (got size {size}, {n_tiles} tiles)"
                         + (" or, with hash_table=True, 5 to 8 tiles" if hash_table else ""))
    if recipe not in RECIPES:
        raise ValueError(f"recipe {recipe!r}: one of {sorted(RECIPES)}")
    if max_depth < 1 or min_depth > max_depth:
        raise ValueError(f"empty band [{min_depth}, {max_depth}]")
    if table and max_depth > OPT_MAX_DEPTH:
        raise ValueError(f"band maximum {max_depth} above {OPT_MAX_DEPTH}, the deepest search optimal_moves runs")
    max_steps = int(kw.get("max_steps", 100))
    if max_depth > max_steps:
        raise ValueError(f"max_depth {max_depth} exceeds max_steps {max_steps}: such a puzzle cannot be won within an episode")
    walk_len = default_walk_len(max_depth) if walk_len is None else int(walk_len)
    if not 0 <= walk_len <= MAX_WALK:
        raise ValueError(f"walk_len {walk_len} outside 0..{MAX_WALK}")
    need = n_walls + (2 if recipe == "uniform" else 1) * n_tiles
    if n_walls < 0 or need > size * size:
        raise ValueError(f"recipe {recipe!r} needs {need} distinct cells, a {size}x{size} board has {size * size}")
    if max_attempts < 1:
        raise ValueError("max_attempts must be positive")
    env = cls(size, n_tiles, n_envs, multi_color, **kw)
    stats = fill(env, n_walls, min_depth=min_depth, max_depth=max_depth, recipe=recipe, walk_len=walk_len, seed=seed,
                 env_index_base=env_index_base, max_attempts=max_attempts, device_bitmap=device_bitmap)
    if stats["unfilled"]:
        raise RuntimeError(f"{stats['unfilled']} of {n_envs} envs unfilled after {stats['rounds']} rounds: "
                           f"{stats['accepted']} of {stats['candidates']} candidates were in the band "
                           f"[{min_depth}, {max_depth}] (yield {stats['accepted'] / stats['candidates']:.3%})"
                           + (f"; {stats['over_bound']} rejections outgrew the search's bound of "
                              f"{stats['bound']} states (-3)" if table else ""))
    env._loaded = True
    env.reset()
    return env
