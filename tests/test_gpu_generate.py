"""GPU tests of the puzzle generator (BatchedTilerSliderEnv.solvable: K7 candidates graded by K6)
and of auto-reset into a pool of puzzles (set_reset_pool: K8 behind K2), against the CPU oracle
and the Python restatement of the generator's streams (tests/gen_port.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import gen_port
from tests.helpers import random_puzzles

pytestmark = pytest.mark.gpu

F_DONE = 1


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def decode(env):
    """Host copies of every env's puzzle: blocked u8[N,S*S], tiles u8[N,T,2], targets (ordered:
    u8[N,T,2]; set: bool[N,S*S])."""
    n = env.n_envs
    return (env.blocked_cells().cpu().numpy(), env.positions(env._init[:n]).cpu().numpy(),
            env.target_positions().cpu().numpy())


def oracle_state(S, multi, blocked, tiles, targets, i):
    b = [divmod(int(c), S) for c in np.flatnonzero(blocked[i])]
    tg = targets[i].tolist() if targets.ndim == 3 else [divmod(int(c), S) for c in np.flatnonzero(targets[i])]
    return orc.OracleState(S, b, tiles[i].tolist(), tg, multi)


GEN_CASES = [  # S, T, W, multi, recipe, min_depth, max_depth
    (3, 1, 1, False, "walk", 1, 4),
    (3, 2, 1, True, "uniform", 1, 6),
    (4, 2, 2, True, "walk", 2, 8),
    (4, 3, 3, False, "uniform", 1, 10),
    (5, 1, 5, False, "walk", 3, 8),
    (5, 3, 4, True, "walk", 4, 12),
    (6, 4, 8, True, "walk", 8, 12),
    (6, 4, 8, True, "walk", 12, 20),
    (6, 4, 8, False, "walk", 4, 20),
    (6, 4, 8, True, "uniform", 1, 30),
    (6, 2, 6, False, "uniform", 2, 9),
    (7, 3, 12, True, "walk", 5, 15),
    (7, 4, 16, False, "walk", 3, 10),
    (8, 4, 30, True, "walk", 6, 14),
    (8, 2, 20, False, "uniform", 1, 20),
    (8, 1, 10, True, "walk", 1, 6),
]


@pytest.mark.parametrize("S,T,W,multi,recipe,min_depth,max_depth", GEN_CASES)
def test_generated_depth_is_exact_and_in_band(ts, S, T, W, multi, recipe, min_depth, max_depth):
    """Every generated puzzle's oracle BFS solve depth equals env.solve_depth and lies in the band."""
    N = 1024
    env = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=min_depth, max_depth=max_depth, recipe=recipe,
                                            seed=S * 100 + T, max_steps=max(100, max_depth))
    depth = env.solve_depth.cpu().numpy()
    assert ((depth >= min_depth) & (depth <= max_depth)).all()
    blocked, tiles, targets = decode(env)
    assert (blocked.sum(1) == W).all()
    for i in range(N):
        st = oracle_state(S, multi, blocked, tiles, targets, i)
        assert st.bfs(max_depth=max_depth, max_states=1 << 21)[2] == depth[i], (i, depth[i])
    assert torch.equal(env.pos, env._init[:N]) and int(env.step_count.sum()) == 0


PIN_CASES = [(3, 2, 1, True), (5, 1, 5, False), (6, 4, 8, True), (6, 3, 8, False), (7, 4, 16, True), (8, 2, 20, False)]


@pytest.mark.parametrize("S,T,W,multi", PIN_CASES)
@pytest.mark.parametrize("recipe", ["uniform", "walk"])
def test_candidates_match_the_python_restatement(ts, S, T, W, multi, recipe):
    """K7's candidates, byte for byte in the packed layout, equal the restated recipe (splitmix64
    stream, partial Fisher-Yates, walk of state-changing moves) encoded by K1; listed slots only."""
    from tiler_slider_b200.generate import write_candidates
    N, base, seed, walk_len = 1021, 5000, 987654321, 13
    for attempt in (0, 3):
        env = ts.BatchedTilerSliderEnv(S, T, N, multi)
        for buf in (env._walls, env._targets, env._init, env._pos):
            buf.fill_(0x5C)
        ids = torch.arange(0, N, 3, dtype=torch.int32, device="cuda")
        write_candidates(env, ids, W, recipe, walk_len, attempt, seed, base)
        blocked, tiles, targets = gen_port.candidate_arrays(orc, S, T, W, multi, recipe, walk_len, seed, attempt,
                                                            (ids.cpu().numpy() + base).tolist())
        ref = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
        sel = ids.long()
        cap, rcap, n = env.capacity, ref.capacity, ids.numel()
        for name in ("_walls", "_targets"):
            nb = getattr(env, name).numel() // cap
            got, want = getattr(env, name), getattr(ref, name)
            for k in range(env._lib.ts_plane_count(nb)):
                w, off = env._lib.ts_plane_width(nb, k), env._lib.ts_plane_offset(nb, k)
                g = got[off * cap:(off + w) * cap].view(cap, w)
                assert torch.equal(g[sel], want[off * rcap:(off + w) * rcap].view(rcap, w)[:n]), (name, k, attempt)
                rest = torch.ones(cap, dtype=torch.bool, device="cuda")
                rest[sel] = False
                assert (g[rest] == 0x5C).all(), (name, "unlisted slot written")
        assert torch.equal(env._init[sel], ref._init[:n]) and torch.equal(env._pos[sel], ref._init[:n])


@pytest.mark.parametrize("S,T,W,multi,band", [(6, 4, 8, True, (1, 30)), (6, 2, 8, False, (2, 6)), (5, 3, 4, True, (3, 9))])
def test_uniform_recipe_keeps_the_synthetic_puzzles_in_the_band(ts, S, T, W, multi, band):
    from tiler_slider_b200.bfs import LocalBfs
    N, seed = 2048, 4242
    syn = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=seed)
    d = LocalBfs(syn).solve(max_depth=band[1]).solve_depth_per_puzzle.cpu().numpy()
    keep = (d >= band[0]) & (d <= band[1])
    assert keep.any()
    gen = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=band[0], max_depth=band[1], recipe="uniform", seed=seed)
    for a, b in zip(decode(syn), decode(gen)):
        assert np.array_equal(a[keep], b[keep])
    assert np.array_equal(gen.solve_depth.cpu().numpy()[keep], d[keep])


@pytest.mark.parametrize("recipe", ["walk", "uniform"])
def test_shard_invariance(ts, recipe):
    """solvable(N) equals solvable(N/2, base 0) followed by solvable(N/2, base N/2)."""
    N, kw = 2048, dict(min_depth=3, max_depth=9, recipe=recipe, seed=77)
    full = ts.BatchedTilerSliderEnv.solvable(N, 5, 2, 5, True, **kw)
    lo = ts.BatchedTilerSliderEnv.solvable(N // 2, 5, 2, 5, True, env_index_base=0, **kw)
    hi = ts.BatchedTilerSliderEnv.solvable(N // 2, 5, 2, 5, True, env_index_base=N // 2, **kw)
    for f, a, b in zip(decode(full), decode(lo), decode(hi)):
        assert np.array_equal(f, np.concatenate([a, b]))
    assert torch.equal(full._init[:N], torch.cat([lo._init[:N // 2], hi._init[:N // 2]]))
    assert torch.equal(full.solve_depth, torch.cat([lo.solve_depth, hi.solve_depth]))


def test_generation_errors(ts):
    E = ts.BatchedTilerSliderEnv
    for args, kw in [((64, 9, 2, 4), {}), ((64, 6, 5, 8), {}), ((64, 6, 0, 8), {}),
                     ((64, 8, 4, 8), {}),                                 # 56^4 arrangements: no on-chip bitmap
                     ((64, 6, 4, 8), dict(min_depth=9, max_depth=8)),
                     ((64, 6, 4, 8), dict(max_depth=40, max_steps=30))]:
        with pytest.raises(ValueError):
            E.solvable(*args, True, **kw)
    with pytest.raises(RuntimeError, match="yield"):          # a walk of 2 moves never needs 29 steps
        E.solvable(256, 6, 4, 8, True, min_depth=29, max_depth=30, walk_len=2, max_attempts=3)


# ---------------------------------------------------------------------------------------------- pool
def oracle_step(st, a, count, max_steps, rewards=orc.DEFAULT_REWARDS):
    """One step of TilerSliderEnv.step on the oracle: (flags, reward, count after)."""
    before = st.current_locations
    st.move(a)
    moved = st.current_locations != before
    won = st.is_won()
    count += 1
    flags = (2 if won else 0) | (0 if moved else 4)
    if count >= max_steps:
        flags |= 8
    if won or count >= max_steps:
        flags |= F_DONE
    reward = rewards[0] if won else rewards[2] if not moved else rewards[1]
    return flags, np.float32(reward), count


def make_pool(ts, kind):
    if kind == "narrow_coloured":
        return ts.BatchedTilerSliderEnv.solvable(200, 6, 4, 8, True, min_depth=1, max_depth=6, seed=5), (6, 4, 8, True)
    if kind == "set_goal":
        return ts.BatchedTilerSliderEnv.solvable(130, 6, 3, 8, False, min_depth=1, max_depth=5, seed=6), (6, 3, 8, False)
    rng = np.random.default_rng(9)
    S, T, W, multi = (12, 3, 30, True) if kind == "wide" else (10, 12, 10, False)
    b, t, g = random_puzzles(rng, 150, S, T, W)
    return ts.BatchedTilerSliderEnv.from_arrays(S, b, t, g, multi), (S, T, W, multi)


@pytest.mark.parametrize("kind,draw_now", [("narrow_coloured", True), ("set_goal", False), ("wide", True), ("generic", False)])
def test_pool_reset_vs_oracle(ts, kind, draw_now):
    """Several hundred auto-reset steps with a pool: every env holds the pool puzzle the restated H
    predicts from its episode count, envs that never finished keep their puzzle, `episodes` counts
    the done events, `solve_depth` follows the pool, and every step's positions / flags / reward
    match the oracle replayed with the puzzles switched at those draws."""
    pool, (S, T, W, multi) = make_pool(ts, kind)
    N, K, max_steps, seed = 509, 240, 7, 31337
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=3, max_steps=max_steps, auto_reset=True,
                                             track_terminal=True)
    first = decode(env)
    env.set_reset_pool(pool, seed=seed, draw_now=draw_now)
    has_depth = pool.solve_depth is not None
    assert (env.solve_depth is not None) == has_depth
    pb, pt, pg = decode(pool)
    pdepth = pool.solve_depth.cpu().numpy() if has_depth else None
    episodes = np.full(N, 1 if draw_now else 0, np.int64)
    cur = [gen_port.pool_draw(seed, e, 0, pool.n_envs) if draw_now else -1 for e in range(N)]
    states = [oracle_state(S, multi, pb, pt, pg, cur[e]) if draw_now else oracle_state(S, multi, *first, e) for e in range(N)]
    count = np.zeros(N, np.int64)
    g = torch.Generator(device="cuda").manual_seed(17)
    acts = torch.randint(0, 4, (K, env.capacity), dtype=torch.uint8, device="cuda", generator=g)
    acts_h = acts.cpu().numpy()
    for k in range(K):
        _, reward, done = env.step(acts[k])
        flags, reward, done = env.flags.cpu().numpy(), reward.cpu().numpy(), done.cpu().numpy()
        term = env.positions(env.terminal_pos).cpu().numpy()
        pos = env.positions().cpu().numpy()
        for e in range(N):
            f, r, count[e] = oracle_step(states[e], int(acts_h[k, e]), count[e], max_steps)
            assert flags[e] == f and reward[e] == r, (kind, k, e)
            assert bool(done[e]) == bool(f & F_DONE)
            assert [tuple(x) for x in (term[e] if done[e] else pos[e]).tolist()] == states[e].current_locations, (kind, k, e)
            if done[e]:
                cur[e] = gen_port.pool_draw(seed, e, int(episodes[e]), pool.n_envs)
                episodes[e] += 1
                states[e] = oracle_state(S, multi, pb, pt, pg, cur[e])
                count[e] = 0
                assert [tuple(x) for x in pos[e].tolist()] == states[e].current_locations
    assert np.array_equal(env.episodes.to(torch.int64).cpu().numpy(), episodes)
    assert (episodes > (1 if draw_now else 0)).any()
    cur = np.array(cur)
    now = decode(env)
    drawn = cur >= 0
    for a, p in zip(now, (pb, pt, pg)):
        assert np.array_equal(a[drawn], p[cur[drawn]])
    for a, f in zip(now, first):                           # never finished, never drawn: the puzzle it started with
        assert np.array_equal(a[~drawn], f[~drawn])
    if has_depth:
        sd = env.solve_depth.cpu().numpy()
        assert np.array_equal(sd[drawn], pdepth[cur[drawn]]) and (sd[~drawn] == -1).all()
    else:
        assert env.solve_depth is None


def test_pool_reset_touches_nothing_outside_the_range(ts):
    """A ragged batch (1,021 envs, capacity 1,024) with its padding poisoned (done bytes set): K8 over
    [0, n) for n = 1021, 510, 3 writes nothing outside the range, and resets every env inside it."""
    pool = ts.BatchedTilerSliderEnv.solvable(64, 6, 4, 8, True, min_depth=1, max_depth=8, seed=1)
    N = 1021
    env = ts.BatchedTilerSliderEnv.synthetic(N, 6, 4, 8, True, seed=2, max_steps=5, auto_reset=True)
    env.set_reset_pool(pool, seed=4)
    cap = env.capacity

    def owner(buf):                                  # env of every byte of a plane-layout buffer
        nb = buf.numel() // cap
        out = torch.empty(nb * cap, dtype=torch.int64, device="cuda")
        for k in range(env._lib.ts_plane_count(nb)):
            w, off = env._lib.ts_plane_width(nb, k), env._lib.ts_plane_offset(nb, k)
            out[off * cap:(off + w) * cap] = torch.arange(cap, device="cuda").repeat_interleave(w)
        return out
    env._episodes[N:] = 77
    env._solve_depth[N:] = -9
    for buf, v in ((env._pos, 0xA5), (env._init, 0xC3), (env._count, 0x5A)):
        buf[N:] = v
    for n_range in (N, 510, 3):
        env._done.fill_(1)
        bufs = {"walls": env._walls, "targets": env._targets, "init": env._init, "pos": env._pos, "count": env._count,
                "episodes": env._episodes, "depth": env._solve_depth}
        before = {k: b.clone() for k, b in bufs.items()}
        a = ts._lib.PoolResetArgs.from_buffer_copy(env._pool_args)
        a.n_envs = n_range
        assert env._lib.ts_pool_reset(C.byref(a), torch.cuda.current_stream().cuda_stream) == 0
        torch.cuda.synchronize()
        for name in ("walls", "targets"):
            outside = owner(bufs[name]) >= n_range
            assert torch.equal(bufs[name][outside], before[name][outside]), (name, n_range)
        for name in ("init", "pos", "count", "episodes", "depth"):
            assert torch.equal(bufs[name][n_range:], before[name][n_range:]), (name, n_range)
        assert torch.equal(env._episodes[:n_range], before["episodes"][:n_range] + 1)
        assert torch.equal(env._pos[:n_range], env._init[:n_range]) and int(env._count[:n_range].sum()) == 0


def test_graph_replay_with_a_pool_equals_eager_steps(ts):
    pool = ts.BatchedTilerSliderEnv.solvable(256, 6, 4, 8, True, min_depth=1, max_depth=6, seed=8)
    N, R = 4099, 24
    kw = dict(seed=12, max_steps=6, auto_reset=True, track_terminal=True)
    a = ts.BatchedTilerSliderEnv.synthetic(N, 6, 4, 8, True, **kw)
    b = ts.BatchedTilerSliderEnv.synthetic(N, 6, 4, 8, True, **kw)
    for e in (a, b):
        e.set_reset_pool(pool, seed=99, draw_now=True)
    g = torch.Generator(device="cuda").manual_seed(5)
    rows = torch.randint(0, 4, (R, a.capacity), dtype=torch.uint8, device="cuda", generator=g)
    graph = a.capture_steps(rows)
    b.reset()
    for rep in range(3):
        graph.replay()
        for k in range(R):
            b.step(rows[k])
        torch.cuda.synchronize()
        for name in ("_pos", "_init", "_walls", "_targets", "_count", "_reward", "_done", "_terminal", "_episodes", "_solve_depth"):
            assert torch.equal(getattr(a, name), getattr(b, name)), (name, rep)
    assert int(a.episodes.to(torch.int64).sum()) > N


def never_win(ts):
    b, t, g = random_puzzles(np.random.default_rng(1), 4, 6, 4, 8)
    return ts.BatchedTilerSliderEnv.from_arrays(6, b, t, g[:, :3], True)      # 3 ordered targets for 4 tiles


def test_pool_arguments(ts):
    pool = ts.BatchedTilerSliderEnv.solvable(64, 6, 4, 8, True, min_depth=1, max_depth=8, seed=1)
    env = ts.BatchedTilerSliderEnv.synthetic(256, 6, 4, 8, True, auto_reset=True)
    for bad in (ts.BatchedTilerSliderEnv.synthetic(64, 6, 3, 8, True),
                ts.BatchedTilerSliderEnv.synthetic(64, 6, 4, 8, False),
                ts.BatchedTilerSliderEnv.synthetic(64, 5, 4, 8, True),
                never_win(ts)):
        with pytest.raises(ValueError):
            env.set_reset_pool(bad)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.synthetic(256, 6, 4, 8, True, auto_reset=False).set_reset_pool(pool)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.synthetic(4, 6, 4, 8, True, auto_reset=True, host_io=True).set_reset_pool(pool)
    env.set_reset_pool(pool)
    with pytest.raises(ValueError):
        env.step_host(torch.zeros(256, dtype=torch.uint8), h_flags=torch.zeros(256, dtype=torch.uint8))
    env.set_reset_pool(None)
    before = env._walls.clone()
    for _ in range(120):
        env.step(torch.randint(0, 4, (256,), dtype=torch.uint8, device="cuda"))
    assert torch.equal(env._walls, before)                      # detached: auto-reset restarts the same puzzle
