"""GPU tests of the on-chip searches at their capacity limits: K9 (optimal_moves) next to the largest
bitmap one CTA can hold, K9, K10 (state_table) and K6 (LocalBfs) with a slab too small for some of
their envs, and K9 on the smallest and fullest boards.  Every expectation comes from the CPU
oracle's BFS; where a slab runs out, the answer is predicted from the oracle's state or level counts
and the kernel's append rule."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.helpers import random_puzzles, reachable_targets
from tests.test_gpu_optimal import oracle_answer, oracle_states, random_steps

pytestmark = pytest.mark.gpu

NOT_SEARCHED = -3


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def puzzles(S, T, walls, n, multi, seed, walk=12):
    """n puzzles of S x S with T tiles for each wall count in `walls`, shuffled together; targets are
    where a random walk of `walk` moves leaves the tiles, so that most are solvable (walk=None: drawn
    at random, so that most are not).  Returns (blocked, tiles, targets)."""
    rng = np.random.default_rng(seed)
    parts = []
    for W in walls:
        blocked, tiles, targets = random_puzzles(rng, n, S, T, W)
        if walk is not None:
            targets = reachable_targets(orc, rng, S, blocked, tiles, multi, walk)
        parts.append((blocked, tiles, targets))
    order = rng.permutation(n * len(walls))
    return tuple(np.concatenate([p[k] for p in parts])[order] for k in range(3))


def free_cells(env):
    return (env.size * env.size - env.blocked_cells().sum(1)).cpu().numpy()


# ---- (a, b) K9 next to the largest bitmap one CTA can hold ------------------------------------------

@pytest.fixture(scope="module", params=[True, False], ids=["ordered", "set"])
def boundary_batch(ts, request):
    """8x8 boards with 4 tiles and F free cells, F in {30, F*-1, F*, F*+1, F*+2}, interleaved, after
    three random steps.  F* = the most free cells whose state space fits the bitmap of one CTA,
    found by asking the planner."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    multi = request.param
    probe = ts.BatchedTilerSliderEnv.synthetic(8, 8, 4, 30, multi, seed=0)
    planner = CudaOptimalMoves(probe)
    fits = [f for f in range(4, 65) if planner.plan(f) is not None]
    f_star = fits[-1]
    assert fits == list(range(4, f_star + 1))
    assert f_star >= 30                     # 8x8 / 4 tiles / 34 walls of test_gpu_optimal and every 6x6 board stay on chip
    groups = sorted({30, f_star - 1, f_star, f_star + 1, f_star + 2})
    blocked, tiles, targets = puzzles(8, 4, [64 - f for f in groups], 32, multi, seed=int(multi) + 40)
    env = ts.BatchedTilerSliderEnv.from_arrays(8, blocked, tiles, targets, multi)
    random_steps(env, 3, seed=5)
    return env, free_cells(env), f_star, groups


def test_bitmap_boundary_mixed_batch(ts, boundary_batch):
    """Envs whose own state space fits the largest bitmap get the oracle's exact answer even when the
    batch holds larger boards; only the larger boards report -3 with an empty mask."""
    env, F, f_star, groups = boundary_batch
    d, m = env.optimal_moves()
    d, m = d.cpu().numpy(), m.cpu().numpy()
    big = F > f_star
    assert big.sum() == 64 and (~big).sum() == 32 * (len(groups) - 2)
    assert (d[big] == NOT_SEARCHED).all() and (m[big] == 0).all()
    states = oracle_states(env)
    for i in np.flatnonzero(~big):
        st, cur = states[i]
        assert (int(d[i]), int(m[i])) == oracle_answer(st, cur), (i, int(F[i]), cur)
    assert (d[~big] >= 1).sum() > 32 * (len(groups) - 2) // 2     # most of them solvable


def test_answers_do_not_depend_on_the_other_envs_of_the_query(ts, boundary_batch):
    """Queried with the whole batch, with the envs that fit only, with each free-cell group alone and
    with a shuffled id list that repeats envs, every env gets the same answer: the plans (bitmap, ring,
    CTAs per SM) differ, the answers may not."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env, F, f_star, groups = boundary_batch
    d_all, m_all = env.optimal_moves()
    d_all, m_all = d_all.cpu().numpy(), m_all.cpu().numpy()
    queries = [np.flatnonzero(F <= f_star)] + [np.flatnonzero(F == f) for f in groups]
    rng = np.random.default_rng(3)
    queries.append(rng.integers(0, env.n_envs, 3 * env.n_envs))
    for ids in queries:
        d, m = env.optimal_moves(ids.tolist())
        assert np.array_equal(d.cpu().numpy(), d_all[ids]) and np.array_equal(m.cpu().numpy(), m_all[ids]), sorted(set(F[ids]))
    planner = CudaOptimalMoves(env)
    assert planner.fitting_free_cells(f_star + 2) == f_star
    assert planner.plan(30)["ctas_per_sm"] > planner.plan(f_star)["ctas_per_sm"]


# ---- (c) K9 with a slab too small for some envs --------------------------------------------------

def k9_with_slab(L, d, exact, q, m):
    """K9's answer when the slab holds q states: the forward search writes every state it discovers
    to the slab and gives up (-3) when a discovery index reaches q, except on the level that meets the
    goal, whose discoveries are never read.  L = level counts of the oracle's BFS from the current
    state over at most m levels, d = its solve depth (-1: no win within m levels)."""
    if 1 <= d <= m:
        return (NOT_SEARCHED, 0) if sum(L[:d]) > q else exact
    last = len(L) - 1                       # the last non-empty level, at most m
    if sum(L[:last + 1]) > q:
        return NOT_SEARCHED, 0
    return (-1, 0) if last < m else (-2, 0)


@pytest.mark.parametrize("multi", [True, False], ids=["ordered", "set"])
def test_optimal_moves_slab_overflow_is_predicted_exactly(ts, multi):
    from tiler_slider_b200.bfs import CudaOptimalMoves

    class SmallSlab(CudaOptimalMoves):
        def __init__(self, env, q, queue_smem=None):
            super().__init__(env, queue_smem=queue_smem)
            self.q = q

        def plan(self, f_max):
            p = super().plan(f_max)
            return None if p is None else {**p, "spill_per_cta": self.q}

    solvable = puzzles(6, 4, [8], 160, multi, seed=int(multi) + 50)
    uniform = puzzles(6, 4, [8], 64, multi, seed=int(multi) + 52, walk=None)
    env = ts.BatchedTilerSliderEnv.from_arrays(6, *(np.concatenate(p) for p in zip(solvable, uniform)), multi)
    random_steps(env, 3, seed=9)
    states = oracle_states(env)
    seen = set()
    for m in (254, 5):
        want_exact, levels = [], []
        for st, cur in states:
            want_exact.append(oracle_answer(st, cur, max_depth=m))
            st.set_locations(cur)
            _, L, d, _ = st.bfs(max_depth=m, max_states=1 << 22)
            levels.append((L, d))
        for q, ring in ((48, None), (300, 32), (2000, None)):
            d, mk = SmallSlab(env, q, ring).query(None, m)
            got = list(zip(d.tolist(), mk.tolist()))
            for i, ((L, dd), exact) in enumerate(zip(levels, want_exact)):
                want = k9_with_slab(L, dd, exact, q, m)
                assert got[i] == want, (m, q, i, L, dd, exact)
                seen.add(("win" if 1 <= dd <= m else "none", want[0] if want[0] < 0 else "exact"))
    # every branch of the prediction was taken
    assert seen >= {("win", "exact"), ("win", NOT_SEARCHED), ("none", NOT_SEARCHED), ("none", -1), ("none", -2)}, seen


@pytest.mark.parametrize("multi", [True, False], ids=["ordered", "set"])
def test_state_table_slab_overflow_is_predicted_exactly(ts, multi):
    """K10's count pass gives an item up (-3, no rows) as soon as a discovery index reaches the q
    entries of its slab, even when the ring would hold the entry: exactly the items of more than q
    states.  Every other item gets the rows and labels of the default plan."""
    from tiler_slider_b200.bfs import CudaStateTable

    class SmallSlab(CudaStateTable):
        def __init__(self, env, q, queue_smem=None):
            super().__init__(env, queue_smem=queue_smem)
            self.q = q

        def plan(self, f_max):
            p = super().plan(f_max)
            return None if p is None else {**p, "spill_per_cta": self.q}

    solvable = puzzles(6, 4, [8], 48, multi, seed=int(multi) + 70)
    uniform = puzzles(6, 4, [8], 16, multi, seed=int(multi) + 72, walk=None)
    env = ts.BatchedTilerSliderEnv.from_arrays(6, *(np.concatenate(p) for p in zip(solvable, uniform)), multi)
    random_steps(env, 3, seed=11)
    count = np.array([st.bfs(max_states=1 << 22)[0] for st, _ in oracle_states(env)])
    full = env.state_table()
    assert (full.status == 0).all()
    rows_per_item = full.offsets.diff().cpu().numpy()
    assert np.array_equal(rows_per_item, count)
    seen = set()
    for q in (48, 2000, 4000):
        for ring in (None, 32):
            offsets, status, pos, distance, mask = SmallSlab(env, q, ring).build(None)
            big = count > q
            assert np.array_equal(status.cpu().numpy(), np.where(big, NOT_SEARCHED, 0)), (q, ring)
            assert np.array_equal(offsets.diff().cpu().numpy(), np.where(big, 0, count)), (q, ring)
            kept = torch.from_numpy(np.repeat(~big, rows_per_item)).cuda()
            assert torch.equal(pos, full.pos[kept]) and torch.equal(distance, full.distance[kept]) \
                and torch.equal(mask, full.mask[kept]), (q, ring)
            seen.update(big.tolist())
    assert seen == {True, False}


# ---- (d) K6 with a slab too small for some puzzles: the hash-partitioned fallback ----------------

def k6_falls_back(L, q, ring, with_paths):
    """Whether K6 gives a puzzle up (status 2) with a slab of q entries and a ring of `ring` entries.
    With paths every discovered state records its parent in the slab, so any discovery index >= q
    overflows.  Without, a state goes to the slab only when it lies `ring` or more past the start of
    the level being expanded; the last state discovered while expanding level k is the farthest."""
    if with_paths:
        return sum(L) > q
    for k in range(len(L) - 1):
        lo, e = sum(L[:k]), sum(L[:k + 2])
        if e - 1 >= q and e - 1 - lo >= ring:
            return True
    return False


def replay_wins_at(S, blocked, tiles, targets, multi, moves):
    st = orc.OracleState(S, blocked, tiles, targets, multi)
    return [k + 1 for k, ch in enumerate(moves) if st.move("UDLR".index(ch))]


@pytest.mark.parametrize("multi", [True, False], ids=["ordered", "set"])
def test_local_bfs_slab_overflow_falls_back_exactly(ts, multi):
    from tiler_slider_b200.bfs import CudaLocalKernels, LocalBfs

    class SmallSlab(CudaLocalKernels):
        def __init__(self, table, q, ring):
            super().__init__(table, queue_smem=ring)
            self.q = q

        def plan(self, lo, hi):
            p = super().plan(lo, hi)
            return None if p is None else {**p, "spill_per_cta": self.q}

    S, n = 6, 96
    blocked, tiles, targets = puzzles(S, 4, [8], n, multi, seed=int(multi) + 60, walk=9)
    table = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    walls = [[(c // S, c % S) for c in np.flatnonzero(blocked[e])] for e in range(n)]
    want = [orc.OracleState(S, walls[e], tiles[e].tolist(), targets[e].tolist(), multi).bfs(max_states=1 << 22)
            for e in range(n)]
    want_states, want_depth = [w[0] for w in want], [w[2] for w in want]
    want_levels = [sum(w[1][k] for w in want if k < len(w[1])) for k in range(max(len(w[1]) for w in want))]
    counts = {}
    for q, ring in ((48, 32), (300, 32), (2000, 64)):
        for with_paths in (True, False):
            k = SmallSlab(table, q, ring)
            res = LocalBfs(kernels=k, n_puzzles=n).solve(with_paths=with_paths)
            assert k.plan(0, n)["queue_smem"] == ring
            fb = sum(k6_falls_back(w[1], q, ring, with_paths) for w in want)
            assert res.fallback_puzzles == fb, (q, ring, with_paths)
            counts[q, with_paths] = fb
            assert res.states_per_puzzle.tolist() == want_states
            assert res.solve_depth_per_puzzle.tolist() == want_depth
            assert res.levels == want_levels
            if with_paths:
                for e in range(n):
                    sol = res.solutions[e]
                    if want_depth[e] < 0:
                        assert sol is None
                    else:
                        assert len(sol) == want_depth[e]
                        assert replay_wins_at(S, walls[e], tiles[e].tolist(), targets[e].tolist(), multi, sol)[:1] == [want_depth[e]]
    # some runs fall back for part of the batch only, and without paths the ring keeps some puzzles on chip
    assert any(0 < fb < n for fb in counts.values())
    assert any(counts[q, False] < counts[q, True] for q, _ in counts)


# ---- (e) K9 on the smallest and fullest boards ----------------------------------------------------

def check_all(env):
    d, m = env.optimal_moves()
    d, m = d.cpu().numpy(), m.cpu().numpy()
    for i, (st, cur) in enumerate(oracle_states(env)):
        assert (int(d[i]), int(m[i])) == oracle_answer(st, cur), (i, cur)
    return d, m


@pytest.mark.parametrize("multi", [True, False], ids=["ordered", "set"])
def test_optimal_moves_on_the_smallest_and_fullest_boards(ts, multi):
    # 1x1, one tile on its target: every move leaves it there
    one = ts.BatchedTilerSliderEnv.from_arrays(1, np.zeros((8, 1), np.uint8), np.zeros((8, 1, 2), np.uint8),
                                               np.zeros((8, 1, 2), np.uint8), multi)
    random_steps(one, 2, seed=1)
    d, m = check_all(one)
    assert (d == 1).all() and (m == 0xF).all()
    # 2x2 with four tiles: nothing moves.  On the goal: distance 1 by any move; a permuted goal is
    # never reached with coloured tiles and is the same goal without colours
    cells = np.array([[0, 0], [0, 1], [1, 0], [1, 1]], np.uint8)
    perms = np.array([[0, 1, 2, 3], [1, 0, 2, 3], [3, 2, 1, 0], [1, 2, 3, 0]])
    full = ts.BatchedTilerSliderEnv.from_arrays(2, np.zeros((4, 4), np.uint8), np.stack([cells] * 4), cells[perms], multi)
    random_steps(full, 2, seed=2)
    d, m = check_all(full)
    assert d[0] == 1 and m[0] == 0xF
    assert (d[1:] == -1).all() if multi else (d[1:] == 1).all()
    # 2x2 with 1 to 4 tiles and 3x3 with 3 or 4 tiles, 0 to 2 walls (4 tiles on 2x2: no room for walls)
    for S, T, walls in ((2, 1, (0, 1, 2)), (2, 2, (0, 1)), (2, 3, (0, 1)), (2, 4, (0,)), (3, 3, (0, 1, 2)), (3, 4, (0, 1, 2))):
        blocked, tiles, targets = puzzles(S, T, walls, 16, multi, seed=S * 10 + T, walk=5)
        env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
        random_steps(env, 3, seed=T)
        d, _ = check_all(env)
        assert (d >= 1).any()
