"""GPU tests of the optimal-move query (BatchedTilerSliderEnv.optimal_moves, K9 ts_optimal_moves):
distances and optimal-move masks of the CURRENT positions against the CPU oracle's BFS, expert
rollouts, the result codes, and the reset pool."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

F_WON = 2
LOWEST_BIT = torch.tensor([0, 0, 1, 0, 2, 0, 1, 0, 3, 0, 1, 0, 2, 0, 1, 0], dtype=torch.uint8)


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def oracle_states(env):
    """One oracle board per env at its current positions."""
    S, n, multi = env.size, env.n_envs, env.multi_color
    blocked = env.blocked_cells().cpu().numpy()
    targets = env.target_positions().cpu().numpy()
    cur = env.positions().cpu().numpy()
    out = []
    for i in range(n):
        b = [divmod(int(c), S) for c in np.flatnonzero(blocked[i])]
        tg = targets[i].tolist() if targets.ndim == 3 else [divmod(int(c), S) for c in np.flatnonzero(targets[i])]
        st = orc.OracleState(S, b, cur[i].tolist(), tg, multi)
        out.append((st, cur[i].tolist()))
    return out


def oracle_answer(st, cur, max_depth=254):
    """(distance, mask) by the oracle's BFS from `cur` and from each of its four successors."""
    st.set_locations(cur)
    d = st.bfs(max_depth=max_depth, max_states=1 << 22)[2]
    mask = 0
    if d >= 1:
        for a in range(4):
            st.set_locations(cur)
            st.move(a)
            if d == 1:
                ok = st.is_won()
            else:
                ok = st.bfs(max_depth=d, max_states=1 << 22)[2] == d - 1
            mask |= int(ok) << a
    st.set_locations(cur)
    return d, mask


def random_steps(env, k, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    for _ in range(k):
        env.step(torch.randint(0, 4, (env.n_envs,), generator=g, dtype=torch.uint8).cuda())


def check_against_oracle(env, dist, mask, sample):
    dist, mask = dist.cpu().numpy(), mask.cpu().numpy()
    states = oracle_states(env)
    for i in sample:
        st, cur = states[i]
        want = oracle_answer(st, cur)
        assert (int(dist[i]), int(mask[i])) == want, (i, cur, want)


ORACLE_CASES = [  # S, T, W, multi
    (3, 1, 1, False), (3, 2, 2, True), (4, 2, 3, False), (4, 3, 4, True), (5, 1, 4, True), (5, 3, 6, False),
    (6, 4, 8, True), (6, 4, 8, False), (7, 2, 14, True), (7, 3, 16, False), (8, 4, 34, True), (8, 2, 24, False),
]


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_distance_and_mask_match_the_oracle(ts, S, T, W, multi):
    """Solvable puzzles and uniform draws (mostly unsolvable with several tiles), stepped a few random
    steps so that the current state differs from init: distance and mask equal the oracle's BFS from
    the current locations."""
    N = 256
    solv = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=1, max_depth=20, seed=S * 10 + T)
    syn = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=S * 10 + T)
    for k, env in enumerate((solv, syn)):
        random_steps(env, 3 + k, seed=S + T)
        dist, mask = env.optimal_moves()
        assert dist.dtype == torch.int32 and mask.dtype == torch.uint8 and dist.shape == mask.shape == (N,)
        assert not (dist == -3).any() and not (dist == -2).any()
        check_against_oracle(env, dist, mask, range(N))


def test_real_levels_match_the_oracle(ts):
    """The reference's real levels (tests/golden/levels_400.txt), grouped by shape, after random steps."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_400.txt")
    groups = {}
    for p in ts.load_puzzle_file(path):
        groups.setdefault((p.size, len(p.initial_locations), p.multiple_colors), []).append(p)
    checked = 0
    for (S, T, multi), ps in groups.items():
        if S > 8 or not 1 <= T <= 4:
            continue
        env = ts.BatchedTilerSliderEnv.from_puzzles(ps)
        random_steps(env, 2, seed=S * T)
        dist, mask = env.optimal_moves()
        assert not (dist == -3).any()
        check_against_oracle(env, dist, mask, range(env.n_envs))
        checked += env.n_envs
    assert checked >= 256


@pytest.mark.parametrize("multi", [True, False])
def test_expert_rollouts(ts, multi):
    """65,536 solvable puzzles in [8, 12]: the first answer equals solve_depth; stepping a random optimal
    move lowers the distance by exactly 1 and wins on exactly step solve_depth; a random non-optimal
    move from the same states never reaches distance d-1."""
    N = 65536
    env = ts.BatchedTilerSliderEnv.solvable(N, 6, 4, 8, multi, min_depth=8, max_depth=12, seed=7)
    depth = env.solve_depth.clone()
    d, m = env.optimal_moves()
    assert torch.equal(d, depth) and (m != 0).all()
    g = torch.Generator(device="cuda").manual_seed(1)
    won_at = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    finished = torch.zeros(N, dtype=torch.bool, device="cuda")
    for k in range(1, 13):
        live = ~finished
        # from the same states: a random non-optimal move (where one exists) never reaches d - 1
        bad = (~m & 0xF) * live.to(torch.uint8)
        saved = env.pos.clone()
        env.raw_move(random_bit(bad, g))
        d_bad, _ = env.optimal_moves()
        assert not ((bad != 0) & (d_bad == d - 1)).any()
        env._pos[:N].copy_(saved)
        # a random optimal move
        env.step(random_bit(m, g))
        won = (env.flags & F_WON) != 0                  # frozen envs report DONE | STALE, not WON
        won_at[won] = k
        d2, m2 = env.optimal_moves()
        still = live & ~won
        assert torch.equal(d2[still], d[still] - 1)
        assert (d[won] == 1).all() and (d2[won] == 1).all()
        finished |= won
        d, m = d2, m2
    assert torch.equal(won_at, depth)


def random_bit(mask, g):
    """A uniformly drawn set bit of each 4-bit mask (0 where the mask is empty)."""
    bits = (mask.unsqueeze(1).to(torch.int32) >> torch.arange(4, device=mask.device, dtype=torch.int32)) & 1
    score = torch.rand(mask.shape[0], 4, device=mask.device, generator=g) * bits
    return torch.where(bits.any(1), score.argmax(1), torch.zeros_like(mask, dtype=torch.int64)).to(torch.uint8)


def test_state_on_the_goal(ts):
    """Envs that won and froze (STALE) sit on the goal: distance 1, and the mask holds the moves that
    leave them there, those that change nothing included (checked against the oracle)."""
    env = ts.BatchedTilerSliderEnv.solvable(512, 5, 2, 4, True, min_depth=1, max_depth=2, seed=3)
    for k in range(4):
        _, m = env.optimal_moves()
        env.step(LOWEST_BIT.cuda()[m.long()])
    assert env.done.all()
    valid = env.valid_moves()
    d, m = env.optimal_moves()
    assert (d == 1).all()
    assert ((m & ~valid & 0xF) != 0).any()          # moves that change nothing are optimal here
    check_against_oracle(env, d, m, range(0, 512, 2))


def test_unsolvable_and_never_win(ts):
    syn = ts.BatchedTilerSliderEnv.synthetic(2048, 6, 4, 8, True, seed=5)
    from tiler_slider_b200.bfs import LocalBfs
    ref = LocalBfs(syn).solve(max_depth=254).solve_depth_per_puzzle
    d, m = syn.optimal_moves()
    assert (ref == -1).sum() > 1000
    assert torch.equal(d[ref == -1], torch.full_like(d[ref == -1], -1)) and (m[ref == -1] == 0).all()
    assert torch.equal(d[ref > 0], ref[ref > 0])
    blocked = np.zeros((64, 25), np.uint8)
    tiles = np.array([[[0, 0], [4, 4]]] * 64, np.uint8)
    targets = np.array([[[0, 4]]] * 64, np.uint8)           # one target for two coloured tiles: never won
    nw = ts.BatchedTilerSliderEnv.from_arrays(5, blocked, tiles, targets, True)
    assert nw.never_win
    random_steps(nw, 3, 0)
    d, m = nw.optimal_moves()
    assert (d == -1).all() and (m == 0).all()


def test_max_depth_cutoff(ts):
    """A small max_depth gives -2 exactly for the envs deeper than it and exact answers for the rest."""
    env = ts.BatchedTilerSliderEnv.solvable(4096, 6, 4, 8, True, min_depth=1, max_depth=16, seed=11)
    random_steps(env, 2, seed=2)
    d_full, m_full = env.optimal_moves()
    for cut in (1, 5, 9):
        d, m = env.optimal_moves(max_depth=cut)
        assert (d_full > cut).any()
        assert torch.equal(d[d_full > cut], torch.full_like(d[d_full > cut], -2))
        assert (m[d_full > cut] == 0).all()
        ok = (d_full >= 1) & (d_full <= cut)
        assert torch.equal(d[ok], d_full[ok]) and torch.equal(m[ok], m_full[ok])
        # no win at all: -1 when the reachable set ran out within `cut` levels, else -2
        assert ((d[d_full == -1] == -1) | (d[d_full == -1] == -2)).all()


def test_too_large_state_space(ts):
    """8x8, 4 tiles, no walls: 64*63*62*61 states do not fit the bitmap: -3 with an empty mask."""
    env = ts.BatchedTilerSliderEnv.synthetic(256, 8, 4, 0, True, seed=1)
    d, m = env.optimal_moves()
    assert (d == -3).all() and (m == 0).all()


def test_ids_order_state_untouched_forced_ring_repeat(ts):
    env = ts.BatchedTilerSliderEnv.solvable(4096, 6, 4, 8, False, min_depth=4, max_depth=20, seed=9, max_steps=30)
    random_steps(env, 4, seed=4)
    before = {name: getattr(env, name).clone() for name in ("_walls", "_targets", "_init", "_pos", "_count", "_done", "_flags",
                                                            "_reward", "_solve_depth")}
    d, m = env.optimal_moves()
    for name, t in before.items():
        assert torch.equal(getattr(env, name), t), name
    d2, m2 = env.optimal_moves()
    assert torch.equal(d, d2) and torch.equal(m, m2)
    ids = torch.randperm(4096, device="cuda")[:1000].to(torch.int32)
    di, mi = env.optimal_moves(ids)
    assert torch.equal(di, d[ids.long()]) and torch.equal(mi, m[ids.long()])
    di, mi = env.optimal_moves(ids.tolist()[::-1])
    assert torch.equal(di, d[ids.long()].flip(0)) and torch.equal(mi, m[ids.long()].flip(0))
    with pytest.raises(IndexError):
        env.optimal_moves([0, 4096])
    from tiler_slider_b200.bfs import CudaOptimalMoves
    small = CudaOptimalMoves(env, queue_smem=32)                 # levels read back from the slab
    ds, ms = small.query(None, 254)
    assert small.plan(28)["queue_smem"] == 32
    assert torch.equal(ds, d) and torch.equal(ms, m)


def test_reset_pool_with_more_free_cells(ts):
    """A pool whose puzzles have more free cells than the batch's own: the bitmap is sized per call,
    so no env reports -3, and envs that just reset report their pool puzzle's depth."""
    N = 8192
    env = ts.BatchedTilerSliderEnv.solvable(N, 6, 3, 12, True, min_depth=1, max_depth=10, seed=21, auto_reset=True,
                                            max_steps=12)
    pool = ts.BatchedTilerSliderEnv.solvable(2048, 6, 3, 4, True, min_depth=3, max_depth=10, seed=22)
    d0, _ = env.optimal_moves()
    assert torch.equal(d0, env.solve_depth)
    env.set_reset_pool(pool, seed=5)
    g = torch.Generator(device="cuda").manual_seed(3)
    fresh_seen = 0
    for k in range(30):
        _, m = env.optimal_moves()
        act = random_bit(m, g)
        explore = torch.rand(N, device="cuda", generator=g) < 0.3
        act = torch.where(explore, torch.randint(0, 4, (N,), device="cuda", generator=g, dtype=torch.uint8), act)
        env.step(act)
        d, m = env.optimal_moves()
        assert not (d == -3).any()
        fresh = env.step_count == 0
        fresh_seen += int(fresh.sum())
        assert torch.equal(d[fresh], env.solve_depth[fresh])
    assert fresh_seen > N
