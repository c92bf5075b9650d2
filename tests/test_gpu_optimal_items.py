"""GPU tests of optimal-move queries on items and of their shortest solutions
(BatchedTilerSliderEnv.optimal_moves(ids, pos, paths=True), K9 ts_optimal_moves): item answers
equal env answers, successors against the CPU oracle and against each other (Bellman), plans that
win in exactly `distance` moves and equal a greedy CPU solver, the result codes on items, the slab
path and the edge cases."""
import os

import numpy as np
import pytest
import torch

from tests.test_gpu_optimal import LOWEST_BIT, ORACLE_CASES, F_WON, oracle_answer, oracle_states, random_steps

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def lowest_bit(mask):
    return LOWEST_BIT.to(mask.device)[mask.long()]


def successor_items(env):
    """The 4N expand() successors of the envs' current positions as items (ids, pos)."""
    succ, _, _ = env.expand()
    ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda").repeat_interleave(4)
    return ids, succ.reshape(-1, env.pos_bytes).contiguous()


def check_plan(env, ids, pos, d, m, plan, max_depth=254):
    """The plan contract: shape, 0..3 on rows < d, 255 elsewhere, row 0 the lowest bit of the mask,
    a replay wins in exactly d moves, and every move is the lowest optimal move of its state."""
    n = d.numel()
    assert plan.shape == (max_depth, n) and plan.dtype == torch.uint8 and plan.is_contiguous()
    rows = torch.arange(max_depth, device="cuda")[:, None]
    inside = rows < d[None, :].long()
    assert (plan[inside] <= 3).all() and (plan[~inside] == 255).all()
    ok = d >= 1
    assert torch.equal(plan[0][ok], lowest_bit(m)[ok])
    final, steps, won, moves, traj = env.playout(ids, pos, actions=plan, record=True)
    assert (won[ok] == 1).all() and torch.equal(steps[ok], d[ok])
    assert torch.equal(moves[inside], plan[inside])
    for k in range(int(d.max()) - 1 if ok.any() else 0):
        dk, mk = env.optimal_moves(ids, pos=traj[k].contiguous())
        live = d > k + 1
        assert torch.equal(dk[live], d[live] - k - 1)
        assert torch.equal(plan[k + 1][live], lowest_bit(mk)[live])
        if env.n_tiles >= 2:                         # the zero rows past an item's end: two tiles on one cell
            assert (dk[steps <= k] == -4).all()


def item_boards(env, ids, pos):
    """(oracle board, locations) of each item."""
    boards = oracle_states(env)
    locs = env.positions(pos).cpu().numpy()
    return [(boards[i][0], locs[j].tolist()) for j, i in enumerate(ids.cpu().tolist())]


def greedy_plan(st, cur):
    """A CPU shortest solution from `cur`: at every state the lowest bit of the oracle's mask."""
    moves = []
    d, m = oracle_answer(st, cur)
    for k in range(max(d, 0)):                  # d moves; the state after the last one is on the goal
        if k:
            _, m = oracle_answer(st, cur)
        a = (m & -m).bit_length() - 1
        moves.append(a)
        st.set_locations(cur)
        st.move(a)
        cur = st.current_locations
    return moves


def check_against_cpu(env, ids, pos, d, m, plan, sample, plan_sample):
    boards = item_boards(env, ids, pos)
    d, m, plan = d.cpu().numpy(), m.cpu().numpy(), plan.cpu().numpy()
    for j in sample:
        st, cur = boards[j]
        assert (int(d[j]), int(m[j])) == oracle_answer(st, cur), (j, cur)
    for j in plan_sample:
        st, cur = boards[j]
        want = greedy_plan(st, cur)
        assert plan[: max(int(d[j]), 0), j].tolist() == want, (j, cur)


# ---- 1. items equal env queries ------------------------------------------------------------------

@pytest.mark.parametrize("multi", [True, False])
def test_items_equal_env_queries(ts, multi):
    env = ts.BatchedTilerSliderEnv.solvable(4096, 6, 4, 8, multi, min_depth=1, max_depth=16, seed=31, max_steps=40)
    random_steps(env, 4, seed=6)
    d0, m0 = env.optimal_moves()
    g = torch.Generator(device="cuda").manual_seed(2)
    ids = torch.randint(0, 4096, (6000,), device="cuda", generator=g, dtype=torch.int32)     # shuffled, repeated
    pos = env.pos[ids.long()].contiguous()
    before = {k: getattr(env, k).clone() for k in ("pos", "step_count", "flags")}
    d, m = env.optimal_moves(ids, pos=pos)
    for k, t in before.items():
        assert torch.equal(getattr(env, k), t), k
    d1, m1 = env.optimal_moves(ids)
    assert torch.equal(d, d1) and torch.equal(m, m1)
    assert torch.equal(d, d0[ids.long()]) and torch.equal(m, m0[ids.long()])
    host = ids[:500].tolist()
    dh, mh = env.optimal_moves(host, pos=pos[:500].clone())
    assert torch.equal(dh, d[:500]) and torch.equal(mh, m[:500])
    da, ma = env.optimal_moves(pos=env.pos.clone())                           # no ids: n_envs rows
    assert torch.equal(da, d0) and torch.equal(ma, m0)
    with pytest.raises(IndexError):
        env.optimal_moves([0, 4096], pos=pos[:2].clone())
    with pytest.raises(ValueError):
        env.optimal_moves(ids, pos=pos[:-1].contiguous())
    with pytest.raises(ValueError):
        env.optimal_moves(ids, pos=pos.to(torch.int32))
    with pytest.raises(ValueError):
        env.optimal_moves(ids, pos=pos.cpu())
    with pytest.raises(ValueError):
        env.optimal_moves(pos=torch.cat([env.pos, env.pos], 1)[:, ::2])       # not contiguous


# ---- 2, 3. successors against the oracle and the Bellman equations; their plans -------------------

@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_successor_items(ts, S, T, W, multi):
    """The 4N expand() successors of solvable and uniform puzzles: distance and mask equal the oracle
    on a sample, every item is Bellman-consistent with its parent, and the plans hold their contract
    and equal the CPU greedy solution on a sample."""
    N = 256
    solv = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=1, max_depth=16, seed=S * 7 + T)
    syn = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=S * 7 + T)
    rng = np.random.default_rng(S * 10 + T)
    for k, env in enumerate((solv, syn)):
        random_steps(env, 2 + k, seed=S + T)
        dp, mp = env.optimal_moves()
        _, moved, won = env.expand()
        ids, pos = successor_items(env)
        d, m, plan = env.optimal_moves(ids, pos=pos, paths=True)
        d2, m2 = env.optimal_moves(ids, pos=pos)
        assert torch.equal(d, d2) and torch.equal(m, m2)
        assert not (d == -3).any() and not (d == -4).any() and not (d == -2).any()
        # Bellman consistency, parent by parent, no oracle
        dc = d.view(N, 4)
        bit = torch.arange(4, device="cuda")
        moved_a = (moved[:, None].long() >> bit) & 1 == 1
        won_a = (won[:, None].long() >> bit) & 1 == 1
        opt_a = (mp[:, None].long() >> bit) & 1 == 1
        two = dp >= 2
        assert torch.equal(opt_a[two], (moved_a & (dc == (dp - 1)[:, None]))[two])
        best = torch.where(dc >= 1, dc, torch.full_like(dc, 1 << 20)).min(1).values
        assert torch.equal(dp[two], 1 + best[two])
        one = dp == 1
        assert torch.equal(opt_a[one], won_a[one])
        assert (dc[dp == -1] == -1).all()
        check_plan(env, ids, pos, d, m, plan)
        sample = rng.choice(4 * N, 24, replace=False)
        check_against_cpu(env, ids, pos, d, m, plan, sample, sample[:6])


def test_real_level_plans(ts):
    """The reference's real levels after random steps: plans hold their contract and equal the CPU
    greedy solution on a sample of every group."""
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
        ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda")
        pos = env.pos.clone()
        d, m, plan = env.optimal_moves(ids, pos=pos, paths=True)
        assert not (d == -3).any() and not (d == -4).any()
        check_plan(env, ids, pos, d, m, plan)
        check_against_cpu(env, ids, pos, d, m, plan, range(0, env.n_envs, 8), range(0, env.n_envs, 16))
        checked += env.n_envs
    assert checked >= 256


# ---- 4. one query replaces the expert loop -------------------------------------------------------

@pytest.mark.parametrize("multi", [True, False])
def test_one_query_replaces_the_expert_loop(ts, multi):
    N = 65536
    env = ts.BatchedTilerSliderEnv.solvable(N, 6, 4, 8, multi, min_depth=8, max_depth=12, seed=7)
    depth = env.solve_depth.clone()
    d, m, plan = env.optimal_moves(paths=True)
    assert torch.equal(d, depth)
    won_at = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    for k in range(14):
        row = plan[k]
        env.step(torch.where(row > 3, torch.zeros_like(row), row))
        won = (env.flags & F_WON) != 0
        assert (won_at[won] == -1).all()                                   # WON once, then frozen
        won_at[won] = k + 1
    assert torch.equal(won_at, depth)


# ---- 5. result codes on items --------------------------------------------------------------------

def test_unsolvable_cutoff_and_never_win_items(ts):
    syn = ts.BatchedTilerSliderEnv.synthetic(2048, 6, 4, 8, True, seed=5)
    ids = torch.arange(2048, dtype=torch.int32, device="cuda").flip(0).contiguous()
    d, m, plan = syn.optimal_moves(ids, pos=syn.pos[ids.long()].contiguous(), paths=True)
    assert (d == -1).sum() > 1000
    assert (plan[:, d < 0] == 255).all() and (m[d < 0] == 0).all()
    solv = ts.BatchedTilerSliderEnv.solvable(1024, 6, 4, 8, True, min_depth=6, max_depth=12, seed=4)
    d, m, plan = solv.optimal_moves(pos=solv.pos.clone(), max_depth=5, paths=True)
    assert plan.shape == (5, 1024)
    assert (d == -2).all() and (m == 0).all() and (plan == 255).all()
    blocked = np.zeros((64, 25), np.uint8)
    tiles = np.array([[[0, 0], [4, 4]]] * 64, np.uint8)
    targets = np.array([[[0, 4]]] * 64, np.uint8)           # one target for two coloured tiles: never won
    nw = ts.BatchedTilerSliderEnv.from_arrays(5, blocked, tiles, targets, True)
    assert nw.never_win
    d, m, plan = nw.optimal_moves(pos=nw.pos.clone(), paths=True)
    assert (d == -1).all() and (m == 0).all() and (plan == 255).all()


def test_not_searched_items(ts):
    big = ts.BatchedTilerSliderEnv.synthetic(64, 8, 4, 0, True, seed=1)    # 64*63*62*61 states
    d, m, plan = big.optimal_moves(pos=big.pos.clone(), paths=True)
    assert (d == -3).all() and (m == 0).all() and (plan == 255).all()
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env = ts.BatchedTilerSliderEnv.solvable(256, 6, 4, 8, False, min_depth=2, max_depth=10, seed=3)
    ids = torch.tensor([0, env.capacity, -1, 5, 1 << 30], dtype=torch.int32, device="cuda")
    pos = env.pos[torch.tensor([0, 1, 2, 5, 3], device="cuda")].contiguous()
    plan = torch.empty((254, 5), dtype=torch.uint8, device="cuda")
    d, m = CudaOptimalMoves(env).query(ids, 254, pos, plan)
    d0, m0 = env.optimal_moves([0, 5])
    assert d.tolist()[1:3] == [-3, -3] and d[4].item() == -3 and (m[[1, 2, 4]] == 0).all()
    assert (plan[:, [1, 2, 4]] == 255).all()
    assert d[[0, 3]].tolist() == d0.tolist() and m[[0, 3]].tolist() == m0.tolist()


@pytest.mark.parametrize("S,T,multi", [(6, 4, True), (6, 3, False), (8, 2, True), (7, 4, False), (3, 2, True)])
def test_bad_states(ts, S, T, multi):
    """A tile on a wall, two tiles on one cell, a byte of 255 and a cell off the board give -4, an
    empty mask and an all-255 plan column; the well-formed items around them keep their answers."""
    W = {3: 2, 6: 8, 7: 14, 8: 24}[S]
    env = ts.BatchedTilerSliderEnv.solvable(64, S, T, W, multi, min_depth=1, max_depth=12, seed=S + T)
    ps = env.pos_stride
    blocked = env.blocked_cells().cpu().numpy()
    good = env.pos.clone()
    rows, kinds = [], []
    for i in range(env.n_envs):
        w = np.flatnonzero(blocked[i])
        p = good[i].clone()
        kind = i % 5
        if kind == 1:                                   # a tile on a wall
            p[T - 1] = int(w[0] // S * ps + w[0] % S)
        elif kind == 2:                                 # two tiles on one cell
            p[T - 1] = p[0]
        elif kind == 3:
            p[0] = 255
        elif kind == 4:                                 # off the board: column S, or row S
            p[0] = (S - 1) * ps + S if i % 2 else S * ps
        rows.append(p)
        kinds.append(kind)
    pos = torch.stack(rows).contiguous()
    kinds = torch.tensor(kinds, device="cuda")
    ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda")
    d, m, plan = env.optimal_moves(ids, pos=pos, paths=True)
    bad = kinds != 0
    if T == 1:
        bad = bad & (kinds != 2)                        # one tile cannot share its cell
    assert (d[bad] == -4).all() and (m[bad] == 0).all() and (plan[:, bad] == 255).all()
    keep = (kinds == 0).nonzero().flatten().to(torch.int32)
    d0, m0, p0 = env.optimal_moves(keep, pos=good[keep.long()].contiguous(), paths=True)
    assert torch.equal(d[keep.long()], d0) and torch.equal(m[keep.long()], m0) and torch.equal(plan[:, keep.long()], p0)
    assert (d0 >= 1).all()


# ---- 6. the slab path ----------------------------------------------------------------------------

def test_slab_path_and_determinism(ts):
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env = ts.BatchedTilerSliderEnv.solvable(4096, 6, 4, 8, False, min_depth=4, max_depth=20, seed=9)
    random_steps(env, 3, seed=4)
    ids, pos = successor_items(env)
    n = ids.numel()
    outs = []
    for q in (CudaOptimalMoves(env), CudaOptimalMoves(env, queue_smem=32), CudaOptimalMoves(env, queue_smem=32)):
        plan = torch.empty((254, n), dtype=torch.uint8, device="cuda")
        d, m = q.query(ids, 254, pos, plan)
        outs.append((d, m, plan))
    assert CudaOptimalMoves(env, queue_smem=32).plan(28)["queue_smem"] == 32
    for d, m, plan in outs[1:]:
        assert torch.equal(d, outs[0][0]) and torch.equal(m, outs[0][1]) and torch.equal(plan, outs[0][2])
    assert (outs[0][0] >= 1).sum() > n // 2


# ---- 7. edge cases -------------------------------------------------------------------------------

def test_no_items_and_states_on_the_goal(ts):
    env = ts.BatchedTilerSliderEnv.solvable(512, 5, 2, 4, True, min_depth=1, max_depth=4, seed=3)
    d, m, plan = env.optimal_moves([], pos=torch.empty((0, env.pos_bytes), dtype=torch.uint8, device="cuda"),
                                   paths=True)
    assert d.shape == (0,) and m.shape == (0,) and plan.shape == (254, 0)
    d, m, plan = env.optimal_moves([], max_depth=7, paths=True)
    assert plan.shape == (7, 0)
    d0, _, plan0 = env.optimal_moves(paths=True)
    final, steps, won = env.playout(actions=plan0)
    assert (won == 1).all()
    ids = torch.arange(512, dtype=torch.int32, device="cuda")
    d, m, plan = env.optimal_moves(ids, pos=final, paths=True)
    _, _, won_a = env.expand(ids, final)
    assert (d == 1).all() and torch.equal(m, won_a)
    assert torch.equal(plan[0], lowest_bit(m)) and (plan[1:] == 255).all()
