"""GPU tests of the hash-table search for 5 to 8 tiles (K11 ts_optimal_moves_table, reached through
optimal_moves(hash_table=True)) and of graded generation on it (solvable(hash_table=True)): answers
against the CPU oracle and BfsSolver, plans, result codes, the -3 bound, table reuse across many items
per CTA, generation and a 5-tile reset pool."""
import numpy as np
import pytest
import torch

from tests.test_gpu_optimal import oracle_answer, oracle_states, random_steps
from tests.test_gpu_optimal_items import check_plan

pytestmark = pytest.mark.gpu

NOT_SEARCHED = -3


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def oracle_of(env, i_list=None):
    """(distance, mask) by the oracle for the current positions of envs i_list (default all)."""
    states = oracle_states(env)
    return [oracle_answer(*states[i]) for i in (range(env.n_envs) if i_list is None else i_list)]


def mixed_batch(ts, S, T, W, multi, n, seed):
    """n solvable(hash_table=True) puzzles then, where the board has the W + 2T cells synthetic()
    draws, n synthetic() ones, after three random steps."""
    parts = [ts.BatchedTilerSliderEnv.solvable(n, S, T, W, multi, min_depth=1, max_depth=10, seed=seed, hash_table=True)]
    if W + 2 * T <= S * S:
        parts.append(ts.BatchedTilerSliderEnv.synthetic(n, S, T, W, multi, seed=seed + 1))
    blocked = torch.cat([e.blocked_cells() for e in parts]).cpu().numpy()
    tiles = torch.cat([e.positions(e._init[:n]) for e in parts]).cpu().numpy()
    tg = [e.target_positions().cpu().numpy() for e in parts]
    if multi:
        targets = np.concatenate(tg)
    else:                                            # set goal: target cells as (row, col) pairs
        targets = np.stack([np.stack(np.divmod(np.flatnonzero(m), S), 1) for m in np.concatenate(tg)]).astype(np.uint8)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    random_steps(env, 3, seed=seed + 2)
    return env


ORACLE_CASES = [  # S, T, W, multi
    (3, 5, 1, True), (3, 8, 0, True), (4, 6, 3, True), (5, 5, 5, True), (7, 5, 10, True),
    (5, 8, 8, False), (6, 5, 8, False), (6, 8, 8, False),
]


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_distance_and_mask_match_the_oracle(ts, S, T, W, multi):
    env = mixed_batch(ts, S, T, W, multi, 12, seed=10 * S + T)
    d, m = env.optimal_moves(hash_table=True)
    assert not ((d == -2) | (d == NOT_SEARCHED)).any()
    got = list(zip(d.tolist(), m.tolist()))
    assert got == oracle_of(env)
    assert (d >= 1).any()


def test_start_distance_equals_bfs_solver_depth(ts):
    from tiler_slider_b200.bfs import solve_batch
    env = mixed_batch(ts, 6, 5, 8, True, 32, seed=3)
    env.reset()
    d, _ = env.optimal_moves(hash_table=True)
    want = solve_batch(env).solve_depth_per_puzzle.cpu()
    assert torch.equal(d.cpu(), want.to(torch.int32))
    assert (d >= 1).any() and (d == -1).any()


@pytest.mark.parametrize("multi", [True, False])
def test_plans_win_in_exactly_distance_moves(ts, multi):
    env = ts.BatchedTilerSliderEnv.solvable(256, 6, 5, 8, multi, min_depth=1, max_depth=14, seed=21, hash_table=True)
    random_steps(env, 2, seed=4)
    ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda")
    pos = env.pos[: env.n_envs].contiguous()
    d0, m0 = env.optimal_moves(ids, pos, hash_table=True)
    d, m, plan = env.optimal_moves(ids, pos, paths=True, hash_table=True)
    assert torch.equal(d, d0) and torch.equal(m, m0)
    assert (d >= 1).any()
    # every later state of a replay is itself queried (check_plan's loop): the hash-table path throughout
    real = env.optimal_moves
    env.optimal_moves = lambda *a, **k: real(*a, hash_table=True, **k)
    try:
        check_plan(env, ids, pos, d, m, plan)
    finally:
        del env.optimal_moves


def test_result_codes(ts):
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env = ts.BatchedTilerSliderEnv.solvable(128, 6, 5, 8, True, min_depth=6, max_depth=12, seed=5, hash_table=True)
    # ids with pos, ids outside the table (-3), a malformed root (-4: two tiles on one cell)
    ids = torch.tensor([3, env.capacity, -1, 7, 1 << 30, 9], dtype=torch.int32, device="cuda")
    pos = env.pos[torch.tensor([3, 0, 0, 7, 0, 9], device="cuda")].clone()
    pos[5, 1] = pos[5, 0]
    d, m = CudaOptimalMoves(env).query(ids, 254, pos.contiguous(), hash_table=True)
    want3, want7 = oracle_of(env, [3, 7])
    assert d.tolist() == [want3[0], -3, -3, want7[0], -3, -4]
    assert m.tolist() == [want3[1], 0, 0, want7[1], 0, 0]
    # a max_depth cut-off (-2) with plans all 255
    d, m, plan = env.optimal_moves(max_depth=5, paths=True, hash_table=True)
    assert (d == -2).all() and (m == 0).all() and (plan == 255).all()
    # a state already on the goal: distance 1 through the moves that keep it there
    final, _, won = env.playout(actions=env.optimal_moves(paths=True, hash_table=True)[2])
    assert (won == 1).all()
    d, m = env.optimal_moves(pos=final, hash_table=True)
    _, _, won_a = env.expand(None, final)
    assert (d == 1).all() and torch.equal(m, won_a)
    # never_win: one target for five coloured tiles
    blocked = np.zeros((64, 36), np.uint8)
    tiles = np.array([[[0, 0], [1, 1], [2, 2], [3, 3], [4, 4]]] * 64, np.uint8)
    nw = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, np.array([[[0, 5]]] * 64, np.uint8), True)
    assert nw.never_win
    d, m, plan = nw.optimal_moves(paths=True, hash_table=True)
    assert (d == -1).all() and (m == 0).all() and (plan == 255).all()


@pytest.mark.parametrize("multi", [True, False])
def test_the_bound_is_predicted_exactly(ts, multi):
    """With table_slots forced to 2q, an item gets -3 exactly when its forward search discovers more
    than q states: the levels before the goal level (all of them when no win is reachable).  Every
    other item gets the default plan's answer."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env = mixed_batch(ts, 6, 5, 8, multi, 24, seed=40 + int(multi))
    states = oracle_states(env)
    need = []
    for st, _ in states:
        n, levels, depth, _ = st.bfs(max_states=1 << 22)
        need.append(sum(levels[:depth]) if depth >= 1 else n)
    need = np.array(need)
    full, full_m = env.optimal_moves(hash_table=True)
    assert not (full == NOT_SEARCHED).any()
    seen = set()
    for q in (32, 512, 4096):
        d, m = CudaOptimalMoves(env, table_slots=2 * q).query(None, 254, hash_table=True)
        big = need > q
        assert np.array_equal(d.cpu().numpy(), np.where(big, NOT_SEARCHED, full.cpu().numpy())), q
        assert np.array_equal(m.cpu().numpy(), np.where(big, 0, full_m.cpu().numpy())), q
        seen.update(big.tolist())
    assert seen == {True, False}


def test_table_reuse_across_hundreds_of_items_per_cta(ts):
    """A plan for one CTA per SM (the largest ring) and 32 puzzles repeated 4,000 times: every CTA
    serves more than a hundred items on average, past the 31 item epochs of its table many times, and
    every answer is its puzzle's."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    env = mixed_batch(ts, 6, 5, 8, True, 16, seed=60)
    want = oracle_of(env)
    ids = torch.arange(32, dtype=torch.int32, device="cuda").repeat(4000)
    search = CudaOptimalMoves(env, ctas_per_sm=1)
    d, m = search.query(ids, 254, hash_table=True)
    assert search._plan_table()["grid"] * 100 < ids.numel()
    got = torch.stack([d, m.int()], 1).view(4000, 32, 2)
    assert (got == torch.tensor(want, dtype=torch.int32, device="cuda")[None]).all()


@pytest.mark.parametrize("multi", [True, False])
def test_solvable_grades_by_the_table_search(ts, multi):
    kw = dict(min_depth=4, max_depth=9, seed=7, hash_table=True)
    env = ts.BatchedTilerSliderEnv.solvable(512, 6, 5, 8, multi, **kw)
    depth = env.solve_depth
    assert ((depth >= 4) & (depth <= 9)).all()
    d, _ = env.optimal_moves(hash_table=True)
    assert torch.equal(d, depth)
    hi = ts.BatchedTilerSliderEnv.solvable(256, 6, 5, 8, multi, env_index_base=256, **kw)
    lo = ts.BatchedTilerSliderEnv.solvable(256, 6, 5, 8, multi, **kw)
    for part, sl in ((lo, slice(0, 256)), (hi, slice(256, 512))):
        assert torch.equal(part.blocked_cells(), env.blocked_cells()[sl])
        assert torch.equal(part.target_positions(), env.target_positions()[sl])
        assert torch.equal(part._init[:256], env._init[sl]) and torch.equal(part.solve_depth, depth[sl])


def test_a_five_tile_reset_pool(ts):
    pool = ts.BatchedTilerSliderEnv.solvable(64, 6, 5, 8, True, min_depth=2, max_depth=8, seed=9, hash_table=True)
    env = ts.BatchedTilerSliderEnv.synthetic(1024, 6, 5, 8, True, auto_reset=True)
    env.set_reset_pool(pool, seed=3, draw_now=True)
    keys = {tuple(b) + tuple(i): k for k, (b, i) in
            enumerate(zip(pool.blocked_cells().cpu().numpy().tolist(), pool._init[:64].cpu().numpy().tolist()))}
    blocked, init = env.blocked_cells().cpu().numpy().tolist(), env._init[:1024].cpu().numpy().tolist()
    js = [keys[tuple(b) + tuple(i)] for b, i in zip(blocked, init)]
    assert torch.equal(env.solve_depth.cpu(), pool.solve_depth.cpu()[js])
    assert torch.equal(env.target_positions().cpu(), pool.target_positions().cpu()[js])
    d, _ = env.optimal_moves(hash_table=True)
    assert torch.equal(d, env.solve_depth)
    assert len(set(js)) > 32
