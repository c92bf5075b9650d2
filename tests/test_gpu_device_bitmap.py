"""GPU tests of the device-memory-bitmap searches (device_bitmap=True): 7x7 and 8x8 boards with four
tiles whose state space outgrows one CTA's shared memory, searched by K6 (LocalBfs, solvable()), K9
(optimal_moves) and K10 (state_table) with the bitmap in device memory.  Every expectation comes
from the CPU oracle's BFS, or from the shared-memory instances on boards both can hold."""
import functools

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.test_gpu_optimal import oracle_answer, oracle_states, random_steps
from tests.test_gpu_optimal_items import lowest_bit, successor_items
from tests.test_gpu_search_limits import free_cells, puzzles, replay_wins_at
from tests.test_gpu_state_table import host_index, item_of_rows, oracle_keys

pytestmark = pytest.mark.gpu

NOT_SEARCHED = -3
F_STAR = 38                         # the most free cells a four-tile shared bitmap holds (test_on_chip_host)
BIG = [(7, (0, 4, 8)), (8, (0, 8, 12, 25))]          # F from 39 to 64: only the device bitmap holds them
MODES = pytest.mark.parametrize("multi", [True, False], ids=["ordered", "set"])


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


@functools.lru_cache(maxsize=None)
def big_batch(S, multi, n=6):
    """n boards of S x S with four tiles for each wall count of BIG, walk targets, three random steps."""
    import tiler_slider_b200 as ts
    walls = dict(BIG)[S]
    blocked, tiles, targets = puzzles(S, 4, walls, n, multi, seed=S * 10 + int(multi), walk=10)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    random_steps(env, 3, seed=S)
    assert (free_cells(env) > F_STAR).all() and free_cells(env).max() == S * S
    return env


def check_plan(env, ids, pos, d, m, plan):
    """test_gpu_optimal_items.check_plan with device_bitmap=True: a replay wins in exactly d moves,
    each move the lowest bit of the mask of the state it is played from."""
    rows = torch.arange(plan.shape[0], device="cuda")[:, None]
    inside = rows < d[None, :].long()
    assert (plan[inside] <= 3).all() and (plan[~inside] == 255).all()
    ok = d >= 1
    assert torch.equal(plan[0][ok], lowest_bit(m)[ok])
    final, steps, won, moves, traj = env.playout(ids, pos, actions=plan, record=True)
    assert (won[ok] == 1).all() and torch.equal(steps[ok], d[ok])
    for k in range(int(d.max()) - 1 if ok.any() else 0):
        dk, mk = env.optimal_moves(ids, pos=traj[k].contiguous(), device_bitmap=True)
        live = d > k + 1
        assert torch.equal(dk[live], d[live] - k - 1)
        assert torch.equal(plan[k + 1][live], lowest_bit(mk)[live])


# ---- K9 against the oracle -------------------------------------------------------------------------

@pytest.mark.parametrize("S", [7, 8])
@MODES
def test_optimal_moves_match_the_oracle(ts, S, multi):
    env = big_batch(S, multi)
    d0, m0 = env.optimal_moves()
    assert (d0 == NOT_SEARCHED).all()                                  # the default is unchanged
    d, m = env.optimal_moves(device_bitmap=True)
    dn, mn = d.cpu().numpy(), m.cpu().numpy()
    for i, (st, cur) in enumerate(oracle_states(env)):
        assert (int(dn[i]), int(mn[i])) == oracle_answer(st, cur), (i, cur)
    assert (dn >= 1).sum() > env.n_envs // 2
    dp, mp, plan = env.optimal_moves(paths=True, device_bitmap=True)
    assert torch.equal(dp, d) and torch.equal(mp, m)
    ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda")
    check_plan(env, ids, None, dp, mp, plan)


@pytest.mark.parametrize("S", [7, 8])
@MODES
def test_successor_items_match_the_oracle(ts, S, multi):
    env = big_batch(S, multi)
    ids, pos = successor_items(env)
    d, m = env.optimal_moves(ids, pos, device_bitmap=True)
    boards = oracle_states(env)
    locs = env.positions(pos).cpu().numpy()
    dn, mn = d.cpu().numpy(), m.cpu().numpy()
    for j in np.random.default_rng(S).choice(len(dn), 24, replace=False):
        st = boards[int(ids[j])][0]
        assert (int(dn[j]), int(mn[j])) == oracle_answer(st, locs[j].tolist()), j


# ---- K10 ---------------------------------------------------------------------------------------------

def bellman_ok(env, tab):
    """test_gpu_state_table.test_bellman_inside_the_table on one table."""
    T = env.n_tiles
    ids = item_of_rows(tab)
    succ, _, won = env.expand(ids.to(torch.int32), tab.pos.contiguous())
    if not env.multi_color:
        succ = succ.sort(-1).values
    d, m = tab.distance.cpu().numpy(), tab.mask.cpu().numpy()
    rows_key = ids.cpu().numpy().astype(np.int64) << 32 | oracle_keys(env, tab.pos).astype(np.int64)
    order = np.argsort(rows_key)
    sk = rows_key[order]
    one = d == 1
    assert T == env.pos_bytes and np.array_equal(m[one], won.cpu().numpy()[one])
    for a in range(4):
        key = ids.cpu().numpy().astype(np.int64) << 32 | oracle_keys(env, succ[:, a]).astype(np.int64)
        at = np.searchsorted(sk, key).clip(0, len(sk) - 1)
        assert (sk[at] == key).all()
        want = (key != rows_key) & (d[order[at]] == d - 1) & (d >= 2)
        assert np.array_equal(((m >> a) & 1).astype(bool) & (d >= 2), want), a


@pytest.mark.parametrize("S", [7, 8])
@MODES
def test_state_tables(ts, S, multi):
    env = big_batch(S, multi)
    assert (env.state_table().status == NOT_SEARCHED).all()           # the default is unchanged
    tab = env.state_table(device_bitmap=True)
    assert (tab.status == 0).all()
    # rows: the oracle's reachable set (canonical in set mode), ascending hash order
    off = tab.offsets.cpu().numpy()
    for i, (st, cur) in enumerate(oracle_states(env)):
        st.set_locations(cur)
        keys = st.bfs(max_states=1 << 22)[3]
        got = oracle_keys(env, tab.pos[off[i]:off[i + 1]])
        assert np.array_equal(np.sort(got), np.sort(keys)), i
    if not multi:
        assert (tab.pos[:, 1:] >= tab.pos[:, :-1]).all()
    items = item_of_rows(tab).cpu().numpy()
    idx = host_index(env, items, tab.pos)
    same = items[1:] == items[:-1]
    assert (idx[1:][same] > idx[:-1][same]).all()
    # labels: K9 on every row, Bellman inside the table
    d, m = env.optimal_moves(item_of_rows(tab).to(torch.int32), pos=tab.pos.contiguous(), device_bitmap=True)
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
    bellman_ok(env, tab)
    # determinism, also after a call on other items has left its states in the uncleared bitmaps
    again = env.state_table(device_bitmap=True)
    ids, pos = successor_items(env)
    assert (env.state_table(ids, pos, device_bitmap=True).status == 0).all()
    third = env.state_table(device_bitmap=True)
    for f in ("offsets", "status", "pos", "distance", "mask"):
        assert torch.equal(getattr(tab, f), getattr(again, f)), f
        assert torch.equal(getattr(tab, f), getattr(third, f)), f


# ---- K6 ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("S", [7, 8])
@MODES
def test_local_bfs(ts, S, multi):
    from tiler_slider_b200.bfs import LocalBfs
    walls = dict(BIG)[S]
    blocked, tiles, targets = puzzles(S, 4, walls, 6, multi, seed=S + 70 + int(multi), walk=9)
    table = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    n = table.n_envs
    wl = [[(c // S, c % S) for c in np.flatnonzero(blocked[e])] for e in range(n)]
    want = [orc.OracleState(S, wl[e], tiles[e].tolist(), targets[e].tolist(), multi).bfs(max_states=1 << 22) for e in range(n)]
    want_levels = [sum(w[1][k] for w in want if k < len(w[1])) for k in range(max(len(w[1]) for w in want))]
    res = LocalBfs(table, device_bitmap=True).solve(with_paths=True)
    assert res.fallback_puzzles == 0
    assert res.states_per_puzzle.tolist() == [w[0] for w in want]
    assert res.solve_depth_per_puzzle.tolist() == [w[2] for w in want]
    assert res.levels == want_levels
    for e in range(n):
        if want[e][2] < 0:
            assert res.solutions[e] is None
        else:
            assert len(res.solutions[e]) == want[e][2]
            assert replay_wins_at(S, wl[e], tiles[e].tolist(), targets[e].tolist(), multi, res.solutions[e])[:1] == [want[e][2]]


# ---- generation ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("S,W", [(8, 8), (7, 4)])
@MODES
def test_solvable_with_device_bitmap(ts, S, W, multi):
    with pytest.raises(ValueError, match="device_bitmap=True"):
        ts.BatchedTilerSliderEnv.solvable(8, S, 4, W, multi, min_depth=8, max_depth=12)
    env = ts.BatchedTilerSliderEnv.solvable(256, S, 4, W, multi, min_depth=8, max_depth=12, device_bitmap=True)
    depth = env.solve_depth[: env.n_envs]
    assert ((depth >= 8) & (depth <= 12)).all()
    d, _ = env.optimal_moves(device_bitmap=True)
    assert torch.equal(d, depth)
    same = ts.BatchedTilerSliderEnv.solvable(256, S, 4, W, multi, min_depth=8, max_depth=12, device_bitmap=True)
    assert torch.equal(env.blocked_cells(), same.blocked_cells())
    assert torch.equal(env.positions(), same.positions()) and torch.equal(env.target_positions(), same.target_positions())


# ---- the same answers on both paths -----------------------------------------------------------------

def forced_gmem(cls):
    """A front-end whose plan is always the gmem plan (as SmallSlab forces a slab in test_gpu_search_limits)."""
    class Forced(cls):
        def plan(self, *a):
            p = super().plan(*a)
            if p is None or p.get("gmem"):
                return p
            g = self._plan_gmem(p["f_max"])
            return g if len(a) == 1 else {**g, "smem_bytes": 4 * g["queue_smem"]}
    return Forced


@pytest.mark.parametrize("S,walls", [(7, (11, 16, 24)), (8, (26, 34, 44))])
@MODES
def test_device_and_shared_instances_agree(ts, S, walls, multi):
    from tiler_slider_b200.bfs import CudaLocalKernels, CudaOptimalMoves, CudaStateTable, LocalBfs
    blocked, tiles, targets = puzzles(S, 4, walls, 12, multi, seed=S * 3 + int(multi), walk=10)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    random_steps(env, 2, seed=S)
    assert (free_cells(env) <= F_STAR).all()
    k9, g9 = CudaOptimalMoves(env), forced_gmem(CudaOptimalMoves)(env)
    n = env.n_envs
    plans = [torch.empty((254, n), dtype=torch.uint8, device="cuda") for _ in range(2)]
    a = k9.query(None, 254, None, plans[0])
    b = g9.query(None, 254, None, plans[1])
    assert g9.plan(S * S - walls[0])["gmem"] and not k9.plan(S * S - walls[0]).get("gmem")
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(plans[0], plans[1])
    assert (a[0] >= 1).any()
    ta, tb = CudaStateTable(env).build(None), forced_gmem(CudaStateTable)(env).build(None)
    assert (ta[1] == 0).all()
    for x, y in zip(ta, tb):
        assert torch.equal(x, y)
    ra = LocalBfs(env).solve()
    kg = forced_gmem(CudaLocalKernels)(env)
    rb = LocalBfs(kernels=kg, n_puzzles=n).solve()
    assert kg.plan(0, n)["gmem"] and ra.fallback_puzzles == rb.fallback_puzzles == 0
    assert torch.equal(ra.states_per_puzzle, rb.states_per_puzzle)
    assert torch.equal(ra.solve_depth_per_puzzle, rb.solve_depth_per_puzzle) and ra.levels == rb.levels


# ---- a batch across the boundary ------------------------------------------------------------------

@MODES
def test_mixed_boundary_batch(ts, multi):
    """8x8 boards with F in {30, F*-1, F*, F*+1, F*+2}: with device_bitmap every env gets the oracle's
    answer, the envs that fit get exactly their default answers, and so does each group alone."""
    groups = [30, F_STAR - 1, F_STAR, F_STAR + 1, F_STAR + 2]
    blocked, tiles, targets = puzzles(8, 4, [64 - f for f in groups], 8, multi, seed=int(multi) + 40)
    env = ts.BatchedTilerSliderEnv.from_arrays(8, blocked, tiles, targets, multi)
    random_steps(env, 3, seed=5)
    F = free_cells(env)
    d, m = env.optimal_moves(device_bitmap=True)
    d, m = d.cpu().numpy(), m.cpu().numpy()
    for i, (st, cur) in enumerate(oracle_states(env)):
        assert (int(d[i]), int(m[i])) == oracle_answer(st, cur), (i, int(F[i]))
    d0, m0 = (x.cpu().numpy() for x in env.optimal_moves())
    fit = F <= F_STAR
    assert np.array_equal(d0[fit], d[fit]) and np.array_equal(m0[fit], m[fit])
    assert (d0[~fit] == NOT_SEARCHED).all()
    tab = env.state_table(device_bitmap=True)
    assert (tab.status == 0).all()
    for f in groups:
        ids = np.flatnonzero(F == f)
        dg, mg = env.optimal_moves(ids.tolist(), device_bitmap=True)
        assert np.array_equal(dg.cpu().numpy(), d[ids]) and np.array_equal(mg.cpu().numpy(), m[ids]), f
        tg = env.state_table(ids.tolist(), device_bitmap=True)
        rows = torch.cat([tab.pos[tab.offsets[i]:tab.offsets[i + 1]] for i in ids.tolist()])
        assert torch.equal(tg.pos, rows), f


def test_planner_on_the_device(ts):
    from tiler_slider_b200.bfs import CudaOptimalMoves, OnChipSearch
    env = ts.BatchedTilerSliderEnv.synthetic(8, 8, 4, 30, True, seed=0)
    k9 = CudaOptimalMoves(env)
    assert max(f for f in range(4, 65) if k9.plan(f) is not None) == F_STAR
    for f in range(F_STAR + 1, 65):
        p = k9._plan_gmem(f)
        assert p is not None and p["gmem"], f
        assert p["grid"] * p["bitmap_words"] * 4 <= OnChipSearch.MAX_SCRATCH_BYTES
        assert p["queue_smem"] & (p["queue_smem"] - 1) == 0 and p["grid"] >= 148
