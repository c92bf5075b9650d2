"""GPU tests of the hash-table state tables for 5 to 8 tiles (K12 ts_state_table_*_table, reached
through state_table(hash_table=True)): the rows against the CPU oracle's reachable sets, the labels
against K11 (optimal_moves(hash_table=True) on the rows) and the oracle, Bellman consistency inside
the table, the row order and its independence of the plan, the max_states bound, table epochs
across many items per CTA, items and result codes, and the README's five-tile reverse curriculum."""
import functools

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.test_gpu_optimal import oracle_answer, oracle_states, random_steps
from tests.test_gpu_state_table import item_of_rows, oracle_keys
from tests.test_gpu_table_search import ORACLE_CASES, mixed_batch

pytestmark = pytest.mark.gpu

NOT_SEARCHED, BAD_STATE = -3, -4
FIELDS = ("offsets", "status", "pos", "distance", "mask")


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def oracle_counts(env):
    """(states reachable from each env's current positions, their sorted oracle keys) by the oracle."""
    out = [st.bfs(max_states=1 << 22) for st, _ in oracle_states(env)]
    return np.array([r[0] for r in out]), [r[3] for r in out]


def default_bound(env):
    from tiler_slider_b200.bfs import CudaStateTable
    return CudaStateTable(env)._plan_table()["spill_per_cta"]


@functools.lru_cache(maxsize=None)
def case(S, T, W, multi):
    """K11's oracle batch of the shape, the oracle's counts and keys, the bound the table needs (None:
    the default one holds every item) and the table."""
    import tiler_slider_b200 as ts
    env = mixed_batch(ts, S, T, W, multi, 12, seed=10 * S + T)
    n, keys = oracle_counts(env)
    ms = None if n.max() <= default_bound(env) else int(n.max())
    return env, n, keys, ms, env.state_table(hash_table=True, max_states=ms)


def k11_labels(env, tab, ms=None):
    """optimal_moves(hash_table=True) of every row (with a bound of ms states when the default one
    is too small for the item's states)."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    ids = item_of_rows(tab).to(torch.int32)
    if ms is None:
        return env.optimal_moves(ids, pos=tab.pos.contiguous(), hash_table=True)
    q = CudaOptimalMoves(env, table_slots=1 << (2 * ms - 1).bit_length())
    plan = q._plan_table()                       # as many CTAs as the tables and slabs fit in 4 GiB
    plan["grid"] = max(1, min(plan["grid"], q.MAX_SCRATCH_BYTES // (12 * plan["table_slots"])))
    return q.query(ids, 254, tab.pos.contiguous(), hash_table=True)


def words(tab):
    return tab.pos.contiguous().view(torch.int64).flatten()


def per_item(tab, i):
    lo, hi = int(tab.offsets[i]), int(tab.offsets[i + 1])
    return tuple(getattr(tab, f)[lo:hi] for f in ("pos", "distance", "mask"))


def assert_same(a, b):
    for f in FIELDS:
        assert torch.equal(getattr(a, f), getattr(b, f)), f


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_reachable_set_matches_the_oracle(ts, S, T, W, multi):
    env, n, keys, ms, tab = case(S, T, W, multi)
    assert (tab.status == 0).all()
    assert tab.pos.shape == (int(tab.offsets[-1]), 8) and tab.pos.dtype == torch.uint8
    assert np.array_equal(tab.offsets.diff().cpu().numpy(), n)
    assert (tab.pos[:, T:] == 0).all()
    off = tab.offsets.cpu().numpy()
    for i in range(env.n_envs):
        got = oracle_keys(env, tab.pos[off[i]:off[i + 1]])
        assert np.array_equal(np.sort(got), np.sort(keys[i])), i


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_labels_equal_optimal_moves(ts, S, T, W, multi):
    """Every row's distance and mask equal K11's answer for that row, bit for bit; a sample also
    equals the oracle's."""
    env, _, _, ms, tab = case(S, T, W, multi)
    d, m = k11_labels(env, tab, ms)
    assert not ((d == -2) | (d == NOT_SEARCHED)).any()
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
    assert (d >= 1).any()
    rows = tab.pos.cpu().numpy()
    items = item_of_rows(tab).cpu().numpy()
    blocked = env.blocked_cells().cpu().numpy()
    targets = env.target_positions().cpu().numpy()
    rng = np.random.default_rng(S * 8 + T)
    for r in rng.choice(len(rows), size=min(8, len(rows)), replace=False):
        i = int(items[r])
        b = [divmod(int(c), S) for c in np.flatnonzero(blocked[i])]
        tg = targets[i].tolist() if targets.ndim == 3 else [divmod(int(c), S) for c in np.flatnonzero(targets[i])]
        cur = [divmod(int(p), env.pos_stride) for p in rows[r, :T]]
        st = orc.OracleState(S, b, cur, tg, multi)
        assert (int(tab.distance[r]), int(tab.mask[r])) == oracle_answer(st, cur), (r, cur)


def canonical_successors(env, tab):
    """expand() of every row (canonical in set mode) as int64 words [M, 4]."""
    T = env.n_tiles
    succ, _, won = env.expand(item_of_rows(tab).to(torch.int32), tab.pos.contiguous())
    if not env.multi_color:
        succ = torch.cat([succ[..., :T].sort(-1).values, succ[..., T:]], -1)
    return succ.contiguous().view(torch.int64)[..., 0], won


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_bellman_inside_the_table(ts, S, T, W, multi):
    """Every successor is a row of its item; distance >= 2: bit a of the mask iff successor a differs
    from the row and has distance - 1; distance 1: the mask is expand()'s won bits."""
    env, _, _, _, tab = case(S, T, W, multi)
    succ, won = canonical_successors(env, tab)
    w, succ = words(tab).cpu().numpy(), succ.cpu().numpy()
    d, m = tab.distance.cpu().numpy(), tab.mask.cpu().numpy()
    one = d == 1
    assert np.array_equal(m[one], won.cpu().numpy()[one])
    off = tab.offsets.cpu().numpy()
    for i in range(env.n_envs):
        lo, hi = off[i], off[i + 1]
        at = lo + np.searchsorted(w[lo:hi], succ[lo:hi]).clip(0, hi - lo - 1)
        assert (w[at] == succ[lo:hi]).all(), i                    # every successor is a row of the item
        for a in range(4):
            want = (succ[lo:hi, a] != w[lo:hi]) & (d[at[:, a]] == d[lo:hi] - 1) & (d[lo:hi] >= 2)
            got = ((m[lo:hi] >> a) & 1).astype(bool) & (d[lo:hi] >= 2)
            assert np.array_equal(got, want), (i, a)


@pytest.mark.parametrize("S,T,W,multi", ORACLE_CASES)
def test_rows_ascending_and_independent_of_the_plan(ts, S, T, W, multi):
    """Per item the rows ascend as little-endian 64-bit words; a second call, a plan of one CTA per
    SM and a ring of 32 entries (levels read back from the slab and the rows) give the same table."""
    from tiler_slider_b200.bfs import CudaStateTable
    from tiler_slider_b200.batch_env import StateTable
    env, _, _, ms, tab = case(S, T, W, multi)
    w = words(tab)
    same = item_of_rows(tab).diff() == 0
    assert (w.diff()[same] > 0).all()
    assert_same(tab, env.state_table(hash_table=True, max_states=ms))
    for kw in (dict(ctas_per_sm=1), dict(queue_smem=32)):
        front = CudaStateTable(env, **kw)
        assert_same(tab, StateTable(*front.build(None, None, False, True, ms)))
        assert front._plan_table(ms)["queue_smem"] == kw.get("queue_smem", front._plan_table(ms)["queue_smem"])


@pytest.mark.parametrize("multi", [True, False])
def test_the_bound_is_predicted_exactly(ts, multi):
    """An item gets -3 and no rows exactly when it reaches more than max_states states, the root
    included; every other item has the rows and labels of the default table."""
    env = mixed_batch(ts, 6, 5, 8, multi, 24, seed=40 + int(multi))
    n, _ = oracle_counts(env)
    full = env.state_table(hash_table=True)
    assert (full.status == 0).all()
    seen = set()
    for q in (32, 512, 4096):
        tab = env.state_table(hash_table=True, max_states=q)
        big = n > q
        assert np.array_equal(tab.status.cpu().numpy(), np.where(big, NOT_SEARCHED, 0)), q
        assert np.array_equal(tab.offsets.diff().cpu().numpy(), np.where(big, 0, n)), q
        for i in np.flatnonzero(~big):
            for g, f in zip(per_item(tab, i), per_item(full, i)):
                assert torch.equal(g, f), (q, i)
        seen.update(big.tolist())
    assert seen == {True, False}
    exact = env.state_table(hash_table=True, max_states=int(n.max()))      # the largest item on the bound
    assert_same(exact, full)
    assert (env.state_table(hash_table=True, max_states=int(n.max()) - 1).status == NOT_SEARCHED).any()


def test_epochs_wrap_in_both_passes(ts):
    """One CTA per SM's plan and 32 small set-goal puzzles repeated 1,500 times: every CTA serves
    well over the 31 epochs of its table in each pass, and every copy's rows are its puzzle's."""
    from tiler_slider_b200.bfs import CudaStateTable
    from tiler_slider_b200.batch_env import StateTable
    rng = np.random.default_rng(8)
    N, S, T = 32, 3, 5
    blocked, tiles, targets = np.zeros((N, S * S), np.uint8), np.zeros((N, T, 2), np.uint8), np.zeros((N, T, 2), np.uint8)
    for i in range(N):
        perm = rng.permutation(S * S)
        blocked[i, perm[0]] = 1
        tg = rng.permutation(perm[1:])[:T]
        tiles[i] = np.stack([perm[1:T + 1] // S, perm[1:T + 1] % S], -1)
        targets[i] = np.stack([tg // S, tg % S], -1)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, False)
    one = env.state_table(hash_table=True)
    reps = 1500
    ids = torch.arange(N, dtype=torch.int32, device="cuda").repeat(reps)
    front = CudaStateTable(env, ctas_per_sm=1)
    tab = StateTable(*front.build(ids, None, False, True))
    assert front._plan_table()["grid"] * 40 < ids.numel()
    assert (tab.status == 0).all()
    assert torch.equal(tab.offsets.diff(), one.offsets.diff().repeat(reps))
    for f in ("pos", "distance", "mask"):
        got = getattr(tab, f).view(reps, -1, *getattr(one, f).shape[1:])
        assert (got == getattr(one, f)[None]).all(), f
    assert (one.distance >= 1).any()


def test_items(ts):
    """Shuffled and repeated ids with roots among the env's own states, and expand() successors as
    roots: each item's rows and labels are those of the same states in the batch's own table."""
    env = ts.BatchedTilerSliderEnv.solvable(256, 6, 5, 8, True, min_depth=2, max_depth=12, seed=17, hash_table=True)
    random_steps(env, 3, seed=5)
    full = env.state_table(hash_table=True)
    assert (full.status == 0).all()
    fw = words(full).cpu().numpy()
    off = full.offsets.cpu()

    fd, fm = full.distance.cpu().numpy(), full.mask.cpu().numpy()

    def check(ids, tab):
        assert (tab.status == 0).all()
        toff, w = tab.offsets.cpu().numpy(), words(tab).cpu().numpy()
        d, m = tab.distance.cpu().numpy(), tab.mask.cpu().numpy()
        for j, e in enumerate(ids.tolist()):
            lo, hi, a, b = int(off[e]), int(off[e + 1]), toff[j], toff[j + 1]
            assert b - a <= hi - lo
            at = lo + np.searchsorted(fw[lo:hi], w[a:b])
            assert (at < hi).all() and (fw[at] == w[a:b]).all(), j     # the states of the env's own table
            assert np.array_equal(d[a:b], fd[at]) and np.array_equal(m[a:b], fm[at]), j

    g = torch.Generator(device="cpu").manual_seed(2)
    ids = torch.randint(0, 256, (200,), generator=g).to(torch.int32)
    ids[100:] = ids[:100]
    pick = off[ids.long()] + (torch.rand(200, generator=g) * off.diff()[ids.long()]).long()
    pos = full.pos[pick.cuda()].contiguous()
    tab = env.state_table(ids.tolist(), pos, hash_table=True)
    check(ids, tab)
    assert_same(tab, env.state_table(ids.tolist(), pos, hash_table=True))
    # expand() successors as roots
    ids = torch.arange(256, dtype=torch.int32, device="cuda")
    succ, _, _ = env.expand(ids, env.pos[:256].contiguous())
    for a in (0, 3):
        check(ids, env.state_table(ids, succ[:, a].contiguous(), hash_table=True))
    # a sub-batch is a slice of the full table
    sub = env.state_table(torch.arange(100, 200, dtype=torch.int32, device="cuda"), hash_table=True)
    lo, hi = int(full.offsets[100]), int(full.offsets[200])
    assert torch.equal(sub.offsets, full.offsets[100:201] - lo)
    for f in ("pos", "distance", "mask"):
        assert torch.equal(getattr(sub, f), getattr(full, f)[lo:hi]), f


@pytest.mark.parametrize("multi", [True, False])
def test_bad_roots(ts, multi):
    """A tile on a wall, two tiles on one cell, a byte of 255 and a zero row: -4 and no rows; the
    items around them keep their tables."""
    env = ts.BatchedTilerSliderEnv.solvable(64, 6, 5, 8, multi, min_depth=1, max_depth=10, seed=3, hash_table=True)
    blocked = env.blocked_cells().cpu().numpy()
    pos = env.pos[:64].clone()
    kinds = torch.arange(64) % 5
    for i in range(64):
        w = int(np.flatnonzero(blocked[i])[0])
        if kinds[i] == 1:
            pos[i, 4] = w // 6 * env.pos_stride + w % 6
        elif kinds[i] == 2:
            pos[i, 4] = pos[i, 0]
        elif kinds[i] == 3:
            pos[i, 0] = 255
        elif kinds[i] == 4:
            pos[i] = 0
    ids = torch.arange(64, dtype=torch.int32, device="cuda")
    tab = env.state_table(ids, pos.contiguous(), hash_table=True)
    d, _ = env.optimal_moves(ids, pos=pos.contiguous(), hash_table=True)
    bad = (kinds != 0).cuda()
    assert (d[bad] == BAD_STATE).all()
    assert torch.equal(tab.status, torch.where(bad, BAD_STATE, 0).to(torch.int32))
    assert (tab.offsets.diff()[bad] == 0).all()
    keep = (~bad).nonzero().flatten().to(torch.int32)
    ref = env.state_table(keep, pos[keep.long()].contiguous(), hash_table=True)
    for f in ("pos", "distance", "mask"):
        assert torch.equal(getattr(tab, f), getattr(ref, f)), f


def test_unsolvable_and_never_win(ts):
    """Uniform coloured draws (mostly unsolvable): rows of an item whose root has no win are all -1,
    and every label is K11's; a never_win batch (a target fewer than tiles) lists the rows of the
    same puzzles with every target, all -1 and mask 0."""
    syn = ts.BatchedTilerSliderEnv.synthetic(48, 6, 5, 8, True, seed=5)
    tab = syn.state_table(hash_table=True)
    d_root, _ = syn.optimal_moves(hash_table=True)
    ok = tab.status == 0
    assert ok.sum() >= 40 and (tab.status[~ok] == NOT_SEARCHED).all()
    assert (d_root[ok] == -1).sum() >= 32
    dead = d_root[item_of_rows(tab)] == -1
    assert (tab.distance[dead] == -1).all() and (tab.mask[dead] == 0).all()
    d, m = k11_labels(syn, tab)
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
    blocked = syn.blocked_cells().cpu().numpy()
    tiles = syn.positions().cpu().numpy()
    targets = syn.target_positions().cpu().numpy()
    full = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, targets, True)
    nw = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, targets[:, :4], True)
    assert nw.never_win
    a, b = full.state_table(hash_table=True), nw.state_table(hash_table=True)
    for f in ("offsets", "status", "pos"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert (b.distance == -1).all() and (b.mask == 0).all()
    assert int(b.offsets[-1]) > 0


def test_root_on_the_goal(ts):
    """Roots already on the goal (tile i on target i): their row has distance 1 and K11's mask."""
    env = ts.BatchedTilerSliderEnv.solvable(128, 5, 5, 5, True, min_depth=1, max_depth=8, seed=3, hash_table=True)
    tg = env.target_positions().to(torch.int32)
    goal = torch.zeros(128, 8, dtype=torch.uint8, device="cuda")
    goal[:, :5] = (tg[..., 0] * env.pos_stride + tg[..., 1]).to(torch.uint8)
    ids = torch.arange(128, dtype=torch.int32, device="cuda")
    tab = env.state_table(ids, goal, hash_table=True)
    d_k11, m_k11 = env.optimal_moves(ids, pos=goal, hash_table=True)
    assert (d_k11 == 1).all()
    on_goal = (tab.pos == goal[item_of_rows(tab)]).all(1)
    assert int(on_goal.sum()) == 128
    assert (tab.distance[on_goal] == 1).all() and torch.equal(tab.mask[on_goal], m_k11)
    d, m = k11_labels(env, tab)
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)


def test_empty_queries(ts):
    env = ts.BatchedTilerSliderEnv.solvable(64, 6, 5, 8, False, min_depth=1, max_depth=10, seed=1, hash_table=True)
    for tab in (env.state_table([], hash_table=True),
                env.state_table(torch.empty(0, dtype=torch.int32, device="cuda"),
                                torch.empty(0, 8, dtype=torch.uint8, device="cuda"), hash_table=True, max_states=64)):
        assert tab.offsets.tolist() == [0] and tab.status.numel() == 0
        assert tab.pos.shape == (0, 8) and tab.distance.numel() == 0 and tab.mask.numel() == 0


@pytest.mark.parametrize("multi", [True, False])
def test_four_tiles_ignore_hash_table(ts, multi):
    env = ts.BatchedTilerSliderEnv.solvable(512, 6, 4, 8, multi, min_depth=2, max_depth=12, seed=11)
    random_steps(env, 2, seed=1)
    assert_same(env.state_table(hash_table=True), env.state_table())


def test_readme_five_tile_reverse_curriculum(ts):
    """The README's example, as written there."""
    import tiler_slider_b200 as ts
    pool5 = ts.BatchedTilerSliderEnv.solvable(1024, 6, 5, 8, True, min_depth=8, max_depth=12, hash_table=True)
    table5 = pool5.state_table(hash_table=True)     # rows ascend per item as int64 words; status -3: more states
                                                    # than max_states (default: the bound of the hash-table plan)
    k = 4
    item = torch.repeat_interleave(torch.arange(pool5.n_envs, device="cuda"), table5.offsets.diff())
    at_k = torch.nonzero(table5.distance == k).flatten()
    row = torch.full((pool5.n_envs,), -1, dtype=torch.int64, device="cuda").scatter_reduce(0, item[at_k], at_k, "amax")
    ids5 = torch.nonzero(row >= 0).flatten().to(torch.int32)       # every enumerated env has such rows: depth >= 8
    d5, _ = pool5.optimal_moves(ids5, pos=table5.pos[row[ids5.long()]], hash_table=True)
    assert (d5 == k).all()
    # beyond the README: every enumerated env got its row
    assert ids5.numel() == int((table5.status == 0).sum()) > 1000
