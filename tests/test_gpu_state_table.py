"""GPU tests of the state tables (BatchedTilerSliderEnv.state_table, K10 ts_state_table): the rows
against the CPU oracle's reachable sets and K6's counts, the labels against K9 (optimal_moves on the
rows) and the oracle, Bellman consistency inside the table, the row order and determinism, items,
the result codes and the ring path."""
import functools
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.test_gpu_optimal import oracle_answer, random_steps

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def walls_for(S, T):
    """Walls that keep every state space on chip (F!/(F-T)! bits in one CTA)."""
    return {3: 1, 4: 3, 5: 5, 6: 8, 7: 14, 8: 34 if T == 4 else 24}[S]


CASES = [(S, T, multi) for S in range(3, 9) for T in range(1, 5) for multi in (True, False)]


def item_of_rows(table):
    """Item index of every row (int64, device)."""
    n = table.status.numel()
    return torch.repeat_interleave(torch.arange(n, device="cuda"), table.offsets.diff())


def oracle_keys(env, rows):
    """Table rows (uint8 [m, pos_bytes]) -> oracle keys (byte i = cell r*S + c of tile i)."""
    S, T, ps = env.size, env.n_tiles, env.pos_stride
    b = rows[:, :T].cpu().numpy().astype(np.uint64)
    cells = b // ps * S + b % ps
    return (cells << (np.arange(T, dtype=np.uint64) * np.uint64(8))).sum(1).astype(np.uint64) if T else np.zeros(len(b), np.uint64)


def host_index(env, env_of_row, rows):
    """Restatement of the kernels' perfect hash (state_index in ts_bfs_local.cuh): digit i = rank of
    tile i's cell among the free cells not taken by tiles 0 .. i-1, radix F - i, tile 0 least
    significant."""
    S, T, ps = env.size, env.n_tiles, env.pos_stride
    free = ~env.blocked_cells().cpu().numpy().astype(bool)[env_of_row]           # [m, S*S]
    F = free.sum(1).astype(np.int64)
    b = rows[:, :T].cpu().numpy().astype(np.int64)
    cell = b // ps * S + b % ps
    rank = np.cumsum(free, 1) - 1
    r = np.take_along_axis(rank, cell, 1)                                           # [m, T]
    idx = np.zeros(len(b), np.int64)
    for i in range(T - 1, -1, -1):
        d = r[:, i] - (r[:, :i] < r[:, i:i + 1]).sum(1)
        idx = idx * (F - i) + d
    return idx


@functools.lru_cache(maxsize=None)
def case(S, T, multi):
    """Solvable puzzles and uniform draws (mostly unsolvable with several tiles), stepped a few
    random steps: the roots are their current positions."""
    W = walls_for(S, T)
    import tiler_slider_b200 as ts
    envs = []
    for k, env in enumerate((ts.BatchedTilerSliderEnv.solvable(24, S, T, W, multi, min_depth=1, max_depth=20, seed=S * 10 + T),
                             ts.BatchedTilerSliderEnv.synthetic(24, S, T, W, multi, seed=S * 10 + T))):
        random_steps(env, 2 + k, seed=S + T)
        envs.append((env, env.state_table()))
    return envs


def labels_by_k9(env, table):
    ids = item_of_rows(table).to(torch.int32)
    return env.optimal_moves(ids, pos=table.pos.contiguous())


@pytest.mark.parametrize("S,T,multi", CASES)
def test_reachable_set_matches_the_oracle(ts, S, T, multi):
    for env, tab in case(S, T, multi):
        assert (tab.status == 0).all()
        blocked = env.blocked_cells().cpu().numpy()
        targets = env.target_positions().cpu().numpy()
        cur = env.positions().cpu().numpy()
        off = tab.offsets.cpu().numpy()
        for i in range(0, env.n_envs, 3):
            b = [divmod(int(c), S) for c in np.flatnonzero(blocked[i])]
            tg = targets[i].tolist() if targets.ndim == 3 else [divmod(int(c), S) for c in np.flatnonzero(targets[i])]
            keys = orc.OracleState(S, b, cur[i].tolist(), tg, multi).bfs(max_states=1 << 22)[3]
            got = oracle_keys(env, tab.pos[off[i]:off[i + 1]])
            assert np.array_equal(np.sort(got), np.sort(keys)), i


@pytest.mark.parametrize("S,T,multi", CASES)
def test_labels_equal_optimal_moves(ts, S, T, multi):
    """Every row's distance and mask equal K9's answer for that row, bit for bit; a sample also
    equals the oracle's."""
    for env, tab in case(S, T, multi):
        d, m = labels_by_k9(env, tab)
        assert not (d == -2).any() and not (d == -3).any()
        assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
        rows = tab.pos.cpu().numpy()
        items = item_of_rows(tab).cpu().numpy()
        blocked = env.blocked_cells().cpu().numpy()
        targets = env.target_positions().cpu().numpy()
        rng = np.random.default_rng(S * 8 + T)
        for r in rng.choice(len(rows), size=min(12, len(rows)), replace=False):
            i = int(items[r])
            b = [divmod(int(c), S) for c in np.flatnonzero(blocked[i])]
            tg = targets[i].tolist() if targets.ndim == 3 else [divmod(int(c), S) for c in np.flatnonzero(targets[i])]
            cur = [divmod(int(p), env.pos_stride) for p in rows[r, :T]]
            st = orc.OracleState(S, b, cur, tg, multi)
            assert (int(tab.distance[r]), int(tab.mask[r])) == oracle_answer(st, cur), (r, cur)


@pytest.mark.parametrize("S,T,multi", CASES)
def test_bellman_inside_the_table(ts, S, T, multi):
    """distance >= 2: bit a of the mask iff successor a (canonical in set mode) differs from the row
    and is a row of the same item with distance - 1; distance 1: the mask is expand()'s won bits."""
    for env, tab in case(S, T, multi):
        ids = item_of_rows(tab)
        succ, _, won = env.expand(ids.to(torch.int32), tab.pos.contiguous())
        if not multi:
            succ = succ.sort(-1).values if T == env.pos_bytes else torch.cat(
                [succ[..., :T].sort(-1).values, succ[..., T:]], -1)
        d = tab.distance.cpu().numpy()
        rows_key = ids.cpu().numpy().astype(np.int64) << 32 | oracle_keys(env, tab.pos).astype(np.int64)
        order = np.argsort(rows_key)
        sk = rows_key[order]
        m = tab.mask.cpu().numpy()
        one = d == 1
        assert np.array_equal(m[one], won.cpu().numpy()[one])
        for a in range(4):
            key = ids.cpu().numpy().astype(np.int64) << 32 | oracle_keys(env, succ[:, a]).astype(np.int64)
            at = np.searchsorted(sk, key).clip(0, len(sk) - 1)
            assert (sk[at] == key).all()                       # every successor is a row of its item
            d_succ = d[order[at]]
            differs = key != rows_key
            want = differs & (d_succ == d - 1) & (d >= 2)
            got = ((m >> a) & 1).astype(bool) & (d >= 2)
            assert np.array_equal(got, want), a


@pytest.mark.parametrize("S,T,multi", CASES[::5])
def test_rows_ascending_and_deterministic(ts, S, T, multi):
    for env, tab in case(S, T, multi):
        items = item_of_rows(tab).cpu().numpy()
        idx = host_index(env, items, tab.pos)
        same = items[1:] == items[:-1]
        assert (idx[1:][same] > idx[:-1][same]).all()
        again = env.state_table()
        for f in ("offsets", "status", "pos", "distance", "mask"):
            assert torch.equal(getattr(tab, f), getattr(again, f)), f


def test_counts_match_local_bfs(ts):
    """Fresh batches (roots = initial positions): the rows per item are K6's states per puzzle."""
    from tiler_slider_b200.bfs import LocalBfs
    for multi in (True, False):
        env = ts.BatchedTilerSliderEnv.solvable(4096, 6, 4, 8, multi, min_depth=8, max_depth=12, seed=3)
        tab = env.state_table()
        assert (tab.status == 0).all() and tab.pos.shape == (int(tab.offsets[-1]), env.pos_bytes)
        assert torch.equal(tab.offsets.diff(), LocalBfs(env).solve().states_per_puzzle)


def test_real_levels(ts):
    """The reference's real levels (tests/golden/levels_400.txt) by shape: the oracle's reachable
    set and K9's labels."""
    groups = {}
    for p in ts.load_puzzle_file(os.path.join(ROOT, "tests", "golden", "levels_400.txt")):
        groups.setdefault((p.size, len(p.initial_locations), p.multiple_colors), []).append(p)
    checked = 0
    for (S, T, multi), ps in groups.items():
        if S > 8 or not 1 <= T <= 4:
            continue
        env = ts.BatchedTilerSliderEnv.from_puzzles(ps)
        tab = env.state_table()
        assert (tab.status == 0).all()
        d, m = labels_by_k9(env, tab)
        assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
        off = tab.offsets.cpu().numpy()
        for i, p in enumerate(ps):
            keys = orc.OracleState(S, p.blocked_locations, p.initial_locations, p.target_locations, multi).bfs(max_states=1 << 22)[3]
            assert np.array_equal(np.sort(oracle_keys(env, tab.pos[off[i]:off[i + 1]])), np.sort(keys)), i
        checked += env.n_envs
    assert checked >= 256


def test_items(ts):
    """Shuffled and repeated ids with different roots, the default (current positions after random
    steps) and a sub-batch: each item's rows and labels are those of the same states in the
    batch's own table (labels belong to states, not roots)."""
    env = ts.BatchedTilerSliderEnv.solvable(512, 6, 4, 8, True, min_depth=2, max_depth=14, seed=17)
    random_steps(env, 3, seed=5)
    full = env.state_table()
    full_items = item_of_rows(full)
    full_key = full_items.cpu().numpy().astype(np.int64) << 32 | oracle_keys(env, full.pos).astype(np.int64)
    # sub-batch: a slice of the full table
    ids = torch.arange(100, 300, dtype=torch.int32, device="cuda")
    sub = env.state_table(ids)
    lo, hi = int(full.offsets[100]), int(full.offsets[300])
    assert torch.equal(sub.offsets, full.offsets[100:301] - lo)
    for f in ("pos", "distance", "mask"):
        assert torch.equal(getattr(sub, f), getattr(full, f)[lo:hi]), f
    # shuffled, repeated ids; roots drawn among each env's own reachable states
    g = torch.Generator(device="cpu").manual_seed(2)
    ids = torch.randint(0, 512, (300,), generator=g).to(torch.int32)
    ids[150:] = ids[:150]
    off = full.offsets.cpu()
    pick = off[ids.long()] + (torch.rand(300, generator=g) * off.diff()[ids.long()]).long()
    pos = full.pos[pick.cuda()].contiguous()
    tab = env.state_table(ids.tolist(), pos)
    assert (tab.status == 0).all()
    items = item_of_rows(tab).cpu().numpy()
    key = ids.numpy().astype(np.int64)[items] << 32 | oracle_keys(env, tab.pos).astype(np.int64)
    order = np.argsort(full_key)
    at = order[np.searchsorted(full_key[order], key)]
    assert np.array_equal(full_key[at], key)
    assert np.array_equal(tab.distance.cpu().numpy(), full.distance.cpu().numpy()[at])
    assert np.array_equal(tab.mask.cpu().numpy(), full.mask.cpu().numpy()[at])
    # a root reachable from the env's root owns a subset: at most as many rows; its own row is present
    assert (tab.offsets.diff().cpu() <= off.diff()[ids.long()]).all()
    with pytest.raises(IndexError):
        env.state_table([0, 512])


@pytest.mark.parametrize("S,T,multi", [(6, 4, True), (6, 4, False), (8, 3, True), (3, 2, False)])
def test_bad_roots(ts, S, T, multi):
    """A tile on a wall, two tiles on one cell, a byte of 255, a cell off the board and the zero rows
    playout(record=True) writes past an item's end: -4 and no rows; the items around them keep
    their tables."""
    env = ts.BatchedTilerSliderEnv.solvable(64, S, T, walls_for(S, T), multi, min_depth=1, max_depth=12, seed=S + T)
    ps = env.pos_stride
    blocked = env.blocked_cells().cpu().numpy()
    good = env.pos.clone()
    _, _, _, _, traj = env.playout(n_steps=40, seed=1, record=True)
    rows, kinds = [], []
    for i in range(env.n_envs):
        w = np.flatnonzero(blocked[i])
        p = good[i].clone()
        kind = i % 6
        if kind == 1:
            p[T - 1] = int(w[0] // S * ps + w[0] % S)
        elif kind == 2:
            p[T - 1] = p[0]
        elif kind == 3:
            p[0] = 255
        elif kind == 4:
            p[0] = (S - 1) * ps + S if i % 2 else S * ps
        elif kind == 5:
            p = traj[-1, i].clone() * 0                 # a zero row of a finished playout
        rows.append(p)
        kinds.append(kind)
    pos = torch.stack(rows).contiguous()
    kinds = torch.tensor(kinds, device="cuda")
    ids = torch.arange(env.n_envs, dtype=torch.int32, device="cuda")
    tab = env.state_table(ids, pos)
    d_k9, _ = env.optimal_moves(ids, pos=pos)
    bad = d_k9 == -4
    assert bad[(kinds >= 1) & (kinds <= 4)].all() and bad[kinds == 5].all()
    assert torch.equal(tab.status, torch.where(bad, -4, 0).to(torch.int32))
    assert (tab.offsets.diff()[bad] == 0).all()
    keep = (~bad).nonzero().flatten().to(torch.int32)
    ref = env.state_table(keep, pos[keep.long()].contiguous())
    for f in ("pos", "distance", "mask"):
        assert torch.equal(getattr(tab, f), getattr(ref, f)), f


def test_too_large_and_mixed_state_spaces(ts):
    """8x8, 4 tiles: boards with no walls do not fit one CTA (-3, no rows); boards with many walls in
    the same batch get the tables they get on their own."""
    S, T, N = 8, 4, 128
    rng = np.random.default_rng(4)
    blocked = np.zeros((N, S * S), np.uint8)
    tiles = np.zeros((N, T, 2), np.uint8)
    targets = np.zeros((N, T, 2), np.uint8)
    for i in range(N):
        W = 0 if i % 4 == 0 else 34
        perm = rng.permutation(S * S)
        blocked[i, perm[:W]] = 1
        tiles[i] = np.stack([perm[W:W + T] // S, perm[W:W + T] % S], -1)
        targets[i] = np.stack([perm[W + T:W + 2 * T] // S, perm[W + T:W + 2 * T] % S], -1)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, True)
    tab = env.state_table()
    big = torch.arange(N, device="cuda") % 4 == 0
    assert (tab.status[big] == -3).all() and (tab.status[~big] == 0).all()
    assert (tab.offsets.diff()[big] == 0).all()
    small = (~big).nonzero().flatten().to(torch.int32)
    alone = env.state_table(small)
    for f in ("pos", "distance", "mask"):
        assert torch.equal(getattr(tab, f), getattr(alone, f)), f
    wide = ts.BatchedTilerSliderEnv.synthetic(64, 8, 4, 0, True, seed=1)
    t2 = wide.state_table()
    assert (t2.status == -3).all() and int(t2.offsets[-1]) == 0 and t2.pos.shape == (0, 4)


def test_unsolvable_and_never_win(ts):
    """Uniform coloured draws (mostly unsolvable) take the shortcut: all -1 for items whose root has
    no win; a never_win batch (one target fewer than tiles) has the rows of the same puzzles with
    every target, all -1 and mask 0."""
    syn = ts.BatchedTilerSliderEnv.synthetic(2048, 6, 4, 8, True, seed=5)
    tab = syn.state_table()
    d_root, _ = syn.optimal_moves()
    items = item_of_rows(tab)
    dead = d_root[items] == -1
    assert (d_root == -1).sum() > 1000
    assert (tab.distance[dead] == -1).all() and (tab.mask[dead] == 0).all()
    d, m = labels_by_k9(syn, tab)
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)
    blocked = syn.blocked_cells().cpu().numpy()[:256]
    tiles = syn.positions().cpu().numpy()[:256]
    targets = syn.target_positions().cpu().numpy()[:256]
    full = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, targets, True)
    nw = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, targets[:, :3], True)
    assert nw.never_win
    a, b = full.state_table(), nw.state_table()
    assert torch.equal(a.offsets, b.offsets) and torch.equal(a.pos, b.pos)
    assert (b.distance == -1).all() and (b.mask == 0).all() and (b.status == 0).all()


def test_root_on_the_goal(ts):
    """Roots already on the goal (ordered: tile i on target i): their row has distance 1 and K9's
    mask, moves that change nothing included."""
    env = ts.BatchedTilerSliderEnv.solvable(256, 5, 2, 4, True, min_depth=1, max_depth=8, seed=3)
    tg = env.target_positions().to(torch.int32)
    goal = torch.zeros(256, env.pos_bytes, dtype=torch.uint8, device="cuda")
    goal[:, :2] = (tg[..., 0] * env.pos_stride + tg[..., 1]).to(torch.uint8)
    ids = torch.arange(256, dtype=torch.int32, device="cuda")
    tab = env.state_table(ids, goal)
    d_k9, m_k9 = env.optimal_moves(ids, pos=goal)
    assert (d_k9 == 1).all()
    items = item_of_rows(tab)
    on_goal = (tab.pos == goal[items]).all(1)
    assert int(on_goal.sum()) == 256
    assert (tab.distance[on_goal] == 1).all() and torch.equal(tab.mask[on_goal], m_k9)
    d, m = labels_by_k9(env, tab)
    assert torch.equal(tab.distance, d) and torch.equal(tab.mask, m)


def test_empty_queries(ts):
    env = ts.BatchedTilerSliderEnv.solvable(64, 6, 3, 8, False, min_depth=1, max_depth=10, seed=1)
    for tab in (env.state_table([]), env.state_table(torch.empty(0, dtype=torch.int32, device="cuda"),
                                                     torch.empty(0, env.pos_bytes, dtype=torch.uint8, device="cuda"))):
        assert tab.offsets.tolist() == [0] and tab.status.numel() == 0
        assert tab.pos.shape == (0, env.pos_bytes) and tab.distance.numel() == 0 and tab.mask.numel() == 0


def test_forced_small_ring(ts):
    """A ring of 32 entries (levels read back from the slab, then from the rows) gives the same
    tables."""
    from tiler_slider_b200.bfs import CudaStateTable
    env = ts.BatchedTilerSliderEnv.solvable(2048, 6, 4, 8, False, min_depth=4, max_depth=16, seed=9)
    random_steps(env, 2, seed=1)
    want = env.state_table()
    small = CudaStateTable(env, queue_smem=32)
    got = small.build(None)
    assert small.plan(28)["queue_smem"] == 32
    for w, g in zip((want.offsets, want.status, want.pos, want.distance, want.mask), got):
        assert torch.equal(w, g)
