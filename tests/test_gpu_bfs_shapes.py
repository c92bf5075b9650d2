"""The hash-partitioned BFS (BfsSolver: bfs_seed, K4 bfs_expand, K5 bfs_hash_insert, bfs_traceback,
ts_bfs_levels) state by state, on every board size 1-8 and every tile count it is compiled for.

Every expectation comes from the CPU oracle (oracle/ts_oracle.c), which shares no code with the
kernels.  The level-by-level tests decode every key the GPU inserted and compare the visited set of
each depth with the oracle's, so a key-packing or canonicalisation bug that merges some states and
splits others fails even where the counts happen to agree.  5 to 8 tiles (no puzzle id in the key,
one puzzle per table) also go through the product paths: paths, depth limits, solve_batch, main.py.
"""
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.helpers import random_puzzles, reachable_targets

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = range(1, 9)
PAIRS = [(S, T) for S in SIZES for T in range(1, min(8, S * S) + 1)]
assert len(PAIRS) == 53                   # every (size, tiles) pair the BFS kernels are compiled for that holds a puzzle
MANY_TILES_SIZES = range(3, 9)            # the board classes 5 to 8 tiles fit: padded 3..6, compact 7 and 8
STATE_CAP = 150_000                       # per puzzle: redraw anything larger (ordered spaces with 5+ tiles grow fast)
WON = np.uint64(1 << 63)
TS_E_UNSUPPORTED = -7                     # include/tiler_slider.h

# walls per board: with 5 to 8 tiles, enough walls that ordered state spaces stay in reach of the oracle
MANY_TILE_WALLS = {3: {5: 1, 6: 1, 7: 1, 8: 0}, 4: {5: 4, 6: 5, 7: 6, 8: 6}, 5: {5: 6, 6: 6, 7: 5, 8: 6},
                   6: {5: 8, 6: 10, 7: 12, 8: 14}, 7: {5: 14, 6: 16, 7: 18, 8: 20}, 8: {5: 24, 6: 26, 7: 28, 8: 28}}


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    t.lib()
    return t


def n_walls(S, T):
    if T >= 5:
        return MANY_TILE_WALLS[S][T]
    return min({1: 0, 2: 1 if T <= 2 else 0, 3: 2}.get(S, S * S // 4), S * S - T)


def blocked_cells(S, row):
    return [(int(c) // S, int(c) % S) for c in np.flatnonzero(row)]


def draw(rng, S, T, W, kind, multi):
    """One puzzle: walls, tiles and targets of a uniform draw (random_puzzles; on boards too full for
    disjoint tiles and targets the targets are any T free cells), targets where a random walk leaves
    the tiles (solvable), or targets = tiles (the board starts on its goal)."""
    if W + 2 * T <= S * S:
        blocked, tiles, targets = (a[0] for a in random_puzzles(rng, 1, S, T, W))
    else:
        perm = rng.permutation(S * S)
        blocked = np.zeros(S * S, np.uint8)
        blocked[perm[:W]] = 1
        tcell, gcell = perm[W:W + T], rng.permutation(perm[W:])[:T]
        tiles = np.stack([tcell // S, tcell % S], -1).astype(np.uint8)
        targets = np.stack([gcell // S, gcell % S], -1).astype(np.uint8)
    if kind == "reachable":
        targets = reachable_targets(orc, rng, S, blocked[None], tiles[None], multi, 12)[0]
    elif kind == "on_goal":
        targets = tiles.copy()
    return blocked, tiles, targets


def oracle_bfs(S, blocked, tiles, targets, multi, max_depth=256):
    st = orc.OracleState(S, blocked_cells(S, blocked), tiles.tolist(), targets.tolist(), multi)
    return st.bfs(max_depth=max_depth, max_states=STATE_CAP, by_level=True)


@functools.lru_cache(maxsize=None)
def cases(S, T, multi):
    """The tables of one (size, tiles, colour mode), each with the oracle's search of every puzzle:
    up to 4 tiles one batch (uniform draws, solvable puzzles, one board on its goal; 260 puzzles on
    the smallest boards so that puzzle ids pass 255), 5 to 8 tiles one table per puzzle.  Ordered
    goal: also a never_win table (one target fewer than tiles), whose visited sets are the same."""
    rng = np.random.default_rng([S, T, int(multi)])
    W = n_walls(S, T)
    if T <= 4:
        n_uniform, n_reachable = (100, 159) if S <= 3 else (4, 6)
    else:
        n_uniform, n_reachable = 1, 2
    puzzles = []
    for kind in ["uniform"] * n_uniform + ["reachable"] * n_reachable + ["on_goal"]:
        for _ in range(60):
            b, t, g = draw(rng, S, T, W, kind, multi)
            try:
                res = oracle_bfs(S, b, t, g, multi)
            except RuntimeError:                      # over STATE_CAP: redraw
                continue
            puzzles.append((kind, b, t, g, res))
            break
        else:
            raise AssertionError(f"no {kind} puzzle under {STATE_CAP} states for S={S} T={T} multi={multi}")
    groups = [puzzles] if T <= 4 else [[p] for p in puzzles]
    tables = [dict(kinds=[p[0] for p in grp], blocked=np.stack([p[1] for p in grp]), tiles=np.stack([p[2] for p in grp]),
                   targets=np.stack([p[3] for p in grp]), oracle=[p[4] for p in grp], never_win=False) for grp in groups]
    if multi:
        base = tables[0] if T <= 4 else tables[1]
        nw = dict(base, kinds=["never_win"] * len(base["kinds"]), targets=base["targets"][:, :T - 1], never_win=True)
        nw["oracle"] = [(n, lv, -1, keys) for n, lv, _, keys in base["oracle"]]   # targets do not change the moves
        tables.append(nw)
    return tables


def env_of(ts, S, tab, multi):
    return ts.BatchedTilerSliderEnv.from_arrays(S, tab["blocked"], tab["tiles"], tab["targets"], multi)


def table_capacity(n_states):
    return 1 << max(8, (2 * n_states).bit_length())


def pack(cells):
    """cells int[N, T] -> oracle keys u64[N] (byte i = cell of tile i, r*S + c)"""
    key = np.zeros(cells.shape[0], np.uint64)
    for i in range(cells.shape[1]):
        key |= cells[:, i].astype(np.uint64) << np.uint64(8 * i)
    return key


def decode(keys, S, T, PS, ordered):
    """GPU keys without bit 63 -> (puzzle id, oracle key).  Byte i is r*PS + c of tile i; unused
    bytes are zero; set goal: the bytes are the canonical (ascending) arrangement."""
    if T <= 4:
        pid, pos, width = keys >> np.uint64(32), keys & np.uint64(0xFFFFFFFF), 32
    else:
        pid, pos, width = np.zeros_like(keys), keys, 64
    if 8 * T < width:
        assert not (pos >> np.uint64(8 * T)).any(), "bytes past the last tile are not zero"
    b = np.stack([(pos >> np.uint64(8 * i)) & np.uint64(0xFF) for i in range(T)], 1).astype(np.int64)
    r, c = b // PS, b % PS
    assert (r < S).all() and (c < S).all(), "a position byte is off the board"
    cells = r * S + c
    if T > 1:
        step = np.diff(cells if not ordered else np.sort(cells, axis=1), axis=1)
        assert (step > 0).all(), "two tiles on one cell" if ordered else "set-goal key not in canonical order"
    return pid, pack(cells)


def goal_key(S, targets, ordered):
    cells = targets[:, :, 0].astype(np.int64) * S + targets[:, :, 1]
    return pack(cells if ordered else np.sort(cells, axis=1))


def search_by_hand(ts, env, capacity):
    """seed, insert, then expand + insert until a level brings nothing new: the new keys of every level"""
    from tiler_slider_b200.bfs import CudaBfsKernels
    k = CudaBfsKernels(env)
    visited = k.new_table(capacity)
    front, _ = k.insert(visited, k.seed())
    levels = []
    while front.numel():
        levels.append(front.clone())
        assert len(levels) < 1000
        front, _ = k.insert(visited, k.expand(levels[-1]))
    return [lv.cpu().numpy().view(np.uint64) for lv in levels]


def rows(pid, depth, key):
    m = np.stack([pid.astype(np.uint64), depth.astype(np.uint64), key.astype(np.uint64)], 1)
    return m[np.lexsort((m[:, 2], m[:, 1], m[:, 0]))]


def check_levels(ts, S, T, multi, tab):
    """One table through seed / expand / insert by hand; returns the number of states compared."""
    P, ordered = tab["tiles"].shape[0], multi
    want_states = sum(o[0] for o in tab["oracle"])
    levels = search_by_hand(ts, env_of(ts, S, tab, multi), table_capacity(want_states))
    keys = np.concatenate(levels)
    depth = np.repeat(np.arange(len(levels)), [lv.size for lv in levels])
    won, plain = (keys & WON) != 0, keys & ~WON
    assert np.unique(plain).size == plain.size, "a key was inserted twice"
    pid, okey = decode(plain, S, T, ts.lib().ts_pos_stride(S), ordered)
    assert (pid < P).all()
    # the visited set of every puzzle, level by level
    want = rows(np.concatenate([np.full(o[0], e) for e, o in enumerate(tab["oracle"])]),
                np.concatenate([np.repeat(np.arange(len(o[1])), o[1]) for o in tab["oracle"]]),
                np.concatenate([o[3] for o in tab["oracle"]]))
    got = rows(pid, depth, okey)
    assert got.shape == want.shape and np.array_equal(got, want), (S, T, multi, tab["kinds"][0])
    # roots come from bfs_seed without the goal bit; every other new key carries is_won of its state
    if tab["never_win"]:
        assert not won.any()
        for e in range(P):
            bl = blocked_cells(S, tab["blocked"][e])
            assert not orc.OracleState(S, bl, tab["tiles"][e].tolist(), tab["targets"][e].tolist(), True).is_won()
    else:
        goal = goal_key(S, tab["targets"], ordered)
        assert np.array_equal(won, (okey == goal[pid.astype(np.int64)]) & (depth > 0))
        for e in range(P):                            # the oracle agrees that the goal state is won
            bl, g = blocked_cells(S, tab["blocked"][e]), tab["targets"][e].tolist()
            assert orc.OracleState(S, bl, g, g, multi).is_won()
    return keys.size


@pytest.mark.parametrize("S", SIZES)
def test_visited_sets_level_by_level(ts, S):
    """Every (S, T) pair of this size in both goal modes: each GPU key decoded, each puzzle's set of
    new states at each depth equal to the oracle's, no key twice, bit 63 = the state is won."""
    covered, compared = set(), {}
    for T in range(1, min(8, S * S) + 1):
        for multi in (True, False):
            for tab in cases(S, T, multi):
                mode = "ordered" if multi else "set"
                compared[(T, mode)] = compared.get((T, mode), 0) + check_levels(ts, S, T, multi, tab)
                covered.add((T, multi))
    assert covered == {(T, m) for T in range(1, min(8, S * S) + 1) for m in (True, False)}
    print(f"\nS={S} states compared: " + ", ".join(f"T={T} {mode}: {n}" for (T, mode), n in sorted(compared.items())))


# ---- 5 to 8 tiles through the product paths ------------------------------------------------------
def many_tile_tables(multi, S_range=MANY_TILES_SIZES, T_range=range(5, 9)):
    for S in S_range:
        for T in T_range:
            for tab in cases(S, T, multi):
                if not tab["never_win"]:
                    yield S, T, tab


def replay_wins(S, blocked, tiles, targets, multi, moves):
    """1-based steps at which the oracle reports a win while replaying `moves`"""
    st = orc.OracleState(S, blocked_cells(S, blocked), tiles.tolist(), targets.tolist(), multi)
    return [k + 1 for k, ch in enumerate(moves) if st.move("UDLR".index(ch))]


def check_solution(S, tab, multi, depth, sol):
    if depth < 0:
        assert sol is None
        return
    assert sol is not None and len(sol) == depth, (sol, depth)
    wins = replay_wins(S, tab["blocked"][0], tab["tiles"][0], tab["targets"][0], multi, sol)
    assert wins[:1] == [depth], (sol, wins)


@pytest.mark.parametrize("multi", [True, False])
def test_paths_with_many_tiles(ts, multi):
    """BfsSolver(...).solve(with_paths=True), device- and host-driven, on every board class for 5 to 8
    tiles: counts, histogram, depth, successor count and a shortest solution that wins on its last move."""
    from tiler_slider_b200.bfs import BfsSolver
    sizes, kinds = set(), {"uniform": 0, "reachable": 0, "on_goal": 0}
    unsolvable = on_goal_solved = 0
    for S, T, tab in many_tile_tables(multi):
        n, lv, depth, _ = tab["oracle"][0]
        for dd in (True, False):
            r = BfsSolver(env_of(ts, S, tab, multi), table_capacity=table_capacity(n)).solve(with_paths=True, device_driven=dd)
            assert r.states_per_puzzle.tolist() == [n] and r.levels == lv and r.n_states == n, (S, T, dd)
            assert r.solve_depth_per_puzzle.tolist() == [depth] and r.solve_depth == depth, (S, T, dd)
            assert r.generated == 4 * n
            check_solution(S, tab, multi, depth, r.solutions[0])
        if tab["kinds"][0] == "on_goal":
            # the goal is tested after a move: a board on its goal needs at least one move (a move that
            # changes nothing, or a cycle back), and when every move leaves the goal for good it is unsolvable
            assert depth != 0
            on_goal_solved += depth > 0
        sizes.add(S)
        kinds[tab["kinds"][0]] += 1
        unsolvable += depth < 0
    assert sizes == set(MANY_TILES_SIZES) and min(kinds.values()) >= len(MANY_TILES_SIZES)
    assert unsolvable >= 1 and on_goal_solved >= 1 and kinds["reachable"] >= 2 * len(MANY_TILES_SIZES)


@pytest.mark.parametrize("multi", [True, False])
def test_depth_limits_with_many_tiles(ts, multi):
    """max_depth 1, 5, 16 and 17 (either side of LEVELS_PER_SYNC = 16): device- and host-driven runs
    agree, and both equal the oracle's histogram cut after level max_depth and its solve depth when
    that is within max_depth."""
    from tiler_slider_b200.bfs import BfsSolver
    assert BfsSolver.LEVELS_PER_SYNC == 16
    sizes, deep, cut_solved = set(), 0, 0
    for S, T, tab in many_tile_tables(multi):
        n, lv, depth, _ = tab["oracle"][0]
        if tab["kinds"][0] != "reachable":
            continue
        deep += len(lv) > 18
        for m in (1, 5, 16, 17):
            want_lv = lv[:m + 1]
            want_depth = depth if 0 < depth <= m else -1
            cut_solved += depth > m
            got = []
            for dd in (True, False):
                r = BfsSolver(env_of(ts, S, tab, multi), table_capacity=table_capacity(n)).solve(max_depth=m, device_driven=dd)
                assert r.levels == want_lv and r.n_states == sum(want_lv), (S, T, m, dd)
                assert r.states_per_puzzle.tolist() == [sum(want_lv)]
                assert r.solve_depth_per_puzzle.tolist() == [want_depth] and r.solve_depth == want_depth, (S, T, m, dd)
                assert r.generated == 4 * sum(lv[:m])
                got.append((r.n_states, r.levels, r.solve_depth, r.generated))
            assert got[0] == got[1]
        sizes.add(S)
    assert sizes == set(MANY_TILES_SIZES)
    assert deep >= 1 and cut_solved >= 1        # some search outlives 17 levels, some solution lies past a cut


def puzzle_of(ts, S, tab, e, multi):
    return ts.Puzzle(S, blocked_cells(S, tab["blocked"][e]), [tuple(int(v) for v in x) for x in tab["tiles"][e]],
                     [tuple(int(v) for v in x) for x in tab["targets"][e]], multi)


def test_solve_batch_with_many_tiles(ts):
    """solve_batch over several puzzles of one shape with 6 and with 8 tiles (one search per puzzle):
    its per-puzzle results are those of one BfsSolver per puzzle and of the oracle, its level
    histogram their element-wise sum."""
    from tiler_slider_b200.bfs import BfsSolver, solve_batch
    sizes = set()
    for S, T, multi in ((3, 6, True), (4, 8, False), (5, 6, False), (6, 8, True), (7, 6, True), (8, 8, False)):
        tabs = [tab for _, _, tab in many_tile_tables(multi, [S], [T])]
        puzzles = [puzzle_of(ts, S, tab, 0, multi) for tab in tabs]
        r = solve_batch(puzzles, with_paths=True)
        want = [tab["oracle"][0] for tab in tabs]
        assert r.states_per_puzzle.tolist() == [w[0] for w in want], (S, T)
        assert r.solve_depth_per_puzzle.tolist() == [w[2] for w in want], (S, T)
        n_lv = max(len(w[1]) for w in want)
        assert r.levels == [sum(w[1][d] for w in want if d < len(w[1])) for d in range(n_lv)]
        assert r.n_states == sum(w[0] for w in want) and r.generated == 4 * r.n_states
        for e, tab in enumerate(tabs):
            one = BfsSolver([puzzles[e]], table_capacity=table_capacity(want[e][0])).solve(with_paths=True)
            assert (one.n_states, one.solve_depth) == (int(r.states_per_puzzle[e]), int(r.solve_depth_per_puzzle[e]))
            assert (one.solutions[0] is None) == (r.solutions[e] is None)
            check_solution(S, tab, multi, want[e][2], r.solutions[e])
        sizes.add(S)
    assert sizes == set(MANY_TILES_SIZES)


def test_main_solve_with_many_tiles(ts, tmp_path):
    """`main.py -input_file F -solve` on puzzles with 5 to 8 tiles: the printed depth and reachable-state
    count are the oracle's, the printed string replays to a win.  (3x3 boards cannot hold 5 tiles and
    5 targets on distinct cells, which the text grammar needs.)"""
    from tiler_slider_b200 import puzzle_to_text
    chosen = []
    for S in range(4, 9):                 # 5 to 8 tiles, both goal modes
        T, multi, rng = 5 + S % 4, S % 2 == 0, np.random.default_rng([S, 99])
        for _ in range(500):              # solvable, and no tile on a target cell (one character per cell)
            b, t, g = draw(rng, S, T, n_walls(S, T), "reachable", multi)
            if {tuple(x) for x in t.tolist()} & {tuple(x) for x in g.tolist()}:
                continue
            try:
                res = oracle_bfs(S, b, t, g, multi)
            except RuntimeError:
                continue
            if res[2] > 0:
                chosen.append((S, dict(blocked=b[None], tiles=t[None], targets=g[None], oracle=[res]), multi))
                break
    assert [c[0] for c in chosen] == list(range(4, 9))
    blocks = [f"multi_color: {'true' if multi else 'false'}\n" + puzzle_to_text(puzzle_of(ts, S, tab, 0, multi))
              for S, tab, multi in chosen]
    f = tmp_path / "puzzles.txt"
    f.write_text("\n---\n".join(blocks) + "\n")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), "-input_file", str(f), "-solve", "-quiet"],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    found = re.findall(r"solution\[(\d+)\]: '([UDLR]*)' \(depth (-?\d+), (\d+) reachable states\)", out.stdout)
    assert len(found) == len(chosen), out.stdout
    for (_, sol, depth, n), (S, tab, multi) in zip(found, chosen):
        n_want, _, depth_want, _ = tab["oracle"][0]
        assert (int(depth), int(n)) == (depth_want, n_want), (S, sol)
        check_solution(S, tab, multi, depth_want, sol)


# ---- refusals and overflow ------------------------------------------------------------------------
def test_refusals_and_table_overflow(ts):
    import ctypes as C
    from tiler_slider_b200._lib import BfsArgs
    from tiler_slider_b200.bfs import BfsSolver, CudaBfsKernels
    two = ts.BatchedTilerSliderEnv.synthetic(2, 6, 5, 8, True, seed=1)
    with pytest.raises(ValueError, match="more than 4 tiles"):
        CudaBfsKernels(two)
    for S, T in ((8, 9), (9, 4)):
        cells = np.arange(2 * T)
        at = np.stack([cells // S, cells % S], -1).astype(np.uint8)
        env = ts.BatchedTilerSliderEnv.from_arrays(S, np.zeros((1, S * S), np.uint8), at[None, :T], at[None, T:], True)
        with pytest.raises(ValueError, match="board sizes up to 8 with 1 to 8 tiles"):
            CudaBfsKernels(env)
    # the C-ABI refuses a T > 4 table that could hold more than one puzzle (its key has no id bits)
    one = ts.BatchedTilerSliderEnv.synthetic(1, 6, 5, 8, True, seed=1)
    out = torch.empty(256, dtype=torch.int64, device=one.device)
    init = torch.zeros(256, 8, dtype=torch.uint8, device=one.device)
    for cap, rc in ((256, TS_E_UNSUPPORTED), (128, 0)):
        a = BfsArgs(size=6, n_tiles=5, goal_mode=one.goal_mode, n_ranks=1, n_items=1, puzzle_capacity=cap,
                    d_init=init.data_ptr(), d_out_keys=out.data_ptr())
        assert ts.lib().ts_bfs_seed(C.byref(a), torch.cuda.current_stream().cuda_stream) == rc
    torch.cuda.synchronize()
    # a table too small for the search: both level loops report it
    S, T, tab = max(many_tile_tables(True), key=lambda x: x[2]["oracle"][0][0])
    assert tab["oracle"][0][0] > 4096
    for dd in (True, False):
        with pytest.raises(RuntimeError, match="table is full"):
            BfsSolver(env_of(ts, S, tab, True), table_capacity=1024).solve(device_driven=dd)
