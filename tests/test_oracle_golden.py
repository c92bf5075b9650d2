"""Pins the CPU oracle (oracle/ts_oracle.c and oracle/py_port.py) to the reference.

Known answers come from (a) the reference's own tests -- the board strings of
tests/test_user_scenarios.py:37-128 and the collision cases of tests/test_state.py:248-311
are restated literally below -- and (b) tests/golden/, recorded by running the unmodified
reference (tests/golden/make_golden.py).  Integer work: the bar is exact equality.
"""
import numpy as np
import pytest

from oracle import oracle as orc
from oracle import py_port

MOVES = {"U": 0, "D": 1, "L": 2, "R": 3}


def render(size, blocked, tiles, targets, multi):
    """TextRender precedence (display.py:63-75): target > tile > blocked > empty."""
    rows = []
    tiles = [tuple(t) for t in tiles]
    targets = [tuple(t) for t in targets]
    blocked = {tuple(b) for b in blocked}
    for i in range(size):
        row = ""
        for j in range(size):
            if (i, j) in targets:
                row += chr((targets.index((i, j)) if multi else 0) + ord("A"))
            elif (i, j) in tiles:
                row += chr((tiles.index((i, j)) if multi else 0) + ord("a"))
            elif (i, j) in blocked:
                row += "X"
            else:
                row += "."
        rows.append(row)
    return "\n".join(rows)


# --- literal golden strings from the reference's tests/test_user_scenarios.py ---------------
SCENARIO_PUZZLE = dict(size=4, blocked=[(1, 0), (2, 3)], tiles=[(0, 3), (3, 2)], targets=[(0, 0), (3, 0)])
SEQ1 = [("R", "A..a\nX...\n...X\nB..b", False), ("D", "A...\nX..a\n...X\nB..b", False),
        ("L", "A...\nXa..\n...X\nB...", False), ("U", "Aa..\nX...\nb..X\nB...", False),
        ("L", "A...\nX...\nb..X\nB...", False), ("D", "A...\nX...\n...X\nB...", True)]
SEQ2 = [("D", "A...\nX..a\n...X\nB.b.", False), ("L", "A...\nXa..\n...X\nB...", False),
        ("D", "A...\nX...\n...X\nBa..", False), ("R", "A...\nX...\n...X\nB.ba", False),
        ("R", "A...\nX...\n...X\nB.ba", False), ("L", "A...\nX...\n...X\nBa..", False)]


@pytest.mark.parametrize("seq", [SEQ1, SEQ2])
@pytest.mark.parametrize("impl", ["c", "py"])
def test_user_scenario_strings(seq, impl):
    p = SCENARIO_PUZZLE
    if impl == "c":
        st = orc.OracleState(p["size"], p["blocked"], p["tiles"], p["targets"], True)
        locs = lambda: st.current_locations
    else:
        st = py_port.PortState(p["size"], p["blocked"], list(p["tiles"]), p["targets"], True)
        locs = lambda: [(int(r), int(c)) for r, c in st.current_locations]
    assert render(4, p["blocked"], locs(), p["targets"], True) == "A..a\nX...\n...X\nB.b."
    for mv, board, won in seq:
        got = st.move(MOVES[mv])
        assert render(4, p["blocked"], locs(), p["targets"], True) == board
        assert bool(got) is won


# --- literal collision cases from the reference's tests/test_state.py:248-311 -----------------
@pytest.mark.parametrize("size,blocked,tiles,mv,expect", [
    (5, [], [(4, 2), (3, 2)], "U", {(0, 2), (1, 2)}),
    (5, [], [(2, 4), (2, 3)], "L", {(2, 0), (2, 1)}),
    (6, [], [(5, 1), (4, 1), (3, 1)], "U", {(0, 1), (1, 1), (2, 1)}),
    (5, [(2, 1)], [(4, 1), (3, 1)], "U", {(3, 1), (4, 1)}),
])
def test_collision_known_answers(size, blocked, tiles, mv, expect):
    st = orc.OracleState(size, blocked, tiles, [(0, 0)] * len(tiles), False)
    st.move(MOVES[mv])
    assert set(st.current_locations) == expect
    # identity: the tile that was nearer the wall stays nearer
    ps = py_port.PortState(size, blocked, list(tiles), [(0, 0)] * len(tiles), False)
    ps.move(MOVES[mv])
    assert [(int(r), int(c)) for r, c in ps.current_locations] == st.current_locations


def test_scenarios_fixture(golden_scenarios):
    for rec in golden_scenarios:
        p = rec["puzzle"]
        st = orc.OracleState(p["size"], p["blocked"], p["tiles"], p["targets"], p["multi_color"])
        assert render(p["size"], p["blocked"], st.current_locations, p["targets"], p["multi_color"]) == rec["initial_board"]
        for step in rec["steps"]:
            won = st.move(MOVES[step["move"]])
            assert [list(x) for x in st.current_locations] == step["positions"]
            assert won == step["info"]["is_won"]
            assert render(p["size"], p["blocked"], st.current_locations, p["targets"], p["multi_color"]) == step["board"]
            assert float(st.get_state_array().sum()) == step["obs_sum"]


def _check_rollout(rec, got):
    assert np.array_equal(got["pos"], rec["pos"]), rec["tag"]
    assert np.array_equal(got["flags"] & 15, rec["flags"]), rec["tag"]
    assert np.array_equal(got["count"], rec["count"]), rec["tag"]


def test_rollouts_fixture_c(golden_rollouts):
    """Reference rollouts under `step; if done: reset` == C oracle with auto_reset."""
    n_checked = 0
    for rec in golden_rollouts:
        got = orc.rollout(rec["S"], rec["multi"], rec["blocked"], rec["tiles"], rec["targets"],
                          rec["actions"], max_steps=rec["max_steps"], auto_reset=True)
        _check_rollout(rec, got)
        n_checked += rec["flags"].size
    assert n_checked > 15000


def test_rollouts_fixture_py(golden_rollouts):
    for rec in golden_rollouts[:12]:
        S, n, K = rec["S"], rec["n"], rec["K"]
        for e in range(min(n, 6)):
            blocked = [(c // S, c % S) for c in np.flatnonzero(rec["blocked"][e])]
            env = py_port.PortEnv(S, blocked, [tuple(map(int, t)) for t in rec["tiles"][e]],
                                  [tuple(map(int, t)) for t in rec["targets"][e]], rec["multi"], rec["max_steps"])
            obs = env.reset()
            for k in range(K):
                obs, done, info = env.step(int(rec["actions"][k, e]))
                assert [[int(r), int(c)] for r, c in env.state.current_locations] == rec["pos"][k, e].tolist()
                assert info["step_count"] == rec["count"][k, e]
                f = rec["flags"][k, e]
                assert (done, info["is_won"], info["invalid_move"], bool(info.get("timeout"))) == \
                    (bool(f & 1), bool(f & 2), bool(f & 4), bool(f & 8))
                if done:
                    obs = env.reset()
            assert np.array_equal(obs, rec["obs_final"][e])


def test_slide_tables(golden_misc):
    for t in golden_misc["slide_tables"]:
        st = orc.OracleState(t["size"], t["blocked"], [(0, 0)], [(0, 0)], False)
        assert np.array_equal(st.move_to, np.array(t["move_to"]))
        ps = py_port.PortState(t["size"], [tuple(b) for b in t["blocked"]], [(0, 0)], [(0, 0)], False)
        assert np.array_equal(ps.move_to, np.array(t["move_to"]))


def test_slide_tables_every_board_class_with_blocked_start_cells(golden_misc):
    """Round-2 fixture: tables of 7x7 ... 16x16 boards; the table is defined for blocked start
    cells too (state.py:85-118 never looks at the start cell itself)."""
    for t in golden_misc["slide_tables_r2"]:
        want = np.array(t["move_to"])
        st = orc.OracleState(t["size"], t["blocked"], [], [], False)
        assert np.array_equal(st.move_to, want), t["size"]
        ps = py_port.PortState(t["size"], [tuple(b) for b in t["blocked"]], [], [], False)
        assert np.array_equal(ps.move_to, want), t["size"]


def _flags_of(step):
    i = step["info"]
    return (orc.F_DONE if step["done"] else 0) | (orc.F_WON if i["is_won"] else 0) | \
        (orc.F_INVALID if i["invalid_move"] else 0) | (orc.F_TIMEOUT if i.get("timeout") else 0)


def test_degenerate_boards(golden_misc):
    """Boards without tiles (won iff no targets: the reference's tests/test_state.py:40-52,
    tests/test_environment.py:569-580) and multi-colour boards whose target count differs from
    the tile count (never won, state.py:183-184), as the reference plays them."""
    for rec in golden_misc["degenerate"]:
        S, multi = rec["size"], rec["multi_color"]
        T, NT = len(rec["tiles"]), len(rec["targets"])
        st = orc.OracleState(S, rec["blocked"], rec["tiles"], rec["targets"], multi)
        assert st.is_won() == rec["won_at_reset"]
        assert np.array_equal(st.get_state_array(), np.array(rec["obs_reset"], np.float32).reshape(S, S, 3))
        assert st.valid_moves() == rec["valid_at_reset"]
        blocked = np.zeros((1, S * S), np.uint8)
        for r, c in rec["blocked"]:
            blocked[0, r * S + c] = 1
        acts = np.array([[MOVES[s["move"]]] for s in rec["steps"]], np.uint8)
        got = orc.rollout(S, multi, blocked, np.array(rec["tiles"], np.uint8).reshape(1, T, 2),
                          np.array(rec["targets"], np.uint8).reshape(1, NT, 2), acts, max_steps=rec["max_steps"])
        env = py_port.PortEnv(S, [tuple(b) for b in rec["blocked"]], [tuple(t) for t in rec["tiles"]],
                              [tuple(t) for t in rec["targets"]], multi, rec["max_steps"])
        env.reset()
        for k, step in enumerate(rec["steps"]):
            assert got["flags"][k, 0] == _flags_of(step), (rec, k)
            assert got["count"][k, 0] == step["info"]["step_count"]
            assert got["pos"][k, 0].tolist() == step["positions"]
            obs, done, info = env.step(MOVES[step["move"]])
            assert done == step["done"] and {k2: (bool(v) if isinstance(v, (bool, np.bool_)) else int(v)) for k2, v in info.items()} == step["info"]
            assert np.array_equal(obs, np.array(step["obs"], np.float32).reshape(S, S, 3))
            assert env.state.is_won() == step["state_is_won"]


def test_slide_table_known_answers():
    """tests/test_state.py:71-157 style: open 5x5 slides to the edges; a wall stops short."""
    st = orc.OracleState(5, [], [(2, 2)], [(0, 0)], False)
    mt = st.move_to
    assert mt[2, 2, 0].tolist() == [0, 2] and mt[2, 2, 1].tolist() == [4, 2]
    assert mt[2, 2, 2].tolist() == [2, 0] and mt[2, 2, 3].tolist() == [2, 4]
    st = orc.OracleState(5, [(0, 2), (2, 4)], [(2, 2)], [(0, 0)], False)
    assert st.move_to[2, 2, 0].tolist() == [1, 2] and st.move_to[2, 2, 3].tolist() == [2, 3]


def test_observations(golden_misc):
    from tests.helpers import parse_text
    for o in golden_misc["observations"]:
        size, blocked, tiles, targets = parse_text(o["text"])
        st = orc.OracleState(size, blocked, tiles, targets, o["multi_color"])
        want = np.array(o["obs"], dtype=np.float32)
        assert np.array_equal(st.get_state_array(), want)
        ps = py_port.PortState(size, blocked, tiles, targets, o["multi_color"])
        assert np.array_equal(ps.observation(), want)


def test_win_logic(golden_misc):
    for w in golden_misc["win_logic"]:
        st = orc.OracleState(3, [], w["tiles"], w["targets"], w["multi_color"])
        assert st.is_won() == w["is_won"], w
        ps = py_port.PortState(3, [], [tuple(t) for t in w["tiles"]], [tuple(t) for t in w["targets"]], w["multi_color"])
        assert ps.is_won() == w["is_won"], w


def test_valid_moves(golden_misc):
    from tests.helpers import parse_text
    for v in golden_misc["valid_moves"]:
        size, blocked, tiles, targets = parse_text(v["text"])
        st = orc.OracleState(size, blocked, tiles, targets, v["multi_color"])
        assert st.valid_moves() == v["valid"]


def test_bfs_known_answers(golden_misc):
    """SURVEY 8(c): 29 / 558 / 950 / 51 reachable states, depths 1 / 8 / 13 / 7."""
    for b in golden_misc["bfs"]:
        st = orc.OracleState(b["size"], b["blocked"], b["tiles"], b["targets"], b["multi_color"])
        n, levels, depth, keys = st.bfs()
        assert (n, levels, depth) == (b["n_states"], b["levels"], b["solve_depth"]), b["name"]
        assert len(np.unique(keys)) == n
    by = {b["name"]: b for b in golden_misc["bfs"]}
    assert by["puzzle_multi_001"]["n_states"] == 29 and by["puzzle_multi_001"]["solve_depth"] == 1
    assert by["puzzle_multi_111"]["n_states"] == 558 and by["puzzle_multi_111"]["solve_depth"] == 8
    assert by["puzzle_multi_180"]["n_states"] == 950 and by["puzzle_multi_180"]["solve_depth"] == 13
    assert by["puzzle_single_151"]["n_states"] == 51 and by["puzzle_single_151"]["solve_depth"] == 7


def test_bfs_keys_by_level(golden_misc):
    """bfs(by_level=True) lists the visited keys level after level: level d is exactly what a
    search cut at depth d has visited and one cut at depth d-1 has not."""
    for b in golden_misc["bfs"]:
        st = orc.OracleState(b["size"], b["blocked"], b["tiles"], b["targets"], b["multi_color"])
        n, levels, depth, keys = st.bfs()
        n2, levels2, depth2, ordered = st.bfs(by_level=True)
        assert (n2, levels2, depth2) == (n, levels, depth)
        assert np.array_equal(np.sort(ordered), keys)
        start = 0
        for d, count in enumerate(levels):
            want = np.setdiff1d(st.bfs(max_depth=d)[3], st.bfs(max_depth=d - 1)[3] if d else [])
            assert np.array_equal(np.sort(ordered[start:start + count]), want), (b["name"], d)
            start += count


def test_success_and_timeout_same_step():
    """SURVEY 7.0 probe: max_steps=1 and a winning move set both flags."""
    blocked = np.zeros((1, 9), np.uint8)
    got = orc.rollout(3, False, blocked, np.array([[[0, 0]]], np.uint8), np.array([[[0, 2]]], np.uint8),
                      np.array([[3]], np.uint8), max_steps=1)
    assert got["flags"][0, 0] == orc.F_DONE | orc.F_WON | orc.F_TIMEOUT
    assert got["count"][0, 0] == 0 and got["reward"][0, 0] == orc.DEFAULT_REWARDS[0]


def test_stale_freeze_without_auto_reset():
    blocked = np.zeros((1, 9), np.uint8)
    acts = np.array([[3], [2], [1]], np.uint8)
    got = orc.rollout(3, False, blocked, np.array([[[0, 0]]], np.uint8), np.array([[[0, 2]]], np.uint8), acts)
    assert got["flags"][:, 0].tolist() == [orc.F_DONE | orc.F_WON, orc.F_DONE | orc.F_STALE, orc.F_DONE | orc.F_STALE]
    assert got["pos"][:, 0, 0].tolist() == [[0, 2]] * 3
    assert got["reward"][:, 0].tolist() == [1.0, 0.0, 0.0]


def test_c_oracle_and_python_port_agree_on_random_boards():
    """The two restatements were written independently (C with an explicit used list, Python
    with the reference's own containers); on 150 random boards of every size 1..12, both colour
    modes, 0-8 tiles' worth of traffic they must agree step by step, including the flags."""
    from tests.helpers import random_puzzles
    rng = np.random.default_rng(99)
    checked = 0
    for trial in range(150):
        S = int(rng.integers(1, 13))
        T = int(rng.integers(1, min(8, S * S) + 1))
        W = int(rng.integers(0, max(1, (S * S - 2 * T) // 2 + 1))) if S * S - 2 * T > 0 else 0
        if W + 2 * T > S * S:
            continue
        multi = bool(rng.integers(0, 2))
        max_steps = int(rng.integers(1, 12))
        blocked, tiles, targets = random_puzzles(rng, 1, S, T, W)
        K = 24
        actions = rng.integers(0, 4, size=(K, 1), dtype=np.uint8)
        got = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=True)
        b = [(c // S, c % S) for c in np.flatnonzero(blocked[0])]
        env = py_port.PortEnv(S, b, [tuple(map(int, t)) for t in tiles[0]], [tuple(map(int, t)) for t in targets[0]],
                              multi, max_steps)
        env.reset()
        for k in range(K):
            _, done, info = env.step(int(actions[k, 0]))
            assert [[int(r), int(c)] for r, c in env.state.current_locations] == got["pos"][k, 0].tolist()
            f = int(got["flags"][k, 0])
            assert (done, info["is_won"], info["invalid_move"], bool(info.get("timeout"))) == \
                (bool(f & 1), bool(f & 2), bool(f & 4), bool(f & 8))
            assert info["step_count"] == got["count"][k, 0]
            if done:
                env.reset()
            checked += 1
    assert checked > 2500


def _levels():
    import os
    from tests.helpers import parse_text
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_400.txt")
    out, grid, multi = [], [], False
    for ln in open(here).read().splitlines() + ["---"]:
        s = ln.strip()
        if s.startswith("#") or not s:
            continue
        if s.startswith("multi_color:"):
            multi = s.split(":")[1].strip() == "true"
        elif set(s) <= {"-"}:
            size, blocked, tiles, targets = parse_text("\n".join(grid))
            out.append((size, blocked, tiles, targets, multi))
            grid, multi = [], False
        else:
            grid.append(s)
    return out


def test_level_corpus_bfs():
    """Real puzzles: the reference's 400 levels (decoded by its own image parser,
    tests/golden/make_levels.py).  For every 8th level a plain BFS over the reference's move
    recorded state count, level histogram and solve depth (tests/golden/make_levels_bfs.py); the
    C oracle's BFS must reproduce them.  Every level of the shipped corpus is solvable."""
    import json
    import os
    levels = _levels()
    assert len(levels) == 400
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_bfs.json")))
    for g in gold:
        size, blocked, tiles, targets, multi = levels[g["index"]]
        n, lv, depth, _ = orc.OracleState(size, blocked, tiles, targets, multi).bfs()
        assert (n, lv, depth) == (g["n_states"], g["levels"], g["solve_depth"]), g["index"]
    solved = sum(orc.OracleState(*lv).bfs()[2] > 0 for lv in levels)
    assert solved == 400


def test_valid_move_rule_used_by_the_kernels():
    """The valid-move kernels run no slide: they use 'a move changes the state iff some tile has an
    empty cell right ahead of it' (ts_valid.cuh).  Pin that rule on the CPU against the oracle's
    copy-and-try get_valid_moves (environment.py:149-171) on random boards of every size."""
    rng = np.random.default_rng(2)
    delta = [(-1, 0), (1, 0), (0, -1), (0, 1)]
    n = 0
    for S in range(1, 17):
        for _ in range(40):
            cells = rng.permutation(S * S)
            W = int(rng.integers(0, max(1, S * S // 3) + 1))
            T = int(rng.integers(0, min(8, S * S - W) + 1))
            blocked = [(int(c) // S, int(c) % S) for c in cells[:W]]
            tiles = [(int(c) // S, int(c) % S) for c in cells[W:W + T]]
            st = orc.OracleState(S, blocked, tiles, tiles, False)
            occ, wall = set(tiles), set(blocked)
            rule = [d for d, (dr, dc) in enumerate(delta)
                    if any(0 <= r + dr < S and 0 <= c + dc < S and (r + dr, c + dc) not in wall and (r + dr, c + dc) not in occ
                           for r, c in tiles)]
            assert rule == st.valid_moves(), (S, blocked, tiles)
            n += 1
    assert n == 640
