"""ts_playout (BatchedTilerSliderEnv.playout) on the B200.

- The plan policy is the step: for every board class (test_gpu_expand.PIN_SHAPES: every bitboard size,
  every wide-record length, the generic tile counts, tile-less boards, never_win), final / steps / won
  equal what step() leaves on a copy (auto_reset off, max_steps 64: pos, step_count, the WON flag),
  traj[k] the positions after step k, moves the plan; a sample is checked against oracle.rollout.
- Real levels: LocalBfs's shortest solutions, padded with 255, win in exactly solve-depth moves; cut
  one move short they do not win.
- The random policy is the restated draw (synth_stream / splitmix64 of tests/gen_port.py, the oracle's
  valid_moves() and move()), bit for bit, for every kernel class and two seeds; boards where nothing
  can move play no move.
- Items: shuffled ids with repeats and explicit positions equal a batch gathered from the listed puzzles;
  ids past capacity give the zero result; n_steps = 0.
- Guards: poisoned guard regions around every output; nothing outside the write set and no env buffer
  (padding included) changes.
- Random playouts that win never beat optimal_moves()'s distance; never_win batches never win.
- One CUDA graph of step() + playout(out=...) replays like the direct calls.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import gen_port
from tests.test_gpu_expand import PIN_SHAPES, assert_untouched, build, env_buffers, gathered
from tests.test_gpu_ranges import GUARD, POISON

pytestmark = pytest.mark.gpu

F_WON = 2
SEEDS = [0, (1 << 40) + 12345]


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def stepped_copy(ts, S, arrays, multi, start, plan):
    """What step() does with the plan on a copy of the batch: (pos after each step [L, N, PW], step_count,
    won ever, flags).  auto_reset off: an env that won is frozen (STALE) and keeps its positions."""
    blocked, tiles, targets = arrays
    ref = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=64, auto_reset=False)
    ref._pos[: start.shape[0]] = start
    L, N = plan.shape
    traj = torch.empty(L, N, ref.pos_bytes, dtype=torch.uint8, device="cuda")
    won = torch.zeros(N, dtype=torch.bool, device="cuda")
    for k in range(L):
        ref.step(plan[k])
        traj[k] = ref.pos
        won |= (ref.flags & F_WON) != 0
    return traj, ref.step_count.to(torch.int32), won.to(torch.uint8), ref.pos.clone()


def check_records(final, steps, moves, traj, PW):
    """moves 255 and traj zero for k >= steps; final = traj[steps - 1] (or the start, checked by the caller)."""
    L, N = moves.shape
    k = torch.arange(L, device="cuda")[:, None]
    after = k >= steps[None, :].long()
    assert torch.equal(moves[after], torch.full_like(moves[after], 255))
    assert not traj[after].any()
    played = steps > 0
    last = (steps.long() - 1).clamp(min=0)
    assert torch.equal(final[played], traj[last, torch.arange(N, device="cuda")][played])


@pytest.mark.parametrize("S,T,NT,W,multi", PIN_SHAPES)
def test_plan_is_the_step(ts, S, T, NT, W, multi):
    N, L = 1001, 40
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=S * 1000 + T * 10 + NT + 7)
    start = env.pos.clone()
    g = torch.Generator(device="cuda").manual_seed(S + 31 * T)
    plan = torch.randint(0, 4, (L, N), dtype=torch.uint8, device="cuda", generator=g)
    before = env_buffers(env)
    final, steps, won, moves, traj = env.playout(actions=plan, record=True)
    assert_untouched(env, before, "playout")
    assert final.shape == (N, env.pos_bytes) and steps.dtype == torch.int32 and moves.shape == (L, N) and traj.shape == (L, N, env.pos_bytes)
    w_traj, w_steps, w_won, w_final = stepped_copy(ts, S, arrays, multi, start, plan)
    assert torch.equal(steps, w_steps)
    assert torch.equal(won, w_won)
    assert torch.equal(final, w_final)
    k = torch.arange(L, device="cuda")[:, None]
    live = k < steps[None, :].long()
    assert torch.equal(traj[live], w_traj[live])
    assert torch.equal(moves[live], plan[live])
    check_records(final, steps, moves, traj, env.pos_bytes)
    if env.never_win:
        assert not won.any()
    # the C oracle on a sample: start at the playout's start positions, same plan
    n = 40
    blocked, _, targets = arrays
    want = orc.rollout(S, multi, blocked[:n], env.positions(start[:n]).cpu().numpy(), targets[:n], plan[:, :n].cpu().numpy(),
                       max_steps=64, auto_reset=False)
    assert np.array_equal(want["final_count"], steps[:n].cpu().numpy())
    assert np.array_equal(want["final_pos"], env.positions(final[:n]).cpu().numpy().astype(np.int16))
    assert np.array_equal(((want["flags"] & F_WON) != 0).any(0), won[:n].cpu().numpy() != 0)


def test_real_solutions_win_in_exactly_their_length(ts):
    """LocalBfs's shortest solutions of the real levels, padded with 255 into one plan per shape group,
    win in exactly solve-depth moves from the initial positions; cut one move short they never win (a
    shorter win would contradict the shortest solution)."""
    from tiler_slider_b200.bfs import LocalBfs
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_400.txt")
    groups = {}
    for p in ts.load_puzzle_file(path):
        groups.setdefault((p.size, len(p.initial_locations), len(p.target_locations), p.multiple_colors), []).append(p)
    code = {"U": 0, "D": 1, "L": 2, "R": 3}
    solved = 0
    for key, ps in groups.items():
        env = ts.BatchedTilerSliderEnv.from_puzzles(ps)
        res = LocalBfs(env).solve(with_paths=True)
        sols = res.solutions
        L = max(len(s) for s in sols if s is not None)
        plan = np.full((L, env.n_envs), 255, np.uint8)
        cut = np.full((L, env.n_envs), 255, np.uint8)
        for i, s in enumerate(sols):
            if s is None:
                continue
            plan[: len(s), i] = [code[c] for c in s]
            cut[: len(s) - 1, i] = plan[: len(s) - 1, i]
        final, steps, won = env.playout(actions=torch.from_numpy(plan).cuda())
        _, steps_cut, won_cut = env.playout(actions=torch.from_numpy(cut).cuda())
        depth = res.solve_depth_per_puzzle.cpu().numpy()
        ok = np.array([s is not None for s in sols])
        assert (depth[ok] >= 1).all(), key
        assert np.array_equal(won.cpu().numpy()[ok], np.ones(ok.sum(), np.uint8)), key
        assert np.array_equal(steps.cpu().numpy()[ok], depth[ok]), key
        assert not won_cut.cpu().numpy()[ok].any(), key
        assert np.array_equal(steps_cut.cpu().numpy()[ok], depth[ok] - 1), key
        solved += int(ok.sum())
    assert solved >= 256


def restate_random(S, multi, blocked, start, targets, seed, idx, L):
    """(final [T, 2], steps, won, moves [L], traj [L, T, 2]) of item `idx` under the random policy: the
    stream synth_stream(seed, idx), one splitmix64 draw per move, the floor(r*n / 2^32)-th valid move."""
    T = start.shape[0]
    st = orc.OracleState(S, [(c // S, c % S) for c in np.flatnonzero(blocked)], start.tolist(), targets.tolist(), multi)
    rng = gen_port.synth_stream(seed, idx)
    moves = np.full(L, 255, np.uint8)
    traj = np.zeros((L, T, 2), np.int64)
    won, steps = False, 0
    while steps < L and not won:
        valid = st.valid_moves()
        if not valid:
            break
        rng, z = gen_port.splitmix64(rng)
        d = valid[((z >> 32) * len(valid)) >> 32]
        won = st.move(d)
        moves[steps] = d
        traj[steps] = np.array(st.current_locations, np.int64).reshape(T, 2)
        steps += 1
    final = traj[steps - 1] if steps else start.astype(np.int64)
    return final, steps, won, moves, traj


# one shape per kernel class and goal rule, boards where nothing can move (1x1 with its tile, a 2x2 full
# of tiles, tile-less boards), never_win
RANDOM_SHAPES = [
    (6, 4, 4, 8, True), (5, 1, 1, 4, False), (4, 3, 3, 2, False), (8, 3, 3, 12, False), (7, 7, 7, 8, True),
    (9, 2, 2, 20, True), (12, 8, 8, 30, True), (12, 4, 4, 30, False), (14, 7, 7, 30, True), (16, 8, 8, 40, False),
    (8, 12, 12, 10, False), (10, 20, 20, 12, True), (6, 0, 2, 8, False), (6, 0, 0, 8, True),
    (1, 1, 1, 0, True), (2, 4, 4, 0, True), (6, 3, 5, 8, True),
]


@pytest.mark.parametrize("S,T,NT,W,multi", RANDOM_SHAPES)
@pytest.mark.parametrize("seed", SEEDS)
def test_random_is_the_restated_draw(ts, S, T, NT, W, multi, seed):
    N, L = 257, 24
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=S * 100 + T + NT)
    blocked, _, targets = arrays
    start = env.positions().cpu().numpy()
    before = env_buffers(env)
    final, steps, won, moves, traj = env.playout(n_steps=L, seed=seed, record=True)
    assert_untouched(env, before, "playout")
    f, s, w, m = env.positions(final).cpu().numpy(), steps.cpu().numpy(), won.cpu().numpy(), moves.cpu().numpy()
    tr = env.positions(traj.reshape(-1, env.pos_bytes)).reshape(L, N, T, 2).cpu().numpy()
    for i in range(N):
        wf, ws, ww, wm, wt = restate_random(S, multi, blocked[i], start[i], targets[i], seed, i, L)
        assert s[i] == ws and bool(w[i]) == ww, (i, s[i], ws, w[i], ww)
        assert np.array_equal(f[i], wf), i
        assert np.array_equal(m[:, i], wm), i
        assert np.array_equal(tr[:, i], wt), i
    check_records(final, steps, moves, traj, env.pos_bytes)
    assert not traj[torch.arange(L, device="cuda")[:, None] >= steps[None, :].long()].any()
    if T == 0 or (S, T) in ((1, 1), (2, 4)):
        assert not steps.any() and not won.any() and torch.equal(final, env.pos)     # nothing can move
    else:
        assert (steps > 0).any()


@pytest.mark.parametrize("S,T,NT,W,multi", [(6, 4, 4, 8, True), (6, 3, 3, 8, False), (12, 8, 8, 30, True),
                                           (10, 20, 20, 12, False), (6, 0, 2, 8, True), (6, 3, 5, 8, True)])
def test_items_equal_the_gathered_puzzles(ts, S, T, NT, W, multi):
    """Shuffled ids with repeats at expand() successors: each result equals the playout of a batch built
    from the listed puzzles at the listed positions, with the same item indices, under both policies."""
    N, n, L = 600, 2000, 20
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=11 + S + T)
    g = torch.Generator().manual_seed(4)
    ids = torch.randint(0, N, (n,), generator=g)
    succ, _, _ = env.expand(ids)
    pos = succ[torch.arange(n, device="cuda"), (ids % 4).cuda()].contiguous()
    ref = gathered(ts, S, arrays, multi, ids, pos)
    gd = torch.Generator(device="cuda").manual_seed(5)
    plan = torch.randint(0, 4, (L, n), dtype=torch.uint8, device="cuda", generator=gd)
    plan[L // 2:, ::7] = 255                                      # ragged plans
    before = env_buffers(env)
    for given in (ids, ids.to(torch.int32).cuda()):
        for kw in (dict(actions=plan), dict(n_steps=L, seed=9)):
            got = env.playout(given, pos, record=True, **kw)
            want = ref.playout(record=True, **kw)
            for a, b in zip(got, want):
                assert torch.equal(a, b), kw
    assert_untouched(env, before, "items")
    # ids only: each listed env from its current positions
    got = env.playout(ids[:N], n_steps=L, seed=3)
    want = gathered(ts, S, arrays, multi, ids[:N], env.pos[ids[:N].cuda()]).playout(n_steps=L, seed=3)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    # ids past capacity (device ids are not checked on the host): the zero result
    bad = torch.tensor([0, env.capacity, -3, env.capacity + 1000, 1], dtype=torch.int32, device="cuda")
    final, steps, won, moves, traj = env.playout(bad, n_steps=L, record=True)
    dense = env.playout(torch.tensor([0, 1], dtype=torch.int32, device="cuda"), n_steps=L, record=True)
    assert not final[1:4].any() and not steps[1:4].any() and not won[1:4].any() and not traj[:, 1:4].any()
    assert (moves[:, 1:4] == 255).all()
    # (the stream is the item index: items 0 and 4 are not items 0 and 1 of `dense`; check item 0 only)
    assert torch.equal(final[0], dense[0][0]) and steps[0] == dense[1][0]
    # n_steps = 0 and an empty plan: the start positions, 0 moves, not won
    for kw in (dict(n_steps=0), dict(actions=torch.empty(0, N, dtype=torch.uint8, device="cuda"))):
        final, steps, won, moves, traj = env.playout(record=True, **kw)
        assert torch.equal(final, env.pos) and not steps.any() and not won.any() and moves.shape == (0, N) and traj.shape == (0, N, env.pos_bytes)


@pytest.mark.parametrize("S,T,NT,W,multi", [(6, 4, 4, 8, True), (5, 1, 1, 4, False), (12, 8, 8, 30, False),
                                           (15, 5, 5, 40, True), (8, 12, 12, 10, True), (6, 0, 0, 8, False)])
@pytest.mark.parametrize("n", [1, 3, 129, 1000])
@pytest.mark.parametrize("policy", ["plan", "random"])
def test_guards_and_env_buffers_are_untouched(ts, S, T, NT, W, multi, n, policy):
    """Outputs are views into poisoned buffers with GUARD bytes on both sides; ids mix live envs, padding
    envs [n_envs, capacity) and ids past capacity.  Only the write set changes, ids past capacity get the
    zero result, and no env buffer -- padding included -- changes."""
    N, L = 301, 12
    env, _ = build(ts, S, T, NT, W, multi, N, seed=n + S + 3)
    PW, cap = env.pos_bytes, env.capacity
    g = torch.Generator().manual_seed(n)
    ids = torch.randint(0, N, (n,), generator=g, dtype=torch.int32)
    if n > 1:
        ids[1] = N + 2                   # padding env: meaningless result, but only inside the write set
    if n > 2:
        ids[2] = cap + 7                 # past capacity: the zero result
    ids[-1] = -1 if n > 3 else ids[-1]
    kw = dict(n_steps=L, seed=77) if policy == "random" else \
        dict(actions=torch.randint(0, 5, (L, n), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n)))
    want = env.playout(ids.cuda(), record=True, **kw)
    sizes = [n * PW, 4 * n, n, L * n, L * n * PW]
    bufs = [torch.full((2 * GUARD + k,), POISON, dtype=torch.uint8, device="cuda") for k in sizes]
    body = [b[GUARD:-GUARD] for b in bufs]
    out = (body[0].view(n, PW), body[1].view(torch.int32), body[2], body[3].view(L, n), body[4].view(L, n, PW))
    guards = [torch.cat([b[:GUARD], b[-GUARD:]]).clone() for b in bufs]
    before = env_buffers(env)
    res = env.playout(ids.cuda(), record=True, out=out, **kw)
    assert all(r is o for r, o in zip(res, out))
    assert_untouched(env, before, "playout")
    for b, gd in zip(bufs, guards):
        assert torch.equal(torch.cat([b[:GUARD], b[-GUARD:]]), gd)
    for a, b in zip(res, want):
        assert torch.equal(a, b)
    outside = ((ids < 0) | (ids >= cap)).cuda()
    assert not res[0][outside].any() and not res[1][outside].any() and not res[2][outside].any()
    assert (res[3][:, outside] == 255).all() and not res[4][:, outside].any()
    # without the records only final / steps / won are written
    bufs3 = [torch.full((2 * GUARD + k,), POISON, dtype=torch.uint8, device="cuda") for k in sizes[:3]]
    body3 = [b[GUARD:-GUARD] for b in bufs3]
    res3 = env.playout(ids.cuda(), out=(body3[0].view(n, PW), body3[1].view(torch.int32), body3[2]), **kw)
    for b in bufs3:
        assert (b[:GUARD] == POISON).all() and (b[-GUARD:] == POISON).all()
    for a, b in zip(res3, want[:3]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("multi", [True, False])
def test_random_wins_never_beat_the_optimal_distance(ts, multi):
    N = 4096
    env = ts.BatchedTilerSliderEnv.solvable(N, 6, 4, 8, multi, min_depth=1, max_depth=10, seed=41)
    dist, _ = env.optimal_moves()
    assert (dist >= 1).all()
    n_won = 0
    for seed in SEEDS:
        _, steps, won = env.playout(n_steps=200, seed=seed)
        w = won.bool()
        assert (steps[w] >= dist[w]).all()
        n_won += int(w.sum())
    assert n_won > 0
    # never_win: multi colour with a target count other than the tile count
    rng = np.random.default_rng(2)
    from tests.test_gpu_ranges import make_puzzles
    blocked, tiles, targets = make_puzzles(rng, 2000, 6, 3, 4, 8)
    nw = ts.BatchedTilerSliderEnv.from_arrays(6, blocked, tiles, targets, True)
    assert nw.never_win
    _, steps, won = nw.playout(n_steps=100, seed=1)
    assert not won.any() and (steps == 100).float().mean() > 0.5
    _, steps, won = nw.playout(actions=torch.randint(0, 4, (50, 2000), dtype=torch.uint8, device="cuda"))
    assert not won.any() and (steps == 50).all()


def test_graph_of_step_and_playout_replays_like_the_calls(ts):
    S, T, W, N, K, L, n = 6, 4, 8, 3000, 3, 16, 1000
    kw = dict(seed=21, max_steps=5, auto_reset=True)
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    gen = torch.Generator(device="cuda").manual_seed(7)
    rows = torch.randint(0, 4, (K, a.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    ids = torch.randint(0, N, (n,), dtype=torch.int32, device="cuda", generator=gen)
    plan = torch.randint(0, 5, (L, n), dtype=torch.uint8, device="cuda", generator=gen)
    PW = a.pos_bytes

    def calls(env, k, out=None):
        env.step(rows[k])
        o = (None, None) if out is None else out
        p = env.playout(ids, actions=plan, record=True, out=o[0])
        r = env.playout(ids, n_steps=L, seed=5 + k, out=o[1])
        return list(p) + list(r)

    want = [[t.clone() for t in calls(b, k)] for k in range(K)]

    def outs():
        u8, i32 = torch.uint8, torch.int32
        rec = (torch.empty(n, PW, dtype=u8, device="cuda"), torch.empty(n, dtype=i32, device="cuda"), torch.empty(n, dtype=u8, device="cuda"),
               torch.empty(L, n, dtype=u8, device="cuda"), torch.empty(L, n, PW, dtype=u8, device="cuda"))
        rnd = (torch.empty(n, PW, dtype=u8, device="cuda"), torch.empty(n, dtype=i32, device="cuda"), torch.empty(n, dtype=u8, device="cuda"))
        return rec, rnd
    bufs = [outs() for _ in range(K)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                     # warm-up outside the capture
        calls(a, 0, bufs[0])
    torch.cuda.current_stream().wait_stream(side)
    a.reset()
    for o in bufs:
        for t in o[0] + o[1]:
            t.fill_(0x5A)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for k in range(K):
            calls(a, k, bufs[k])
    graph.replay()
    torch.cuda.synchronize()
    for k in range(K):
        got = list(bufs[k][0]) + list(bufs[k][1])
        for i, (g_, w_) in enumerate(zip(got, want[k])):
            assert torch.equal(g_, w_), (k, i)
