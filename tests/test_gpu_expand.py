"""ts_expand and the item form of observe_planes on the B200.

- Pin to the step: for every board class (S 1..16, every wide-record length, 0..8, 12, 20 and 32
  tiles, both goal modes, never_win, duplicate set targets, tile-less boards, the reference's real
  levels), succ[:, a], the moved bit and the won bit equal the positions, !INVALID and WON that
  raw_move(a) leaves on a copy of the positions; a sample is checked against the C oracle.
- Items: shuffled ids with repeats, and positions from an earlier expansion (two levels), equal the
  dense results of the gathered puzzles; ids past capacity give zeros; padding ids write only the
  write set.
- Guards: poisoned guard regions around every output, item counts 1, 3, 129 and ragged; nothing
  outside the write set and no env buffer (padding included) changes.
- Item planes equal observe_planes of a batch built from the listed puzzles at the listed positions.
- A BFS made of expand() and torch.unique reproduces optimal_moves() (distance and mask).
- One CUDA graph of step + expand(out) + item observe_planes(out) replays like the calls.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.test_gpu_ranges import GUARD, POISON, make_puzzles

pytestmark = pytest.mark.gpu

F_WON, F_INVALID = 2, 4
DTYPES = [torch.uint8, torch.bfloat16, torch.float16, torch.float32]


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def build(ts, S, T, NT, W, multi, N, seed, walk=3):
    """N dense boards (make_puzzles: duplicate and covered targets included), then `walk` random raw
    moves so that the positions are not the initial ones."""
    rng = np.random.default_rng(seed)
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(walk):
        env.raw_move(torch.randint(0, 4, (N,), dtype=torch.uint8, device="cuda", generator=g))
    return env, (blocked, tiles, targets)


def composed(env):
    """The composition expand() replaces: clone pos, four times raw_move + copy out, restore."""
    saved = env._pos.clone()
    succ, moved, won = [], torch.zeros(env.n_envs, dtype=torch.uint8, device="cuda"), torch.zeros(env.n_envs, dtype=torch.uint8, device="cuda")
    for a in range(4):
        env._pos.copy_(saved)
        f = env.raw_move(torch.full((env.n_envs,), a, dtype=torch.uint8, device="cuda"))
        succ.append(env.pos.clone())
        moved |= ((f & F_INVALID) == 0).to(torch.uint8) << a
        won |= ((f & F_WON) != 0).to(torch.uint8) << a
    env._pos.copy_(saved)
    return torch.stack(succ, 1), moved, won


def env_buffers(env):
    names = ["_walls", "_targets", "_init", "_pos", "_count", "_reward", "_done", "_flags", "_obs_targets", "_terminal"]
    return {k: getattr(env, k).clone() for k in names if getattr(env, k) is not None}


def assert_untouched(env, before, tag):
    for k, v in env_buffers(env).items():
        assert torch.equal(before[k], v), (tag, k)


def check_oracle_sample(env, arrays, succ, moved, won, multi, n=40):
    blocked, _, targets = arrays
    S, T = env.size, env.n_tiles
    pos = env.positions().cpu().numpy()
    sc = env.positions(succ.reshape(-1, env.pos_bytes)).reshape(env.n_envs, 4, T, 2).cpu().numpy()
    mv, wn = moved.cpu().numpy(), won.cpu().numpy()
    for e in range(min(n, env.n_envs)):
        bl = [(c // S, c % S) for c in np.flatnonzero(blocked[e])]
        for a in range(4):
            st = orc.OracleState(S, bl, pos[e].tolist(), targets[e].tolist(), multi)
            st.move(a)
            now = np.array(st.current_locations, dtype=np.int64).reshape(T, 2)
            assert np.array_equal(now, sc[e, a]), (e, a)
            assert bool((mv[e] >> a) & 1) == (not np.array_equal(now, pos[e].reshape(T, 2))), (e, a)
            assert bool((wn[e] >> a) & 1) == bool(st.is_won()), (e, a)


# (S, T, NT, W, multi): every bitboard size, every wide record length (S 9..16: 5, 5, 6, 6, 7, 7, 8, 8 pair
# words), the generic tile counts, tile-less boards, and never_win batches (multi colour, NT != T)
PIN_SHAPES = [
    (1, 1, 1, 0, True), (2, 2, 2, 1, False), (3, 3, 3, 2, True), (4, 4, 4, 3, False), (5, 1, 1, 4, False),
    (5, 5, 5, 4, True), (6, 4, 4, 8, True), (6, 4, 4, 8, False), (6, 2, 2, 0, False), (7, 6, 6, 10, False),
    (7, 7, 7, 8, True), (8, 8, 8, 12, True), (8, 3, 3, 12, False),
    (9, 2, 2, 20, True), (10, 5, 5, 20, False), (11, 8, 8, 25, True), (12, 8, 8, 30, True), (12, 4, 4, 30, False),
    (13, 6, 6, 30, False), (14, 7, 7, 30, True), (15, 3, 3, 40, True), (16, 8, 8, 40, False), (16, 1, 1, 40, True),
    (6, 12, 12, 8, True), (8, 12, 12, 10, False), (10, 20, 20, 12, True), (12, 32, 32, 30, True), (16, 32, 32, 40, False),
    (6, 0, 0, 8, True), (6, 0, 2, 8, False), (12, 0, 0, 30, False), (12, 0, 3, 30, True),
    (6, 3, 5, 8, True), (12, 4, 2, 30, True), (8, 12, 10, 10, True),
]


@pytest.mark.parametrize("S,T,NT,W,multi", PIN_SHAPES)
def test_expand_is_the_step(ts, S, T, NT, W, multi):
    N = 1001                                                  # ragged: raw_move's last env takes the generic kernel
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=S * 1000 + T * 10 + NT)
    before = env_buffers(env)
    succ, moved, won = env.expand()
    assert_untouched(env, before, "expand")
    assert succ.shape == (N, 4, env.pos_bytes) and moved.shape == won.shape == (N,)
    want = composed(env)
    assert torch.equal(succ, want[0])
    assert torch.equal(moved, want[1])
    assert torch.equal(won, want[2])
    assert torch.equal(moved, env.valid_moves())
    if env.never_win:
        assert not won.any()
    check_oracle_sample(env, arrays, succ, moved, won, multi)


def test_expand_real_levels_are_the_step(ts):
    """The reference's real levels (tests/golden/levels_400.txt), grouped by shape, after random moves."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_400.txt")
    groups = {}
    for p in ts.load_puzzle_file(path):
        groups.setdefault((p.size, len(p.initial_locations), len(p.target_locations), p.multiple_colors), []).append(p)
    checked = 0
    for (S, T, NT, multi), ps in groups.items():
        env = ts.BatchedTilerSliderEnv.from_puzzles(ps)
        g = torch.Generator(device="cuda").manual_seed(S * 10 + T)
        for k in range(3):
            succ, moved, won = env.expand()
            want = composed(env)
            assert torch.equal(succ, want[0]) and torch.equal(moved, want[1]) and torch.equal(won, want[2]), (S, T, multi, k)
            env.raw_move(torch.randint(0, 4, (env.n_envs,), dtype=torch.uint8, device="cuda", generator=g))
        checked += env.n_envs
    assert checked >= 256


def gathered(ts, S, arrays, multi, ids, pos):
    """A batch whose env i is puzzle ids[i] at positions pos[i]."""
    blocked, tiles, targets = arrays
    i = ids.cpu().numpy()
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked[i], tiles[i], targets[i], multi)
    env._pos[: len(i)] = pos
    return env


@pytest.mark.parametrize("S,T,NT,W,multi", [(6, 4, 4, 8, True), (6, 3, 3, 8, False), (12, 8, 8, 30, True),
                                           (10, 20, 20, 12, False), (6, 0, 2, 8, True), (6, 3, 5, 8, True)])
def test_items_equal_the_gathered_puzzles(ts, S, T, NT, W, multi):
    N = 700
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=5 + S + T)
    dense = env.expand()
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(0, N, (2500,), generator=g)            # shuffled, with repeats
    for given in (ids, ids.tolist(), ids.to(torch.int64).cuda(), ids.to(torch.int32).cuda()):
        s1, m1, w1 = env.expand(given)
        assert torch.equal(s1, dense[0][ids.cuda()]) and torch.equal(m1, dense[1][ids.cuda()]) and torch.equal(w1, dense[2][ids.cuda()])
    # level 2 from the level-1 words: the items of puzzle ids[j // 4] at succ[j // 4, j % 4]
    ids2 = ids.repeat_interleave(4)
    pos2 = s1.reshape(-1, env.pos_bytes)
    before = env_buffers(env)
    s2, m2, w2 = env.expand(ids2.cuda().to(torch.int32), pos2)
    assert_untouched(env, before, "level 2")
    ref = gathered(ts, S, arrays, multi, ids2, pos2)
    want = composed(ref)
    assert torch.equal(s2, want[0]) and torch.equal(m2, want[1]) and torch.equal(w2, want[2])
    # explicit positions without ids: item i is env i
    p = s1[:N, 2].contiguous()
    s3, m3, w3 = env.expand(pos=p)
    ref = gathered(ts, S, arrays, multi, torch.arange(N), p)
    want = composed(ref)
    assert torch.equal(s3, want[0]) and torch.equal(m3, want[1]) and torch.equal(w3, want[2])


@pytest.mark.parametrize("S,T,NT,W,multi", [(6, 4, 4, 8, True), (5, 1, 1, 4, False), (12, 8, 8, 30, False),
                                           (15, 5, 5, 40, True), (8, 12, 12, 10, True), (6, 0, 0, 8, False)])
@pytest.mark.parametrize("n", [1, 3, 129, 1000])
@pytest.mark.parametrize("with_pos", [False, True])
def test_guards_and_env_buffers_are_untouched(ts, S, T, NT, W, multi, n, with_pos):
    """Outputs are views into poisoned buffers with GUARD bytes on both sides; ids mix live envs, padding
    envs [n_envs, capacity) and ids past capacity.  Only succ / moved / won of the n items change, the ids
    past capacity read as zeros, and no env buffer -- padding included -- changes."""
    N = 301
    env, _ = build(ts, S, T, NT, W, multi, N, seed=n + S)
    PW, cap = env.pos_bytes, env.capacity
    g = torch.Generator().manual_seed(n)
    ids = torch.randint(0, N, (n,), generator=g, dtype=torch.int32)
    if n > 1:
        ids[1] = N + 2                   # padding env: meaningless result, but only inside the write set
    if n > 2:
        ids[2] = cap + 7                 # past capacity: zeros
    ids[-1] = -1 if n > 3 else ids[-1]
    dense = env.expand()
    pos = None
    if with_pos:
        pos = dense[0][ids.clamp(0, N - 1).long(), ids.abs().long() % 4].contiguous()
    bufs = [torch.full((2 * GUARD + k,), POISON, dtype=torch.uint8, device="cuda") for k in (4 * n * PW, n, n)]
    out = (bufs[0][GUARD:-GUARD].view(n, 4, PW), bufs[1][GUARD:-GUARD], bufs[2][GUARD:-GUARD])
    guards = [torch.cat([b[:GUARD], b[-GUARD:]]).clone() for b in bufs]
    before = env_buffers(env)
    res = env.expand(ids.cuda(), pos, out=out)
    assert all(r is o for r, o in zip(res, out))
    assert_untouched(env, before, "expand")
    for b, gd in zip(bufs, guards):
        assert torch.equal(torch.cat([b[:GUARD], b[-GUARD:]]), gd)
    live = ((ids >= 0) & (ids < N)).cuda()
    outside = ((ids < 0) | (ids >= cap)).cuda()
    assert not out[0][outside].any() and not out[1][outside].any() and not out[2][outside].any()
    if not with_pos:
        li = ids.cuda()[live].long()
        assert torch.equal(out[0][live], dense[0][li]) and torch.equal(out[1][live], dense[1][li]) and torch.equal(out[2][live], dense[2][li])


@pytest.mark.parametrize("S,T,NT,W,multi", [(6, 4, 4, 8, True), (6, 3, 3, 8, False), (12, 6, 6, 30, True),
                                           (10, 20, 20, 12, True), (6, 3, 5, 8, True), (5, 0, 2, 4, False)])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_item_planes_equal_the_gathered_batch(ts, S, T, NT, W, multi, dtype):
    N = 500
    env, arrays = build(ts, S, T, NT, W, multi, N, seed=17 + S + T)
    g = torch.Generator().manual_seed(9)
    ids = torch.randint(0, N, (300,), generator=g)
    succ, _, _ = env.expand(ids)
    ids4, pos4 = ids.repeat_interleave(4), succ.reshape(-1, env.pos_bytes)
    before = env_buffers(env)
    planes = env.observe_planes(dtype=dtype, ids=ids4.cuda().to(torch.int32), pos=pos4)
    assert_untouched(env, before, "planes")
    want = gathered(ts, S, arrays, multi, ids4, pos4).observe_planes(dtype=dtype)
    assert planes.shape == want.shape and torch.equal(planes, want)
    # ids only: each listed env at its current positions; host ids
    p_ids = env.observe_planes(dtype=dtype, ids=ids.tolist())
    assert torch.equal(p_ids, env.observe_planes(dtype=dtype)[ids.cuda()])
    # an id past capacity: an all-zero image; preallocated out
    bad = torch.tensor([0, env.capacity, -5, 1], dtype=torch.int32, device="cuda")
    out = torch.full((4, env.plane_count, S, S), 7, dtype=dtype, device="cuda")
    assert env.observe_planes(out, dtype=dtype, ids=bad) is out
    assert not out[1:3].any()
    assert torch.equal(out[[0, 3]], env.observe_planes(dtype=dtype)[[0, 1]])


def bfs_distance(env, ids, pos, max_depth):
    """Distance to the goal of each item (id, pos), from expand() and torch.unique only: level by level,
    keys (item << 32 | word), a goal seen after a move ends the item's search.  -1: none within max_depth."""
    n = ids.numel()
    dist = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    word = lambda p: p.contiguous().view(torch.int32).reshape(-1).to(torch.int64) & 0xFFFFFFFF   # noqa: E731
    item = torch.arange(n, device="cuda")
    fid, fpos = ids, pos
    visited = (item << 32) | word(pos)
    shifts = torch.arange(4, device="cuda")
    for d in range(1, max_depth + 1):
        succ, moved, won = env.expand(fid, fpos)
        hit = torch.unique(item[won != 0])
        dist[hit[dist[hit] < 0]] = d
        c_item = item.repeat_interleave(4)
        c_moved = ((moved.long()[:, None] >> shifts) & 1).reshape(-1).bool()
        sel = c_moved & (dist[c_item] < 0)
        keys = torch.unique((c_item[sel] << 32) | word(succ.reshape(-1, env.pos_bytes)[sel]))
        keys = keys[~torch.isin(keys, visited)]
        if keys.numel() == 0:
            break
        visited = torch.cat([visited, keys])
        item = keys >> 32
        fid = ids[item]
        fpos = (((keys & 0xFFFFFFFF)[:, None] >> (8 * shifts)) & 0xFF).to(torch.uint8).contiguous()
    return dist


@pytest.mark.parametrize("multi", [True, False])
def test_bfs_from_expand_reproduces_optimal_moves(ts, multi):
    N = 1024
    env = ts.BatchedTilerSliderEnv.solvable(N, 6, 4, 8, multi, min_depth=1, max_depth=8, seed=31)
    d_ref, m_ref = env.optimal_moves()
    assert (d_ref >= 1).all()
    ids = torch.arange(N, dtype=torch.int32, device="cuda")
    dist = bfs_distance(env, ids, env.pos.clone(), 8)
    assert torch.equal(dist.to(torch.int32), d_ref)
    succ, moved, won = env.expand()
    d_succ = bfs_distance(env, ids.repeat_interleave(4), succ.reshape(-1, env.pos_bytes), 9).reshape(N, 4)
    bits = torch.arange(4, device="cuda")
    wins = ((won.long()[:, None] >> bits) & 1).bool()
    on_path = torch.where(dist[:, None] == 1, wins, d_succ == dist[:, None] - 1)
    mask = (on_path.long() << bits).sum(1).to(torch.uint8)
    assert torch.equal(mask, m_ref)


def test_graph_of_step_expand_and_item_planes_replays_like_the_calls(ts):
    S, T, W, N, K = 6, 4, 8, 3000, 4
    kw = dict(seed=21, max_steps=5, auto_reset=True)
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    gen = torch.Generator(device="cuda").manual_seed(7)
    rows = torch.randint(0, 4, (K, a.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    ids = torch.randint(0, N, (1000,), dtype=torch.int32, device="cuda", generator=gen)
    ids4 = ids.repeat_interleave(4)
    PW, C = a.pos_bytes, a.plane_count

    def calls(env, k, out=None):
        env.step(rows[k])
        o = None if out is None else out[0]
        succ, moved, won = env.expand(ids, out=o)
        planes = env.observe_planes(None if out is None else out[1], dtype=torch.bfloat16, ids=ids4, pos=succ.reshape(-1, PW))
        return succ, moved, won, planes

    want = [[t.clone() for t in calls(b, k)] for k in range(K)]
    outs = [((torch.empty(1000, 4, PW, dtype=torch.uint8, device="cuda"), torch.empty(1000, dtype=torch.uint8, device="cuda"),
              torch.empty(1000, dtype=torch.uint8, device="cuda")),
             torch.empty(4000, C, S, S, dtype=torch.bfloat16, device="cuda")) for _ in range(K)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                     # warm-up outside the capture
        calls(a, 0, outs[0])
    torch.cuda.current_stream().wait_stream(side)
    a.reset()
    for o in outs:
        for t in o[0]:
            t.fill_(0xEE)
        o[1].fill_(3)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for k in range(K):
            calls(a, k, outs[k])
    graph.replay()
    torch.cuda.synchronize()
    for k in range(K):
        got = list(outs[k][0]) + [outs[k][1]]
        for g_, w_ in zip(got, want[k]):
            assert torch.equal(g_, w_), k
