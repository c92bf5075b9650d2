"""GPU parity tests: the CUDA path (through the C-ABI, via BatchedTilerSliderEnv) against the
CPU oracle and the reference-generated golden fixtures.  Integer / byte work: the bar is
bit-exact equality everywhere; the float32 observation holds small integers, so it is
compared with exact equality too (no tolerance).
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.helpers import random_puzzles

pytestmark = pytest.mark.gpu

F_DONE, F_WON, F_INVALID, F_TIMEOUT, F_STALE = 1, 2, 4, 8, 16


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def run_gpu(ts, S, multi, blocked, tiles, targets, actions, max_steps, auto_reset):
    """Drive the batch env with the action matrix; return post-move/pre-reset positions,
    flags, pre-increment counts and rewards per step, like the oracle's rollout."""
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=max_steps,
                                               auto_reset=auto_reset, track_terminal=True)
    K, N = actions.shape
    T = tiles.shape[1]
    acts = torch.as_tensor(actions).cuda()
    pos = np.zeros((K, N, T, 2), np.int16)
    flags = np.zeros((K, N), np.uint8)
    count = np.zeros((K, N), np.int32)
    reward = np.zeros((K, N), np.float32)
    for k in range(K):
        before = env.step_count.to(torch.int32).clone()
        state, r, d = env.step(acts[k])
        f = env.flags
        assert torch.equal(d, (f & F_DONE) != 0)
        post = env.positions()
        if auto_reset:
            term = env.positions(env.terminal_pos)
            post = torch.where(d[:, None, None], term, post)
        pos[k] = post.cpu().numpy()
        flags[k] = f.cpu().numpy()
        count[k] = before.cpu().numpy()
        reward[k] = r.cpu().numpy()
    return dict(pos=pos, flags=flags, count=count, reward=reward,
                final_pos=env.positions().cpu().numpy().astype(np.int16),
                final_count=env.step_count.to(torch.int32).cpu().numpy())


def assert_same(got, want, tag=""):
    for key in ("pos", "flags", "count", "reward", "final_pos", "final_count"):
        if key in want:
            assert np.array_equal(got[key], want[key]), f"{tag}: {key} differs"


def test_golden_rollouts(ts, golden_rollouts):
    """Reference-recorded rollouts (tests/golden/rollouts.npz) replayed on the GPU."""
    n = 0
    for rec in golden_rollouts:
        if not ts.lib().ts_supported(rec["S"], rec["T"]):
            continue
        got = run_gpu(ts, rec["S"], rec["multi"], rec["blocked"], rec["tiles"], rec["targets"], rec["actions"],
                      rec["max_steps"], True)
        assert np.array_equal(got["pos"], rec["pos"]), rec["tag"]
        assert np.array_equal(got["flags"], rec["flags"]), rec["tag"]
        assert np.array_equal(got["count"], rec["count"]), rec["tag"]
        n += rec["flags"].size
    assert n > 10000


SHAPES = [  # S, T, W, multi, N, K, max_steps
    (5, 1, 5, False, 8192, 128, 100),      # config 2
    (6, 4, 8, True, 8192, 128, 100),       # config 3
    (6, 4, 8, False, 4096, 96, 100),
    (4, 2, 2, True, 4096, 64, 7),
    (3, 3, 1, False, 2048, 64, 5),
    (2, 2, 0, True, 1024, 32, 3),
    (1, 1, 0, False, 256, 8, 2),
    (5, 4, 3, True, 4096, 64, 300),        # int32 step counter
    (6, 8, 6, True, 4096, 64, 100),
    (6, 3, 0, False, 2048, 64, 100),
    (7, 5, 10, True, 4096, 64, 50),
    (8, 8, 12, True, 4096, 64, 100),
    (8, 6, 20, False, 2048, 64, 13),
    (7, 7, 4, False, 2048, 64, 100),
    (12, 8, 36, True, 8192, 128, 100),     # config 4 (wide boards)
    (12, 8, 36, False, 4096, 64, 100),
    (9, 4, 20, True, 2048, 64, 9),
    (10, 3, 0, False, 2048, 64, 100),
    (16, 8, 60, True, 2048, 64, 300),
    (16, 5, 100, False, 2048, 64, 100),
    (13, 1, 40, False, 2048, 64, 100),
    (11, 6, 25, True, 2048, 64, 100),      # wide wall records: 9,10 -> 5 pair words, 11,12 -> 6, 13,14 -> 7, 15,16 -> 8
    (14, 8, 50, False, 2048, 64, 100),     # widest board with edge sentinels inside the 16-bit line
    (14, 2, 0, True, 2048, 48, 20),
    (15, 7, 70, True, 2048, 64, 100),      # plain lines, like 16
    (10, 8, 30, True, 2048, 64, 100),
    (5, 2, 3, True, 1021, 300, 255),       # widest 1-byte step counter; N not a multiple of 4
    (5, 2, 3, False, 1023, 300, 256),      # first 4-byte step counter
    (6, 4, 8, True, 777, 40, 1),           # every step times out
    (10, 20, 12, False, 1024, 48, 100),    # more than 8 tiles: the per-env generic kernels (the reference's own 20-tile board shape)
    (16, 32, 50, True, 512, 40, 300),
    (6, 12, 6, True, 1021, 64, 20),
    (8, 9, 10, False, 515, 48, 100),
    (12, 16, 20, True, 512, 40, 100),
    (3, 9, 0, True, 256, 16, 9),           # a full board: nothing can ever move
]


@pytest.mark.parametrize("S,T,W,multi,N,K,max_steps", SHAPES)
@pytest.mark.parametrize("auto_reset", [True, False])
def test_random_vs_oracle(ts, S, T, W, multi, N, K, max_steps, auto_reset):
    """>= 1e6 checked env-steps for the bench shapes: positions per tile, is_won,
    invalid_move, timeout, done, stale, pre-increment step_count, reward."""
    if not ts.lib().ts_supported(S, T):
        pytest.skip("shape not built")
    rng = np.random.default_rng(1000 * S + 10 * T + W + (7 if multi else 0))
    blocked, tiles, targets = random_puzzles(rng, N, S, T, W) if W + 2 * T <= S * S else crowded(rng, N, S, T, W)
    actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
    want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=auto_reset)
    got = run_gpu(ts, S, multi, blocked, tiles, targets, actions, max_steps, auto_reset)
    assert_same(got, want, f"S{S}T{T}")


def crowded(rng, N, S, T, W):
    """Boards too full for disjoint tiles and targets: targets drawn independently."""
    blocked, tiles, _ = random_puzzles(rng, N, S, T, W) if W + T <= S * S else (None, None, None)
    _, targets, _ = random_puzzles(rng, N, S, T, 0)
    return blocked, tiles, targets


def test_targets_under_tiles_and_crowded(ts):
    rng = np.random.default_rng(5)
    for S, T, W, multi in [(1, 1, 0, False), (2, 2, 1, True), (3, 8, 0, False), (3, 8, 1, True), (4, 8, 8, False)]:
        N, K = 512, 24
        blocked, tiles, targets = crowded(rng, N, S, T, W)
        actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
        want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=9, auto_reset=True)
        got = run_gpu(ts, S, multi, blocked, tiles, targets, actions, 9, True)
        assert_same(got, want, f"crowded S{S}T{T}")


def test_set_goal_with_duplicate_and_missing_targets(ts):
    """Single colour is set equality (state.py:185-186): duplicate targets collapse, a target
    count different from the tile count can never (or only by collapse) be met."""
    S = 3
    blocked = np.zeros((2, 9), np.uint8)
    tiles = np.array([[[0, 0]], [[0, 0]]], np.uint8)
    targets = np.array([[[0, 2], [0, 2]], [[0, 2], [2, 2]]], np.uint8)
    acts = np.array([[3, 3], [1, 1]], np.uint8)
    want = orc.rollout(S, False, blocked, tiles, targets, acts)
    got = run_gpu(ts, S, False, blocked, tiles, targets, acts, 100, False)
    assert_same(got, want)
    assert want["flags"][0, 0] & F_WON and not (want["flags"][:, 1] & F_WON).any()


DEGENERATE = [  # S, T, NT, W, multi, max_steps
    (5, 0, 0, 3, False, 100), (5, 0, 2, 3, False, 6), (5, 0, 0, 3, True, 100), (5, 0, 3, 0, True, 5),
    (6, 3, 2, 6, True, 9), (6, 2, 4, 6, True, 100), (4, 1, 0, 2, True, 7), (6, 2, 3, 6, False, 100), (6, 3, 1, 4, False, 12),
    (12, 0, 0, 20, False, 100), (12, 0, 2, 20, True, 4), (12, 3, 2, 30, True, 100), (12, 2, 5, 30, True, 8),
    (12, 3, 2, 30, False, 100), (16, 2, 3, 40, False, 10), (9, 1, 1, 10, False, 100),
]


@pytest.mark.parametrize("S,T,NT,W,multi,max_steps", DEGENERATE)
@pytest.mark.parametrize("auto_reset", [True, False])
def test_degenerate_batches_vs_oracle(ts, S, T, NT, W, multi, max_steps, auto_reset):
    """Boards without tiles (nothing moves; won iff there are no targets, state.py:183-186) and
    boards whose target count differs from the tile count (ordered goal: never won,
    state.py:183-184; set goal: duplicates collapse, state.py:185-186): every field of the step,
    the observation, the valid-move mask and the goal check against the oracle."""
    rng = np.random.default_rng(77 * S + 5 * T + NT + (3 if multi else 0))
    N, K = 515, 24
    perm = np.argsort(rng.random((N, S * S)), axis=1)
    blocked = np.zeros((N, S * S), np.uint8)
    np.put_along_axis(blocked, perm[:, :W], 1, axis=1)
    tc = perm[:, W:W + T]
    tiles = np.stack([tc // S, tc % S], -1).astype(np.uint8)
    gc = perm[:, W + T:W + T + NT].copy()
    if NT >= 2:
        gc[::3, 1] = gc[::3, 0]                              # every third board has a duplicate target
    if NT >= 1 and T >= 1:
        gc[1::4, 0] = tc[1::4, 0]                             # some targets under tiles
    targets = np.stack([gc // S, gc % S], -1).astype(np.uint8)
    actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
    want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=auto_reset)
    got = run_gpu(ts, S, multi, blocked, tiles, targets, actions, max_steps, auto_reset)
    assert_same(got, want, f"degenerate S{S} T{T} NT{NT}")
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=1000)
    obs, vm, won = env.observe().cpu().numpy(), env.valid_moves().cpu().numpy(), env.goal_check().cpu().numpy()
    for e in range(0, N, 5):
        b = [(c // S, c % S) for c in np.flatnonzero(blocked[e])]
        st = orc.OracleState(S, b, tiles[e].tolist(), targets[e].tolist(), multi)
        assert np.array_equal(obs[e], st.get_state_array()), e
        assert [d for d in range(4) if vm[e] >> d & 1] == st.valid_moves()
        assert bool(won[e]) == st.is_won()
    assert tuple(env.target_positions().shape) == ((N, NT, 2) if env.goal_mode == ts.GOAL_ORDERED else (N, S * S))


def test_limits_are_value_errors_not_fallbacks(ts):
    """More than 32 tiles / boards above 16x16 / more than 32 ordered targets on a mismatched board
    are outside the kernels' domain: ValueError, never a host computation."""
    blocked = np.zeros((1, 9), np.uint8)
    blocked = np.zeros((1, 49), np.uint8)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.from_arrays(7, blocked, np.zeros((1, 33, 2), np.uint8), np.zeros((1, 33, 2), np.uint8), True)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.from_arrays(7, blocked, np.zeros((1, 1, 2), np.uint8), np.zeros((1, 33, 2), np.uint8), True)
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv(17, 1, 4)


def test_sub_range_steps_touch_nothing_outside_the_range(ts):
    """The capacity contract of include/tiler_slider.h: ts_step reads and writes exactly
    [first_env, first_env + n_envs).  A batch of 3,001 envs (capacity 3,072) has its padding
    poisoned, and is stepped (a) whole, (b) through the ragged sub-range [0, 510) or [0, 3) only --
    the envs outside the range, padding included, must stay bit for bit as they were, the envs
    inside must match the oracle -- and (c) through the consecutive sub-ranges [0, 128),
    [128, 512), [512, 2048) and the ragged [2048, 3001): every buffer must equal the whole-batch
    step bit for bit, so ranges that start at a non-zero first_env step exactly their own envs.
    Covers the bitboard kernels (4-env groups + the per-env kernel for the ragged end), the wide
    kernel, and the generic kernels (9..32 tiles on narrow and wide boards, and boards without
    tiles)."""
    import ctypes as C
    for S, T, W, multi, auto_reset in [(6, 4, 8, True, True), (6, 4, 8, False, False), (5, 1, 5, False, True),
                                       (8, 6, 12, True, False), (12, 8, 36, True, True), (3, 2, 1, True, True),
                                       (4, 2, 2, True, True), (8, 8, 12, True, True), (6, 3, 4, True, False),
                                       (6, 12, 6, True, True), (10, 20, 12, False, False), (5, 0, 3, False, True),
                                       (9, 4, 20, False, False), (16, 8, 60, True, True)]:
        N, K, max_steps = 3001, 10, 6
        rng = np.random.default_rng(S * 100 + T)
        blocked, tiles, targets = random_puzzles(rng, N, S, T, W)
        actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
        want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=auto_reset)
        whole = []                            # every buffer after each whole-batch step
        for ends in ((N,), (510,), (3,), (128, 512, 2048, N)):
            env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=max_steps,
                                                       auto_reset=auto_reset, track_terminal=True)
            cap, n_range = env.capacity, ends[-1]
            bufs = {k: getattr(env, k) for k in ("_pos", "_count", "_reward", "_done", "_flags", "_terminal")}
            poison = {"_pos": 0xA5, "_count": 0x5A, "_reward": -123.5, "_done": 0x77, "_flags": 0, "_terminal": 0xC3}
            for k, buf in bufs.items():       # the padding envs (flags stay 0: a set DONE bit would mean "frozen")
                buf[N:] = poison[k]
            acts = torch.zeros(K, cap, dtype=torch.uint8, device="cuda")
            acts[:, :N] = torch.as_tensor(actions).cuda()
            for k in range(K):
                before = {name: buf.clone() for name, buf in bufs.items()}
                a = env._step_args(acts[k].data_ptr())
                for lo, hi in zip((0,) + ends[:-1], ends):
                    a.first_env, a.n_envs = lo, hi - lo
                    assert ts.lib().ts_step(C.byref(a), torch.cuda.current_stream().cuda_stream) == 0
                for name, buf in bufs.items():
                    assert torch.equal(buf[n_range:], before[name][n_range:]), (S, T, name, ends, k)
                if ends == (N,):
                    whole.append({name: buf.clone() for name, buf in bufs.items()})
                elif n_range == N:
                    for name, buf in bufs.items():
                        assert torch.equal(buf, whole[k][name]), (S, T, name, ends, k)
                d = env._done[:n_range].bool()
                post = env.positions(env._pos[:n_range])
                if auto_reset:
                    post = torch.where(d[:, None, None], env.positions(env._terminal[:n_range]), post)
                assert np.array_equal(post.cpu().numpy(), want["pos"][k][:n_range])
                assert np.array_equal(env._flags[:n_range].cpu().numpy(), want["flags"][k][:n_range])
                assert np.array_equal(env._reward[:n_range].cpu().numpy(), want["reward"][k][:n_range])


def test_fast_path_without_status_byte(ts):
    """track_flags=False (auto-reset only): the step stores state, reward and done but no status
    byte -- one byte less per env-step.  Same positions / reward / done as the tracked batch and
    the oracle; is_won() comes from the reward."""
    for S, T, W, multi in [(6, 4, 8, True), (5, 1, 5, False), (12, 8, 36, True), (8, 3, 10, False)]:
        N, K = 4099, 40
        kw = dict(seed=31, max_steps=9, auto_reset=True, track_terminal=True)
        a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, **kw)
        b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, track_flags=False, **kw)
        assert not b.track_flags and b._step_args(b._actions.data_ptr()).d_flags is None
        g = torch.Generator(device="cuda").manual_seed(8)
        acts = torch.randint(0, 4, (K, a.capacity), dtype=torch.uint8, device="cuda", generator=g)
        for k in range(K):
            a.step(acts[k])
            b.step(acts[k])
            assert torch.equal(a.pos, b.pos) and torch.equal(a.reward, b.reward) and torch.equal(a.done, b.done)
            assert torch.equal(a.terminal_pos[a.done], b.terminal_pos[b.done]) and torch.equal(a.step_count, b.step_count)
            assert torch.equal(a.is_won(), b.is_won())
        with pytest.raises(RuntimeError):
            b.flags
    # without auto-reset the done state lives in the status byte: the request is ignored
    c = ts.BatchedTilerSliderEnv.synthetic(64, 5, 1, 5, False, auto_reset=False, track_flags=False)
    assert c.track_flags


def test_one_byte_counter_boundary(ts):
    """max_steps 254 / 255: the SWAR counter of a frozen env must not carry into its neighbour
    (255 without auto-reset therefore uses the 4-byte counter)."""
    for max_steps, auto_reset in [(254, False), (255, False), (255, True), (254, True)]:
        S, T, W, N, K = 4, 1, 2, 64, 300
        rng = np.random.default_rng(max_steps)
        blocked, tiles, targets = random_puzzles(rng, N, S, T, W)
        targets[:] = tiles                     # a tile starts on its target: a win needs a move away and back
        actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
        want = orc.rollout(S, False, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=auto_reset)
        got = run_gpu(ts, S, False, blocked, tiles, targets, actions, max_steps, auto_reset)
        assert_same(got, want, f"max_steps {max_steps}")
    e = ts.BatchedTilerSliderEnv.synthetic(8, 4, 1, 2, False, max_steps=255, auto_reset=False)
    assert e.count_bytes == 4
    assert ts.BatchedTilerSliderEnv.synthetic(8, 4, 1, 2, False, max_steps=255, auto_reset=True).count_bytes == 1


def test_observation_valid_moves_goal(ts):
    rng = np.random.default_rng(11)
    for S, T, W, multi in [(5, 1, 5, False), (6, 4, 8, True), (6, 4, 8, False), (4, 2, 2, True), (8, 8, 10, True),
                           (12, 8, 36, True), (12, 8, 36, False), (16, 3, 50, False), (9, 5, 20, False),
                           (11, 2, 30, True), (14, 8, 40, False), (15, 4, 60, True), (10, 20, 12, False), (12, 16, 30, True),
                           (6, 9, 5, True)]:
        N, K = 256, 12
        blocked, tiles, targets = random_puzzles(rng, N, S, T, W)
        actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
        env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=1000)
        states = []
        for e in range(N):
            b = [(c // S, c % S) for c in np.flatnonzero(blocked[e])]
            states.append(orc.OracleState(S, b, tiles[e].tolist(), targets[e].tolist(), multi))
        for k in range(K + 1):
            obs = env.observe().cpu().numpy()
            vm = env.valid_moves().cpu().numpy()
            won = env.goal_check().cpu().numpy()
            for e in range(N):
                assert np.array_equal(obs[e], states[e].get_state_array())
                assert [d for d in range(4) if vm[e] >> d & 1] == states[e].valid_moves()
                assert bool(won[e]) == states[e].is_won()
            if k < K:
                fl = env.raw_move(torch.as_tensor(actions[k]).cuda()).cpu().numpy()
                for e in range(N):
                    w = states[e].move(int(actions[k, e]))
                    assert bool(fl[e] & F_WON) == w


def test_synth_well_formed_and_shard_invariant(ts):
    S, T, W = 6, 4, 8
    full = ts.BatchedTilerSliderEnv.synthetic(4096, S, T, W, True, seed=77)
    blocked = full.blocked_cells().cpu().numpy()
    pos = full.positions().cpu().numpy().astype(int)
    tg = full.target_positions().cpu().numpy().astype(int)
    assert (blocked.sum(1) == W).all()
    cells = pos[..., 0] * S + pos[..., 1]
    tcells = tg[..., 0] * S + tg[..., 1]
    for e in range(0, 4096, 37):
        occupied = set(np.flatnonzero(blocked[e])) | set(cells[e]) | set(tcells[e])
        assert len(occupied) == W + 2 * T
    # the same global env index gives the same puzzle whatever the shard
    part = ts.BatchedTilerSliderEnv.synthetic(1024, S, T, W, True, seed=77, env_index_base=2048)
    assert torch.equal(part.pos, full.pos[2048:3072])
    assert torch.equal(part.blocked_cells(), full.blocked_cells()[2048:3072])
    other = ts.BatchedTilerSliderEnv.synthetic(1024, S, T, W, True, seed=78)
    assert not torch.equal(other.pos, full.pos[:1024])
    # set mode: targets as a bitboard of exactly T cells, disjoint from tiles and walls
    single = ts.BatchedTilerSliderEnv.synthetic(512, S, T, W, False, seed=3)
    tb = single.target_positions().cpu().numpy()
    assert (tb.sum(1) == T).all() and not (tb & single.blocked_cells().cpu().numpy()).any()


def test_synthetic_rollout_vs_oracle(ts):
    """The bench workload itself: device-generated puzzles decoded to the host and replayed by
    the oracle (config 2 and config 3 shapes)."""
    for S, T, W, multi in [(5, 1, 5, False), (6, 4, 8, True), (6, 4, 8, False), (12, 8, 36, True)]:
        N, K = 8192, 128
        env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=1002, max_steps=100, auto_reset=True,
                                                 track_terminal=True)
        blocked = env.blocked_cells().cpu().numpy().astype(np.uint8)
        tiles = env.positions().cpu().numpy()
        if env.goal_mode == ts.GOAL_ORDERED:
            targets = env.target_positions().cpu().numpy()
        else:
            tgt_cells = env.target_positions().cpu().numpy()
            targets = np.stack([np.flatnonzero(r) for r in tgt_cells])
            targets = np.stack([targets // S, targets % S], -1).astype(np.uint8)
        g = torch.Generator(device="cuda").manual_seed(2002)
        actions = torch.randint(0, 4, (K, N), dtype=torch.uint8, device="cuda", generator=g)
        want = orc.rollout(S, multi, blocked, tiles, targets, actions.cpu().numpy(), max_steps=100, auto_reset=True)
        for k in range(K):
            _, r, d = env.step(actions[k])
            post = torch.where(d[:, None, None], env.positions(env.terminal_pos), env.positions())
            assert np.array_equal(post.cpu().numpy(), want["pos"][k])
            assert np.array_equal(env.flags.cpu().numpy(), want["flags"][k])
            assert np.array_equal(r.cpu().numpy(), want["reward"][k])


def test_full_size_properties(ts):
    """BASELINE config 3 at its full size (16,777,216 envs, 6x6, 4 coloured tiles, 8 walls):
    size-independent properties of the move --
      * well-formedness is preserved: tiles stay in bounds, distinct, never on a wall;
      * idempotence: repeating the same action moves nothing (every env reports invalid_move);
      * reversal symmetry: after UP, DOWN brings every tile to the cell a single DOWN would not
        pass -- checked as 'DOWN after UP == DOWN after (UP, DOWN, UP, DOWN)' (a slide to the far
        side forgets the history along that axis);
      * determinism: two independently built envs end with the same checksum;
    plus the first 4,096 envs against the oracle."""
    S, T, W, N = 6, 4, 8, 16_777_216
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=1002, max_steps=255, auto_reset=False)
    walls = env.blocked_cells()

    def check_well_formed():
        p = env.positions().to(torch.int64)
        cell = p[..., 0] * S + p[..., 1]
        assert int(p.max()) < S and int(p.min()) >= 0
        assert not bool(walls.gather(1, cell).any())
        srt = cell.sort(dim=1).values
        assert bool((srt[:, 1:] != srt[:, :-1]).all())

    def act(d):
        return torch.full((env.capacity,), d, dtype=torch.uint8, device="cuda")

    gen = torch.Generator(device="cuda").manual_seed(7)
    n_chk = 4096
    blocked = walls[:n_chk].cpu().numpy().astype(np.uint8)
    tiles0 = env.positions()[:n_chk].cpu().numpy()
    targets = env.target_positions()[:n_chk].cpu().numpy()
    rand_actions = torch.randint(0, 4, (6, env.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    for k in range(6):
        env.step(rand_actions[k])
    check_well_formed()
    want = orc.rollout(S, True, blocked, tiles0, targets, rand_actions[:, :n_chk].cpu().numpy(), max_steps=255)
    assert np.array_equal(env.positions()[:n_chk].cpu().numpy(), want["final_pos"])
    live = (env.flags & F_DONE) == 0
    for d in range(4):
        env.step(act(d))
        first = env.pos.clone()
        env.step(act(d))                                   # same action again: nothing may move
        still_live = live & ((env.flags & F_STALE) == 0)
        assert torch.equal(env.pos, first)
        assert bool(((env.flags & F_INVALID) != 0)[still_live].all())
        live = (env.flags & F_DONE) == 0
    check_well_formed()
    env.reset()
    env.step(act(0)); env.step(act(1))
    once = env.pos.clone()
    env.step(act(0)); env.step(act(1))
    assert torch.equal(env.pos[live_after_reset(env)], once[live_after_reset(env)])
    checksum = int((env.pos.to(torch.int64) * torch.arange(1, 5, device="cuda")).sum())
    env2 = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=1002, max_steps=255, auto_reset=False)
    for d in (0, 1, 0, 1):
        env2.step(act(d))
    assert int((env2.pos.to(torch.int64) * torch.arange(1, 5, device="cuda")).sum()) == checksum


def live_after_reset(env):
    return (env.flags & (F_DONE | F_STALE)) == 0


def test_real_levels_step_parity(ts):
    """The reference's 400 real levels (tests/golden/levels_400.txt, decoded by its own image
    parser): 96 random steps each with auto-reset and max_steps 25, every field against the oracle."""
    import os
    puzzles = ts.load_puzzle_file(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "levels_400.txt"))
    groups = {}
    for p in puzzles:
        groups.setdefault((p.size, len(p.initial_locations), p.multiple_colors), []).append(p)
    rng = np.random.default_rng(400)
    total = 0
    for (S, T, multi), ps in groups.items():
        n, K = len(ps), 96
        blocked = np.zeros((n, S * S), np.uint8)
        for i, p in enumerate(ps):
            for r, c in p.blocked_locations:
                blocked[i, r * S + c] = 1
        tiles = np.array([p.initial_locations for p in ps], np.uint8).reshape(n, T, 2)
        targets = np.array([p.target_locations for p in ps], np.uint8).reshape(n, T, 2)
        actions = rng.integers(0, 4, size=(K, n), dtype=np.uint8)
        want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=25, auto_reset=True)
        env = ts.BatchedTilerSliderEnv.from_puzzles(ps, max_steps=25, auto_reset=True, track_terminal=True)
        for k in range(K):
            _, r, d = env.step(torch.as_tensor(actions[k]).cuda())
            post = torch.where(d[:, None, None], env.positions(env.terminal_pos), env.positions())
            assert np.array_equal(post.cpu().numpy(), want["pos"][k])
            assert np.array_equal(env.flags.cpu().numpy(), want["flags"][k])
            assert np.array_equal(r.cpu().numpy(), want["reward"][k])
        total += n * K
    assert total == 400 * 96


def test_side_stream_and_unaligned_action_views(ts):
    """Calls follow torch's current stream, and an action tensor that cannot be handed to the
    kernel as it is (odd offset view, int64 dtype, host tensor) is staged, not rejected."""
    S, T, W, N, K = 6, 4, 8, 5000, 12
    ref = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=21, auto_reset=True)
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=21, auto_reset=True)
    g = torch.Generator(device="cuda").manual_seed(5)
    acts = torch.randint(0, 4, (K, ref.capacity), dtype=torch.uint8, device="cuda", generator=g)
    pad = torch.zeros(N + 7, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    for k in range(K):
        ref.step(acts[k])
        kind = k % 3
        if kind == 0:
            pad[3:3 + N] = acts[k, :N]
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                env.step(pad[3:3 + N])                       # misaligned device view, side stream
            torch.cuda.current_stream().wait_stream(side)
        elif kind == 1:
            env.step(acts[k, :N].to(torch.int64))            # wrong dtype
        else:
            env.step(acts[k, :N].cpu().numpy())              # host array
        assert torch.equal(env.pos, ref.pos) and torch.equal(env.flags, ref.flags)
        assert torch.equal(env.reward, ref.reward) and torch.equal(env.step_count, ref.step_count)


def test_cuda_graph_replay_matches_eager(ts):
    S, T, W, N, R = 5, 1, 5, 10_000, 8
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, False, seed=4, auto_reset=True)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, False, seed=4, auto_reset=True)
    rows = torch.randint(0, 4, (R, a.capacity), dtype=torch.uint8, device="cuda")
    graph = a.capture_steps(rows)
    a.reset()
    for _ in range(3):
        graph.replay()
        for k in range(R):
            b.step(rows[k])
        torch.cuda.synchronize()
        assert torch.equal(a.pos, b.pos) and torch.equal(a.step_count, b.step_count)
        assert torch.equal(a.reward, b.reward) and torch.equal(a.flags, b.flags)


def test_step_host_matches_step(ts):
    S, T, W, N = 6, 4, 8, 50_000
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=9, auto_reset=True)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=9, auto_reset=True)
    h_act = torch.empty(N, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    h_done = torch.empty(N, dtype=torch.uint8).pin_memory()
    rng = np.random.default_rng(1)
    for k in range(20):
        h_act.copy_(torch.from_numpy(rng.integers(0, 4, N, dtype=np.uint8)))
        _, r, d = a.step(h_act.cuda())
        b.step_host(h_act, h_rew, h_done, chunk_envs=8192)
        assert torch.equal(a.pos, b.pos)
        assert torch.equal(r.cpu(), h_rew) and torch.equal(d.cpu(), h_done.bool())
    c = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, seed=9, auto_reset=True)
    h_flags = torch.empty(N, dtype=torch.uint8).pin_memory()
    lut = torch.tensor([c.rewards[1], 0, c.rewards[0], 0, c.rewards[2], 0, c.rewards[0], 0], dtype=torch.float32)
    rng = np.random.default_rng(1)
    for k in range(20):
        h_act.copy_(torch.from_numpy(rng.integers(0, 4, N, dtype=np.uint8)))
        c.step_host(h_act, h_flags=h_flags, chunk_envs=8192)
    # after the same 20 action vectors the compact path is in the same state as the others, and
    # its status byte reproduces done and reward
    assert torch.equal(c.pos, a.pos)
    assert torch.equal((h_flags & 1).bool(), h_done.bool())
    assert torch.equal(lut[((h_flags >> 1) & 3).long() * 2], h_rew)


def test_argument_errors(ts):
    import ctypes as C
    from tiler_slider_b200 import _lib
    env = ts.BatchedTilerSliderEnv.synthetic(256, 5, 1, 5, False)
    a = env._step_args(env._actions.data_ptr())
    a.capacity = 100
    assert ts.lib().ts_step(C.byref(a), None) == -3
    a = env._step_args(env._actions.data_ptr() + 1)
    assert ts.lib().ts_step(C.byref(a), None) == -5
    a = env._step_args(env._actions.data_ptr())
    a.size = 17
    assert ts.lib().ts_step(C.byref(a), None) == -1
    assert b"size" in ts.lib().ts_last_error_string()
    with pytest.raises(ValueError):
        env.step(torch.zeros(3, dtype=torch.uint8))
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.from_puzzles([ts.Puzzle(3, [(0, 0)], [(0, 0)], [(1, 1)])])
    with pytest.raises(ValueError):
        ts.BatchedTilerSliderEnv.from_puzzles([ts.Puzzle(3, [], [(0, 0), (0, 0)], [(1, 1), (2, 2)])])


@pytest.mark.parametrize("S,T,W,multi,N,seed", [(5, 1, 5, False, 1_048_576, 1001), (12, 8, 36, True, 4_194_304, 1003)])
def test_baseline_configs_at_their_literal_sizes(ts, S, T, W, multi, N, seed):
    """BASELINE configs 2 and 4 at their full env counts (1,048,576 / 4,194,304): the first and the
    last 4,096 envs against the oracle over 24 steps, and size-independent properties over the
    whole batch -- tiles stay on distinct open cells, repeating an action moves nothing, and the
    fast path (no status byte) ends in the same state."""
    K, n_chk = 24, 4096
    kw = dict(seed=seed, max_steps=100, auto_reset=True, track_terminal=True)
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, **kw)
    fast = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, track_flags=False, **kw)
    walls = env.blocked_cells()
    g = torch.Generator(device="cuda").manual_seed(seed + 1000)
    actions = torch.randint(0, 4, (K, env.capacity), dtype=torch.uint8, device="cuda", generator=g)
    want = {}
    for name, sl in (("head", slice(0, n_chk)), ("tail", slice(N - n_chk, N))):
        blocked = walls[sl].cpu().numpy().astype(np.uint8)
        tiles = env.positions()[sl].cpu().numpy()
        if env.goal_mode == ts.GOAL_ORDERED:
            targets = env.target_positions()[sl].cpu().numpy()
        else:
            cells = np.stack([np.flatnonzero(r) for r in env.target_positions()[sl].cpu().numpy()])
            targets = np.stack([cells // S, cells % S], -1).astype(np.uint8)
        want[name] = (sl, orc.rollout(S, multi, blocked, tiles, targets, actions[:, sl].cpu().numpy(), max_steps=100, auto_reset=True))
    for k in range(K):
        _, r, d = env.step(actions[k])
        fast.step(actions[k])
        for sl, w in want.values():
            post = torch.where(d[sl][:, None, None], env.positions(env.terminal_pos[sl]), env.positions(env.pos[sl]))
            assert np.array_equal(post.cpu().numpy(), w["pos"][k])
            assert np.array_equal(env.flags[sl].cpu().numpy(), w["flags"][k]) and np.array_equal(r[sl].cpu().numpy(), w["reward"][k])
    assert torch.equal(env.pos, fast.pos) and torch.equal(env.reward, fast.reward) and torch.equal(env.done, fast.done)
    p = env.positions().to(torch.int64)
    cell = p[..., 0] * S + p[..., 1]
    assert int(p.max()) < S and not bool(walls.gather(1, cell).any())
    if T > 1:
        srt = cell.sort(dim=1).values
        assert bool((srt[:, 1:] != srt[:, :-1]).all())
    same = torch.full((env.capacity,), 2, dtype=torch.uint8, device="cuda")
    env.step(same)
    before = env.pos.clone()
    live = ~env.done
    env.step(same)
    assert torch.equal(env.pos[live & ~env.done], before[live & ~env.done])
    assert bool(((env.flags & F_INVALID) != 0)[live].all())


def test_fuzz_random_shapes_vs_oracle(ts):
    """Seeded fuzz over the whole shape space the kernels cover: board size 1..16, 0..32 tiles, target
    counts equal to / different from the tile count, duplicate targets, both colour modes, auto-reset
    on / off, step limits around the counter-width boundaries, batch sizes that are not multiples of
    4 -- every field of every step against the oracle."""
    rng = np.random.default_rng(20261018)
    n_cases = 0
    for case in range(70):
        S = int(rng.integers(1, 17))
        T = int(rng.integers(0, min(8, S * S) + 1)) if rng.random() < 0.75 else int(rng.integers(9, 33)) if S * S >= 32 else int(rng.integers(0, S * S + 1))
        W = int(rng.integers(0, max(1, (S * S - T) // 2) + 1)) if S * S - T > 0 else 0
        multi = bool(rng.integers(0, 2))
        NT = T if rng.random() < 0.6 else int(rng.integers(0, min(32, S * S) + 1))
        auto_reset = bool(rng.integers(0, 2))
        max_steps = int(rng.choice([1, 2, 5, 17, 100, 254, 255, 256, 300]))
        N, K = int(rng.integers(1, 700)), int(rng.integers(4, 40))
        perm = np.argsort(rng.random((N, S * S)), axis=1)
        blocked = np.zeros((N, S * S), np.uint8)
        np.put_along_axis(blocked, perm[:, :W], 1, axis=1)
        tc = perm[:, W:W + T]
        tiles = np.stack([tc // S, tc % S], -1).astype(np.uint8)
        gc = rng.integers(0, S * S, size=(N, NT))                       # targets anywhere: under tiles, on walls, duplicated
        targets = np.stack([gc // S, gc % S], -1).astype(np.uint8)
        actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
        want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=max_steps, auto_reset=auto_reset)
        got = run_gpu(ts, S, multi, blocked, tiles, targets, actions, max_steps, auto_reset)
        assert_same(got, want, f"fuzz case {case}: S{S} T{T} NT{NT} W{W} multi{multi} ar{auto_reset} ms{max_steps} N{N}")
        n_cases += 1
    assert n_cases == 70


@pytest.mark.parametrize("S,T,W,multi", [(6, 4, 8, True), (12, 8, 36, True), (5, 1, 5, False), (8, 5, 14, False)])
def test_long_rollout_with_many_resets(ts, S, T, W, multi):
    """2,000 steps of 2,048 envs with auto-reset (about 20 episodes per env at max_steps = 100, more
    where boards are won): final positions, final step counters and the per-step flag / reward
    checksums must equal the oracle's -- no drift over resets, counters or the fast path."""
    N, K = 2048, 2000
    rng = np.random.default_rng(S * 7 + T)
    blocked, tiles, targets = random_puzzles(rng, N, S, T, W)
    actions = rng.integers(0, 4, size=(K, N), dtype=np.uint8)
    want = orc.rollout(S, multi, blocked, tiles, targets, actions, max_steps=100, auto_reset=True)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=100, auto_reset=True)
    fast = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi, max_steps=100, auto_reset=True, track_flags=False)
    acts = torch.zeros(K, env.capacity, dtype=torch.uint8, device="cuda")
    acts[:, :N] = torch.as_tensor(actions).cuda()
    flag_sum = torch.zeros(N, dtype=torch.int64, device="cuda")
    rew_sum = torch.zeros(N, dtype=torch.float64, device="cuda")
    for k in range(K):
        _, r, _ = env.step(acts[k])
        fast.step(acts[k])
        flag_sum += env.flags.to(torch.int64) * (k % 251 + 1)
        rew_sum += r.to(torch.float64)
    assert np.array_equal(env.positions().cpu().numpy(), want["final_pos"])
    assert np.array_equal(env.step_count.to(torch.int32).cpu().numpy(), want["final_count"])
    w = (want["flags"].astype(np.int64) * (np.arange(K) % 251 + 1)[:, None]).sum(0)
    assert np.array_equal(flag_sum.cpu().numpy(), w)
    assert np.array_equal(rew_sum.cpu().numpy(), want["reward"].astype(np.float64).sum(0))
    assert torch.equal(fast.pos, env.pos) and torch.equal(fast.step_count, env.step_count)
    assert (want["flags"] & F_DONE).sum() > 15 * N
