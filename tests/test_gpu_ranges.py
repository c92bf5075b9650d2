"""The range contract of include/tiler_slider.h, entry point by entry point: every batch call covers
[first_env, first_env + n_envs) of a batch, and each writes exactly its documented set --

  ts_encode, ts_synth, ts_step       the envs of the range
  ts_observe                         d_obs[0 .. n_envs), d_obs RELATIVE to first_env
  ts_valid_moves, ts_goal_check      d_mask / d_won ABSOLUTE; the bitboard kernels (S <= 8, 1..8
                                     tiles) may also store the correct result of the up-to-3 envs
                                     after the range that share its last 4-env group
  ts_step_host                       device buffers as ts_step, host buffers relative to the range

Every output buffer gets GUARD poisoned bytes on both sides (float buffers: a NaN bit pattern, so
that a stray 0.0 or 1.0 shows), padding envs are poisoned too, and after each call every byte
outside the allowed write set must be unchanged, bit for bit.  Inside the range the results are
compared with the oracle (ts_oracle.c) or a plain numpy restatement pinned to it.  The calls go
through the C-ABI with the batch's own input buffers.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

GUARD = 64                 # bytes on each side of an output buffer (keeps the body 16-byte aligned)
POISON = 0xA5              # byte sentinel: no mask (0..15), won byte (0/1), flag byte or position is 0xA5
NAN_BITS = 0x7FC0DEAD      # float sentinel: a quiet NaN no kernel computes


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def stream():
    return torch.cuda.current_stream().cuda_stream


def round_up(n, m):
    return (n + m - 1) // m * m


class Guarded:
    """Device buffer of n_bytes between two GUARD-byte guards, all filled with a sentinel."""

    def __init__(self, n_bytes, fill=POISON, float_fill=False):
        assert n_bytes % 4 == 0 or not float_fill
        self.n = n_bytes
        if float_fill:
            self.whole = torch.full(((2 * GUARD + n_bytes) // 4,), NAN_BITS, dtype=torch.int32, device="cuda").view(torch.uint8)
        else:
            self.whole = torch.full((2 * GUARD + n_bytes,), fill, dtype=torch.uint8, device="cuda")
        assert self.whole.data_ptr() % 16 == 0
        self.before = self.whole.clone()

    @property
    def ptr(self):
        return self.whole.data_ptr() + GUARD

    @property
    def body(self):
        return self.whole[GUARD: GUARD + self.n]

    def guards_intact(self):
        w, b = self.whole, self.before
        return torch.equal(w[:GUARD], b[:GUARD]) and torch.equal(w[GUARD + self.n:], b[GUARD + self.n:])


def make_puzzles(rng, N, S, T, NT, W):
    """Dense boards: W walls and T tiles on distinct cells, NT targets anywhere (on walls, under tiles,
    duplicated).  Every third board has its targets on its tiles (won at reset when NT == T), every
    sixth of those in reversed order (a set goal is still met, an ordered one is not)."""
    perm = np.argsort(rng.random((N, S * S)), axis=1)
    blocked = np.zeros((N, S * S), np.uint8)
    np.put_along_axis(blocked, perm[:, :W], 1, axis=1)
    tc = perm[:, W:W + T]
    gc = rng.integers(0, S * S, size=(N, NT))
    if NT == T and T > 0:
        gc[::3] = tc[::3]
        gc[::6] = tc[::6, ::-1]
    tiles = np.stack([tc // S, tc % S], -1).astype(np.uint8)
    targets = np.stack([gc // S, gc % S], -1).astype(np.uint8)
    return blocked, tiles, targets


def oracle_states(S, blocked, tiles, targets, multi):
    return [orc.OracleState(S, [(c // S, c % S) for c in np.flatnonzero(blocked[e])], tiles[e].tolist(),
                            targets[e].tolist(), multi) for e in range(blocked.shape[0])]


# ---------------------------------------------------------------------------------------------------
# 1. ts_observe
# ---------------------------------------------------------------------------------------------------
def obs_envs_per_block(S):
    """Envs per block of the observation kernel, restated from obs_envs_per_block in
    tiler_slider_b200/csrc/ts_observe.cu:22-27 (about 28 KB of floats, at most 64, a multiple of 4)."""
    e = min(7168 // (S * S * 3), 64) & ~3
    return max(e, 4)


def ref_observation(S, blocked, tiles, targets, multi):
    """GameState.get_state_array (state.py:188-211) over a batch: ch0 blocked, ch1 tile index+1
    (multi colour) or 1, ch2 target index+1 or 1, later indices overwriting earlier ones."""
    N, T, NT = blocked.shape[0], tiles.shape[1], targets.shape[1]
    obs = np.zeros((N, S, S, 3), np.float32)
    obs[..., 0] = blocked.reshape(N, S, S)
    e = np.arange(N)
    for k in range(T):
        obs[e, tiles[:, k, 0], tiles[:, k, 1], 1] = k + 1 if multi else 1
    for k in range(NT):
        obs[e, targets[:, k, 0], targets[:, k, 1], 2] = k + 1 if multi else 1
    return obs


def obs_cases(S):
    """n_envs whose last block is (a) full, (b) partial with a float count divisible by 4 (bulk copy),
    (c) partial with a float count that is not (float4 loop + scalar tail; odd S only, 1..3 envs)."""
    E, per = obs_envs_per_block(S), 3 * S * S
    cases = {"full": 2 * E, "bulk": E + next(r for r in range(1, E) if r * per % 4 == 0)}
    if S % 2:
        cases.update({f"tail{r}": E + r for r in (1, 2, 3)})
    for name, n in cases.items():
        last = n - (n - 1) // E * E
        floats = last * per
        if name == "full":
            assert last == E
        elif name == "bulk":
            assert last < E and floats % 4 == 0
        else:
            assert last < E and floats % 4 != 0 and last % 4 == int(name[-1])
    return cases


OBS_SHAPES = [(S, 1 if S == 1 else min(8, S * S // 3), 1 if S == 1 else min(8, S * S // 3), S * S // 4, multi)
              for S in range(1, 17) for multi in (True, False)] + [
    (6, 12, 12, 6, True), (13, 20, 20, 30, False),      # 9..32 tiles
    (7, 3, 5, 6, True), (11, 2, 0, 20, True),          # never-win ordered batches: 5 targets for 3 tiles, none for 2
    (5, 0, 2, 3, False),                                # no tiles
]


@pytest.mark.parametrize("S,T,NT,W,multi", OBS_SHAPES)
def test_observe_sub_ranges_and_block_tails(ts, S, T, NT, W, multi):
    """ts_observe on ranges starting at env 0, 4 and 132 (ending short of the capacity) whose last
    block takes each of the kernel's three store paths; every float of every env against the numpy
    restatement of get_state_array, the guards around d_obs untouched."""
    rng = np.random.default_rng(1000 + 40 * S + 2 * T + NT + multi)
    N = 300
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    want = ref_observation(S, blocked, tiles, targets, multi)
    for e, st in zip(range(0, N, 37), oracle_states(S, blocked[::37], tiles[::37], targets[::37], multi)):
        assert np.array_equal(want[e], st.get_state_array()), e       # the restatement is the oracle's
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    assert env.never_win == (multi and NT != T)
    want_bits = torch.from_numpy(want).view(torch.int32)
    per = S * S * 3
    for name, n in obs_cases(S).items():
        for lo in (0, 4, 132):
            assert lo + n < env.capacity
            out = Guarded(n * per * 4, float_fill=True)
            a = env._observe_args(out.body)
            a.first_env, a.n_envs, a.d_obs = lo, n, out.ptr
            assert ts.lib().ts_observe(C.byref(a), stream()) == 0
            got = out.body.view(torch.int32).view(n, S, S, 3).cpu()
            assert torch.equal(got, want_bits[lo:lo + n]), (name, lo)
            assert out.guards_intact(), (name, lo)


def test_observe_out_is_validated(ts):
    """observe(out) checks the tensor before any launch: wrong shape, dtype, device or layout is a
    ValueError and the tensor stays as it was; a 16-byte-misaligned view is refused by ts_observe."""
    from tiler_slider_b200 import TilerSliderError
    S, N = 5, 99
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, 2, 3, True, seed=3)
    want = env.observe()
    out = torch.full((N, S, S, 3), float("nan"), device="cuda")
    assert env.observe(out) is out and torch.equal(out, want)
    pinned = torch.full((N, S, S, 3), float("nan")).pin_memory()
    env.observe(pinned)
    torch.cuda.synchronize()
    assert torch.equal(pinned, want.cpu())
    bad = [torch.full((N + 1, S, S, 3), 7.0, device="cuda"),
           torch.full((N - 1, S, S, 3), 7.0, device="cuda"),
           torch.full((N, S * S * 3), 7.0, device="cuda"),
           torch.full((N, S, S, 3), 7.0, dtype=torch.float16, device="cuda"),
           torch.full((N, S, S, 3), 7.0, dtype=torch.float64, device="cuda"),
           torch.full((N, S, S, 3), 7.0),                                     # host memory, not pinned
           torch.full((N, S, S, 6), 7.0, device="cuda")[..., :3],             # non-contiguous
           torch.full((S, S, N, 3), 7.0, device="cuda").permute(2, 0, 1, 3)]  # non-contiguous, right shape
    if torch.cuda.device_count() > 1:
        bad.append(torch.full((N, S, S, 3), 7.0, device="cuda:1"))
    for t in bad:
        with pytest.raises(ValueError):
            env.observe(t)
        torch.cuda.synchronize()
        assert bool((t == 7.0).all())
    buf = torch.full((N * S * S * 3 + 4,), 7.0, device="cuda")
    view = buf[1:1 + N * S * S * 3].view(N, S, S, 3)                         # contiguous, 4 bytes off alignment
    with pytest.raises(TilerSliderError, match="code -5"):
        env.observe(view)
    torch.cuda.synchronize()
    assert bool((buf == 7.0).all())


# ---------------------------------------------------------------------------------------------------
# 2. ts_valid_moves and ts_goal_check
# ---------------------------------------------------------------------------------------------------
QUERY_SHAPES = [  # S, T, NT, W, multi
    (5, 1, 1, 5, False), (6, 4, 4, 8, True), (6, 4, 4, 8, False), (8, 8, 8, 12, True), (3, 2, 2, 1, False),
    (7, 5, 5, 10, False), (6, 3, 2, 6, True),                                    # bitboard; the last never wins
    (12, 4, 4, 30, True), (16, 8, 8, 60, False), (9, 3, 3, 20, False), (14, 6, 6, 40, True),
    (12, 3, 5, 30, True),                                                        # wide (both wall-record forms); never wins
    (6, 12, 12, 6, True), (12, 16, 16, 20, False), (10, 20, 20, 12, True), (4, 9, 9, 0, False),   # generic
    (5, 0, 0, 3, False), (5, 0, 2, 3, False), (12, 0, 2, 20, True), (12, 0, 0, 20, True),         # no tiles
]
QUERY_RANGES = [(0, 509), (4, 510), (128, 131), (512, 640)]


@pytest.mark.parametrize("S,T,NT,W,multi", QUERY_SHAPES)
def test_queries_write_their_range_and_nothing_else(ts, S, T, NT, W, multi):
    """ts_valid_moves / ts_goal_check on sub-ranges of a 640-env batch (capacity 640, so one range
    ends exactly at the capacity): inside the range the oracle's valid_moves() / is_won(); the
    bitboard kernels may also store the correct answer for the envs up to the end of the range's last
    4-env group; every other byte of the guarded, poisoned mask stays as it was."""
    rng = np.random.default_rng(2000 + 40 * S + 2 * T + NT + multi)
    N = 640
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    assert env.capacity == N
    # move once so that positions differ from the packed initial ones (the kernels read d_pos)
    actions = rng.integers(0, 4, N, dtype=np.uint8)
    env.raw_move(torch.as_tensor(actions).cuda())
    states = oracle_states(S, blocked, tiles, targets, multi)
    for st, d in zip(states, actions):
        st.move(int(d))
    want = {"valid": np.array([sum(1 << d for d in st.valid_moves()) for st in states], np.uint8),
            "won": np.array([st.is_won() for st in states], np.uint8)}
    slack = 3 if S <= 8 and 1 <= T <= 8 else 0
    for lo, hi in QUERY_RANGES:
        for kind in ("valid", "won"):
            out = Guarded(N)
            if kind == "valid":
                a = ts._lib.ValidArgs(size=S, n_tiles=T, first_env=lo, n_envs=hi - lo, capacity=N,
                                      d_walls=env._walls.data_ptr(), d_pos=env._pos.data_ptr(), d_mask=out.ptr)
                assert ts.lib().ts_valid_moves(C.byref(a), stream()) == 0
            else:
                a = ts._lib.GoalArgs(size=S, n_tiles=T, goal_mode=env.goal_mode, never_win=int(env.never_win),
                                     first_env=lo, n_envs=hi - lo, capacity=N, d_targets_packed=env._targets.data_ptr(),
                                     d_pos=env._pos.data_ptr(), d_won=out.ptr)
                assert ts.lib().ts_goal_check(C.byref(a), stream()) == 0
            got = out.body.cpu().numpy()
            tag = (kind, lo, hi)
            assert np.array_equal(got[lo:hi], want[kind][lo:hi]), tag
            end = min(round_up(hi, 4), N) if slack else hi
            extra = got[hi:end]
            assert ((extra == POISON) | (extra == want[kind][hi:end])).all(), tag
            assert (got[:lo] == POISON).all() and (got[end:] == POISON).all(), tag
            assert out.guards_intact(), tag


# ---------------------------------------------------------------------------------------------------
# 3. ts_encode and ts_synth
# ---------------------------------------------------------------------------------------------------
def owner_maps(lib, S, pw, goal_mode, cap):
    """For every byte of the walls / targets / init / pos buffers: the env it belongs to."""
    def words(per_env):
        return np.arange(cap * per_env) // per_env

    def planes(nb):
        return np.concatenate([np.arange(lib.ts_plane_width(nb, k) * cap) // lib.ts_plane_width(nb, k)
                               for k in range(lib.ts_plane_count(nb))])
    if S > 8:
        per_axis = lib.ts_walls_bytes(S) // 2
        walls = np.tile(words(per_axis), 2)                  # [axis][env][line]
        tg = words(pw) if goal_mode == 0 else words(lib.ts_target_board_bytes(S))
    else:
        walls = planes(lib.ts_board_bytes(S))
        tg = words(pw) if goal_mode == 0 else planes(lib.ts_board_bytes(S))
    return {"walls": walls, "targets": tg, "init": words(pw), "pos": words(pw)}


def board_bits(lib, S, raw, cap):
    """Plane-layout bitboards (S <= 8) -> bool[cap, S, S] cells."""
    nb, bs = lib.ts_board_bytes(S), lib.ts_board_stride(S)
    cols, off = [], 0
    for k in range(lib.ts_plane_count(nb)):
        w = lib.ts_plane_width(nb, k)
        cols.append(raw[off * cap:(off + w) * cap].reshape(cap, w))
        off += w
    bits = np.unpackbits(np.concatenate(cols, axis=1), axis=1, bitorder="little")
    return bits[:, :S * bs].reshape(cap, S, bs)[:, :, :S].astype(bool)


def check_decodes_to(ts, env_like, bufs, lo, hi, blocked, tiles, targets):
    """Inside [lo, hi) the packed buffers decode to the dense description of envs lo..hi-1."""
    lib = ts.lib()
    S, T, cap, ps, pw, mode = env_like
    n = hi - lo
    cells = blocked[lo:hi].reshape(n, S, S).astype(bool)
    walls = bufs["walls"]
    if S > 8:
        L = lib.ts_walls_bytes(S) // 4
        lines = walls.view(np.uint16).reshape(2, cap, L)[:, lo:hi, :S].astype(np.uint32)
        lead = 1 if S <= 14 else 0
        bits = ((lines[..., None] >> (np.arange(S) + lead)) & 1).astype(bool)   # [axis, env, line, bit]
        assert np.array_equal(bits[1], cells)                                  # rows: line r, bit c
        assert np.array_equal(bits[0].transpose(0, 2, 1), cells)               # columns: line c, bit r
    else:
        assert np.array_equal(board_bits(lib, S, walls, cap)[lo:hi], cells)
    packed = (tiles[lo:hi, :, 0].astype(np.int64) * ps + tiles[lo:hi, :, 1]) if T else np.zeros((n, 0), np.int64)
    for name in ("init", "pos"):
        w = bufs[name].reshape(cap, pw)[lo:hi]
        assert np.array_equal(w[:, :T], packed) and not w[:, T:].any(), name
    NT = targets.shape[1]
    tg = bufs["targets"]
    if mode == 0:
        k = min(NT, T)
        w = tg.reshape(cap, pw)[lo:hi]
        want = targets[lo:hi, :k, 0].astype(np.int64) * ps + targets[lo:hi, :k, 1]
        assert np.array_equal(w[:, :k], want) and not w[:, k:].any()
    else:
        tcells = np.zeros((n, S * S), bool)
        if NT:
            tcells[np.arange(n)[:, None], targets[lo:hi, :, 0].astype(int) * S + targets[lo:hi, :, 1]] = True
        tcells = tcells.reshape(n, S, S)
        if S > 8:
            rec = tg.view(np.uint16).reshape(cap, 17)[lo:hi].astype(np.uint32)
            bits = ((rec[:, :16, None] >> np.arange(16)) & 1).astype(bool)
            assert np.array_equal(bits[:, :S, :S], tcells) and not bits[:, S:].any() and not bits[:, :, S:].any()
            assert np.array_equal(rec[:, 16], tcells.reshape(n, -1).sum(1))    # distinct target cells
        else:
            assert np.array_equal(board_bits(lib, S, tg, cap)[lo:hi], tcells)


LOAD_SHAPES = [  # S, T, NT, W, multi
    (6, 4, 4, 8, True), (6, 4, 4, 8, False), (3, 2, 3, 1, False), (8, 8, 8, 12, True), (7, 3, 2, 6, True),
    (12, 8, 8, 36, True), (16, 3, 3, 50, False), (12, 5, 7, 30, False), (15, 6, 6, 40, True),
    (10, 20, 20, 12, False), (6, 12, 12, 6, True), (5, 0, 0, 3, False), (13, 0, 2, 20, True),
]
LOAD_RANGES = [(4, 510), (128, 131), (512, 640)]


def guarded_like(env):
    return {"walls": Guarded(env._walls.numel()), "targets": Guarded(env._targets.numel()),
            "init": Guarded(env._init.numel()), "pos": Guarded(env._pos.numel())}


def check_write_set(owners, g, ref, lo, hi, tag):
    """The buffer equals the poison everywhere except the bytes of envs lo..hi-1, which equal ref's."""
    for name, buf in g.items():
        got = buf.body.cpu().numpy()
        inside = (owners[name] >= lo) & (owners[name] < hi)
        assert (got[~inside] == POISON).all(), (tag, name)
        assert np.array_equal(got[inside], ref[name][inside]), (tag, name)
        assert buf.guards_intact(), (tag, name)


@pytest.mark.parametrize("S,T,NT,W,multi", LOAD_SHAPES)
def test_encode_and_synth_sub_ranges(ts, S, T, NT, W, multi):
    """ts_encode and ts_synth on sub-ranges of poisoned, guarded buffers: every plane and record of
    the range (bitboard planes or both axes of the wide lines; ordered words, set planes or the wide
    17-word record with its distinct-target count; init and pos) -- encode: decodes back to the
    dense input and equals the whole-batch encode; synth with env_index_base = first_env: equals the
    same slice of a whole-batch synth; both: no byte of another env or of a guard changes."""
    lib = ts.lib()
    rng = np.random.default_rng(3000 + 40 * S + 2 * T + NT + multi)
    N = 640
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    whole = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    ref = {"walls": whole._walls, "targets": whole._targets, "init": whole._init, "pos": whole._pos}
    ref = {k: v.reshape(-1).cpu().numpy() for k, v in ref.items()}
    cap, pw, mode = whole.capacity, whole.pos_bytes, whole.goal_mode
    owners = owner_maps(lib, S, pw, mode, cap)
    for name, o in owners.items():
        assert o.size == ref[name].size and o.max() == cap - 1, name
    dev = {k: torch.as_tensor(v).cuda() for k, v in (("b", blocked), ("t", tiles), ("g", targets))}
    for lo, hi in LOAD_RANGES:
        g = guarded_like(whole)
        a = ts._lib.EncodeArgs(size=S, n_tiles=T, n_targets=NT, goal_mode=mode, first_env=lo, n_envs=hi - lo, capacity=cap,
                               d_blocked=dev["b"][lo:hi].data_ptr(), d_tiles=dev["t"][lo:hi].data_ptr() if T else None,
                               d_targets=dev["g"][lo:hi].data_ptr() if NT else None,
                               d_walls=g["walls"].ptr, d_targets_packed=g["targets"].ptr, d_init=g["init"].ptr, d_pos=g["pos"].ptr)
        assert lib.ts_encode(C.byref(a), stream()) == 0
        check_write_set(owners, g, ref, lo, hi, ("encode", lo, hi))
        check_decodes_to(ts, (S, T, cap, whole.pos_stride, pw, mode), {k: b.body.cpu().numpy() for k, b in g.items()},
                         lo, hi, blocked, tiles, targets)
    if W + 2 * T > S * S:
        return
    syn = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=99)
    ref = {k: getattr(syn, "_" + k).reshape(-1).cpu().numpy() for k in ("walls", "targets", "init", "pos")}
    owners = owner_maps(lib, S, syn.pos_bytes, syn.goal_mode, cap)
    for lo, hi in LOAD_RANGES:
        g = guarded_like(syn)
        a = ts._lib.SynthArgs(size=S, n_tiles=T, n_walls=W, goal_mode=syn.goal_mode, first_env=lo, n_envs=hi - lo,
                              capacity=cap, env_index_base=lo, seed=99, d_walls=g["walls"].ptr,
                              d_targets_packed=g["targets"].ptr, d_init=g["init"].ptr, d_pos=g["pos"].ptr)
        assert lib.ts_synth(C.byref(a), stream()) == 0
        check_write_set(owners, g, ref, lo, hi, ("synth", lo, hi))


# ---------------------------------------------------------------------------------------------------
# 4. ts_step_host against ts_step
# ---------------------------------------------------------------------------------------------------
DEV_POISON = {"_pos": 0xA5, "_count": 0x5A, "_reward": -123.5, "_done": 0x77, "_flags": 0xC3}
HOST_SHAPES = [(6, 4, 8, True), (12, 4, 30, False), (10, 20, 12, True), (5, 0, 3, False)]   # bitboard, wide, generic, no tiles


class HostCtx:
    def __init__(self, lib, n_streams):
        self.lib, self.h = lib, C.c_void_p()
        assert lib.ts_host_ctx_create(C.byref(self.h), n_streams) == 0

    def close(self):
        self.lib.ts_host_ctx_destroy(self.h)


def pinned(n, dtype, fill):
    return torch.full((n,), fill, dtype=dtype).pin_memory()


def same_bits(x, y):
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return torch.equal(x, y)


def run_step_host_twins(ts, S, T, W, multi, auto_reset, outputs, lo, n, chunks, ctxs, K=12):
    """Twin batches: `a` stepped by ts_step on [lo, lo+n), `b` by ts_step_host on the same range with
    `outputs` downloaded into pinned host buffers that carry a poisoned tail; every device buffer
    of b must equal a's after each step (outside the range: as before), every host output a's range."""
    lib = ts.lib()
    N, TAIL = 1000, 40
    kw = dict(seed=5, max_steps=5, auto_reset=auto_reset)
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, **kw)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, **kw)
    names = list(DEV_POISON)
    for name in names:                      # padding envs of both, poisoned alike
        getattr(a, name)[N:] = DEV_POISON[name]
        getattr(b, name)[N:] = DEV_POISON[name]
    rng = np.random.default_rng(S * 10 + T + 2 * auto_reset)
    h_act = pinned(n + TAIL, torch.uint8, 0xEE)
    finished = 0
    for k in range(K):
        h_act[:n] = torch.from_numpy(rng.integers(0, 4, n, dtype=np.uint8))
        h_rew = pinned(n + TAIL, torch.int32, NAN_BITS).view(torch.float32) if "reward" in outputs else None
        h_done = pinned(n + TAIL, torch.uint8, POISON) if "done" in outputs else None
        h_flags = pinned(n + TAIL, torch.uint8, POISON) if "flags" in outputs else None
        a._actions[lo:lo + n] = h_act[:n].cuda()
        sa = a._step_args(a._actions.data_ptr())
        sa.first_env, sa.n_envs = lo, n
        assert lib.ts_step(C.byref(sa), stream()) == 0
        torch.cuda.synchronize()
        sb = b._step_args(b._actions.data_ptr())
        sb.first_env, sb.n_envs = lo, n
        chunk, ctx = chunks[k % len(chunks)], ctxs[k % len(ctxs)]
        rc = lib.ts_step_host(ctx.h, C.byref(sb), h_act.data_ptr(), None if h_rew is None else h_rew.data_ptr(),
                              None if h_done is None else h_done.data_ptr(), None if h_flags is None else h_flags.data_ptr(), chunk)
        assert rc == 0, lib.ts_last_error_string()
        tag = (S, T, auto_reset, outputs, lo, n, k, chunk)
        for name in names:
            assert same_bits(getattr(b, name), getattr(a, name)), (tag, name)
        for h, name in ((h_rew, "_reward"), (h_done, "_done"), (h_flags, "_flags")):
            if h is None:
                continue
            assert same_bits(h[:n], getattr(a, name)[lo:lo + n].cpu()), (tag, name)
            tail = h[n:].view(torch.int32) if h.dtype == torch.float32 else h[n:]
            assert bool((tail == (NAN_BITS if h.dtype == torch.float32 else POISON)).all()), (tag, name, "tail")
        assert bool((h_act[n:] == 0xEE).all())
        finished += int((a._flags[lo:lo + n] & 1).sum())
    assert finished > 0, "the run should finish episodes"


@pytest.mark.parametrize("S,T,W,multi", HOST_SHAPES)
@pytest.mark.parametrize("auto_reset", [True, False])
def test_step_host_matches_step_bit_for_bit(ts, S, T, W, multi, auto_reset):
    """ts_step_host over [0, 1000) for each kernel class, with auto-reset on and off (off: the status
    byte is state the kernel reads back), each output set (reward + done, flags only, all three),
    chunks of 128, 384 (the last chunk ragged) and 1152 (one chunk, more streams than chunks), on
    contexts of 1 and 3 streams."""
    lib = ts.lib()
    ctxs = [HostCtx(lib, 1), HostCtx(lib, 3)]
    try:
        for outputs in (("reward", "done"), ("flags",), ("reward", "done", "flags")):
            run_step_host_twins(ts, S, T, W, multi, auto_reset, outputs, 0, 1000, (128, 384, 1152), ctxs)
    finally:
        for c in ctxs:
            c.close()


def test_step_host_sub_range(ts):
    """ts_step_host with first_env = 132: the host buffers are relative to the range, the device
    buffers absolute; the envs outside [132, 832) keep their state."""
    lib = ts.lib()
    ctxs = [HostCtx(lib, 3), HostCtx(lib, 1)]
    try:
        for S, T, W, multi in HOST_SHAPES:
            run_step_host_twins(ts, S, T, W, multi, False, ("reward", "done", "flags"), 132, 700, (256, 128, 1024), ctxs)
    finally:
        for c in ctxs:
            c.close()
