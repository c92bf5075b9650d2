"""ts_observe_planes / BatchedTilerSliderEnv.observe_planes: the channel-first 0/1 observation.

  - reference pin: on every board size in both colour modes, 9..32 tiles, never-win batches and
    tile-less boards, in all four dtypes, the planes equal a numpy restatement of the format; mapped
    back through the relation of include/tiler_slider.h that restatement is ref_observation, the
    restatement of get_state_array that test_gpu_ranges pins to the oracle;
  - ranges and guards through the C-ABI: sub-ranges from env 0, 4 and 132 whose last block takes
    each store path of the kernel, images larger than one block's stage, guard bytes (NaN patterns
    for the float dtypes) unchanged bit for bit;
  - live state: after every step of auto-reset batches (with and without a reset pool) the planes
    map back to that step's observe(), and an observe_planes call changes no env buffer;
  - a CUDA graph of steps and observe_planes(out) replays to the planes of uncaptured calls;
  - observe_planes(out) refuses wrong buffers before any launch.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_gpu_ranges import GUARD, make_puzzles, oracle_states, ref_observation

pytestmark = pytest.mark.gpu

DTYPES = [torch.uint8, torch.bfloat16, torch.float16, torch.float32]
# guard / poison element of each dtype: a byte pattern no plane holds (float types: a NaN)
POISON_BITS = {torch.uint8: (0xA5, torch.uint8), torch.bfloat16: (0x7FA5, torch.int16),
               torch.float16: (0x7EA5, torch.int16), torch.float32: (0x7FC0DEAD, torch.int32)}
STAGE = 28672              # bytes a block of the kernel owns (PLANES_STAGE, csrc/ts_observe_planes.cu)


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def stream():
    return torch.cuda.current_stream().cuda_stream


def ordered_goal(T, NT, multi):
    return multi or (T == 1 and NT == 1)


def ref_planes(S, blocked, tiles, targets, multi):
    """The format of include/tiler_slider.h restated in numpy: uint8 [N, C, S, S]."""
    N, T, NT = blocked.shape[0], tiles.shape[1], targets.shape[1]
    e = np.arange(N)
    if ordered_goal(T, NT, multi):
        out = np.zeros((N, 1 + T + NT, S, S), np.uint8)
        for k in range(T):
            out[e, 1 + k, tiles[:, k, 0], tiles[:, k, 1]] = 1
        for k in range(NT):
            out[e, 1 + T + k, targets[:, k, 0], targets[:, k, 1]] = 1
    else:
        out = np.zeros((N, 3, S, S), np.uint8)
        for k in range(T):
            out[e, 1, tiles[:, k, 0], tiles[:, k, 1]] = 1
        for k in range(NT):
            out[e, 2, targets[:, k, 0], targets[:, k, 1]] = 1
    out[:, 0] = blocked.reshape(N, S, S)
    return out


def planes_to_hwc(planes, T, ordered):
    """The relation of include/tiler_slider.h: planes -> get_state_array's float32 [N, S, S, 3]
    (numpy or torch, any dtype)."""
    lib = torch if isinstance(planes, torch.Tensor) else np
    p = planes.float() if lib is torch else planes.astype(np.float32)
    if not ordered:
        return p[:, :3].permute(0, 2, 3, 1) if lib is torch else p[:, :3].transpose(0, 2, 3, 1)
    C = p.shape[1]
    w = lib.arange(1, C, dtype=lib.float32)
    if lib is torch:
        w = w.to(p.device)
    w = (w - (w > T) * T)[None, :, None, None]              # tile i: i+1, target j: j+1
    ch1 = (p[:, 1:1 + T] * w[:, :T]).sum(1)
    if C == 1 + T:
        ch2 = lib.zeros_like(p[:, 0])
    else:
        ch2 = (p[:, 1 + T:] * w[:, T:])
        ch2 = ch2.amax(1) if lib is torch else ch2.max(1)
    return lib.stack((p[:, 0], ch1, ch2), -1)


def as_dtype_bytes(planes_u8, dtype):
    """Expected bytes of the uint8 restatement in `dtype`, as a flat uint8 tensor."""
    return torch.from_numpy(planes_u8).to(dtype).contiguous().view(torch.uint8).reshape(-1)


class GuardedPlanes:
    """Device buffer of n elements of `dtype` between two GUARD-byte guards, all poisoned."""

    def __init__(self, n, dtype):
        bits, store = POISON_BITS[dtype]
        width = torch.empty((), dtype=dtype).element_size()
        self.n_bytes = n * width
        total = 2 * GUARD + self.n_bytes
        total += -total % 4
        sw = torch.empty((), dtype=store).element_size()
        self.whole = torch.full((total // sw,), bits, dtype=store, device="cuda").view(torch.uint8)
        assert self.whole.data_ptr() % 16 == 0
        self.before = self.whole.clone()

    @property
    def ptr(self):
        return self.whole.data_ptr() + GUARD

    @property
    def body(self):
        return self.whole[GUARD: GUARD + self.n_bytes]

    def guards_intact(self):
        w, b = self.whole, self.before
        return torch.equal(w[:GUARD], b[:GUARD]) and torch.equal(w[GUARD + self.n_bytes:], b[GUARD + self.n_bytes:])


# ---------------------------------------------------------------------------------------------------
# 1. the format against the restatement, and the restatement against get_state_array
# ---------------------------------------------------------------------------------------------------
PIN_SHAPES = [(S, 1 if S == 1 else min(8, S * S // 3), 1 if S == 1 else min(8, S * S // 3), S * S // 4, multi)
              for S in range(1, 17) for multi in (True, False)] + [
    (6, 12, 12, 6, True), (13, 20, 20, 30, False), (16, 32, 32, 60, True), (12, 32, 32, 40, False),   # 9..32 tiles
    (5, 1, 1, 5, False), (7, 3, 5, 6, True), (11, 2, 0, 20, True), (8, 4, 2, 10, True),   # 1/1 single colour; never-win: NT > T, none, NT < T
    (14, 3, 32, 20, True),                                                                # never-win, 32 targets
    (5, 0, 2, 3, False), (12, 0, 3, 10, True), (4, 0, 0, 2, True),                       # no tiles
]


@pytest.mark.parametrize("S,T,NT,W,multi", PIN_SHAPES)
def test_planes_equal_the_restatement_in_every_dtype(ts, S, T, NT, W, multi):
    """Every element of observe_planes() in each dtype equals the numpy restatement; mapped back
    through the relation, the restatement is ref_observation (spot-checked against the oracle here
    too) and the planes are the batch's own observe()."""
    rng = np.random.default_rng(5000 + 40 * S + 2 * T + NT + multi)
    N = 300
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    want = ref_planes(S, blocked, tiles, targets, multi)
    ordered = ordered_goal(T, NT, multi)
    hwc = ref_observation(S, blocked, tiles, targets, multi)
    # duplicate targets included: ch2's maximum keeps the largest index at a cell, which is the one
    # the reference's loop writes last
    assert np.array_equal(planes_to_hwc(want, T, ordered), hwc)
    for e, st in zip(range(0, N, 41), oracle_states(S, blocked[::41], tiles[::41], targets[::41], multi)):
        assert np.array_equal(hwc[e], st.get_state_array()), e
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    assert env.plane_count == want.shape[1]
    obs = env.observe()
    for dtype in DTYPES:
        got = env.observe_planes(dtype=dtype)
        assert got.dtype == dtype and got.shape == want.shape and got.is_contiguous()
        assert torch.equal(got.contiguous().view(torch.uint8).reshape(-1).cpu(), as_dtype_bytes(want, dtype)), dtype
        assert torch.equal(planes_to_hwc(got, T, ordered), obs), dtype


# ---------------------------------------------------------------------------------------------------
# 2. sub-ranges, block tails, images larger than a stage, guards
# ---------------------------------------------------------------------------------------------------
def planes_cases(env_bytes):
    """Env counts n whose call ends in each store path of the kernel: the last block's byte count
    `last` = a full stage; short, a multiple of 16 (one bulk copy); short, not a multiple of 16 and
    >= 16 (bulk copy + stored tail); below 16 (stored tail only, after at least one full block).
    The smallest such n of each kind that exists, up to n = STAGE (every residue the image size
    allows is reached by then) or 16 MB of output."""
    cases = {}
    for n in range(1, min(STAGE, (1 << 24) // env_bytes + 1) + 1):
        total = n * env_bytes
        last = total - (total - 1) // STAGE * STAGE
        kind = ("full" if last == STAGE else "bulk" if last % 16 == 0 else
                "bulk_tail" if last > 16 else "tail" if total > STAGE else None)
        if kind and kind not in cases:
            cases[kind] = n
        if len(cases) == 4:
            break
    return cases


RANGE_SHAPES = [  # S, T, NT, W, multi
    (5, 1, 1, 5, False), (6, 4, 4, 8, True), (3, 2, 2, 1, False), (7, 3, 5, 6, True),
    (12, 8, 8, 36, True), (13, 20, 20, 30, False), (11, 2, 0, 20, True), (5, 0, 2, 3, False),
    (16, 32, 32, 60, True),                    # 66,560 B per env in fp32: more than two stages
    (16, 32, 32, 60, False), (9, 32, 32, 20, True),
]


def test_range_cases_cover_every_store_path():
    """Over the shapes and dtypes of the range test, every store path is taken (u8 5x5 / 1 tile:
    75-byte images, which no power of two divides)."""
    seen = set()
    for S, T, NT, W, multi in RANGE_SHAPES:
        C_ = 1 + T + NT if ordered_goal(T, NT, multi) else 3
        for width in (1, 2, 4):
            seen |= set(planes_cases(C_ * S * S * width))
    assert seen == {"full", "bulk", "bulk_tail", "tail"}
    assert 16 * 16 * 65 * 4 > 2 * STAGE


@pytest.mark.parametrize("S,T,NT,W,multi", RANGE_SHAPES)
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_planes_sub_ranges_block_tails_and_guards(ts, S, T, NT, W, multi, dtype):
    """ts_observe_planes on ranges starting at env 0, 4 and 132 (ending short of the capacity), for
    env counts whose last block takes each store path: the bytes of the range equal the restatement
    (d_out relative to first_env), the guards on both sides are untouched."""
    C_ = 1 + T + NT if ordered_goal(T, NT, multi) else 3
    width = torch.empty((), dtype=dtype).element_size()
    per = C_ * S * S
    cases = planes_cases(per * width)
    N = 132 + max(cases.values()) + 4
    rng = np.random.default_rng(6000 + 40 * S + 2 * T + NT + multi)
    blocked, tiles, targets = make_puzzles(rng, N, S, T, NT, W)
    want = as_dtype_bytes(ref_planes(S, blocked, tiles, targets, multi), dtype)
    env = ts.BatchedTilerSliderEnv.from_arrays(S, blocked, tiles, targets, multi)
    assert env.plane_count == C_
    pb = per * width
    for name, n in cases.items():
        for lo in (0, 4, 132):
            assert lo + n < env.capacity
            out = GuardedPlanes(n * per, dtype)
            a = env._observe_planes_args(None, dtype)
            a.first_env, a.n_envs, a.d_out = lo, n, out.ptr
            assert ts.lib().ts_observe_planes(C.byref(a), stream()) == 0
            got = out.body.cpu()
            assert torch.equal(got, want[lo * pb:(lo + n) * pb]), (name, lo, n)
            assert out.guards_intact(), (name, lo, n)


# ---------------------------------------------------------------------------------------------------
# 3. live state: stepping batches, reset pools
# ---------------------------------------------------------------------------------------------------
LIVE_SHAPES = [(6, 4, 8, True), (6, 3, 8, False), (12, 4, 30, False), (12, 6, 30, True), (10, 20, 12, True)]   # narrow, wide, generic


def env_buffers(env):
    names = ["_walls", "_targets", "_init", "_pos", "_count", "_reward", "_done", "_flags", "_episodes", "_solve_depth", "_obs_targets"]
    return {k: getattr(env, k).clone() for k in names if getattr(env, k) is not None}


def check_live(env, T, tag, dtype):
    before = env_buffers(env)
    planes = env.observe_planes(dtype=dtype)
    after = env_buffers(env)
    for k in before:
        assert torch.equal(before[k], after[k]), (tag, k)
    ordered = env.goal_mode == 0
    assert torch.equal(planes_to_hwc(planes, T, ordered), env.observe()), tag
    if ordered:     # one cell per tile and target plane
        assert bool((planes[:, 1:].float().sum((2, 3)) == 1).all()), tag


@pytest.mark.parametrize("S,T,W,multi", LIVE_SHAPES)
@pytest.mark.parametrize("with_pool", [False, True])
def test_planes_follow_stepping_batches(ts, S, T, W, multi, with_pool):
    """Auto-reset batches stepped 30 times (max_steps 6, so episodes end by timeout as well as by
    wins); with a pool, finished envs load a new puzzle, so walls and targets change under the
    observation.  After every step the planes map back to observe()."""
    N = 3000
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=11, max_steps=6, auto_reset=True)
    if with_pool:
        pool = ts.BatchedTilerSliderEnv.synthetic(257, S, T, W, multi, seed=12)
        env.set_reset_pool(pool, seed=3, draw_now=True)
    gen = torch.Generator(device="cuda").manual_seed(S * 100 + T)
    finished = 0
    for k in range(30):
        actions = torch.randint(0, 4, (env.capacity,), dtype=torch.uint8, device="cuda", generator=gen)
        _, _, done = env.step(actions)
        finished += int(done.sum())
        check_live(env, T, (k, with_pool), DTYPES[k % 4])
    assert finished > 0
    if with_pool:
        assert int(env.episodes.sum()) > N


# ---------------------------------------------------------------------------------------------------
# 4. CUDA graphs
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.uint8], ids=str)
def test_graph_of_steps_and_planes_replays_like_the_calls(ts, dtype):
    """A graph capturing 8 x (step + observe_planes(out[k])) replays to the planes that the same
    calls write on a twin batch without capture."""
    S, T, W, N, K = 6, 4, 8, 5000, 8
    kw = dict(seed=21, max_steps=5, auto_reset=True)
    a = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    b = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, True, **kw)
    gen = torch.Generator(device="cuda").manual_seed(7)
    rows = torch.randint(0, 4, (K, a.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    shape = (N, a.plane_count, S, S)
    want = torch.stack([(b.step(rows[k]), b.observe_planes(dtype=dtype))[1] for k in range(K)])
    outs = torch.full((K,) + shape, 3, dtype=dtype, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                     # warm-up outside the capture
        a.step(rows[0])
        a.observe_planes(outs[0], dtype=dtype)
    torch.cuda.current_stream().wait_stream(side)
    a.reset()
    outs.fill_(3)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for k in range(K):
            a.step(rows[k])
            a.observe_planes(outs[k], dtype=dtype)
    assert bool((outs == 3).all())                    # captured, not run
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(outs, want)


# ---------------------------------------------------------------------------------------------------
# 5. validation of observe_planes(out)
# ---------------------------------------------------------------------------------------------------
def test_planes_out_is_validated(ts):
    """observe_planes(out) checks the tensor before any launch: wrong shape, dtype, device or layout
    is a ValueError and the tensor stays as it was; so is a dtype the kernel does not write; a
    16-byte-misaligned view is refused by ts_observe_planes."""
    from tiler_slider_b200 import TilerSliderError
    S, N = 5, 99
    env = ts.BatchedTilerSliderEnv.synthetic(N, S, 2, 3, True, seed=3)
    C_ = env.plane_count
    assert C_ == 5
    for dtype in DTYPES:
        want = env.observe_planes(dtype=dtype)
        out = torch.full((N, C_, S, S), 7, dtype=dtype, device="cuda")
        assert env.observe_planes(out, dtype=dtype) is out and torch.equal(out, want)
        pinned = torch.full((N, C_, S, S), 7, dtype=dtype).pin_memory()
        env.observe_planes(pinned, dtype=dtype)
        torch.cuda.synchronize()
        assert torch.equal(pinned, want.cpu())
    bad = [torch.full((N + 1, C_, S, S), 7.0, device="cuda"),
           torch.full((N - 1, C_, S, S), 7.0, device="cuda"),
           torch.full((N, C_ + 1, S, S), 7.0, device="cuda"),
           torch.full((N, C_ * S * S), 7.0, device="cuda"),
           torch.full((N, C_, S, S), 7.0, dtype=torch.float16, device="cuda"),    # dtype differs from the requested float32
           torch.full((N, C_, S, S), 7.0),                                         # host memory, not pinned
           torch.full((N, C_, S, 2 * S), 7.0, device="cuda")[..., :S],            # non-contiguous
           torch.full((N, S, S, C_), 7.0, device="cuda").permute(0, 3, 1, 2)]     # non-contiguous, right shape
    if torch.cuda.device_count() > 1:
        bad.append(torch.full((N, C_, S, S), 7.0, device="cuda:1"))
    for t in bad:
        with pytest.raises(ValueError):
            env.observe_planes(t)
        torch.cuda.synchronize()
        assert bool((t == 7.0).all())
    for dtype in (torch.float64, torch.int32, torch.bool, torch.int8):
        with pytest.raises(ValueError, match="dtype"):
            env.observe_planes(dtype=dtype)
        with pytest.raises(ValueError):
            env.observe_planes(torch.full((N, C_, S, S), 7, dtype=dtype, device="cuda"), dtype=dtype)
    for dtype in DTYPES:
        n = N * C_ * S * S
        buf = torch.full((n + 16,), 7, dtype=dtype, device="cuda")
        view = buf[1:1 + n].view(N, C_, S, S)                                     # contiguous, off alignment
        with pytest.raises(TilerSliderError, match="code -5"):
            env.observe_planes(view, dtype=dtype)
        torch.cuda.synchronize()
        assert bool((buf == 7).all())
