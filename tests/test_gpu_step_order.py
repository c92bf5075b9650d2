"""ts_step_args.order: a step launch may walk its range ascending (0) or descending (1), and
BatchedTilerSliderEnv.step() alternates the two so that each step starts on the envs the previous one
left in L2.  The order must not change any result: for every step kernel class, twin batches stepped
with order 0, with order 1 and through step()'s alternation hold the same bytes in every buffer after
every step.  A descending sub-range writes nothing outside its range, and captured graphs of odd and
even length equal the eager steps."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_gpu_ranges import DEV_POISON, Guarded, same_bits

pytestmark = pytest.mark.gpu

# (S, T, walls, multi): padded bitboards S <= 6, compact S = 7 and 8, wide S = 9..14 (wall records of
# ceil(S/2) pair words) and S = 15, 16 (plain 8-word lines), the generic kernel (0 tiles, > 8 tiles);
# T = 1..8 with both goal modes (multi: ordered, single colour: set)
CLASSES = [(3, 1, 1, False), (4, 2, 3, True), (5, 3, 4, False), (6, 4, 8, True), (6, 4, 8, False),
           (7, 5, 6, True), (7, 7, 5, False), (8, 6, 8, False), (8, 8, 6, True),
           (9, 2, 10, True), (12, 8, 36, True), (14, 3, 20, False),
           (15, 5, 30, False), (16, 1, 30, True), (16, 8, 40, True),
           (10, 20, 12, True), (5, 0, 3, False)]
N = 2051                  # several blocks of every kernel, a partial last block and a ragged 4-env group
K = 64
BUFFERS = ("_pos", "_reward", "_done", "_flags", "_count", "_terminal")


@pytest.fixture(scope="module")
def ts():
    import tiler_slider_b200 as t
    assert torch.cuda.is_available()
    t.lib()
    return t


def stream():
    return torch.cuda.current_stream().cuda_stream


def make(ts, S, T, W, multi, auto_reset, max_steps, n=N):
    return ts.BatchedTilerSliderEnv.synthetic(n, S, T, W, multi, seed=S * 100 + T, max_steps=max_steps,
                                              auto_reset=auto_reset, track_terminal=True)


def launch(ts, env, actions, order, lo=0, n=None):
    a = env._step_args(actions.data_ptr())
    a.first_env, a.n_envs, a.order = lo, env.n_envs - lo if n is None else n, order
    assert ts.lib().ts_step(C.byref(a), stream()) == 0, ts.lib().ts_last_error_string()


def assert_same(x, y, tag):
    for name in BUFFERS:
        assert same_bits(getattr(x, name), getattr(y, name)), (tag, name)


@pytest.mark.parametrize("S,T,W,multi", CLASSES)
@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("max_steps", [7, 300], ids=["u8count", "u32count"])
def test_order_does_not_change_the_rollout(ts, S, T, W, multi, auto_reset, max_steps):
    asc, desc, alt = (make(ts, S, T, W, multi, auto_reset, max_steps) for _ in range(3))
    assert asc.count_bytes == (1 if max_steps < 255 else 4)
    gen = torch.Generator(device="cuda").manual_seed(7 * S + T)
    finished = 0
    for k in range(K):
        row = torch.randint(0, 4, (asc.capacity,), dtype=torch.uint8, device="cuda", generator=gen)
        launch(ts, asc, row, 0)
        launch(ts, desc, row, 1)
        alt.step(row[: alt.n_envs])
        assert alt._cached_args.order == (k + 1) % 2
        assert_same(asc, desc, (k, "descending"))
        assert_same(asc, alt, (k, "alternating"))
        finished += int(asc._done[:N].sum())
    assert finished > 0 or max_steps > K, "with max_steps 7 every env times out within the rollout"


@pytest.mark.parametrize("S,T,W,multi", [(6, 4, 8, True), (8, 6, 8, False), (12, 4, 30, False), (16, 3, 30, True),
                                         (10, 20, 12, True)])
@pytest.mark.parametrize("auto_reset", [True, False])
def test_descending_sub_range_writes_only_its_envs(ts, S, T, W, multi, auto_reset):
    """[132, 833): starts inside the first block and ends in a ragged 4-env group.  Everything outside
    the range is poisoned and must stay so; inside, the descending twin equals the ascending one.  The
    reward buffer sits between poisoned guards."""
    lo, n = 132, 701
    twins = [make(ts, S, T, W, multi, auto_reset, 7) for _ in range(2)]
    guarded = []
    for e in twins:
        g = Guarded(e.capacity * 4, float_fill=True)
        g.body.view(torch.float32)[lo: lo + n] = e._reward[lo: lo + n]
        e._reward = g.body.view(torch.float32)
        e._cached_args = None
        guarded.append(g)
        for name, v in DEV_POISON.items():
            buf = getattr(e, name)
            if name != "_reward":
                buf[:lo] = v
                buf[lo + n:] = v
        e._terminal[:lo] = 0x3C
        e._terminal[lo + n:] = 0x3C
    outside = [{name: torch.cat([getattr(e, name)[:lo], getattr(e, name)[lo + n:]]).clone() for name in BUFFERS} for e in twins]
    rng = np.random.default_rng(S + T)
    for k in range(24):
        row = torch.from_numpy(rng.integers(0, 4, twins[0].capacity, dtype=np.uint8)).cuda()
        launch(ts, twins[0], row, 0, lo, n)
        launch(ts, twins[1], row, 1, lo, n)
        for e, out, g in zip(twins, outside, guarded):
            assert g.guards_intact(), (k, "reward guards")
            for name in BUFFERS:
                buf = getattr(e, name)
                assert same_bits(torch.cat([buf[:lo], buf[lo + n:]]), out[name]), (k, name, "outside the range")
        assert_same(twins[0], twins[1], k)


@pytest.mark.parametrize("S,T,W,multi", [(6, 4, 8, True), (12, 8, 36, True)])
@pytest.mark.parametrize("R", [5, 6])
def test_captured_steps_equal_eager_steps(ts, S, T, W, multi, R):
    """A graph bakes the order of each launch it holds: an even one alternates across replays, an odd
    one repeats a direction at each replay boundary.  Either way two replays equal 2R eager steps."""
    eager, graphed = (make(ts, S, T, W, multi, True, 7) for _ in range(2))
    gen = torch.Generator(device="cuda").manual_seed(R)
    rows = torch.randint(0, 4, (R, eager.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    g = graphed.capture_steps(rows)
    for rep in range(2):
        g.replay()
        for k in range(R):
            eager.step(rows[k][: eager.n_envs])
        torch.cuda.synchronize()
        assert_same(eager, graphed, rep)
