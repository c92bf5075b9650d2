"""Python restatement of the puzzle generator's random streams (include/tiler_slider.h, K7
ts_synth_candidates and K8 ts_pool_reset), used by the tests to predict the device's candidates
and pool draws.  The moves of the walk recipe come from the C oracle."""
import numpy as np

M64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15


def mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def splitmix64(state):
    """(next state, output) of one splitmix64 draw."""
    state = (state + GOLDEN) & M64
    return state, mix64(state)


def attempt_seed(seed, attempt):
    if attempt == 0:
        return seed & M64
    return splitmix64((seed ^ (0xA0761D6478BD642F * attempt)) & M64)[1]


def synth_stream(seed, gidx):
    return splitmix64((seed ^ (0xD1B54A32D192ED03 * (gidx + 1))) & M64)[0]


def partial_fisher_yates(rng, cells, draws):
    perm = list(range(cells))
    for d in range(draws):
        rng, z = splitmix64(rng)
        j = d + (((z >> 32) * (cells - d)) >> 32)
        perm[d], perm[j] = perm[j], perm[d]
    return rng, perm


def candidate(orc, S, T, W, multi, recipe, walk_len, seed, attempt, gidx):
    """(blocked cells, tiles [(r, c)], targets [(r, c)]) of one candidate."""
    rng = synth_stream(attempt_seed(seed, attempt), gidx)
    if recipe == "uniform":
        rng, perm = partial_fisher_yates(rng, S * S, W + 2 * T)
        rc = [divmod(c, S) for c in perm[W:W + 2 * T]]
        return perm[:W], rc[:T], rc[T:]
    rng, perm = partial_fisher_yates(rng, S * S, W + T)
    blocked = [divmod(c, S) for c in perm[:W]]
    tiles = [divmod(c, S) for c in perm[W:W + T]]
    st = orc.OracleState(S, blocked, tiles, tiles, multi)
    for _ in range(walk_len):
        valid = st.valid_moves()
        if not valid:
            break
        rng, z = splitmix64(rng)
        st.move(valid[((z >> 32) * len(valid)) >> 32])
    return perm[:W], tiles, st.current_locations


def candidate_arrays(orc, S, T, W, multi, recipe, walk_len, seed, attempt, gidxs):
    """blocked u8[N,S*S], tiles u8[N,T,2], targets u8[N,T,2] for the global indices gidxs."""
    n = len(gidxs)
    blocked = np.zeros((n, S * S), np.uint8)
    tiles = np.zeros((n, T, 2), np.uint8)
    targets = np.zeros((n, T, 2), np.uint8)
    for i, g in enumerate(gidxs):
        b, t, g_ = candidate(orc, S, T, W, multi, recipe, walk_len, seed, attempt, int(g))
        blocked[i, b] = 1
        tiles[i] = t
        targets[i] = g_
    return blocked, tiles, targets


def pool_draw(seed, gidx, episode, n_pool):
    """Index of the pool puzzle K8 gives env `gidx` at the start of episode number `episode`."""
    h = mix64(mix64((seed ^ (((gidx + 1) * 0xD1B54A32D192ED03) & M64)) & M64) ^ (((episode + 1) * GOLDEN) & M64))
    return (h * n_pool) >> 64
