// ts_generate.cu -- puzzles worth playing: K7 ts_synth_candidates (candidate puzzles for the
// generator that keeps those K6 grades into a band of shortest-solution lengths) and K8
// ts_pool_reset (auto-reset into a pool of puzzles).  Entry points and argument checks: ts_api.cu.
//
// No reference counterpart: the reference draws puzzles with create_simple_env
// (explainrl/environment/environment.py:221-226, K0 here), of which about 1 % are solvable for the
// benchmark shape, and its reset (environment.py:89-97) restarts the same puzzle.
//
// K7: one thread per listed env slot, positions in (T+3)/4 32-bit words (1..4 tiles: K6 grades the
// candidates; 5..8 tiles, ts_synth_candidates_t8: K11 does).  The uniform recipe IS K0's draw (synth_env, ts_synth.cuh),
// with a fresh seed per attempt after the first.  The walk recipe keeps K0's walls and tiles and
// slides the tiles with slide_env<S,T> -- the step's own device code -- along a random walk of
// state-changing moves; the targets are where the tiles end up, so every candidate is solvable.
// K8: one thread per 16 envs reads their done bytes with one 16-byte load, a warp exits when none
// is set (about 1 % of the envs finish per step); a finished env draws a pool puzzle from a hash of
// (seed, global env index, episode number) and gets its walls / targets / initial positions.  It
// is launched with programmatic dependent launch right behind the step, like the step itself.
#include "ts_synth.cuh"

namespace ts {

constexpr int GEN_THREADS = 128;
constexpr int POOL_THREADS = 256;
constexpr int POOL_ENVS = 16;           // envs per K8 thread: one 16-byte load of done bytes

// seed of attempt a: attempt 0 is K0's seed, later attempts a fresh one
__device__ __forceinline__ uint64_t attempt_seed(uint64_t seed, uint32_t attempt) {
    if (attempt == 0) return seed;
    uint64_t s = seed ^ (0xA0761D6478BD642Full * (uint64_t)attempt);
    return splitmix64(s);
}

template <int S, int T>
__global__ void __launch_bounds__(GEN_THREADS) synth_candidates_kernel(const ts_synth_candidates_args a) {
    constexpr int CELLS = S * S, PW = pos_bytes(T), PS = pos_stride(S), BS = board_stride(S), NB = board_bytes(S);
    static_assert(T >= 1 && T <= 8 && S <= 8, "1..8 tiles, one 64-bit board");
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_items) return;
    const int64_t slot = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    if (slot < 0 || slot >= a.capacity) return;
    const size_t env = (size_t)slot, cap = (size_t)a.capacity;
    const uint64_t gidx = (uint64_t)(a.env_index_base + slot);
    const uint64_t seed = attempt_seed(a.seed, (uint32_t)a.attempt);
    if (a.recipe == TS_RECIPE_UNIFORM) {
        synth_env(S, T, a.n_walls, a.goal_mode, seed, gidx, cap, env, a.d_walls, a.d_targets_packed, a.d_init, a.d_pos);
        return;
    }
    // ---- walk: K0's walls and tiles, then walk_len state-changing moves drawn from the same stream
    const int W = a.n_walls;
    uint64_t rng = synth_stream(seed, gidx);
    uint8_t perm[CELLS];
    synth_cells(rng, CELLS, W + T, perm);
    uint64_t walls = 0;
    if constexpr (padded_board(S)) walls = Padded<S>::SENT;         // the stored sentinels (ts_common.cuh)
    for (int d = 0; d < W; ++d) walls |= 1ull << ((perm[d] / S) * BS + perm[d] % S);
    constexpr int PR = (T + 3) / 4;                                  // 32-bit position words
    uint32_t q[PR] = {};
#pragma unroll
    for (int t = 0; t < T; ++t) q[t / 4] |= (uint32_t)((perm[W + t] / S) * PS + perm[W + t] % S) << (8 * (t % 4));
    const uint32_t init = q[0], init_hi = q[PR - 1];           // init_hi: tiles 4..7 (5..8 tiles)
    for (int s = 0; s < a.walk_len; ++s) {
        uint32_t nxt[4][PR], mask = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            uint32_t x[PR];
#pragma unroll
            for (int w = 0; w < PR; ++w) x[w] = q[w];
            slide_env<S, T>(x, walls, (uint32_t)d >> 1, ((uint32_t)d & 1u) ^ 1u);
            uint32_t changed = 0;
#pragma unroll
            for (int w = 0; w < PR; ++w) {
                nxt[d][w] = x[w];
                changed |= x[w] ^ q[w];
            }
            mask |= (uint32_t)(changed != 0u) << d;
        }
        const int n = __popc(mask);
        if (n == 0) break;                                           // nothing can move: the walk ends here
        const uint32_t r = (uint32_t)(splitmix64(rng) >> 32);
        uint32_t m = mask;
        for (int k = (int)(((uint64_t)r * (uint32_t)n) >> 32); k > 0; --k) m &= m - 1u;   // k-th state-changing move
        const int d = __ffs(m) - 1;
#pragma unroll
        for (int w = 0; w < PR; ++w) q[w] = d == 0 ? nxt[0][w] : d == 1 ? nxt[1][w] : d == 2 ? nxt[2][w] : nxt[3][w];
    }
    for (int b = 0; b < NB; ++b) a.d_walls[board_byte_addr(NB, cap, env, b)] = (uint8_t)(walls >> (8 * b));
#pragma unroll
    for (int t = 0; t < PW; ++t) {
        a.d_init[env * PW + t] = (uint8_t)((t < 4 ? init : init_hi) >> (8 * (t % 4)));
        a.d_pos[env * PW + t] = (uint8_t)((t < 4 ? init : init_hi) >> (8 * (t % 4)));
    }
    if (a.goal_mode == TS_GOAL_ORDERED) {
#pragma unroll
        for (int t = 0; t < PW; ++t) a.d_targets_packed[env * PW + t] = (uint8_t)(q[t / 4] >> (8 * (t % 4)));
    } else {
        uint64_t tb = 0;                                             // target board: no sentinels
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const uint32_t p = (q[t / 4] >> (8 * (t % 4))) & 0xFFu;
            tb |= 1ull << (padded_board(S) ? p : (p >> 4) * (uint32_t)S + (p & 15u));
        }
        for (int b = 0; b < NB; ++b) a.d_targets_packed[board_byte_addr(NB, cap, env, b)] = (uint8_t)(tb >> (8 * b));
    }
}

cudaError_t candidates_dispatch(const ts_synth_candidates_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_items + GEN_THREADS - 1) / GEN_THREADS);
    auto go = [&](auto S, auto T) {
        synth_candidates_kernel<decltype(S)::value, decltype(T)::value><<<blocks, GEN_THREADS, 0, st>>>(a);
        return cudaGetLastError();
    };
    if (a.n_tiles <= 4) return dispatch_small(a.size, a.n_tiles, go);
    // 5..8 tiles (ts_synth_candidates_t8): boards of size 3..8, the ones that hold them
    return dispatch_size(a.size, [&](auto S) {
        constexpr int SV = decltype(S)::value;
        if constexpr (SV < 3) return cudaErrorInvalidValue;
        else return dispatch_tiles<5, 8>(a.n_tiles, [&](auto T) { return go(S, T); });
    });
}

// ---- K8 pool reset -------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// w bytes (1, 2, 4, 8 or a multiple of 16), both ends aligned to min(w, 16)
__device__ __forceinline__ void copy_elem(uint8_t* dst, const uint8_t* src, int w) {
    if (w >= 16) {
        for (int k = 0; k < w / 16; ++k) reinterpret_cast<uint4*>(dst)[k] = reinterpret_cast<const uint4*>(src)[k];
    } else if (w == 8) {
        *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(src);
    } else if (w == 4) {
        *reinterpret_cast<uint32_t*>(dst) = *reinterpret_cast<const uint32_t*>(src);
    } else if (w == 2) {
        *reinterpret_cast<uint16_t*>(dst) = *reinterpret_cast<const uint16_t*>(src);
    } else {
        *dst = *src;
    }
}

// board of nb <= 8 bytes (S <= 8) in the plane layout -- planes of width 8, 4, 2, 1, widest first:
// element `j` of a buffer of stride pcap -> element `env` of one of stride cap
__device__ __forceinline__ void copy_planes(uint8_t* dst, size_t cap, size_t env, const uint8_t* src, size_t pcap, size_t j, int nb) {
    int off = 0;
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1)
        if (nb & w) {
            copy_elem(dst + (size_t)off * cap + env * (size_t)w, src + (size_t)off * pcap + j * (size_t)w, w);
            off += w;
        }
}

__device__ __forceinline__ void pool_reset_env(const ts_pool_reset_args& a, size_t env) {
    const size_t cap = (size_t)a.capacity, pcap = (size_t)a.pool_capacity;
    const int S = a.size, pw = pos_bytes(a.n_tiles);
    const uint32_t ep = a.d_episode[env];
    a.d_episode[env] = ep + 1u;
    const uint64_t g = (uint64_t)a.env_index_base + env;
    const uint64_t h = mix64(mix64(a.seed ^ ((g + 1ull) * 0xD1B54A32D192ED03ull)) ^ (((uint64_t)ep + 1ull) * 0x9E3779B97F4A7C15ull));
    const size_t j = (size_t)__umul64hi(h, (uint64_t)a.n_pool);
    // walls
    if (wide_board(S)) {                       // u16 [axis][capacity][L lines]: two records of 2L bytes (a multiple of 4)
        const int L = 2 * wide_line_words(S);
        for (int axis = 0; axis < 2; ++axis) {
            uint32_t* d = reinterpret_cast<uint32_t*>(a.d_walls + 2 * ((size_t)axis * cap * L + env * L));
            const uint32_t* s = reinterpret_cast<const uint32_t*>(a.d_pool_walls + 2 * ((size_t)axis * pcap * L + j * L));
            for (int k = 0; k < L / 2; ++k) d[k] = s[k];
        }
    } else {
        copy_planes(a.d_walls, cap, env, a.d_pool_walls, pcap, j, board_bytes(S));
    }
    // targets
    if (a.goal_mode == TS_GOAL_ORDERED) {
        copy_elem(a.d_targets_packed + env * pw, a.d_pool_targets + j * pw, pw);
    } else if (wide_board(S)) {                // u16 [capacity][17]
        uint16_t* d = reinterpret_cast<uint16_t*>(a.d_targets_packed) + env * WIDE_TARGET_WORDS;
        const uint16_t* s = reinterpret_cast<const uint16_t*>(a.d_pool_targets) + j * WIDE_TARGET_WORDS;
        for (int k = 0; k < WIDE_TARGET_WORDS; ++k) d[k] = s[k];
    } else {
        copy_planes(a.d_targets_packed, cap, env, a.d_pool_targets, pcap, j, board_bytes(S));
    }
    // initial positions; the episode starts there
    copy_elem(a.d_init + env * pw, a.d_pool_init + j * pw, pw);
    copy_elem(a.d_pos + env * pw, a.d_pool_init + j * pw, pw);
    if (a.count_bytes == 1) static_cast<uint8_t*>(a.d_step_count)[env] = 0;
    else static_cast<int32_t*>(a.d_step_count)[env] = 0;
    if (a.d_solve_depth && a.d_pool_depth) a.d_solve_depth[env] = a.d_pool_depth[j];
}

// bit i set when byte i of w is not zero (the four flags gathered by one multiply, no carries)
__device__ __forceinline__ uint32_t nonzero_bytes(uint32_t w) {
    return ((__vcmpne4(w, 0u) & 0x01010101u) * 0x01020408u) >> 24;
}

// One thread per 16 envs reads their done bytes; a warp whose 512 envs have none set exits.  The
// finished envs of a warp are then listed in shared memory and reset one per lane, so that a step
// in which a few envs finished costs one short pass per warp, and one in which all of them did
// walks consecutive envs across the lanes.
__global__ void __launch_bounds__(POOL_THREADS) pool_reset_kernel(const ts_pool_reset_args a) {
    __shared__ uint16_t list[POOL_THREADS / 32][32 * POOL_ENVS];
    dependent_launch_sync();                   // the step in front of this launch has finished writing done
    const int64_t lo = a.first_env, hi = a.first_env + a.n_envs;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const int64_t e0 = (lo & ~(int64_t)(POOL_ENVS - 1)) + POOL_ENVS * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
    uint32_t m = 0;                            // bit k: env e0 + k is in the range and finished
    if (e0 < hi) {
        m = 0xFFFFu;                           // d_done = NULL: every env
        if (a.d_done) {
            const uint4 v = __ldcs(reinterpret_cast<const uint4*>(a.d_done + e0));
            m = nonzero_bytes(v.x) | nonzero_bytes(v.y) << 4 | nonzero_bytes(v.z) << 8 | nonzero_bytes(v.w) << 12;
        }
        if (e0 < lo) m &= 0xFFFFu << (lo - e0);
        if (hi - e0 < POOL_ENVS) m &= (1u << (hi - e0)) - 1u;
    }
    if (__ballot_sync(0xFFFFFFFFu, m != 0u) == 0u) return;   // the common case: nobody in these 512 envs finished
    const uint32_t c = (uint32_t)__popc(m);
    uint32_t x = c;                                           // inclusive prefix sum of the counts over the lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    const uint32_t total = __shfl_sync(0xFFFFFFFFu, x, 31);
    for (uint32_t pos = x - c; m; m &= m - 1u) list[warp][pos++] = (uint16_t)(lane * POOL_ENVS + (uint32_t)(__ffs(m) - 1));
    __syncwarp();
    const int64_t wbase = e0 - (int64_t)lane * POOL_ENVS;
    for (uint32_t t = lane; t < total; t += 32) pool_reset_env(a, (size_t)(wbase + list[warp][t]));
}

cudaError_t pool_reset_dispatch(const ts_pool_reset_args& a, cudaStream_t st) {
    const int64_t base = a.first_env & ~(int64_t)(POOL_ENVS - 1);
    const int64_t threads = (a.first_env + a.n_envs - base + POOL_ENVS - 1) / POOL_ENVS;
    launch_dependent(pool_reset_kernel, (unsigned)((threads + POOL_THREADS - 1) / POOL_THREADS), POOL_THREADS, st, a);
    return cudaGetLastError();
}

}  // namespace ts
