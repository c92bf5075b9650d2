// ts_observe.cu -- K3: dense observation, GameState.get_state_array
// (explainrl/environment/state.py:188-211): float32 [N][S][S][3] (HWC) -- ch0 blocked (0/1), ch1
// tile index+1 (ordered goal) or 1 (set goal), ch2 target index+1 or 1; later indices overwrite
// earlier ones (state.py:202-209).
//
// A pure HBM writer: 12*S*S bytes per env against ~14 bytes read, and almost every float is
// zero.  So the kernel does not compute floats, it scatters the few non-zeros: a block owns E
// consecutive envs (about 28 KB of output), zero-fills their image in shared memory with
// 16-byte stores, drops in the walls (one work item per (env, row), only the set bits are
// visited), the tiles and the targets (one thread per env, in index order, so that a later
// index overwrites an earlier one exactly as the reference's loops do), and hands the finished
// image to the SM's copy engine (cp.async.bulk) in one piece.
// History (profiles/experiments/observe_throughput.py, 6x6 / 4 tiles, GB/s written): thread per
// cell with runtime S and per-byte loops 1227; thread per cell, compile-time S, SWAR matching
// 2442; staged image, bit test per cell, 256-thread store loop 5050; this kernel 5810.
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

constexpr int OBS_THREADS = 256;
__host__ __device__ constexpr int obs_envs_per_block(int S) {
    int e = 7168 / (S * S * 3);
    e = e > 64 ? 64 : e;
    e &= ~3;                       // multiple of 4: a block's output starts 16-byte aligned for odd S too
    return e < 4 ? 4 : e;
}

template <int S>
__global__ void __launch_bounds__(OBS_THREADS) observe_kernel(const ts_observe_args a) {
    constexpr int CELLS = S * S, PER_ENV = CELLS * 3, NB = board_bytes(S), E = obs_envs_per_block(S);
    __shared__ __align__(16) float stage[E * PER_ENV];
    const int64_t env0 = (int64_t)blockIdx.x * E;
    const int n_here = (int)min((int64_t)E, a.n_envs - env0);
    const size_t cap = (size_t)a.capacity;
    const bool ordered = a.goal_mode == TS_GOAL_ORDERED;
    const int T = a.n_tiles, pw = pos_bytes(T);
    const int n_floats = n_here * PER_ENV;

    for (int k = threadIdx.x; k < (E * PER_ENV) / 4; k += OBS_THREADS)
        reinterpret_cast<float4*>(stage)[k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    __syncthreads();

    // walls (and set-goal targets): one work item per (env, row) -- the row's bits are fetched once and
    // only the SET bits are visited (a board is mostly empty: 8 walls in 36 cells), instead of one
    // board load and one bit test per cell
    for (int j = threadIdx.x; j < n_here * S; j += OBS_THREADS) {
        const int e = j / S, r = j - e * S;
        const size_t env = (size_t)(a.first_env + env0 + e);
        uint32_t wrow, trow = 0;
        if constexpr (wide_board(S)) {
            wrow = (uint32_t)reinterpret_cast<const uint16_t*>(a.d_walls)[(cap + env) * (2 * wide_line_words(S)) + r] >> wide_line_lead(S);   // plane 1 = rows
            if (!ordered) trow = reinterpret_cast<const uint16_t*>(a.d_targets_packed)[env * WIDE_TARGET_WORDS + r];
        } else {
            wrow = (uint32_t)(load_board_elem<NB>(a.d_walls, cap, env) >> (r * board_stride(S)));
            if (!ordered) trow = (uint32_t)(load_board_elem<NB>(a.d_targets_packed, cap, env) >> (r * board_stride(S)));
        }
        constexpr uint32_t ROW = (1u << S) - 1u;      // drops the sentinels past column S-1
        float* img = stage + (e * CELLS + r * S) * 3;
        for (uint32_t m = wrow & ROW; m; m &= m - 1u) img[(__ffs(m) - 1) * 3] = 1.0f;
        for (uint32_t m = trow & ROW; m; m &= m - 1u) img[(__ffs(m) - 1) * 3 + 2] = 1.0f;
    }
    // tiles and ordered targets: one thread per env, ascending index (later overwrites earlier).
    // Ordered targets: n_targets = 0 means "as many as tiles, packed like the position word";
    // otherwise (target count != tile count: a board that can never be won, state.py:183-184)
    // d_targets_packed holds pos_bytes(n_targets)-byte words of n_targets targets, -1 = none.
    const int NT = a.n_targets == 0 ? T : (a.n_targets < 0 ? 0 : a.n_targets);
    const int tpw = pos_bytes(NT);
    for (int e = threadIdx.x; e < n_here; e += OBS_THREADS) {
        const size_t env = (size_t)(a.first_env + env0 + e);
        const uint8_t* pp = a.d_pos + env * pw;
        float* img = stage + e * PER_ENV;
        for (int k = 0; k < T; ++k) {
            const int b = pp[k];
            img[((b / pos_stride(S)) * S + b % pos_stride(S)) * 3 + 1] = ordered ? (float)(k + 1) : 1.0f;
        }
        if (ordered) {
            const uint8_t* tp = a.d_targets_packed + env * tpw;
            for (int k = 0; k < NT; ++k) {
                const int t = tp[k];
                img[((t / pos_stride(S)) * S + t % pos_stride(S)) * 3 + 2] = (float)(k + 1);
            }
        }
    }
    float* out = a.d_obs + env0 * PER_ENV;          // 16-byte aligned: E * PER_ENV is a multiple of 4
    // Stream-out by the copy engine of the SM: one elected thread hands the whole staged image
    // (up to 28 KB, contiguous in HBM) to cp.async.bulk (TMA 1-D, SASS UBLKCP) instead of 256 threads
    // looping over 16-byte stores.  The writers publish their shared-memory stores to the async
    // proxy first; the issuing thread stays until the engine has read the stage.  (A block whose
    // image is not a multiple of 16 bytes -- the ragged last block of an odd board size -- keeps the loop.)
    if ((n_floats & 3) == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(out), "r"((uint32_t)__cvta_generic_to_shared(stage)), "r"((uint32_t)n_floats * 4u) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        return;
    }
    __syncthreads();
    for (int k = threadIdx.x; k * 4 < n_floats; k += OBS_THREADS) {
        if (k * 4 + 3 < n_floats) __stcs(reinterpret_cast<float4*>(out) + k, reinterpret_cast<const float4*>(stage)[k]);
        else for (int j = k * 4; j < n_floats; ++j) out[j] = stage[j];
    }
}

template <int S> static void launch_observe(const ts_observe_args& a, cudaStream_t st) {
    constexpr int E = obs_envs_per_block(S);
    observe_kernel<S><<<(unsigned)((a.n_envs + E - 1) / E), OBS_THREADS, 0, st>>>(a);
}

cudaError_t observe_dispatch(const ts_observe_args& a, cudaStream_t st) {
    switch (a.size) {
#define TS_OBS(S) case S: launch_observe<S>(a, st); break;
        TS_OBS(1) TS_OBS(2) TS_OBS(3) TS_OBS(4) TS_OBS(5) TS_OBS(6) TS_OBS(7) TS_OBS(8)
        TS_OBS(9) TS_OBS(10) TS_OBS(11) TS_OBS(12) TS_OBS(13) TS_OBS(14) TS_OBS(15) TS_OBS(16)
#undef TS_OBS
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace ts
