// ts_step.cuh -- K2, the fused step kernel (bitboard variant, boards of at most 64 bits).
//
// One launch advances every env of the range by one externally supplied action and fuses
//   GameState.move            explainrl/environment/state.py:120-170   (slide_env)
//   GameState.is_won          explainrl/environment/state.py:172-186   (goal compare)
//   TilerSliderEnv.step       explainrl/environment/environment.py:119-143
//                             invalid_move, done, step counter, timeout
//   TilerSliderEnv.reset      explainrl/environment/environment.py:89-97 (optional auto-reset)
// plus the repo-defined reward.  Thread = 4 consecutive envs; all traffic is 32/64/128-bit
// coalesced.  The kernel is bound by the integer ALU pipe, not by HBM (profiles/), so the
// per-env bookkeeping is done SWAR on the four packed status bytes of the thread's envs.
#pragma once
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

constexpr int STEP_THREADS = 256;

// Resident CTAs per SM requested from ptxas.  The kernel needs every warp it can get to
// cover the load latency at the top of each thread (measured: 8 CTAs x 256 threads = full
// occupancy runs the 6x6/4-tile step 15% faster than the 40-register default), but only the
// variants that fit 32 registers without spilling are forced there.
template <int S, int T, int GOAL, bool AR, int CW>
constexpr int step_min_blocks() {
    if (padded_board(S) && T <= 4 && GOAL == TS_GOAL_ORDERED && CW == 1) return 8;
    if (T <= 4) return 6;
    return 4;
}

// bit 7 of every byte of the result = (byte of a) >= (byte of b); b given as its low 7 bits
// (b_lo) and its bit 7 (b_hi), both replicated per byte
__device__ __forceinline__ uint32_t swar_ge_u8(uint32_t a, uint32_t b_lo, uint32_t b_hi) {
    const uint32_t t = (a | 0x80808080u) - b_lo;           // bit7: (a & 0x7f) >= (b & 0x7f); no cross-byte borrow
    return ((a & ~b_hi) | (~(a ^ b_hi) & t)) & 0x80808080u;
}

// Everything one thread loads for its 4 envs.
template <int S, int T, int GOAL, int CW>
struct StepInputs {
    static constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    uint32_t praw[PW];
    uint32_t traw[PW];
    BoardGroup<NB> walls, tboard;
    uint32_t act4, cnt4, prev_flags;
    uint32_t cntw[GROUP];
};

// The fused step of one 4-env group: slide, goal, bookkeeping, reward, auto-reset, stores.
// AR: auto-reset on (flags are write-only) / off (done envs are frozen and report STALE)
// CW: bytes of the step counter (1: SWAR bookkeeping, 4: per-env)
// dir_tab: the four DirParams (one per action) in shared memory, padded boards only; one
// conflict-free LDS.128 per env replaces the per-env decode of the action bits.
template <int S, int T, int GOAL, bool AR, int CW>
__device__ __forceinline__ void step_group(const ts_step_args& a, uint32_t g, StepInputs<S, T, GOAL, CW>& in,
                                           const uint4* dir_tab) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4, NB = board_bytes(S);
    constexpr int NWORDS = (NB + 3) / 4;
    const size_t e0 = (size_t)g * GROUP;
    uint32_t (&praw)[PW] = in.praw;
    uint32_t (&cntw)[GROUP] = in.cntw;
    const uint32_t cnt4 = in.cnt4;
    // scalars out of the parameter block first: through the reference the compiler may not
    // speculate the loads and turns the selects below into branches
    const float r_win = a.r_win, r_step = a.r_step, r_invalid = a.r_invalid;
    const int max_steps = a.max_steps;

    uint32_t pnew[PW];
#pragma unroll
    for (int j = 0; j < PW; ++j) pnew[j] = praw[j];
    uint32_t wm4 = 0;        // per byte: F_WON | F_INVALID of this step
    uint32_t to7 = 0;        // per byte: bit 7 = timeout (CW == 4 path fills it per env)
    float rew[GROUP];
    const bool can_win = a.never_win == 0;
    const uint32_t h4 = actions_h4(in.act4), f4 = actions_f4(in.act4);

#pragma unroll
    for (int e = 0; e < GROUP; ++e) {
        uint32_t q[PR], q0[PR], bw[NWORDS];
        group_elem<PW>(praw, e, q0);
#pragma unroll
        for (int w = 0; w < PR; ++w) q[w] = q0[w];
        in.walls.get(e, bw);
        bool moved = false;
        if constexpr (padded_board(S)) {
            const uint4 d = dir_tab[(in.act4 >> (8 * e)) & 3u];
            moved = slide_padded<S, T>(q, board64(bw), DirParams{d.x, d.y, d.z, d.w});   // no q0 kept alive
        } else {
            slide_env<S, T>(q, board64(bw), (h4 >> (8 * e)) & 0xFFu, (f4 >> (8 * e)) & 0xFFu);
#pragma unroll
            for (int w = 0; w < PR; ++w) moved |= q[w] != q0[w];
        }
        bool won = can_win;
        if constexpr (GOAL == TS_GOAL_ORDERED) {
            uint32_t tq[PR];
            group_elem<PW>(in.traw, e, tq);
#pragma unroll
            for (int w = 0; w < PR; ++w) won &= q[w] == tq[w];
        } else {
            uint32_t tw[NWORDS];
            in.tboard.get(e, tw);
            won &= occupancy<S, T>(q) == board64(tw);
        }
        rew[e] = won ? r_win : (moved ? r_step : r_invalid);
        uint32_t wm = won ? F_WON : 0u;
        if (!moved) wm |= F_INVALID;
        wm4 = mad_u32(wm, 1u << (8 * e), wm4);
        if constexpr (CW == 4) {
            cntw[e] += 1u;
            if ((int)cntw[e] >= max_steps) to7 |= 0x80u << (8 * e);
        }
        group_set<PW>(pnew, e, q);
    }

    // ---- SWAR bookkeeping on the four status bytes (environment.py:133-141) -------------------
    uint32_t c1 = 0;
    if constexpr (CW == 1) {
        c1 = cnt4 + 0x01010101u;                              // step_count += 1 (never wraps: count < max_steps <= 255)
        const uint32_t ms = (uint32_t)max_steps;
        to7 = swar_ge_u8(c1, (ms & 0x7Fu) * 0x01010101u, (ms & 0x80u) * 0x01010101u);
    }
    uint32_t done1 = ((wm4 >> 1) | (to7 >> 7)) & 0x01010101u;     // won or timeout
    uint32_t flags4 = wm4 | (to7 >> 4) | done1;
    if constexpr (!AR) {
        // envs that were already done are frozen: positions, counter and status untouched
        const uint32_t stale1 = in.prev_flags & 0x01010101u;
        if (stale1) {
            const uint32_t sm = stale1 * 0xFFu;
            flags4 = (flags4 & ~sm) | (stale1 * (F_DONE | F_STALE));
            done1 |= stale1;
            c1 = (c1 & ~sm) | (cnt4 & sm);
#pragma unroll
            for (int e = 0; e < GROUP; ++e) {
                if ((stale1 >> (8 * e)) & 1u) {
                    uint32_t q0[PR];
                    group_elem<PW>(praw, e, q0);
                    group_set<PW>(pnew, e, q0);
                    rew[e] = 0.0f;
                    if constexpr (CW == 4) cntw[e] -= 1u;
                }
            }
        }
    }

    // ---- auto-reset (environment.py:89-97) and the optional terminal snapshot ----------------
    if (done1 != 0) {
        if (a.d_terminal_pos) st_words<PW>(a.d_terminal_pos + e0 * PW, pnew);
        if constexpr (AR) {
            uint32_t iraw[PW];
            ld_words<PW>(a.d_init + e0 * PW, iraw);
            c1 &= ~(done1 * 0xFFu);
#pragma unroll
            for (int e = 0; e < GROUP; ++e) {
                if ((done1 >> (8 * e)) & 1u) {
                    uint32_t q[PR];
                    group_elem<PW>(iraw, e, q);
                    group_set<PW>(pnew, e, q);
                    if constexpr (CW == 4) cntw[e] = 0;
                }
            }
        }
    }

    // ---- stores --------------------------------------------------------------------------------
    st_words<PW>(a.d_pos + e0 * PW, pnew);
    if constexpr (CW == 1) __stcs(reinterpret_cast<unsigned int*>(a.d_step_count) + g, c1);
    else __stcs(reinterpret_cast<uint4*>(a.d_step_count) + g, make_uint4(cntw[0], cntw[1], cntw[2], cntw[3]));
    __stcs(reinterpret_cast<float4*>(a.d_reward) + g, make_float4(rew[0], rew[1], rew[2], rew[3]));
    if (a.d_done) __stcs(reinterpret_cast<unsigned int*>(a.d_done + e0), done1);
    if (a.d_flags) __stcs(reinterpret_cast<unsigned int*>(a.d_flags + e0), flags4);
}

// fill the per-block table of direction parameters (threads 0..3) -- call before any early return
template <int S> __device__ __forceinline__ void fill_dir_tab(uint4* dir_tab) {
    if constexpr (padded_board(S)) {
        if (threadIdx.x < 4) {
            const DirParams d = dir_params<S>(threadIdx.x >> 1, ~threadIdx.x & 1u);
            dir_tab[threadIdx.x] = make_uint4(d.st, d.lm, d.fm, d.fk);
        }
        __syncthreads();
    }
}

// ---- direct kernel: every thread loads its own group straight from global memory --------------
template <int S, int T, int GOAL, bool AR, int CW>
__global__ void __launch_bounds__(STEP_THREADS, (step_min_blocks<S, T, GOAL, AR, CW>())) step_kernel(const __grid_constant__ ts_step_args a) {
    constexpr int PW = pos_bytes(T);
    __shared__ uint4 dir_tab[4];
    fill_dir_tab<S>(dir_tab);
    // 32-bit group index: every address below is base + g * constant, one IMAD.WIDE each
    // (ts_step rejects capacities of 2^32 groups or more)
    // whole 4-env groups only: ts_step hands the ragged end of a range (n_envs % 4 envs) to
    // generic_step_kernel (ts_generic.cu), so nothing outside [first_env, first_env + n_envs) is touched
    // order 1 walks the range from its end, so a step that follows an ascending one starts on the
    // groups it left in L2 (ts_step_args.order): i -> n_groups - 1 - i = (i ^ m) + n_groups with
    // m = ~0, the form under which the kernels of boards up to 6x6 fit their registers without spills.
    // ts_step has checked first_env, n_envs >= 0.
    const uint32_t n_groups = (uint32_t)((uint64_t)a.n_envs / GROUP);
    const uint32_t i = blockIdx.x * STEP_THREADS + threadIdx.x;
    if (i >= n_groups) return;
    const uint32_t m = 0u - (uint32_t)a.order;
    const uint32_t g = (i ^ m) + ((uint32_t)((uint64_t)a.first_env / GROUP) + (n_groups & m));
    const size_t cap = (size_t)a.capacity;
    const size_t e0 = (size_t)g * GROUP;
    dependent_launch_sync();     // nothing is read before the launch ahead of us has completed (ts_common.cuh)

    StepInputs<S, T, GOAL, CW> in;
    // targets and step counters are only needed after the slide; under the 32-register cap the
    // compiler sinks their loads to that point, so pull the lines into L2 now (no register cost)
    if constexpr (GOAL == TS_GOAL_ORDERED) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.d_targets_packed + e0 * PW));
    // (the counter's address is formed inside the asm, so the compiler forms it again for the load
    // instead of keeping it live across the slide: that register is what keeps the kernel spill-free)
    asm volatile("{ .reg .u64 p; mad.wide.u32 p, %1, %2, %0; prefetch.global.L2 [p]; }" ::"l"(a.d_step_count), "r"(g), "n"(GROUP * CW));
    ld_words<PW>(a.d_pos + e0 * PW, in.praw);
    in.walls.load(a.d_walls, cap, g);
    if constexpr (GOAL == TS_GOAL_ORDERED) ld_words<PW>(a.d_targets_packed + e0 * PW, in.traw);
    else in.tboard.load(a.d_targets_packed, cap, g);
    in.act4 = __ldcs(reinterpret_cast<const unsigned int*>(a.d_actions + e0));
    in.cnt4 = 0;
    if constexpr (CW == 1) {
        in.cnt4 = __ldcs(reinterpret_cast<const unsigned int*>(a.d_step_count) + g);
    } else {
        const uint4 c = __ldcs(reinterpret_cast<const uint4*>(a.d_step_count) + g);
        in.cntw[0] = c.x; in.cntw[1] = c.y; in.cntw[2] = c.z; in.cntw[3] = c.w;
    }
    in.prev_flags = 0;
    if constexpr (!AR) in.prev_flags = __ldcs(reinterpret_cast<const unsigned int*>(a.d_flags + e0));
    step_group<S, T, GOAL, AR, CW>(a, g, in, dir_tab);
}

template <int S, int T, int GOAL>
inline void launch_step_goal(const ts_step_args& a, unsigned blocks, cudaStream_t stream) {
    const bool ar = a.auto_reset != 0, narrow = a.count_bytes == 1;
    if (ar && narrow) launch_dependent(step_kernel<S, T, GOAL, true, 1>, blocks, STEP_THREADS, stream, a);
    else if (ar) launch_dependent(step_kernel<S, T, GOAL, true, 4>, blocks, STEP_THREADS, stream, a);
    else if (narrow) launch_dependent(step_kernel<S, T, GOAL, false, 1>, blocks, STEP_THREADS, stream, a);
    else launch_dependent(step_kernel<S, T, GOAL, false, 4>, blocks, STEP_THREADS, stream, a);
}

template <int S, int T>
inline cudaError_t launch_step(const ts_step_args& a, cudaStream_t stream) {
    const size_t n_groups = (size_t)(a.n_envs / GROUP);          // the caller passes whole groups (ts_step splits off the rest)
    const unsigned blocks = (unsigned)((n_groups + STEP_THREADS - 1) / STEP_THREADS);
    if (blocks == 0) return cudaSuccess;
    if (a.goal_mode == TS_GOAL_ORDERED) launch_step_goal<S, T, TS_GOAL_ORDERED>(a, blocks, stream);
    else launch_step_goal<S, T, TS_GOAL_SET>(a, blocks, stream);
    return cudaGetLastError();
}

}  // namespace ts
