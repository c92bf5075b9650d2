// ts_expand.cu -- ts_expand on boards of size <= 8 with 1..8 tiles: the four successors of an item
// (env id, position word), whether each move changed anything and whether it wins.  Boards of size
// 9..16 are expanded by wide_expand_kernel (ts_wide.cu), 0 and 9..32 tiles by generic_expand_kernel
// (ts_generic.cu), as ts_step splits its work.
//
// Results reproduced: GameState.move (explainrl/environment/state.py:120-170) once per move and
// GameState.is_won (state.py:172-186) of each result -- the slide_env core and the goal compare of
// step_group (ts_step.cuh), so successor, moved and won bits equal what ts_step leaves in pos and
// flags for that action.
//
// Thread = one item.  Walls and targets are read once (load_board_elem: the env's element of every
// byte plane), the position word once; the four slides run in registers, and the 4*PW-byte output
// row leaves in one or two vector stores.  Unlike K4 (bfs_expand_kernel, ts_bfs.cu) nothing is
// canonicalised: set-goal successors keep the tile order, and a move that changes nothing gives the
// unchanged word.
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

constexpr int EXPAND_THREADS = 256;

template <int S, int T>
__global__ void __launch_bounds__(EXPAND_THREADS) expand_kernel(const __grid_constant__ ts_expand_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4, NB = board_bytes(S);
    const int64_t i = (int64_t)blockIdx.x * EXPAND_THREADS + threadIdx.x;
    if (i >= a.n_items) return;
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint32_t s[4][PR] = {};
    uint32_t moved = 0, won = 0;
    if (e >= 0 && e < a.capacity) {            // ids outside the table: zero row, nothing read (as K7 and K9)
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        uint32_t q0[PR], tq[PR];
        if (a.d_item_pos) ld_pos<PW>(a.d_item_pos, (size_t)i, q0);
        else ld_pos<PW>(a.d_pos, env, q0);
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, env);
        const bool ordered = a.goal_mode == TS_GOAL_ORDERED, can_win = a.never_win == 0;
        uint64_t tboard = 0;
        if (ordered) ld_pos<PW>(a.d_targets_packed, env, tq);
        else tboard = load_board_elem<NB>(a.d_targets_packed, cap, env);
#pragma unroll
        for (uint32_t d = 0; d < 4; ++d) {
            uint32_t q[PR];
#pragma unroll
            for (int w = 0; w < PR; ++w) q[w] = q0[w];
            bool mv = false;
            // the step's own "moved": the slide's counts on padded boards, a changed word on compact ones
            if constexpr (padded_board(S)) {
                mv = slide_padded<S, T>(q, walls, dir_params<S>(d >> 1, ~d & 1u));
            } else {
                slide_compact<S, T>(q, walls, d >> 1, ~d & 1u);
#pragma unroll
                for (int w = 0; w < PR; ++w) mv |= q[w] != q0[w];
            }
            bool w_ = can_win;
            if (ordered) {
#pragma unroll
                for (int w = 0; w < PR; ++w) w_ &= q[w] == tq[w];
            } else {
                w_ &= occupancy<S, T>(q) == tboard;
            }
            moved |= (mv ? 1u : 0u) << d;
            won |= (w_ ? 1u : 0u) << d;
#pragma unroll
            for (int w = 0; w < PR; ++w) s[d][w] = q[w];
        }
    }
    st_succ4<PW>(a.d_succ + (size_t)i * (4 * PW), s);
    if (a.d_moved) a.d_moved[i] = (uint8_t)moved;
    if (a.d_won) a.d_won[i] = (uint8_t)won;
}

cudaError_t expand_dispatch(const ts_expand_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_items + EXPAND_THREADS - 1) / EXPAND_THREADS);
    return dispatch_small<MAX_TILES>(a.size, a.n_tiles, [&](auto S, auto T) {
        expand_kernel<decltype(S)::value, decltype(T)::value><<<blocks, EXPAND_THREADS, 0, st>>>(a);
        return cudaGetLastError();
    });
}

}  // namespace ts
