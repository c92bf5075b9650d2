// ts_playout.cu -- ts_playout on boards of size <= 8 with 1..8 tiles: up to n_steps moves of an item
// (env id, position word), taken from a plan or drawn at random, with the goal checked after every
// move.  Boards of size 9..16 are played by wide_playout_kernel (ts_wide.cu), 0 and 9..32 tiles by
// generic_playout_kernel (ts_generic.cu), as ts_step splits its work.
//
// Results reproduced: GameState.move (explainrl/environment/state.py:120-170) once per move and
// GameState.is_won (state.py:172-186) after it -- the slide_env core and the goal compare of
// step_group (ts_step.cuh), so each move leaves what ts_step leaves in pos for that action.
//
// Thread = one item.  Walls, targets and the position word are read once and stay in registers for
// every move; a move reads one plan byte (the plan policy: a warp reads 32 consecutive bytes of the
// step-major plan) or nothing (the random policy: the valid-move mask of ts_valid_moves, from the
// occupancy the goal test needs anyway, and one draw of the item's stream).  The policy is a template
// parameter: the plan kernel carries no random-number code.
#include "ts_playout.cuh"
#include "ts_valid.cuh"

namespace ts {

constexpr int PLAYOUT_THREADS = 256;

template <int S, int T, int POLICY>
__global__ void __launch_bounds__(PLAYOUT_THREADS) playout_kernel(const __grid_constant__ ts_playout_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4, NB = board_bytes(S);
    constexpr bool RANDOM = POLICY == TS_PLAYOUT_RANDOM;
    const int64_t i = (int64_t)blockIdx.x * PLAYOUT_THREADS + threadIdx.x;
    if (i >= a.n_items) return;
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint32_t q[PR] = {};
    int steps = 0;
    bool won = false;
    if (e >= 0 && e < a.capacity) {            // ids outside the table: zero result, nothing read (as ts_expand)
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        if (a.d_item_pos) ld_pos<PW>(a.d_item_pos, (size_t)i, q);
        else ld_pos<PW>(a.d_pos, env, q);
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, env);
        const bool ordered = a.goal_mode == TS_GOAL_ORDERED, can_win = a.never_win == 0;
        uint32_t tq[PR] = {};
        uint64_t tboard = 0;
        if (ordered) ld_pos<PW>(a.d_targets_packed, env, tq);
        else tboard = load_board_elem<NB>(a.d_targets_packed, cap, env);
        uint64_t rng = 0, occ = 0;
        if constexpr (RANDOM) {
            rng = synth_stream(a.seed, (uint64_t)i);
            occ = occupancy<S, T>(q);
        }
        while (steps < a.n_steps && !won) {
            uint32_t d;
            if constexpr (RANDOM) {
                const uint32_t mask = valid_mask_of<S>(occ, walls);
                if (!mask) break;                  // nothing can move: the playout ends here
                d = draw_move(rng, mask);
            } else {
                d = __ldcs(a.d_plan + playout_row(a, steps, i));
                if (d >= 4) break;                 // the end of the plan
            }
            slide_env<S, T>(q, walls, d >> 1, ~d & 1u);
            if (RANDOM || !ordered) occ = occupancy<S, T>(q);
            won = can_win;
            if (ordered) {
#pragma unroll
                for (int w = 0; w < PR; ++w) won &= q[w] == tq[w];
            } else {
                won &= occ == tboard;
            }
            playout_record<PW>(a, steps, i, d, q);
            ++steps;
        }
    }
    st_pos<PW>(a.d_final, (size_t)i, q);
    a.d_steps[i] = steps;
    a.d_won[i] = won ? 1 : 0;
    playout_tail<PW>(a, steps, i);
}

cudaError_t playout_dispatch(const ts_playout_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_items + PLAYOUT_THREADS - 1) / PLAYOUT_THREADS);
    return dispatch_small<MAX_TILES>(a.size, a.n_tiles, [&](auto S, auto T) {
        constexpr int s = decltype(S)::value, t = decltype(T)::value;
        if (a.policy == TS_PLAYOUT_RANDOM) playout_kernel<s, t, TS_PLAYOUT_RANDOM><<<blocks, PLAYOUT_THREADS, 0, st>>>(a);
        else playout_kernel<s, t, TS_PLAYOUT_PLAN><<<blocks, PLAYOUT_THREADS, 0, st>>>(a);
        return cudaGetLastError();
    });
}

}  // namespace ts
