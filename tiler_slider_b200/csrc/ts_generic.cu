// ts_generic.cu -- step / valid-move / goal / expand / playout kernels for everything the specialised kernels do not cover:
//   (a) the ragged end of a range on bitboard-class boards (S <= 8): step_kernel works on whole
//       4-env groups, so ts_step hands the last n_envs % 4 envs of a call to generic_step_kernel --
//       nothing outside [first_env, first_env + n_envs) is ever read-modified-written;
//   (b) boards without tiles (T = 0, any S): the reference accepts them -- nothing moves, every
//       move is invalid, and the board is won iff it has no targets either
//       (explainrl/environment/state.py:183-186, tests/test_state.py:40-52,
//       tests/test_environment.py:569-580 of the reference);
//   (c) boards with 9 .. 32 tiles (any S <= 16): the reference puts no limit on the tile count
//       (its tests build a 20-tile board, tests/test_state.py:627-642); the register kernels are
//       instantiated for T <= 8, more tiles take this path (position words of 16 / 32 bytes).
// Thread = one env, runtime S and T, plain loops over row words held in local arrays: the closed
// form of GameState.move (state.py:120-170; ts_common.cuh) written out cell by cell -- a tile
// advances by the number of EMPTY cells between itself and the first wall / edge ahead -- and the
// bookkeeping of TilerSliderEnv.step (explainrl/environment/environment.py:119-143) and reset
// (:89-97) exactly as step_group (ts_step.cuh) does it.  Not a fast path.
#include "ts_common.cuh"
#include "ts_playout.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

// a bitboard-class board (S <= 8) of one env as a 64-bit word (runtime plane layout)
__device__ __forceinline__ uint64_t load_board64(const uint8_t* base, int S, size_t cap, size_t env) {
    const int nb = board_bytes(S);
    uint64_t b = 0;
    for (int k = 0; k < nb; ++k) b |= (uint64_t)base[board_byte_addr(nb, cap, env, k)] << (8 * k);
    return b;
}
__device__ __forceinline__ uint64_t cell_mask64(int S) {
    uint64_t m = 0;
    for (int r = 0; r < S; ++r) m |= (uint64_t)((1u << S) - 1u) << (r * board_stride(S));
    return m;
}
// rows[r] = row r of env's WALL board, cell (r, c) at bit c -- every board class
__device__ __forceinline__ void wall_rows(uint32_t* rows, const uint8_t* d_walls, int S, size_t cap, size_t env) {
    const uint32_t cells = (1u << S) - 1u;
    if (wide_board(S)) {
        const uint16_t* lines = reinterpret_cast<const uint16_t*>(d_walls) + (cap + env) * (size_t)(2 * wide_line_words(S));   // plane 1 = rows
        for (int r = 0; r < S; ++r) rows[r] = ((uint32_t)lines[r] >> wide_line_lead(S)) & cells;
    } else {
        const uint64_t b = load_board64(d_walls, S, cap, env);
        for (int r = 0; r < S; ++r) rows[r] = (uint32_t)(b >> (r * board_stride(S))) & cells;
    }
}
// rows[r] = row r of env's set-goal TARGET board
__device__ __forceinline__ void target_rows(uint32_t* rows, const uint8_t* d_tb, int S, size_t cap, size_t env) {
    const uint32_t cells = (1u << S) - 1u;
    if (wide_board(S)) {
        const uint16_t* lines = reinterpret_cast<const uint16_t*>(d_tb) + env * WIDE_TARGET_WORDS;
        for (int r = 0; r < S; ++r) rows[r] = lines[r];
    } else {
        const uint64_t b = load_board64(d_tb, S, cap, env);
        for (int r = 0; r < S; ++r) rows[r] = (uint32_t)(b >> (r * board_stride(S))) & cells;
    }
}

// GameState.is_won (state.py:183-186) of positions p[0..T): ordered = byte-wise equality with the
// packed targets; set = the occupancy rows equal the target rows (exact set equality)
__device__ __forceinline__ bool goal_met(const uint8_t* p, int S, int T, int goal_mode, const uint8_t* d_targets, size_t cap, size_t env) {
    const int pw = pos_bytes(T), ps = pos_stride(S);
    if (goal_mode == TS_GOAL_ORDERED) {
        for (int t = 0; t < T; ++t)
            if (p[t] != d_targets[env * pw + t]) return false;
        return true;
    }
    if (!wide_board(S)) {                       // occupancy == target bitboard, both in one word
        const int bs = board_stride(S);
        uint64_t occ = 0;
        for (int t = 0; t < T; ++t) occ |= 1ull << ((p[t] / ps) * bs + p[t] % ps);
        return occ == (load_board64(d_targets, S, cap, env) & cell_mask64(S));
    }
    uint32_t occ[MAX_SIZE], tgt[MAX_SIZE];
    target_rows(tgt, d_targets, S, cap, env);
    for (int r = 0; r < S; ++r) occ[r] = 0;
    for (int t = 0; t < T; ++t) occ[p[t] / ps] |= 1u << (p[t] % ps);
    for (int r = 0; r < S; ++r)
        if (occ[r] != tgt[r]) return false;
    return true;
}

// the env's walls in the form generic_slide reads: the 64-bit board on boards up to 8x8, rows on wide ones
struct GenericWalls {
    uint64_t b;
    uint32_t rows[MAX_SIZE];
};
__device__ __forceinline__ void load_generic_walls(GenericWalls& w, const uint8_t* d_walls, int S, int T, size_t cap, size_t env) {
    if (T > 0 && !wide_board(S)) w.b = load_board64(d_walls, S, cap, env);
    else if (T > 0) wall_rows(w.rows, d_walls, S, cap, env);
}

// One slide of the T tiles p0 -> p under `action` (state.py:137-170), cell by cell; true iff a tile moved.
// T = 0: nothing moves.
__device__ __forceinline__ bool generic_slide(const uint8_t* p0, uint8_t* p, int S, int T, uint32_t action, const GenericWalls& wl) {
    const int ps = pos_stride(S);
    const int dr = action == 0 ? -1 : action == 1 ? 1 : 0, dc = action == 2 ? -1 : action == 3 ? 1 : 0;   // state.py:31-34
    bool moved = false;
    if (T > 0 && !wide_board(S)) {             // the whole board in one word: register bit tests (ragged ends, the single-env adapter)
        const int bs = board_stride(S);
        const uint64_t walls = wl.b;
        uint64_t occ = 0;
        for (int t = 0; t < T; ++t) occ |= 1ull << ((p0[t] / ps) * bs + p0[t] % ps);
        for (int t = 0; t < T; ++t) {
            const int r = p0[t] / ps, c = p0[t] % ps;
            int n = 0;
            for (int rr = r + dr, cc = c + dc; rr >= 0 && rr < S && cc >= 0 && cc < S; rr += dr, cc += dc) {
                const int bit = rr * bs + cc;
                if ((walls >> bit) & 1ull) break;
                if (!((occ >> bit) & 1ull)) ++n;
            }
            p[t] = (uint8_t)((r + n * dr) * ps + (c + n * dc));
            moved |= n != 0;
        }
    } else if (T > 0) {                        // wide boards with more than 8 tiles: row words in local arrays
        const uint32_t* walls = wl.rows;
        uint32_t occ[MAX_SIZE];
        for (int r = 0; r < S; ++r) occ[r] = 0;
        for (int t = 0; t < T; ++t) occ[p0[t] / ps] |= 1u << (p0[t] % ps);
        for (int t = 0; t < T; ++t) {
            const int r = p0[t] / ps, c = p0[t] % ps;
            int n = 0;
            for (int rr = r + dr, cc = c + dc; rr >= 0 && rr < S && cc >= 0 && cc < S; rr += dr, cc += dc) {
                if ((walls[rr] >> cc) & 1u) break;
                if (!((occ[rr] >> cc) & 1u)) ++n;
            }
            p[t] = (uint8_t)((r + n * dr) * ps + (c + n * dc));
            moved |= n != 0;
        }
    }
    return moved;
}

__global__ void __launch_bounds__(128) generic_step_kernel(const ts_step_args a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i), cap = (size_t)a.capacity;
    const int S = a.size, T = a.n_tiles, pw = pos_bytes(T);
    const uint32_t action = a.d_actions[env] & 3u;

    uint8_t p0[MAX_TILES_ANY], p[MAX_TILES_ANY];
    for (int t = 0; t < T; ++t) p[t] = p0[t] = a.d_pos[env * pw + t];
    GenericWalls wl;
    load_generic_walls(wl, a.d_walls, S, T, cap, env);
    const bool moved = generic_slide(p0, p, S, T, action, wl);
    const bool won = a.never_win == 0 && goal_met(p, S, T, a.goal_mode, a.d_targets_packed, cap, env);
    // bookkeeping (environment.py:126-141)
    const bool narrow = a.count_bytes == 1;
    uint32_t count = narrow ? (uint32_t)reinterpret_cast<const uint8_t*>(a.d_step_count)[env]
                            : reinterpret_cast<const uint32_t*>(a.d_step_count)[env];
    count += 1u;
    const bool timeout = (int)count >= a.max_steps;
    bool done = won || timeout;
    uint32_t flags = (done ? F_DONE : 0u) | (won ? F_WON : 0u) | (moved ? 0u : F_INVALID) | (timeout ? F_TIMEOUT : 0u);
    float reward = won ? a.r_win : (moved ? a.r_step : a.r_invalid);
    if (!a.auto_reset && (a.d_flags[env] & F_DONE)) {   // frozen: the reference raises here (environment.py:113-114)
        flags = F_DONE | F_STALE;
        reward = 0.0f;
        count -= 1u;
        done = true;
        for (int t = 0; t < T; ++t) p[t] = p0[t];
    }
    if (done) {
        if (a.d_terminal_pos) for (int t = 0; t < pw; ++t) a.d_terminal_pos[env * pw + t] = t < T ? p[t] : 0;
        if (a.auto_reset) {                              // environment.py:89-97
            for (int t = 0; t < T; ++t) p[t] = a.d_init[env * pw + t];
            count = 0;
        }
    }
    for (int t = 0; t < pw; ++t) a.d_pos[env * pw + t] = t < T ? p[t] : 0;
    if (narrow) reinterpret_cast<uint8_t*>(a.d_step_count)[env] = (uint8_t)count;
    else reinterpret_cast<uint32_t*>(a.d_step_count)[env] = count;
    a.d_reward[env] = reward;
    if (a.d_done) a.d_done[env] = done ? 1 : 0;
    if (a.d_flags) a.d_flags[env] = (uint8_t)flags;
}

// GameState.is_won of the current positions (boards without tiles: won iff there are no targets; the
// caller's never_win carries "ordered mode with a target count different from the tile count")
__global__ void __launch_bounds__(128) generic_goal_kernel(const ts_goal_args a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i);
    const int T = a.n_tiles, pw = pos_bytes(T);
    uint8_t p[MAX_TILES_ANY];
    for (int t = 0; t < T; ++t) p[t] = a.d_pos[env * pw + t];
    a.d_won[env] = (a.never_win == 0 && goal_met(p, a.size, T, a.goal_mode, a.d_targets_packed, (size_t)a.capacity, env)) ? 1 : 0;
}

// get_valid_moves (environment.py:149-171): a move changes the state iff some tile has an empty
// cell right ahead of it (see valid_mask_of, ts_valid.cuh)
__global__ void __launch_bounds__(128) generic_valid_kernel(const ts_valid_args a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i), cap = (size_t)a.capacity;
    const int S = a.size, T = a.n_tiles, pw = pos_bytes(T), ps = pos_stride(S);
    uint32_t open[MAX_SIZE];
    uint8_t p[MAX_TILES_ANY];
    wall_rows(open, a.d_walls, S, cap, env);
    for (int r = 0; r < S; ++r) open[r] = ~open[r] & ((1u << S) - 1u);
    for (int t = 0; t < T; ++t) {
        p[t] = a.d_pos[env * pw + t];
        open[p[t] / ps] &= ~(1u << (p[t] % ps));
    }
    uint32_t mask = 0;
    for (int t = 0; t < T; ++t) {
        const int r = p[t] / ps, c = p[t] % ps;
        if (r > 0 && ((open[r - 1] >> c) & 1u)) mask |= 1u;
        if (r + 1 < S && ((open[r + 1] >> c) & 1u)) mask |= 2u;
        if (c > 0 && ((open[r] >> (c - 1)) & 1u)) mask |= 4u;
        if (c + 1 < S && ((open[r] >> (c + 1)) & 1u)) mask |= 8u;
    }
    a.d_mask[env] = (uint8_t)mask;
}

// ts_expand for 0 and 9..32 tiles (any S): the step's slide and goal test once per move.  An id
// outside [0, capacity) reads nothing and writes zero successors and masks.
__global__ void __launch_bounds__(128) generic_expand_kernel(const ts_expand_args a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n_items) return;
    const int S = a.size, T = a.n_tiles, pw = pos_bytes(T);
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint8_t* out = a.d_succ + (size_t)i * (4 * pw);
    uint32_t moved = 0, won = 0;
    if (e >= 0 && e < a.capacity) {
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        const uint8_t* src = a.d_item_pos ? a.d_item_pos + (size_t)i * pw : a.d_pos + env * pw;
        uint8_t p0[MAX_TILES_ANY], p[MAX_TILES_ANY];
        for (int t = 0; t < T; ++t) p0[t] = src[t];
        GenericWalls wl;
        load_generic_walls(wl, a.d_walls, S, T, cap, env);
        for (uint32_t d = 0; d < 4; ++d) {
            if (generic_slide(p0, p, S, T, d, wl)) moved |= 1u << d;
            if (a.never_win == 0 && goal_met(p, S, T, a.goal_mode, a.d_targets_packed, cap, env)) won |= 1u << d;
            for (int t = 0; t < pw; ++t) out[d * pw + t] = t < T ? p[t] : 0;
        }
    } else {
        for (int t = 0; t < 4 * pw; ++t) out[t] = 0;
    }
    if (a.d_moved) a.d_moved[i] = (uint8_t)moved;
    if (a.d_won) a.d_won[i] = (uint8_t)won;
}

cudaError_t generic_expand_dispatch(const ts_expand_args& a, cudaStream_t st) {
    if (a.n_items <= 0) return cudaSuccess;
    generic_expand_kernel<<<(unsigned)((a.n_items + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

// ts_playout for 0 and 9..32 tiles (any S): the step's slide and goal test once per move.  The random
// policy takes its mask from the four slides of the current positions, then plays the drawn one.  An
// id outside [0, capacity) reads nothing: zero positions, 0 moves, not won.
__global__ void __launch_bounds__(128) generic_playout_kernel(const ts_playout_args a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n_items) return;
    const int S = a.size, T = a.n_tiles, pw = pos_bytes(T);
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint8_t p[MAX_TILES_ANY], nxt[MAX_TILES_ANY];
    for (int t = 0; t < MAX_TILES_ANY; ++t) p[t] = 0;
    int steps = 0;
    bool won = false;
    if (e >= 0 && e < a.capacity) {
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        const uint8_t* src = a.d_item_pos ? a.d_item_pos + (size_t)i * pw : a.d_pos + env * pw;
        for (int t = 0; t < T; ++t) p[t] = src[t];
        GenericWalls wl;
        load_generic_walls(wl, a.d_walls, S, T, cap, env);
        uint64_t rng = a.policy == TS_PLAYOUT_RANDOM ? synth_stream(a.seed, (uint64_t)i) : 0;
        while (steps < a.n_steps && !won) {
            uint32_t d;
            if (a.policy == TS_PLAYOUT_RANDOM) {
                uint32_t mask = 0;
                for (uint32_t m = 0; m < 4; ++m)
                    if (generic_slide(p, nxt, S, T, m, wl)) mask |= 1u << m;
                if (!mask) break;
                d = draw_move(rng, mask);
            } else {
                d = a.d_plan[playout_row(a, steps, i)];
                if (d >= 4) break;
            }
            generic_slide(p, nxt, S, T, d, wl);
            for (int t = 0; t < T; ++t) p[t] = nxt[t];
            won = a.never_win == 0 && goal_met(p, S, T, a.goal_mode, a.d_targets_packed, cap, env);
            const size_t row = playout_row(a, steps, i);
            if (a.d_moves) a.d_moves[row] = (uint8_t)d;
            if (a.d_traj)
                for (int t = 0; t < pw; ++t) a.d_traj[row * pw + t] = t < T ? p[t] : 0;
            ++steps;
        }
    }
    for (int t = 0; t < pw; ++t) a.d_final[(size_t)i * pw + t] = t < T ? p[t] : 0;
    a.d_steps[i] = steps;
    a.d_won[i] = won ? 1 : 0;
    for (int k = steps; k < a.n_steps && (a.d_moves || a.d_traj); ++k) {
        const size_t row = playout_row(a, k, i);
        if (a.d_moves) a.d_moves[row] = 255;
        if (a.d_traj)
            for (int t = 0; t < pw; ++t) a.d_traj[row * pw + t] = 0;
    }
}

cudaError_t generic_playout_dispatch(const ts_playout_args& a, cudaStream_t st) {
    if (a.n_items <= 0) return cudaSuccess;
    generic_playout_kernel<<<(unsigned)((a.n_items + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t generic_step_dispatch(const ts_step_args& a, cudaStream_t st) {
    if (a.n_envs <= 0) return cudaSuccess;
    generic_step_kernel<<<(unsigned)((a.n_envs + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t generic_goal_dispatch(const ts_goal_args& a, cudaStream_t st) {
    if (a.n_envs <= 0) return cudaSuccess;
    generic_goal_kernel<<<(unsigned)((a.n_envs + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t generic_valid_dispatch(const ts_valid_args& a, cudaStream_t st) {
    if (a.n_envs <= 0) return cudaSuccess;
    generic_valid_kernel<<<(unsigned)((a.n_envs + 127) / 128), 128, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace ts
