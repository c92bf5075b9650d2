// ts_wide.cu -- step / valid-move / goal kernels for wide boards (9 <= S <= 16, T <= 8), the
// shape of BASELINE config 4 (12x12, 8 tiles, dense walls).
//
// Results reproduced: GameState.move (explainrl/environment/state.py:120-170), is_won
// (state.py:172-186), TilerSliderEnv.step bookkeeping (explainrl/environment/environment.py:
// 119-143), reset (environment.py:89-97), get_valid_moves (environment.py:149-171).
//
// A wide board does not fit a 64-bit word, so the bitboard tricks of ts_common.cuh do not
// apply.  Layout (one record of ceil(S/2) pair words per env and axis, axis-major planes):
//   walls[x][env][line]  u16, x = axis: plane 1 holds the rows (line r, cell (r,c) at bit c+1)
//                        and serves LEFT/RIGHT, plane 0 holds the columns (line c, cell (r,c) at
//                        bit r+1) and serves UP/DOWN.  A step reads exactly ONE record
//                        (select-source load).  For S <= 14 every line carries an edge sentinel
//                        at BOTH ends (bit 0 and bit S+1), so that for UP/LEFT one BREV of a
//                        pair word (two lines) turns both lines around with a sentinel still
//                        ahead of every slide; cells then sit at bit 14-c of the other half.
//                        S = 15, 16 have no room for that: plain lines (cell at bit c, no
//                        sentinel), reversed and re-aligned in registers (slide_wide16).
//                        History (profiles/): DRAM serves these reads at 128-byte granularity.
//                        With [env][4 orientations] of 32 bytes the whole 128-byte line around the
//                        one sector a step needs was fetched (612 MB read per 4.2M-env launch
//                        instead of 210 MB); four orientation planes cut that by a quarter, two
//                        axis planes + in-register reversal by half -- and since neighbouring envs
//                        pick their axis independently, nearly every line of BOTH planes is still
//                        touched, so what counts is the footprint: records hold only the
//                        ceil(S/2) pair words a board of this size has (24 bytes for 12x12).
//   tboard[env][17]      u16: 16 rows of target cells + the number of distinct targets (set goal only)
//   position byte        row*16 + col
// Thread = one env.  The 16 line words of the chosen orientation and the occupancy lines
// built from the tile positions live in shared memory as [word][thread] columns: a thread
// only ever touches its own column, so the dynamic line index costs no bank conflict
// (bank = thread % 32 whatever the line) and needs no barrier.
#include "ts_common.cuh"
#include "ts_playout.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

constexpr int WIDE_THREADS = 256;
constexpr int WIDE_MIN_BLOCKS = 8;

struct WideSmem {
    uint32_t w[8][WIDE_THREADS];   // wall lines, two 16-bit lines per word
    uint32_t o[8][WIDE_THREADS];   // occupancy lines of the current move
};

// S = 15, 16 (plain lines, 8 pair words).  Fetch the env's 32-byte wall record of the move's axis (plane 1 =
// rows for LEFT/RIGHT, plane 0 = columns for UP/DOWN), turn it toward the move direction and park
// it in the thread's smem column.  Stored lines run toward DOWN / RIGHT; for UP / LEFT (f = 1)
// every line is reversed in registers: brev flips the pair word (both halves reversed and
// swapped), PRMT swaps the halves back, a shift re-aligns the S cells.
__device__ __forceinline__ void load_oriented_walls(WideSmem& sm, const uint4* sector, int S, uint32_t f) {
    const uint4 b0 = __ldg(sector), b1 = __ldg(sector + 1);
    uint32_t w[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    if (f) {
        const uint32_t cells2 = ((1u << S) - 1u) * 0x00010001u;          // the S cell bits of both halves
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = (__byte_perm(__brev(w[k]), 0, 0x1032) >> (16 - S)) & cells2;
    }
    uint32_t* wcol = &sm.w[0][threadIdx.x];
#pragma unroll
    for (int k = 0; k < 8; ++k) wcol[k * WIDE_THREADS] = w[k];
}

__device__ __forceinline__ uint32_t half_of(uint32_t word, uint32_t half) {
    return __byte_perm(word, 0, 0x4410u + half * 0x22u);   // half ? word >> 16 : word & 0xffff
}

// One slide of all T tiles of the calling thread's env, S = 15 or 16 (no room for two stored
// sentinels in a 16-bit line: lines are extracted and the edge bit is OR-ed in).  `board` = the 32-byte
// orientation sector for `action`.  q: position bytes (row*16+col), updated in place.
template <int T>
__device__ __forceinline__ void slide_wide16(WideSmem& sm, uint32_t (&q)[(T + 3) / 4], const uint4* board, int S, uint32_t action) {
    constexpr int PR = (T + 3) / 4;
    const int tid = threadIdx.x;
    const uint32_t h = (action >> 1) & 1u, f = ~action & 1u;
    load_oriented_walls(sm, board, S, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sm.o[k][tid] = 0;

    // (line, offset) per byte: high nibble = line, low nibble = offset toward the move direction
    const uint32_t ks = 0x01010101u * (uint32_t)(S - 1);
    uint32_t Q[PR], ACC[PR];
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        uint32_t x = h ? q[w] : swap_nibbles(q[w]);
        if (f) x = (x & 0xF0F0F0F0u) | (ks - (x & 0x0F0F0F0Fu));
        Q[w] = x;
        ACC[w] = 0;
    }
    uint32_t line[T], off[T];
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t b = byte_of<i % 4>(Q[i / 4]);
        line[i] = b >> 4;
        off[i] = b & 15u;
        sm.o[line[i] >> 1][tid] |= 1u << (off[i] + 16u * (line[i] & 1u));
    });
    const uint32_t sentinel = 1u << S;
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t ww = half_of(sm.w[line[i] >> 1][tid], line[i] & 1u) | sentinel;
        const uint32_t oo = half_of(sm.o[line[i] >> 1][tid], line[i] & 1u);
        const uint32_t x = ww >> (off[i] + 1u);          // walls past the tile; the sentinel ends the line
        const uint32_t run = (x - 1u) & ~x;              // cells before the first wall
        ACC[i / 4] += (uint32_t)__popc(run & ~(oo >> (off[i] + 1u))) << (8 * (i % 4));
    });
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        uint32_t x = Q[w] + ACC[w];                      // offset += #empty cells; never carries (<= S-1)
        if (f) x = (x & 0xF0F0F0F0u) | (ks - (x & 0x0F0F0F0Fu));
        q[w] = h ? x : swap_nibbles(x);
    }
    if constexpr (T % 4 != 0) q[PR - 1] &= 0xFFFFFFFFu >> (8 * (4 - T % 4));   // keep unused bytes zero
}

// One slide, 9 <= S <= 14.  Every stored line has its cells at bits 1..S between two edge
// sentinels (bit 0, bit S+1), two lines per 32-bit pair word.  DOWN / RIGHT use the words as they
// are: a tile at offset c of line l is bit 16*(l&1) + c+1 of pair l>>1.  UP / LEFT use BREV of
// the words: the same tile is then bit 16*(1-(l&1)) + 14-c, and the line's bit-0 sentinel has
// become the bit-15 sentinel ahead of it.  Either way "bit index within the pair" is the low 5
// bits of the byte b = l*16 + off (bit 4 flipped for UP / LEFT), which is what the funnel shifts
// consume directly, and the slide is: x = walls >> b has the tile's own (wall-free) cell at bit 0
// and the first wall or sentinel ahead as its lowest set bit; (x-1) & ~x are the cells up to
// there; those not occupied (the tile itself is occupied) are the empty cells it moves over.
template <int T, int LW>
__device__ __forceinline__ void slide_wide(WideSmem& sm, uint32_t (&q)[(T + 3) / 4], const uint32_t* rec, uint32_t action) {
    constexpr int PR = (T + 3) / 4;
    const uint32_t h = (action >> 1) & 1u, f = ~action & 1u;
    uint32_t* wcol = &sm.w[0][threadIdx.x];     // this thread's column: pair k at wcol[k * WIDE_THREADS]
    uint32_t* ocol = &sm.o[0][threadIdx.x];
    {
        uint32_t w[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};   // LW = 5..7 pair words; records are 4*LW bytes apart
        if constexpr (LW % 2 == 0) {            // 8-byte aligned records
#pragma unroll
            for (int k = 0; k < LW / 2; ++k) {
                const uint2 v = __ldg(reinterpret_cast<const uint2*>(rec) + k);
                w[2 * k] = v.x;
                w[2 * k + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < LW; ++k) w[k] = __ldg(rec + k);
        }
        const uint32_t fmask = 0u - f;
#pragma unroll
        for (int k = 0; k < LW; ++k) {          // pairs >= LW hold no line of the board
            uint32_t r;
            asm("brev.b32 %0, %1;" : "=r"(r) : "r"(w[k]));
            wcol[k * WIDE_THREADS] = w[k] ^ ((w[k] ^ r) & fmask);   // f ? r : w[k] as one LOP3
            ocol[k * WIDE_THREADS] = 0;
        }
    }
    // offset of every tile toward the move direction: c+1, or 14-c for UP / LEFT (SWAR, one
    // multiply-add: bytes stay in 1..14, so nothing carries)
    const uint32_t fm = 1u - 2u * f;
    const uint32_t fk = 0x01010101u + f * 0x0D0D0D0Du;        // +1 | 14
    const uint32_t fu = 0xFEFEFEFFu + f * 0x0F0F0F0Fu;        // -1 | 14 : off -> c on the way back
    const uint32_t fx = f * 0x10101010u;                      // BREV swapped the two lines of a pair
    uint32_t LN[PR], OF[PR], B[PR], PM[PR], ACC[PR];
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        const uint32_t hi = (q[w] >> 4) & 0x0F0F0F0Fu, lo = q[w] & 0x0F0F0F0Fu;   // rows, cols
        LN[w] = h ? hi : lo;
        OF[w] = (h ? lo : hi) * fm + fk;
        B[w] = (LN[w] * 16u + OF[w]) ^ fx;
        PM[w] = B[w] & 0xE0E0E0E0u;                           // pair index * 32 per byte
        ACC[w] = 0;
    }
    uint32_t* oc[T];
    uint32_t sh[T];
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        sh[i] = B[i / 4] >> (8 * (i % 4));                    // funnel shifts read the low 5 bits
        oc[i] = ocol + byte_of<i % 4>(PM[i / 4]) * (WIDE_THREADS / 32);
        // 1 << (sh & 31) into the pair word; ATOMS.OR is one instruction where a read-modify-write
        // is three (measured: 53.7 vs 55.0 us per 4.2M-env step), and nothing else touches the column
        atomicOr(oc[i], __funnelshift_l(0u, 1u, sh[i]));
    });
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t x = __funnelshift_r(*(oc[i] - 8 * WIDE_THREADS), 0u, sh[i]);   // the wall pair sits 8 rows below
        const uint32_t y = __funnelshift_r(*oc[i], 0u, sh[i]);
        ACC[i / 4] = mad_u32((uint32_t)__popc((x - 1u) & ~x & ~y), 1u << (8 * (i % 4)), ACC[i / 4]);
    });
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        const uint32_t ofn = (OF[w] + ACC[w]) * fm + fu;      // new column / row
        q[w] = (h ? LN[w] : ofn) * 16u + (h ? ofn : LN[w]);
    }
    if constexpr (T % 4 != 0) q[PR - 1] &= 0xFFFFFFFFu >> (8 * (4 - T % 4));   // keep unused bytes zero
}

// set goal (state.py:185-186): every tile stands on a target cell AND the board has exactly T
// distinct target cells (word 16 of the record, written by ts_encode / ts_synth) -- tiles are on
// distinct cells, so the two together are set equality.  The record keeps the true target cells
// whatever their number: ts_observe draws channel 2 from it.
template <int T>
__device__ __forceinline__ bool on_targets_wide(const uint32_t (&q)[(T + 3) / 4], const uint8_t* tboard, size_t env) {
    const uint16_t* rows = reinterpret_cast<const uint16_t*>(tboard) + env * WIDE_TARGET_WORDS;
    bool all = __ldg(rows + 16) == (uint16_t)T;
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t b = byte_of<i % 4>(q[i / 4]);
        all &= ((__ldg(rows + (b >> 4)) >> (b & 15u)) & 1u) != 0;
    });
    return all;
}

// AR: auto-reset on / off (off: finished envs are frozen and report STALE); LW = ceil(S/2) pair
// words per wall record (8: board size 15 or 16, plain lines without stored sentinels).
// 32-bit env index: ts_step rejects larger batches.
template <int T, int GOAL, bool AR, int LW>
__global__ void __launch_bounds__(WIDE_THREADS, WIDE_MIN_BLOCKS) wide_step_kernel(const __grid_constant__ ts_step_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4;
    __shared__ WideSmem sm;
    const uint32_t n = (uint32_t)a.n_envs;
    const uint32_t i = blockIdx.x * WIDE_THREADS + threadIdx.x;
    if (i >= n) return;
    const uint32_t env = (uint32_t)a.first_env + (a.order ? n - 1u - i : i);   // ts_step_args.order
    dependent_launch_sync();
    const uint32_t action = a.d_actions[env] & 3u;
    uint32_t q0[PR], q[PR];
    ld_pos<PW>(a.d_pos, env, q0);
#pragma unroll
    for (int w = 0; w < PR; ++w) q[w] = q0[w];
    const bool narrow = a.count_bytes == 1;
    uint32_t count = narrow ? (uint32_t)reinterpret_cast<const uint8_t*>(a.d_step_count)[env]
                            : reinterpret_cast<const uint32_t*>(a.d_step_count)[env];
    bool stale = false;
    if constexpr (!AR) stale = (a.d_flags[env] & F_DONE) != 0;
    const float r_win = a.r_win, r_step = a.r_step, r_invalid = a.r_invalid;

    const uint32_t* rec = reinterpret_cast<const uint32_t*>(a.d_walls) + ((size_t)(action >> 1) * (size_t)a.capacity + env) * LW;
    if constexpr (LW == 8) slide_wide16<T>(sm, q, reinterpret_cast<const uint4*>(rec), a.size, action);
    else slide_wide<T, LW>(sm, q, rec, action);

    bool moved = false, won = a.never_win == 0;
#pragma unroll
    for (int w = 0; w < PR; ++w) moved |= q[w] != q0[w];
    if constexpr (GOAL == TS_GOAL_ORDERED) {
        uint32_t tq[PR];
        ld_pos<PW>(a.d_targets_packed, env, tq);
#pragma unroll
        for (int w = 0; w < PR; ++w) won &= q[w] == tq[w];
    } else {
        won &= on_targets_wide<T>(q, a.d_targets_packed, env);
    }
    count += 1u;
    const bool timeout = (int)count >= a.max_steps;
    bool done = won || timeout;
    uint32_t flags = (done ? F_DONE : 0u) | (won ? F_WON : 0u) | (moved ? 0u : F_INVALID) | (timeout ? F_TIMEOUT : 0u);
    float reward = won ? r_win : (moved ? r_step : r_invalid);
    if constexpr (!AR) {
        if (stale) {   // frozen: the reference raises here (environment.py:113-114)
            flags = F_DONE | F_STALE;
            reward = 0.0f;
            count -= 1u;
            done = true;
#pragma unroll
            for (int w = 0; w < PR; ++w) q[w] = q0[w];
        }
    }
    if (done) {
        if (a.d_terminal_pos) st_pos<PW>(a.d_terminal_pos, env, q);
        if constexpr (AR) {   // environment.py:89-97
            ld_pos<PW>(a.d_init, env, q);
            count = 0;
        }
    }
    st_pos<PW>(a.d_pos, env, q);
    if (narrow) reinterpret_cast<uint8_t*>(a.d_step_count)[env] = (uint8_t)count;
    else reinterpret_cast<uint32_t*>(a.d_step_count)[env] = count;
    a.d_reward[env] = reward;
    if (a.d_done) a.d_done[env] = done ? 1 : 0;
    if (a.d_flags) a.d_flags[env] = (uint8_t)flags;
}

// Valid-move mask of a wide board without running a slide (see valid_mask_of, ts_valid.cuh): a move
// changes the state iff some tile has an empty cell right ahead.  Occupancy rows are built in the
// thread's shared-memory column (pair words: rows 2k | 2k+1 << 16, cell c at bit c), the wall rows come
// from the rows plane alone; LEFT / RIGHT shift inside the rows, UP / DOWN shift the rows past each
// other with one funnel shift per pair word.
template <int T, int LW>
__device__ __forceinline__ uint32_t valid_mask_wide(WideSmem& sm, const uint32_t (&q)[(T + 3) / 4], const uint32_t* rows_rec, int S) {
    uint32_t* ocol = &sm.o[0][threadIdx.x];
#pragma unroll
    for (int k = 0; k < LW; ++k) ocol[k * WIDE_THREADS] = 0;
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t b = byte_of<i % 4>(q[i / 4]);          // row * 16 + col
        atomicOr(ocol + (b >> 5) * WIDE_THREADS, 1u << ((b & 15u) + (b & 16u)));
    });
    const uint32_t lead = LW == 8 ? 0u : 1u;                     // S <= 14: cells at bits 1..S between two sentinels
    const uint32_t row_cells = (1u << S) - 1u;
    uint32_t o[LW + 2], open[LW];
    o[0] = o[LW + 1] = 0;
#pragma unroll
    for (int k = 0; k < LW; ++k) {
        o[k + 1] = ocol[k * WIDE_THREADS];
        const uint32_t cells = row_cells | ((2 * k + 1 < S ? row_cells : 0u) << 16);     // the rows this pair really has
        open[k] = cells & ~(__ldg(rows_rec + k) >> lead) & ~o[k + 1];
    }
    uint32_t up = 0, down = 0, left = 0, right = 0;
#pragma unroll
    for (int k = 0; k < LW; ++k) {
        up |= __funnelshift_r(o[k + 1], o[k + 2], 16) & open[k];      // row r+1 seen from row r
        down |= __funnelshift_l(o[k], o[k + 1], 16) & open[k];        // row r-1 seen from row r
        left |= ((o[k + 1] >> 1) & 0x7FFF7FFFu) & open[k];
        right |= ((o[k + 1] << 1) & 0xFFFEFFFEu) & open[k];
    }
    return (up ? 1u : 0u) | (down ? 2u : 0u) | (left ? 4u : 0u) | (right ? 8u : 0u);
}

template <int T>
__global__ void __launch_bounds__(WIDE_THREADS) wide_valid_kernel(const __grid_constant__ ts_valid_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4;
    __shared__ WideSmem sm;
    const int64_t i = (int64_t)blockIdx.x * WIDE_THREADS + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i);
    uint32_t q0[PR];
    ld_pos<PW>(a.d_pos, env, q0);
    const int lw = wide_line_words(a.size);
    const uint32_t* rec = reinterpret_cast<const uint32_t*>(a.d_walls) + ((size_t)a.capacity + env) * (size_t)lw;   // plane 1 = rows
    uint32_t mask;
    switch (lw) {
        case 5: mask = valid_mask_wide<T, 5>(sm, q0, rec, a.size); break;
        case 6: mask = valid_mask_wide<T, 6>(sm, q0, rec, a.size); break;
        case 7: mask = valid_mask_wide<T, 7>(sm, q0, rec, a.size); break;
        default: mask = valid_mask_wide<T, 8>(sm, q0, rec, a.size); break;
    }
    a.d_mask[env] = (uint8_t)mask;
}

template <int T>
__global__ void __launch_bounds__(WIDE_THREADS) wide_goal_kernel(const __grid_constant__ ts_goal_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4;
    const int64_t i = (int64_t)blockIdx.x * WIDE_THREADS + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i);
    uint32_t q[PR];
    ld_pos<PW>(a.d_pos, env, q);
    bool won = a.never_win == 0;
    if (a.goal_mode == TS_GOAL_ORDERED) {
        uint32_t tq[PR];
        ld_pos<PW>(a.d_targets_packed, env, tq);
#pragma unroll
        for (int w = 0; w < PR; ++w) won &= q[w] == tq[w];
    } else {
        won &= on_targets_wide<T>(q, a.d_targets_packed, env);
    }
    a.d_won[env] = won ? 1 : 0;
}

// ts_expand on wide boards: thread = one item (env id, position word); the four moves are four
// slides of the step's, each reading the wall record of its axis, and the step's goal compare.
// An id outside [0, capacity) reads nothing and writes zero successors and masks.
template <int T, int LW>
__global__ void __launch_bounds__(WIDE_THREADS) wide_expand_kernel(const __grid_constant__ ts_expand_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4;
    __shared__ WideSmem sm;
    const int64_t i = (int64_t)blockIdx.x * WIDE_THREADS + threadIdx.x;
    if (i >= a.n_items) return;
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint32_t s[4][PR] = {};
    uint32_t moved = 0, won = 0;
    if (e >= 0 && e < a.capacity) {
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        uint32_t q0[PR], tq[PR];
        if (a.d_item_pos) ld_pos<PW>(a.d_item_pos, (size_t)i, q0);
        else ld_pos<PW>(a.d_pos, env, q0);
        const bool ordered = a.goal_mode == TS_GOAL_ORDERED, can_win = a.never_win == 0;
        if (ordered) ld_pos<PW>(a.d_targets_packed, env, tq);
#pragma unroll
        for (uint32_t d = 0; d < 4; ++d) {
            uint32_t q[PR];
#pragma unroll
            for (int w = 0; w < PR; ++w) q[w] = q0[w];
            const uint32_t* rec = reinterpret_cast<const uint32_t*>(a.d_walls) + ((size_t)(d >> 1) * cap + env) * LW;
            if constexpr (LW == 8) slide_wide16<T>(sm, q, reinterpret_cast<const uint4*>(rec), a.size, d);
            else slide_wide<T, LW>(sm, q, rec, d);
            bool mv = false, w_ = can_win;
#pragma unroll
            for (int w = 0; w < PR; ++w) mv |= q[w] != q0[w];
            if (ordered) {
#pragma unroll
                for (int w = 0; w < PR; ++w) w_ &= q[w] == tq[w];
            } else {
                w_ &= on_targets_wide<T>(q, a.d_targets_packed, env);
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

// ts_playout on wide boards: thread = one item (env id, position word), positions in registers for
// every move; a move is the step's slide on the wall record of its axis and the step's goal compare.
// The random policy takes the mask of ts_valid_moves (valid_mask_wide, rows record) before each move.
// The records are re-read every move (a thread reads the same 4*LW bytes again, which is expected to hit
// L1; not measured against records held in registers or shared memory).
// An id outside [0, capacity) reads nothing: zero positions, 0 moves, not won.
template <int T, int LW, int POLICY>
__global__ void __launch_bounds__(WIDE_THREADS) wide_playout_kernel(const __grid_constant__ ts_playout_args a) {
    constexpr int PW = pos_bytes(T), PR = (T + 3) / 4;
    __shared__ WideSmem sm;
    const int64_t i = (int64_t)blockIdx.x * WIDE_THREADS + threadIdx.x;
    if (i >= a.n_items) return;
    const int64_t e = a.d_env_ids ? (int64_t)a.d_env_ids[i] : i;
    uint32_t q[PR] = {};
    int steps = 0;
    bool won = false;
    if (e >= 0 && e < a.capacity) {
        const size_t env = (size_t)e, cap = (size_t)a.capacity;
        if (a.d_item_pos) ld_pos<PW>(a.d_item_pos, (size_t)i, q);
        else ld_pos<PW>(a.d_pos, env, q);
        const bool ordered = a.goal_mode == TS_GOAL_ORDERED, can_win = a.never_win == 0;
        uint32_t tq[PR] = {};
        if (ordered) ld_pos<PW>(a.d_targets_packed, env, tq);
        const uint32_t* cols = reinterpret_cast<const uint32_t*>(a.d_walls) + env * LW;           // plane 0: UP / DOWN
        const uint32_t* rows = reinterpret_cast<const uint32_t*>(a.d_walls) + (cap + env) * LW;   // plane 1: LEFT / RIGHT
        uint64_t rng = 0;
        if constexpr (POLICY == TS_PLAYOUT_RANDOM) rng = synth_stream(a.seed, (uint64_t)i);
        while (steps < a.n_steps && !won) {
            uint32_t d;
            if constexpr (POLICY == TS_PLAYOUT_RANDOM) {
                const uint32_t mask = valid_mask_wide<T, LW>(sm, q, rows, a.size);
                if (!mask) break;
                d = draw_move(rng, mask);
            } else {
                d = __ldcs(a.d_plan + playout_row(a, steps, i));
                if (d >= 4) break;
            }
            const uint32_t* rec = d >> 1 ? rows : cols;
            if constexpr (LW == 8) slide_wide16<T>(sm, q, reinterpret_cast<const uint4*>(rec), a.size, d);
            else slide_wide<T, LW>(sm, q, rec, d);
            won = can_win;
            if (ordered) {
#pragma unroll
                for (int w = 0; w < PR; ++w) won &= q[w] == tq[w];
            } else {
                won &= on_targets_wide<T>(q, a.d_targets_packed, env);
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

template <int T, int GOAL, int LW> static void launch_wide_step_lw(const ts_step_args& a, unsigned blocks, cudaStream_t st) {
    if (a.auto_reset != 0) launch_dependent(wide_step_kernel<T, GOAL, true, LW>, blocks, WIDE_THREADS, st, a);
    else launch_dependent(wide_step_kernel<T, GOAL, false, LW>, blocks, WIDE_THREADS, st, a);
}
template <int T, int GOAL> static void launch_wide_step_goal(const ts_step_args& a, unsigned blocks, cudaStream_t st) {
    switch (wide_line_words(a.size)) {
        case 5: launch_wide_step_lw<T, GOAL, 5>(a, blocks, st); break;
        case 6: launch_wide_step_lw<T, GOAL, 6>(a, blocks, st); break;
        case 7: launch_wide_step_lw<T, GOAL, 7>(a, blocks, st); break;
        default: launch_wide_step_lw<T, GOAL, 8>(a, blocks, st); break;
    }
}
template <int T> static cudaError_t launch_wide_step(const ts_step_args& a, cudaStream_t st) {
    // 32-bit env index: ts_step refuses such a range with TS_E_BAD_RANGE before it gets here; kept as a backstop
    if (a.first_env + a.n_envs >= ((int64_t)1 << 32)) return cudaErrorInvalidValue;
    const unsigned blocks = (unsigned)((a.n_envs + WIDE_THREADS - 1) / WIDE_THREADS);
    if (a.goal_mode == TS_GOAL_ORDERED) launch_wide_step_goal<T, TS_GOAL_ORDERED>(a, blocks, st);
    else launch_wide_step_goal<T, TS_GOAL_SET>(a, blocks, st);
    return cudaGetLastError();
}

#define TS_WIDE_SWITCH(CALL)                                   \
    switch (a.n_tiles) {                                       \
        case 1: CALL(1); break; case 2: CALL(2); break;        \
        case 3: CALL(3); break; case 4: CALL(4); break;        \
        case 5: CALL(5); break; case 6: CALL(6); break;        \
        case 7: CALL(7); break; case 8: CALL(8); break;        \
        default: return cudaErrorInvalidValue;                 \
    }

cudaError_t wide_step_dispatch(const ts_step_args& a, cudaStream_t st) {
#define CALL(T) return launch_wide_step<T>(a, st)
    TS_WIDE_SWITCH(CALL)
#undef CALL
    return cudaErrorInvalidValue;
}

cudaError_t wide_valid_dispatch(const ts_valid_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_envs + WIDE_THREADS - 1) / WIDE_THREADS);
#define CALL(T) wide_valid_kernel<T><<<blocks, WIDE_THREADS, 0, st>>>(a)
    TS_WIDE_SWITCH(CALL)
#undef CALL
    return cudaGetLastError();
}

template <int T> static void launch_wide_expand(const ts_expand_args& a, unsigned blocks, cudaStream_t st) {
    switch (wide_line_words(a.size)) {
        case 5: wide_expand_kernel<T, 5><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        case 6: wide_expand_kernel<T, 6><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        case 7: wide_expand_kernel<T, 7><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        default: wide_expand_kernel<T, 8><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
    }
}

cudaError_t wide_expand_dispatch(const ts_expand_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_items + WIDE_THREADS - 1) / WIDE_THREADS);
#define CALL(T) launch_wide_expand<T>(a, blocks, st)
    TS_WIDE_SWITCH(CALL)
#undef CALL
    return cudaGetLastError();
}

template <int T, int POLICY> static void launch_wide_playout(const ts_playout_args& a, unsigned blocks, cudaStream_t st) {
    switch (wide_line_words(a.size)) {
        case 5: wide_playout_kernel<T, 5, POLICY><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        case 6: wide_playout_kernel<T, 6, POLICY><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        case 7: wide_playout_kernel<T, 7, POLICY><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
        default: wide_playout_kernel<T, 8, POLICY><<<blocks, WIDE_THREADS, 0, st>>>(a); break;
    }
}

cudaError_t wide_playout_dispatch(const ts_playout_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_items + WIDE_THREADS - 1) / WIDE_THREADS);
#define CALL(T)                                                                                              \
    if (a.policy == TS_PLAYOUT_RANDOM) launch_wide_playout<T, TS_PLAYOUT_RANDOM>(a, blocks, st);             \
    else launch_wide_playout<T, TS_PLAYOUT_PLAN>(a, blocks, st)
    TS_WIDE_SWITCH(CALL)
#undef CALL
    return cudaGetLastError();
}

cudaError_t wide_goal_dispatch(const ts_goal_args& a, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.n_envs + WIDE_THREADS - 1) / WIDE_THREADS);
#define CALL(T) wide_goal_kernel<T><<<blocks, WIDE_THREADS, 0, st>>>(a)
    TS_WIDE_SWITCH(CALL)
#undef CALL
    return cudaGetLastError();
}

}  // namespace ts
