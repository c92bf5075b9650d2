// ts_synth.cuh -- device code shared by the load-time kernels of ts_api.cu (K1 ts_encode, K0
// ts_synth) and the puzzle generator of ts_generate.cu: the board writers and K0's draw.
//
// Reference map (paths relative to the reference checkout):
//   synth_env   explainrl/environment/environment.py:221-226  create_simple_env recipe
#pragma once
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

// value of bit `bit` of a stored WALL board: blocked cells, plus (padded boards) the sentinel
// column S of every row and every bit past the last row
__device__ __forceinline__ int wall_bit(const uint8_t* blocked_cells, int S, int bit) {
    const int bs = board_stride(S);
    const int r = bit / bs, c = bit % bs;
    if (r >= S) return padded_board(S) ? 1 : 0;
    if (c >= S) return 1;
    return blocked_cells[r * S + c] ? 1 : 0;
}

// Write the wall board(s) of one env from a 0/1 cell map (all three board classes).
__device__ inline void store_walls(uint8_t* d_walls, size_t cap, size_t env, int S, const uint8_t* cellmap) {
    if (wide_board(S)) {
        const int lines = 2 * wide_line_words(S);      // S rounded up to even
        uint16_t* w = reinterpret_cast<uint16_t*>(d_walls) + env * lines;   // [axis][env][line]
        const size_t plane = cap * lines;
        const int lead = wide_line_lead(S);           // S <= 14: cells at bits 1..S between two sentinels
        for (int l = 0; l < lines; ++l) {
            uint32_t col = 0, row = 0;
            if (l < S && lead) col = row = 1u | (1u << (S + 1));   // edge sentinels (ts_wide.cu)
            if (l < S)
                for (int k = 0; k < S; ++k) {
                    if (cellmap[k * S + l]) col |= 1u << (k + lead);    // column l, bit = row
                    if (cellmap[l * S + k]) row |= 1u << (k + lead);    // row l, bit = column
                }
            w[0 * plane + l] = (uint16_t)col;
            w[1 * plane + l] = (uint16_t)row;
        }
        return;
    }
    const int nb = board_bytes(S);
    for (int b = 0; b < nb; ++b) {
        uint32_t v = 0;
        for (int k = 0; k < 8; ++k) v |= (uint32_t)wall_bit(cellmap, S, 8 * b + k) << k;
        d_walls[board_byte_addr(nb, cap, env, b)] = (uint8_t)v;
    }
}

// Write the set-goal target board of one env from its target cells (row*S+col each).
__device__ inline void store_target_board(uint8_t* d_tb, size_t cap, size_t env, int S, int T, const int* cells, int n) {
    if (wide_board(S)) {
        uint16_t rows[16];
        for (int r = 0; r < 16; ++r) rows[r] = 0;
        for (int t = 0; t < n; ++t) rows[cells[t] / S] |= (uint16_t)(1u << (cells[t] % S));
        int distinct = 0;
        for (int r = 0; r < 16; ++r) distinct += __popc((uint32_t)rows[r]);
        // the wide kernels test "every tile on a target cell"; that is set equality only when
        // there are exactly T distinct targets (state.py:185-186): the count travels in word 16
        uint16_t* o = reinterpret_cast<uint16_t*>(d_tb) + env * WIDE_TARGET_WORDS;
        for (int r = 0; r < 16; ++r) o[r] = rows[r];
        o[16] = (uint16_t)distinct;
        return;
    }
    const int nb = board_bytes(S), bs = board_stride(S);
    for (int b = 0; b < nb; ++b) {
        uint32_t v = 0;
        for (int t = 0; t < n; ++t) {
            const int bit = (cells[t] / S) * bs + (cells[t] % S);
            if ((bit >> 3) == b) v |= 1u << (bit & 7);
        }
        d_tb[board_byte_addr(nb, cap, env, b)] = (uint8_t)v;
    }
}

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// K0's random stream of the env with global index `gidx`: a counter-based hash of (seed, gidx)
__device__ __forceinline__ uint64_t synth_stream(uint64_t seed, uint64_t gidx) {
    uint64_t rng = seed ^ (0xD1B54A32D192ED03ull * (gidx + 1));
    splitmix64(rng);
    return rng;
}

// The first `draws` entries of a uniformly random permutation of the `cells` cells (partial
// Fisher-Yates), one 32-bit draw of the stream per entry.
__device__ __forceinline__ void synth_cells(uint64_t& rng, int cells, int draws, uint8_t* perm) {
    for (int c = 0; c < cells; ++c) perm[c] = (uint8_t)c;
    for (int d = 0; d < draws; ++d) {  // partial Fisher-Yates: prefix of a uniform permutation
        const uint32_t r = (uint32_t)(splitmix64(rng) >> 32);
        const int j = d + (int)(((uint64_t)r * (uint32_t)(cells - d)) >> 32);
        const uint8_t t = perm[d];
        perm[d] = perm[j];
        perm[j] = t;
    }
}

// K0's puzzle for one env: the first W cells of the permutation blocked, the next T tiles, the
// next T targets; written to env slot `env` of the packed buffers.
__device__ inline void synth_env(int S, int T, int W, int goal_mode, uint64_t seed, uint64_t gidx, size_t cap, size_t env,
                                 uint8_t* d_walls, uint8_t* d_targets_packed, uint8_t* d_init, uint8_t* d_pos) {
    const int pw = pos_bytes(T), cells = S * S;
    uint64_t rng = synth_stream(seed, gidx);
    uint8_t perm[MAX_SIZE * MAX_SIZE];
    synth_cells(rng, cells, W + 2 * T, perm);
    const int ps = pos_stride(S);
    uint8_t cellmap[MAX_SIZE * MAX_SIZE];
    for (int c = 0; c < cells; ++c) cellmap[c] = 0;
    for (int d = 0; d < W; ++d) cellmap[perm[d]] = 1;
    store_walls(d_walls, cap, env, S, cellmap);
    for (int t = 0; t < pw; ++t) {
        uint8_t v = 0;
        if (t < T) { const int c = perm[W + t]; v = (uint8_t)((c / S) * ps + (c % S)); }
        d_init[env * pw + t] = v;
        d_pos[env * pw + t] = v;
    }
    if (goal_mode == TS_GOAL_ORDERED) {
        for (int t = 0; t < pw; ++t) {
            uint8_t v = 0;
            if (t < T) { const int c = perm[W + T + t]; v = (uint8_t)((c / S) * ps + (c % S)); }
            d_targets_packed[env * pw + t] = v;
        }
    } else {
        int tcells[MAX_TILES_ANY];
        for (int t = 0; t < T; ++t) tcells[t] = perm[W + T + t];
        store_target_board(d_targets_packed, cap, env, S, T, tcells, T);
    }
}

}  // namespace ts
