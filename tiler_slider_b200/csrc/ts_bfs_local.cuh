// ts_bfs_local.cuh -- device helpers of the on-chip searches (K6 ts_bfs_local.cu, K9 ts_optimal.cu):
// canonical set-goal states, position byte -> bitboard bit, and the perfect hash of a state over the
// free cells of its puzzle that keys the shared-memory bitmap.
#pragma once
#include "ts_common.cuh"

namespace ts {

// canonical form of a set-goal state: its T position bytes sorted ascending (tiles are interchangeable)
template <int T> __device__ __forceinline__ void sort_bytes4(uint32_t& q) {
    uint32_t b[T];
    static_for<0, T>([&](auto I) { constexpr int i = decltype(I)::value; b[i] = byte_of<i>(q); });
#pragma unroll
    for (int round = 0; round < T; ++round)
#pragma unroll
        for (int i = round & 1; i + 1 < T; i += 2) {
            const uint32_t lo = min(b[i], b[i + 1]), hi = max(b[i], b[i + 1]);
            b[i] = lo; b[i + 1] = hi;
        }
    q = 0;
    static_for<0, T>([&](auto I) { constexpr int i = decltype(I)::value; q |= b[i] << (8 * i); });
}

// bitboard bit of position byte p
template <int S> __device__ __forceinline__ uint32_t pos_to_bit(uint32_t p) {
    if constexpr (padded_board(S)) return p;                       // stride S+1 both ways
    else return (p >> 4) * (uint32_t)S + (p & 15u);
}
template <int S> __host__ __device__ constexpr uint64_t cell_mask() {
    uint64_t m = 0;
    for (int r = 0; r < S; ++r)
        for (int c = 0; c < S; ++c) m |= 1ull << (r * board_stride(S) + c);
    return m;
}

// perfect hash of a state: its tiles stand on DISTINCT free cells, so digit i = rank of tile i
// among the cells not taken by tiles 0..i-1, mixed radix F, F-1, ... (28^4 bits would not leave
// room for three CTAs per SM, 28*27*26*25 bits do).  lut = position byte -> rank among the free cells.
template <int T> __device__ __forceinline__ uint32_t state_index(const uint8_t (&lut)[128], uint32_t F, uint32_t q) {
    uint32_t r[T];
    static_for<0, T>([&](auto I) { constexpr int i = decltype(I)::value; r[i] = lut[byte_of<i>(q)]; });
    uint32_t idx = 0;
    static_for<0, T>([&](auto I) {
        constexpr int i = T - 1 - decltype(I)::value;          // most significant digit first
        uint32_t d = r[i];
#pragma unroll
        for (int j = 0; j < i; ++j) d -= (r[j] < r[i]) ? 1u : 0u;
        idx = idx * (F - (uint32_t)i) + d;
    });
    return idx;
}

}  // namespace ts
