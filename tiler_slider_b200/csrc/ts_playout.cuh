// ts_playout.cuh -- device code shared by the three ts_playout kernels (ts_playout.cu, ts_wide.cu,
// ts_generic.cu): the random policy's draw and the optional per-move records.
#pragma once
#include "ts_synth.cuh"

namespace ts {

// The move K7's walk rule (ts_generate.cu) draws from `mask` (bit d set: move d changes the
// positions; not 0): one 32-bit draw r of the stream, then the floor(r*n / 2^32)-th of the n set
// bits, lowest first.
__device__ __forceinline__ uint32_t draw_move(uint64_t& rng, uint32_t mask) {
    const uint32_t r = (uint32_t)(splitmix64(rng) >> 32);
    for (int k = (int)(((uint64_t)r * (uint32_t)__popc(mask)) >> 32); k > 0; --k) mask &= mask - 1u;
    return (uint32_t)(__ffs(mask) - 1);
}

// element k (step-major) of item i in the [n_steps][n_items] record arrays
__device__ __forceinline__ size_t playout_row(const ts_playout_args& a, int k, int64_t i) {
    return (size_t)k * (size_t)a.n_items + (size_t)i;
}

// the optional records of move k of item i: the move played and the positions after it
template <int PW>
__device__ __forceinline__ void playout_record(const ts_playout_args& a, int k, int64_t i, uint32_t d, const uint32_t (&q)[(PW + 3) / 4]) {
    const size_t row = playout_row(a, k, i);
    if (a.d_moves) __stcs(a.d_moves + row, (unsigned char)d);
    if (a.d_traj) st_pos<PW>(a.d_traj, row, q);
}

// the records of the moves k = from .. n_steps-1 that item i did not play: 255 and zero positions
template <int PW> __device__ __forceinline__ void playout_tail(const ts_playout_args& a, int from, int64_t i) {
    if (!a.d_moves && !a.d_traj) return;
    const uint32_t zero[(PW + 3) / 4] = {};
    for (int k = from; k < a.n_steps; ++k) playout_record<PW>(a, k, i, 255u, zero);
}

}  // namespace ts
