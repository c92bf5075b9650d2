// ts_bfs_local.cu -- K6: breadth-first search of MANY SMALL puzzles, one CTA per puzzle, entirely
// on chip (BASELINE config 5 for batches).
//
// Why: dedup is per puzzle and a puzzle is small (6x6 / 4 tiles / 8 walls: 3,300 states on
// average, < 2e4 at the 99.9th percentile), yet the hash-partitioned search (ts_bfs.cu) sends
// every successor to one visited table in HBM -- one random 32-byte sector (and its write-back)
// per successor, 9 % of the HBM roofline.  Here the visited set of a puzzle never leaves the SM:
//   * it is a BITMAP over a perfect hash of the state: a tile can only stand on one of the F free
//     cells of ITS puzzle, so state -> sum(rank(tile i) * F^i) with rank = index of the cell
//     among the free cells NOT TAKEN BY TILES 0..i-1 (mixed radix F, F-1, ...) is collision free, and
//     F!/(F-T)! bits fit shared memory (28*27*26*25 bits = 60 KB for the benchmark shape, three CTAs
//     per SM; 5 KB for the reference's real levels).  Dedup = one shared-memory atomicOr per
//     successor, no probing, no table overflow;
//   * the frontier is an append-only queue of 32-bit states in discovery order (= BFS order); the
//     level being expanded and the one being appended live in a shared-memory ring, whatever
//     exceeds it spills to a per-CTA slab in HBM with purely sequential traffic; level boundaries
//     are two indices;
//   * persistent CTAs draw puzzles from a ticket counter (puzzle sizes vary 100x).
// Thread = one (state, move) pair, so a level of n states offers 4n-way parallelism; new states
// are appended with one shared-memory atomic per warp; one __syncthreads per level (three rotating
// per-level counters).  Successor function = GameState.move (explainrl/environment/state.py:
// 120-170) through slide_env<S,T>, goal test = is_won (state.py:172-186): the same device code as
// the step kernel.  Semantics identical to the hash-partitioned search: set-goal states are
// canonicalised by sorting, the solve depth is the first depth at which ANY successor (new or not)
// meets the goal.  BFS itself has no counterpart in the reference (parity unpinned; results pinned
// to a plain BFS over the reference's move, tests/golden/).
//
// A puzzle that does not fit (F^T bits above the bitmap the launch was given, queue spill
// exhausted) is reported in d_status and left to the hash-partitioned search.
#include "ts_bfs_local.cuh"

namespace ts {

template <int S, int T>
__global__ void __launch_bounds__(SEARCH_THREADS) bfs_local_kernel(const ts_bfs_local_args a) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    static_assert(T >= 1 && T <= 4, "32-bit states");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = dyn;
    uint32_t* const queue = dyn + a.bitmap_words;
#include "ts_bfs_local_body.inc"
}


// Device instance of K6 (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh): CTA b's bitmap is
// d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.  A CTA alone touches its
// slice, and __syncthreads orders the block's global accesses as it orders its shared ones.
template <int S, int T>
__global__ void __launch_bounds__(SEARCH_THREADS) bfs_local_gmem_kernel(const ts_bfs_local_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    static_assert(gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words;
    uint32_t* const queue = dyn;
#include "ts_bfs_local_body.inc"
}

static constexpr auto K6 = [](auto S, auto T) { return bfs_local_kernel<decltype(S)::value, decltype(T)::value>; };
static constexpr auto K6_GMEM = [](auto S, auto T) { return bfs_local_gmem_kernel<decltype(S)::value, decltype(T)::value>; };

}  // namespace ts

using namespace ts;

static int local_check(const ts_bfs_local_args* a) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > 8) return TS_E_UNSUPPORTED;
    if (int rc = check_search_plan(*a)) return rc;
    return a->spill_per_cta < 0 ? TS_E_BAD_ARGUMENT : 0;
}

// the checks of a launch before its empty-batch return
static int local_launch_check(const ts_bfs_local_args* a) {
    if (int rc = local_check(a)) return rc;
    if (a->n_puzzles < 0 || a->puzzle_capacity <= 0 || a->puzzle_capacity % CAP_ALIGN || a->max_depth < 0 || a->n_levels < 1) return TS_E_BAD_ARGUMENT;
    if (!a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_states_per_puzzle || !a->d_solve_depth || !a->d_status ||
        !a->d_levels || !a->d_counters || (a->spill_per_cta && !a->d_spill))
        return TS_E_NULL_POINTER;
    if (a->d_lengths && (!a->d_moves || !a->d_parent_scratch || a->max_moves < 1)) return TS_E_NULL_POINTER;
    return 0;
}

extern "C" {

int ts_bfs_local_smem_bytes(const ts_bfs_local_args* a) {
    if (int rc = local_check(a)) return rc;
    return (int)search_smem_bytes(*a);
}

int ts_bfs_local_ctas_per_sm(const ts_bfs_local_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = local_check(a)) return rc;
    return search_ctas_per_sm(K6, *a, ctas_per_sm, n_sm);
}

int ts_bfs_local(const ts_bfs_local_args* a, int grid, void* stream) {
    if (int rc = local_launch_check(a)) return rc;
    if (a->n_puzzles == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)search_kernel(K6, *a, grid, nullptr, (cudaStream_t)stream);
}

int ts_bfs_local_gmem_ctas_per_sm(const ts_bfs_local_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = local_check(a)) return rc;
    return search_gmem_ctas_per_sm(K6_GMEM, *a, ctas_per_sm, n_sm);
}

int ts_bfs_local_gmem(const ts_bfs_local_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = local_launch_check(a)) return rc;
    if (int rc = check_gmem(*a, d_bitmap)) return rc;
    if (a->n_puzzles == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)search_gmem_kernel(K6_GMEM, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
