// ts_optimal.cu -- K9: exact distance to the goal and the set of optimal first moves of many items
// (env id, positions: the env's current ones or a caller's word), one CTA per item, on chip, and
// optionally a shortest solution per item.  Built on K6's machinery (ts_bfs_local.cu; the CTA
// shape, hash, plan check and launch are in ts_bfs_local.cuh): persistent CTAs drawing items from a
// ticket counter, the visited set a shared-memory bitmap over the perfect hash of a state among the
// free cells of its puzzle, the frontier ring with a per-CTA HBM slab, the successor function
// slide_env<S,T> and goal test of the step.
//
//   0. Root: the item's word must be a well-formed state (every tile on an in-board free cell, no
//      two on one cell), else TS_OPT_BAD_STATE -- the hash below is only defined for those.
//   1. Forward: BFS from the root (set goal: states canonicalised by sorting), stopped
//      after the level in which a successor first meets the goal; that level number is d.  Every
//      state appended is also written to the slab (the ring only holds the levels in flight), so
//      that levels 1 .. d-1 can be read again; their boundaries stay in shared memory.
//   2. Backward: the bitmap is cleared and keyed again by the same hash, now as the set of "good"
//      states, those from which a shortest solution continues.  Level d-1: good when some move
//      wins.  Level k = d-2 .. 1: good when some successor that differs from it is marked.  A
//      successor of a level-k state lies at level <= k+1, so only level k+1's marks can be hit; the
//      marks of level k itself must not be (a same-level successor is one step farther from the
//      goal), so all flags of level k are computed first (written over the level's slab entries)
//      and set after a barrier.  One bitmap serves every level without clearing.  A good state's
//      slab entry is its hash << 2 | the lowest of those moves (only levels > k are marked, so they
//      are exactly its optimal moves); the mark loop reads entry >> 2.
//   3. Root: d == 1: the moves that win; otherwise the moves whose successor is marked (the root is
//      never marked, so a move that changes nothing is never optimal there).
//   4. Plan (d_plan set): from the root, play the lowest optimal move; the state reached at level k
//      is good, so level k's slab range holds its entry, and that entry's move is the next one.
//      This gives the lexicographically smallest shortest solution (UP < DOWN < LEFT < RIGHT).
// The forward pass stops at the goal level instead of enumerating the reachable set, and the
// backward pass slides each state of levels 1 .. d-1 once more.  No reference counterpart (parity
// unpinned; results pinned to a plain CPU BFS, tests/test_gpu_optimal.py).
#include "ts_bfs_local.cuh"

namespace ts {

constexpr uint32_t OPT_NONE = 0xFFFFFFFFu;
constexpr uint32_t WON = 1u, OVER = 2u;

// PLAN: the instance that writes d_plan (a compile-time parameter, so that the query without plans
// carries none of the plan's code: its slab entries are bare hashes, as they were before plans)
template <int S, int T, bool PLAN>
__global__ void __launch_bounds__(SEARCH_THREADS) optimal_moves_kernel(const ts_optimal_moves_args a) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    constexpr uint32_t KEY_SHIFT = PLAN ? 2u : 0u;        // slab entry of a good state: hash << KEY_SHIFT | move
    static_assert(T >= 1 && T <= 4, "32-bit states");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = dyn;
    uint32_t* const queue = dyn + a.bitmap_words;
#include "ts_optimal_body.inc"
}

// the most free cells among the listed envs (sizes the bitmap of a launch)
template <int S>
__global__ void max_free_cells_kernel(const ts_optimal_moves_args a, int32_t* out) {
    constexpr int NB = board_bytes(S);
    uint32_t best = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n_items; i += (long long)gridDim.x * blockDim.x) {
        const long long env = a.d_env_ids ? (long long)a.d_env_ids[i] : i;
        if (env < 0 || env >= a.capacity) continue;
        const uint64_t walls = load_board_elem<NB>(a.d_walls, (size_t)a.capacity, (size_t)env);
        best = max(best, (uint32_t)__popcll(~walls & cell_mask<S>()));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) best = max(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if ((threadIdx.x & 31u) == 0u && best) atomicMax(out, (int32_t)best);
}

// Device instance of K9 (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh): CTA b's bitmap is
// d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.  __syncthreads orders the
// block's global accesses as it orders its shared ones, so the flag / mark phases of the backward
// pass need no fence.  The largest hash is 64*63*62*61 - 1 < 15,249,024 (F = 64), so a plan's slab
// entry hash << 2 | move stays below 2^26.
// (at least 5 CTAs per SM: without that bound ptxas takes 40 registers for two of the four instances
// and spills 16 bytes; with it they take 45-48 and none spill)
template <int S, int T, bool PLAN>
__global__ void __launch_bounds__(SEARCH_THREADS, 5) optimal_moves_gmem_kernel(const ts_optimal_moves_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    constexpr uint32_t KEY_SHIFT = PLAN ? 2u : 0u;        // slab entry of a good state: hash << KEY_SHIFT | move
    static_assert(gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words;
    uint32_t* const queue = dyn;
#include "ts_optimal_body.inc"
}

static constexpr auto K9 = [](auto S, auto T) { return optimal_moves_kernel<decltype(S)::value, decltype(T)::value, false>; };
static constexpr auto K9_PLAN = [](auto S, auto T) { return optimal_moves_kernel<decltype(S)::value, decltype(T)::value, true>; };
static constexpr auto K9_GMEM = [](auto S, auto T) { return optimal_moves_gmem_kernel<decltype(S)::value, decltype(T)::value, false>; };
static constexpr auto K9_GMEM_PLAN = [](auto S, auto T) { return optimal_moves_gmem_kernel<decltype(S)::value, decltype(T)::value, true>; };

}  // namespace ts

using namespace ts;

// shape and shared-memory plan
static int optimal_check_plan(const ts_optimal_moves_args* a) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;                                 // wide boards: no 64-bit board word
    return check_search_plan(*a);
}

// the env table the listed envs are read from
static int optimal_check_table(const ts_optimal_moves_args* a) {
    if (a->capacity <= 0 || a->capacity % TS_CAP_ALIGN) return TS_E_BAD_CAPACITY;
    if (a->n_items < 0 || (!a->d_env_ids && a->n_items > a->capacity)) return TS_E_BAD_RANGE;
    if (!a->d_walls || !a->d_targets_packed || !a->d_pos) return TS_E_NULL_POINTER;
    return 0;
}

// the checks of a launch before its empty-query return
static int optimal_check_launch(const ts_optimal_moves_args* a) {
    if (int rc = optimal_check_plan(a)) return rc;
    if (int rc = optimal_check_table(a)) return rc;
    if (a->max_depth < 1 || a->max_depth > TS_OPT_MAX_DEPTH || a->spill_per_cta < 1 || a->spill_per_cta > 0xFFFFFFFFll)
        return TS_E_BAD_ARGUMENT;
    if (!a->d_spill || !a->d_counters || !a->d_distance || !a->d_mask) return TS_E_NULL_POINTER;
    return 0;
}

extern "C" {

int ts_optimal_moves_smem_bytes(const ts_optimal_moves_args* a) {
    if (int rc = optimal_check_plan(a)) return rc;
    return (int)search_smem_bytes(*a);
}

int ts_optimal_moves_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = optimal_check_plan(a)) return rc;
    return a->d_plan ? search_ctas_per_sm(K9_PLAN, *a, ctas_per_sm, n_sm) : search_ctas_per_sm(K9, *a, ctas_per_sm, n_sm);
}

int ts_optimal_max_free_cells(const ts_optimal_moves_args* a, int32_t* d_max_free, void* stream) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;
    if (int rc = optimal_check_table(a)) return rc;
    if (!d_max_free) return TS_E_NULL_POINTER;
    if (a->n_items == 0) return 0;
    const long long blocks = (a->n_items + 255) / 256;
    return (int)dispatch_size(a->size, [&](auto S) {
        max_free_cells_kernel<decltype(S)::value><<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, (cudaStream_t)stream>>>(*a, d_max_free);
        return cudaGetLastError();
    });
}

int ts_optimal_moves(const ts_optimal_moves_args* a, int grid, void* stream) {
    if (int rc = optimal_check_launch(a)) return rc;
    if (a->n_items == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)(a->d_plan ? search_kernel(K9_PLAN, *a, grid, nullptr, (cudaStream_t)stream)
                           : search_kernel(K9, *a, grid, nullptr, (cudaStream_t)stream));
}

int ts_optimal_moves_gmem_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = optimal_check_plan(a)) return rc;
    return a->d_plan ? search_gmem_ctas_per_sm(K9_GMEM_PLAN, *a, ctas_per_sm, n_sm) : search_gmem_ctas_per_sm(K9_GMEM, *a, ctas_per_sm, n_sm);
}

int ts_optimal_moves_gmem(const ts_optimal_moves_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = optimal_check_launch(a)) return rc;
    if (int rc = check_gmem(*a, d_bitmap)) return rc;
    if (a->n_items == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)(a->d_plan ? search_gmem_kernel(K9_GMEM_PLAN, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream)
                           : search_gmem_kernel(K9_GMEM, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream));
}

}  // extern "C"
