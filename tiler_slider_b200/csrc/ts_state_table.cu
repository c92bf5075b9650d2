// ts_state_table.cu -- K10: the state table of many items (env id, positions): every state reachable
// from the item's root, each with its exact distance to the goal and its optimal moves (K9's
// definitions), one CTA per item, on chip.  K6/K9's machinery (ts_bfs_local.cuh): persistent CTAs
// drawing items from a ticket counter, the visited set a shared-memory bitmap over the perfect hash
// of a state among the free cells of its puzzle, the frontier ring, slide_env<S,T> and the goal test.
// Two launches with one plan:
//
//   count  root check (TS_OPT_BAD_STATE, K9's rule), then a BFS to exhaustion; the ring spills to a
//          per-CTA slab.  Writes the number of states, or TS_OPT_NOT_SEARCHED.
//   fill   (the caller has turned the counts into row offsets) the same BFS, the item's own output
//          rows serving as the queue beyond the ring (their number is known: no slab, no overflow);
//          then
//     order      the rows are rewritten from the bitmap in ascending hash order: a block-wide scan of
//                the words' popcounts gives each set bit its row, and its index is decoded (mixed
//                radix digits -> ranks among the remaining free cells -> position bytes).  BFS order
//                within a level depends on atomics; this order does not.
//     sweep      retrograde rounds over the rows, the bitmap cleared and reused as the set of
//                resolved states.  Round r = 1, 2, ...: an unresolved row hits the moves that win
//                (r = 1) or whose successor differs from it and is marked (r >= 2); rows with a hit
//                get distance r and the hits as mask; after a barrier the rows resolved in round r
//                are marked.  A marked successor was resolved in round r-1 exactly (one resolved
//                earlier would have resolved the row earlier), so the mask is K9's.  The rows are
//                swept in place (not compacted): an unresolved row costs one load and compare per
//                lane a round, and compaction would need a second copy of the rows and a scan per
//                round.  The sweep stops after a round that resolves nothing; what is left is -1.
//                Skipped when no successor met the goal in the forward pass (never_win included).
// No reference counterpart (results pinned to K9 and a plain CPU BFS, tests/test_gpu_state_table.py).
#include "ts_bfs_local.cuh"

namespace ts {

namespace {
constexpr uint32_t TAB_OVER = 1u;

// a state word as the PW bytes of a row
template <int PW> __device__ __forceinline__ uint32_t load_row(const uint8_t* p) {
    if constexpr (PW == 4) return *reinterpret_cast<const uint32_t*>(p);
    else if constexpr (PW == 2) return *reinterpret_cast<const uint16_t*>(p);
    else return *p;
}
template <int PW> __device__ __forceinline__ void store_row(uint8_t* p, uint32_t q) {
    if constexpr (PW == 4) *reinterpret_cast<uint32_t*>(p) = q;
    else if constexpr (PW == 2) *reinterpret_cast<uint16_t*>(p) = (uint16_t)q;
    else *p = (uint8_t)q;
}
}  // namespace

// FILL: the second launch (rows, order, sweep); otherwise the count pass
template <int S, int T, bool FILL>
__global__ void __launch_bounds__(SEARCH_THREADS) state_table_kernel(const ts_state_table_args a) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S), WARPS = SEARCH_THREADS / 32;
    static_assert(T >= 1 && T <= 4, "32-bit states");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = dyn;
    uint32_t* const queue = dyn + a.bitmap_words;
#include "ts_state_table_body.inc"
}


// Device instance of K10 (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh): CTA b's bitmap is
// d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.  __syncthreads orders the
// block's global accesses as it orders its shared ones, so the mark phases of the sweep need no
// fence.  The order scan's index w * 32 + bit stays below 64*63*62*61 = 15,249,024 (F = 64).
template <int S, int T, bool FILL>
__global__ void __launch_bounds__(SEARCH_THREADS) state_table_gmem_kernel(const ts_state_table_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S), WARPS = SEARCH_THREADS / 32;
    static_assert(gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    uint32_t* const bitmap = d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words;
    uint32_t* const queue = dyn;
#include "ts_state_table_body.inc"
}

static constexpr auto K10_COUNT = [](auto S, auto T) { return state_table_kernel<decltype(S)::value, decltype(T)::value, false>; };
static constexpr auto K10_FILL = [](auto S, auto T) { return state_table_kernel<decltype(S)::value, decltype(T)::value, true>; };
static constexpr auto K10_GMEM_COUNT = [](auto S, auto T) { return state_table_gmem_kernel<decltype(S)::value, decltype(T)::value, false>; };
static constexpr auto K10_GMEM_FILL = [](auto S, auto T) { return state_table_gmem_kernel<decltype(S)::value, decltype(T)::value, true>; };

}  // namespace ts

using namespace ts;

// shape, shared-memory plan and the env table (the checks of ts_optimal_moves)
static int state_table_check(const ts_state_table_args* a, int grid) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;                                 // wide boards: no 64-bit board word
    if (int rc = check_search_plan(*a)) return rc;
    if (a->capacity <= 0 || a->capacity % TS_CAP_ALIGN) return TS_E_BAD_CAPACITY;
    if (a->n_items < 0 || (!a->d_env_ids && a->n_items > a->capacity)) return TS_E_BAD_RANGE;
    if (!a->d_walls || !a->d_targets_packed || !a->d_pos || !a->d_counters || !a->d_status) return TS_E_NULL_POINTER;
    if (a->n_items > 0 && grid < 1) return TS_E_BAD_ARGUMENT;
    return 0;
}

// the launch checks of each pass before its empty-query return
static int count_check(const ts_state_table_args* a, int grid) {
    if (int rc = state_table_check(a, grid)) return rc;
    if (a->spill_per_cta < 1 || a->spill_per_cta > 0xFFFFFFFFll) return TS_E_BAD_ARGUMENT;
    if (!a->d_spill || !a->d_count) return TS_E_NULL_POINTER;
    return 0;
}
static int fill_check(const ts_state_table_args* a, int grid) {
    if (int rc = state_table_check(a, grid)) return rc;
    if (!a->d_offsets || !a->d_rows || !a->d_distance || !a->d_mask) return TS_E_NULL_POINTER;
    return 0;
}
// shape and shared-memory plan (the occupancy queries)
static int occupancy_check(const ts_state_table_args* a) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;
    return check_search_plan(*a);
}

extern "C" {

int ts_state_table_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = occupancy_check(a)) return rc;
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    int count = 0, fill = 0;
    if (int rc = search_ctas_per_sm(K10_COUNT, *a, &count, n_sm)) return rc;
    if (int rc = search_ctas_per_sm(K10_FILL, *a, &fill, n_sm)) return rc;
    *ctas_per_sm = count < fill ? count : fill;
    return 0;
}

int ts_state_table_count(const ts_state_table_args* a, int grid, void* stream) {
    if (int rc = count_check(a, grid)) return rc;
    if (a->n_items == 0) return 0;
    return (int)search_kernel(K10_COUNT, *a, grid, nullptr, (cudaStream_t)stream);
}

int ts_state_table_fill(const ts_state_table_args* a, int grid, void* stream) {
    if (int rc = fill_check(a, grid)) return rc;
    if (a->n_items == 0) return 0;
    return (int)search_kernel(K10_FILL, *a, grid, nullptr, (cudaStream_t)stream);
}

int ts_state_table_gmem_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = occupancy_check(a)) return rc;
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    int count = 0, fill = 0;
    if (int rc = search_gmem_ctas_per_sm(K10_GMEM_COUNT, *a, &count, n_sm)) return rc;
    if (int rc = search_gmem_ctas_per_sm(K10_GMEM_FILL, *a, &fill, n_sm)) return rc;
    *ctas_per_sm = count < fill ? count : fill;
    return 0;
}

int ts_state_table_count_gmem(const ts_state_table_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = count_check(a, grid)) return rc;
    if (int rc = check_gmem(*a, d_bitmap)) return rc;
    if (a->n_items == 0) return 0;
    return (int)search_gmem_kernel(K10_GMEM_COUNT, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream);
}

int ts_state_table_fill_gmem(const ts_state_table_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = fill_check(a, grid)) return rc;
    if (int rc = check_gmem(*a, d_bitmap)) return rc;
    if (a->n_items == 0) return 0;
    return (int)search_gmem_kernel(K10_GMEM_FILL, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
