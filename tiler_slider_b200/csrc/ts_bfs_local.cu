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
// the step kernel, in the successor function K9 and K10 share (ts_bfs_local.cuh).  Semantics
// identical to the hash-partitioned search: set-goal states are canonicalised by sorting, the solve
// depth is the first depth at which ANY successor (new or not) meets the goal.  BFS itself has no counterpart in the reference (parity unpinned; results pinned
// to a plain BFS over the reference's move, tests/golden/).
//
// A puzzle that does not fit (F^T bits above the bitmap the launch was given, queue spill
// exhausted) is reported in d_status and left to the hash-partitioned search.  7x7 and 8x8 boards
// with four tiles also have a device instance (GMEM), whose bitmap is in device memory and may hold
// every state space of those boards (ts_bfs_local.cuh).
#include "ts_bfs_local.cuh"

namespace ts {

// GMEM: the device instance (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh)
template <int S, int T, bool GMEM>
__global__ void __launch_bounds__(SEARCH_THREADS) bfs_local_kernel(const ts_bfs_local_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    static_assert(T >= 1 && T <= 4, "32-bit states");
    static_assert(!GMEM || gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    // GMEM: CTA b's bitmap is d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.  A
    // CTA alone touches its slice, and __syncthreads orders the block's global accesses as it orders
    // its shared ones.
    uint32_t* const bitmap = GMEM ? d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words : dyn;
    uint32_t* const queue = GMEM ? dyn : dyn + a.bitmap_words;
    __shared__ uint8_t lut[128];                 // position byte -> rank among the free cells
    __shared__ uint32_t hist[SEARCH_LEVELS];     // new states per depth, all puzzles this CTA completed
    __shared__ uint32_t plevel[SEARCH_LEVELS];   // ... of the puzzle in flight (added to hist when it completes)
    __shared__ uint32_t cnt[3];                  // entries appended during level L: cnt[L % 3]
    __shared__ uint32_t s_solve, s_over;
    __shared__ unsigned long long s_goal;        // with paths: (parent index << 2 | move) of a goal successor at the solve depth
    __shared__ long long s_ticket;

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    // The queue's shared-memory part is a RING over discovery indices (queue_smem = R, a power of two):
    // BFS only ever reads the level being expanded and appends the next one, so an entry p is kept
    // in ring[p % R] when it is appended within R of the start of the level being expanded (lo), and
    // in the HBM slab spill[p] otherwise; one level later the reader applies the same test with that
    // level's lo (prev_lo).  An append to slot p % R overwrites entry p - R < lo: consumed long ago.
    const uint32_t R = (uint32_t)a.queue_smem, RMASK = R - 1u;
    uint32_t* const spill = a.d_spill + (size_t)blockIdx.x * (size_t)a.spill_per_cta;
    uint32_t* const parents = a.d_parent_scratch ? a.d_parent_scratch + (size_t)blockIdx.x * (size_t)a.spill_per_cta : nullptr;
    const uint32_t q_cap = (uint32_t)a.spill_per_cta;       // discovery indices the slabs can address
    for (uint32_t k = tid; k < SEARCH_LEVELS; k += SEARCH_THREADS) hist[k] = 0;
    unsigned long long generated = 0;            // thread 0: successors generated by completed puzzles
    uint32_t deepest = 0;

    for (;;) {
        __syncthreads();                         // the previous puzzle is finished with shared memory
        if (tid == 0) s_ticket = (long long)atomicAdd((unsigned long long*)&a.d_counters[0], 1ull);
        __syncthreads();
        const long long ticket = s_ticket;
        if (ticket >= a.n_puzzles) break;
        const size_t pid = a.d_puzzle_ids ? (size_t)a.d_puzzle_ids[ticket] : (size_t)ticket;
        const size_t cap = (size_t)a.puzzle_capacity;

        // ---- the puzzle: walls, goal, initial state, free-cell ranks ---------------------------
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, pid);
        uint64_t tboard = 0;
        uint32_t tq = 0, q_init = 0;
        if (a.goal_mode == TS_GOAL_SET) tboard = load_board_elem<NB>(a.d_targets_packed, cap, pid);
        else static_for<0, T>([&](auto I) { constexpr int t = decltype(I)::value; tq |= (uint32_t)a.d_targets_packed[pid * PW + t] << (8 * t); });
        static_for<0, T>([&](auto I) { constexpr int t = decltype(I)::value; q_init |= (uint32_t)a.d_init[pid * PW + t] << (8 * t); });
        if (a.goal_mode == TS_GOAL_SET) sort_bytes4<T>(q_init);
        const uint64_t free_cells = ~walls & cell_mask<S>();
        const uint32_t F = (uint32_t)__popcll(free_cells);
        fill_lut<S>(tid, free_cells, lut);
        // states = arrangements of T distinct tiles on F cells: F (F-1) ... (F-T+1) bits
        unsigned long long bits = 1;
#pragma unroll
        for (int t = 0; t < T; ++t) bits *= (F > (uint32_t)t ? F - (uint32_t)t : 1u);
        const uint32_t words = (uint32_t)((bits + 31) / 32);
        if (words > (uint32_t)a.bitmap_words) {     // does not fit this launch: left to the hash-partitioned search
            if (tid == 0) a.d_status[pid] = 1;
            continue;
        }
        clear_bitmap(bitmap, words, tid);
        if (tid == 0) { cnt[0] = cnt[1] = cnt[2] = 0; s_solve = 0xFFFFFFFFu; s_over = 0; s_goal = ~0ull; }
        __syncthreads();

        // perfect hash of a state over the puzzle's free cells (ts_bfs_local.cuh)
        auto state_index = [&](uint32_t q) { return ts::state_index<T>(lut, F, q); };

        if (tid == 0) {
            const uint32_t idx = state_index(q_init);
            bitmap[idx >> 5] |= 1u << (idx & 31u);
            queue[0] = q_init;
            if (parents) parents[0] = 0xFFFFFFFFu;
            plevel[0] = 1;
        }
        __syncthreads();

        uint32_t lo = 0, hi = 1, depth = 0, prev_lo = 0;
        unsigned long long gen_p = 0;
        bool too_deep = false;
        while (lo < hi && depth < (uint32_t)a.max_depth) {
            if (depth + 1u >= SEARCH_LEVELS) { too_deep = true; break; }
            uint32_t* const my_cnt = &cnt[depth % 3u];
            if (tid == 0) cnt[(depth + 1u) % 3u] = 0;
            const uint32_t n_items = (hi - lo) * 4u;
            for (uint32_t base = 0; base < n_items; base += SEARCH_THREADS) {
                const uint32_t j = base + tid;
                const bool live = j < n_items;
                const uint32_t src = lo + (j >> 2), d = j & 3u;
                bool is_new = false;
                uint32_t qn = 0;
                if (live) {
                    const uint32_t q0 = (src - prev_lo) < R ? queue[src & RMASK] : spill[src];
                    bool won;
                    qn = successor<S, T>(q0, d, walls, a.goal_mode == TS_GOAL_SET, tboard, tq, won);
                    won &= a.never_win == 0;
                    if (won) {
                        const uint32_t before = atomicMin(&s_solve, depth + 1u);
                        if (parents && before > depth + 1u) atomicMin(&s_goal, ((unsigned long long)(depth + 1u) << 32) | ((unsigned long long)src << 2) | d);
                    }
                    if (qn != q0) {               // an unchanged state is its own (visited) parent
                        const uint32_t idx = state_index(qn);
                        const uint32_t bit = 1u << (idx & 31u);
                        is_new = (atomicOr(&bitmap[idx >> 5], bit) & bit) == 0;
                    }
                }
                const unsigned m = __ballot_sync(0xFFFFFFFFu, is_new);
                if (m) {
                    uint32_t pos = 0;
                    if (lane == (uint32_t)(__ffs(m) - 1)) pos = atomicAdd(my_cnt, (uint32_t)__popc(m));
                    pos = __shfl_sync(0xFFFFFFFFu, pos, __ffs(m) - 1);
                    if (is_new) {
                        pos += hi + (uint32_t)__popc(m & ((1u << lane) - 1u));
                        if (pos - lo < R) queue[pos & RMASK] = qn;
                        else if (pos < q_cap) spill[pos] = qn;
                        else s_over = 1;
                        if (parents) {
                            if (pos < q_cap) parents[pos] = (src << 2) | d;
                            else s_over = 1;
                        }
                    }
                }
            }
            __syncthreads();
            const uint32_t n_new = *my_cnt;
            gen_p += 4ull * (hi - lo);
            prev_lo = lo;
            lo = hi;
            hi += n_new;
            ++depth;
            if (s_over) break;
            if (tid == 0) plevel[depth] = n_new;
        }
        if (s_over || too_deep) {                 // spill slab exhausted / deeper than the level buffer: left to the hash-partitioned search
            if (tid == 0) a.d_status[pid] = s_over ? 2 : 3;
            continue;
        }
        __syncthreads();                          // plevel complete
        for (uint32_t k = tid; k <= depth; k += SEARCH_THREADS) hist[k] += plevel[k];
        if (tid == 0) {
            generated += gen_p;
            a.d_status[pid] = 0;
            a.d_states_per_puzzle[pid] = (long long)hi;
            const uint32_t sd = s_solve;
            a.d_solve_depth[pid] = sd == 0xFFFFFFFFu ? -1 : (int32_t)sd;
            deepest = max(deepest, depth);
            if (a.d_lengths) {                    // shortest move string: walk the parent chain back from the goal successor
                int32_t len = -1;
                if (sd != 0xFFFFFFFFu && (long long)sd <= a.max_moves && parents) {
                    __threadfence_block();
                    len = (int32_t)sd;
                    uint8_t* out = a.d_moves + pid * (size_t)a.max_moves;
                    uint32_t link = (uint32_t)(s_goal & 0xFFFFFFFFull);
                    for (int32_t k = len - 1; k >= 0; --k) {
                        out[k] = (uint8_t)(link & 3u);
                        link = parents[link >> 2];
                    }
                }
                a.d_lengths[pid] = len;
            }
        }
    }
    // ---- per-CTA tallies ----------------------------------------------------------------------
    __syncthreads();
    for (uint32_t k = tid; k < SEARCH_LEVELS; k += SEARCH_THREADS)
        if (hist[k] && k < (uint32_t)a.n_levels) atomicAdd((unsigned long long*)&a.d_levels[k], (unsigned long long)hist[k]);
    if (tid == 0) {
        atomicAdd((unsigned long long*)&a.d_counters[1], generated);
        atomicMax((unsigned long long*)&a.d_counters[3], (unsigned long long)deepest);
    }
}

static constexpr auto K6 = [](auto S, auto T, auto G) { return bfs_local_kernel<decltype(S)::value, decltype(T)::value, decltype(G)::value>; };

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

template <bool GMEM> static int local_ctas_per_sm(const ts_bfs_local_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = local_check(a)) return rc;
    return search_ctas_per_sm<GMEM>(K6, *a, ctas_per_sm, n_sm);
}

template <bool GMEM> static int local_launch(const ts_bfs_local_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = local_launch_check(a)) return rc;
    if constexpr (GMEM) {
        if (int rc = check_gmem(*a, d_bitmap)) return rc;
    }
    if (a->n_puzzles == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)search_kernel<GMEM>(K6, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream);
}

extern "C" {

int ts_bfs_local_smem_bytes(const ts_bfs_local_args* a) {
    if (int rc = local_check(a)) return rc;
    return (int)search_smem_bytes(*a);
}

int ts_bfs_local_ctas_per_sm(const ts_bfs_local_args* a, int* ctas_per_sm, int* n_sm) { return local_ctas_per_sm<false>(a, ctas_per_sm, n_sm); }
int ts_bfs_local(const ts_bfs_local_args* a, int grid, void* stream) { return local_launch<false>(a, nullptr, grid, stream); }
int ts_bfs_local_gmem_ctas_per_sm(const ts_bfs_local_args* a, int* ctas_per_sm, int* n_sm) { return local_ctas_per_sm<true>(a, ctas_per_sm, n_sm); }
int ts_bfs_local_gmem(const ts_bfs_local_args* a, uint32_t* d_bitmap, int grid, void* stream) { return local_launch<true>(a, d_bitmap, grid, stream); }

}  // extern "C"
