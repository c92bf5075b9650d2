// ts_optimal.cu -- K9: exact distance to the goal and the set of optimal first moves of many items
// (env id, positions: the env's current ones or a caller's word), one CTA per item, on chip, and
// optionally a shortest solution per item.  Built on K6's machinery (ts_bfs_local.cu; the CTA
// shape, hash, successor function, bitmap clear, plan and table checks and launch are in
// ts_bfs_local.cuh): persistent CTAs drawing items from a ticket counter, the visited set a
// shared-memory bitmap over the perfect hash of a state among the free cells of its puzzle (or, in
// the device instances of 7x7 and 8x8 boards with four tiles, a device-memory one), the frontier ring
// with a per-CTA HBM slab, the successor function slide_env<S,T> and goal test of the step.
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
// carries none of the plan's code: its slab entries are bare hashes, as they were before plans).
// GMEM: the device instance (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh), at least 5 CTAs
// per SM: without that bound ptxas takes 40 registers for two of its four instances and spills 16
// bytes; with it they take 45-48 and none spill.
template <int S, int T, bool PLAN, bool GMEM>
__global__ void __launch_bounds__(SEARCH_THREADS, GMEM ? 5 : 0) optimal_moves_kernel(const ts_optimal_moves_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    constexpr uint32_t KEY_SHIFT = PLAN ? 2u : 0u;        // slab entry of a good state: hash << KEY_SHIFT | move
    static_assert(T >= 1 && T <= 4, "32-bit states");
    static_assert(!GMEM || gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    // GMEM: CTA b's bitmap is d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.
    // __syncthreads orders the block's global accesses as it orders its shared ones, so the flag /
    // mark phases of the backward pass need no fence.  The largest hash is 64*63*62*61 - 1 <
    // 15,249,024 (F = 64), so a plan's slab entry hash << 2 | move stays below 2^26.
    uint32_t* const bitmap = GMEM ? d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words : dyn;
    uint32_t* const queue = GMEM ? dyn : dyn + a.bitmap_words;
    __shared__ uint8_t lut[128];                 // position byte -> rank among the free cells
    __shared__ uint32_t lstart[SEARCH_LEVELS];   // level k = discovery indices [lstart[k], lstart[k+1])
    __shared__ uint32_t cnt[3];                  // entries appended during level L: cnt[L % 3]
    __shared__ uint32_t lflag[3];                // ... and whether a successor met the goal (WON) / the slab overflowed (OVER)
    __shared__ long long s_ticket;
    __shared__ uint32_t s_move;                  // plan: the move played from the current state

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    // ring over discovery indices as in K6: entry p is in ring[p % R] when it was appended within R of
    // the start of the level being expanded, and in the slab in any case
    const uint32_t R = (uint32_t)a.queue_smem, RMASK = R - 1u;
    uint32_t* const slab = a.d_spill + (size_t)blockIdx.x * (size_t)a.spill_per_cta;
    const uint32_t q_cap = (uint32_t)a.spill_per_cta;
    const size_t cap = (size_t)a.capacity;
    unsigned long long fwd = 0, bwd = 0;         // states expanded forward / re-expanded backward (thread 0's count is added)

    for (;;) {
        __syncthreads();                         // the previous env is finished with shared memory
        if (tid == 0) s_ticket = (long long)atomicAdd((unsigned long long*)&a.d_counters[0], 1ull);
        __syncthreads();
        const long long ticket = s_ticket;
        if (ticket >= a.n_items) break;
        // the item's column of the plan: row r
        auto plan_at = [&](uint32_t r) -> uint8_t& { return a.d_plan[(size_t)r * (size_t)a.n_items + (size_t)ticket]; };
        // no solution: distance `code`, mask 0, an all-255 plan column (every thread calls it)
        auto no_solution = [&](int32_t code) {
            if (tid == 0) { a.d_distance[ticket] = code; a.d_mask[ticket] = 0; }
            if constexpr (PLAN)
#pragma unroll 1
                for (uint32_t r = tid; r < (uint32_t)a.max_depth; r += SEARCH_THREADS) plan_at(r) = 0xFF;
        };
        const long long env = a.d_env_ids ? (long long)a.d_env_ids[ticket] : ticket;
        if (env < 0 || env >= a.capacity) { no_solution(TS_OPT_NOT_SEARCHED); continue; }
        const size_t pid = (size_t)env;

        // ---- the item: walls, goal, root state, free-cell ranks ---------------------------------
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, pid);
        const uint64_t free_cells = ~walls & cell_mask<S>();
        uint32_t root;
        if (!read_root<S, T>(a, ticket, pid, free_cells, root)) { no_solution(TS_OPT_BAD_STATE); continue; }
        if (a.never_win) { no_solution(TS_OPT_UNSOLVABLE); continue; }   // no state meets the goal
        uint64_t tboard = 0;
        uint32_t tq = 0;
        if (a.goal_mode == TS_GOAL_SET) tboard = load_board_elem<NB>(a.d_targets_packed, cap, pid);
        else static_for<0, T>([&](auto I) { constexpr int t = decltype(I)::value; tq |= (uint32_t)a.d_targets_packed[pid * PW + t] << (8 * t); });
        if (a.goal_mode == TS_GOAL_SET) sort_bytes4<T>(root);
        const uint32_t F = (uint32_t)__popcll(free_cells);
        fill_lut<S>(tid, free_cells, lut);
        unsigned long long bits = 1;
#pragma unroll
        for (int t = 0; t < T; ++t) bits *= (F > (uint32_t)t ? F - (uint32_t)t : 1u);
        const uint32_t words = (uint32_t)((bits + 31) / 32);
        if (words > (uint32_t)a.bitmap_words) { no_solution(TS_OPT_NOT_SEARCHED); continue; }
        clear_bitmap(bitmap, words, tid);
        if (tid == 0) { cnt[0] = cnt[1] = cnt[2] = 0; lflag[0] = lflag[1] = lflag[2] = 0; }
        __syncthreads();

        // state after move m (set goal: canonical); won = it meets the goal (ts_bfs_local.cuh)
        auto successor = [&](uint32_t q0, uint32_t m, bool& won) { return ts::successor<S, T>(q0, m, walls, a.goal_mode == TS_GOAL_SET, tboard, tq, won); };
        auto marked = [&](uint32_t q) {
            const uint32_t idx = state_index<T>(lut, F, q);
            return (bitmap[idx >> 5] >> (idx & 31u)) & 1u;
        };

        if (tid == 0) {
            const uint32_t idx = state_index<T>(lut, F, root);
            bitmap[idx >> 5] |= 1u << (idx & 31u);
            queue[0] = root;
            slab[0] = root;
            lstart[0] = 0;
        }
        __syncthreads();

        // ---- 1. forward: BFS levels until a successor meets the goal ---------------------------
        uint32_t lo = 0, hi = 1, depth = 0, prev_lo = 0;
        int32_t dist = TS_OPT_CUTOFF;
        for (;;) {
            if (lo == hi) { dist = TS_OPT_UNSOLVABLE; break; }
            if (depth == (uint32_t)a.max_depth) break;
            uint32_t* const my_cnt = &cnt[depth % 3u];
            uint32_t* const my_flag = &lflag[depth % 3u];
            if (tid == 0) cnt[(depth + 1u) % 3u] = lflag[(depth + 1u) % 3u] = 0;
            const uint32_t n_items = (hi - lo) * 4u;
            for (uint32_t base = 0; base < n_items; base += SEARCH_THREADS) {
                const uint32_t j = base + tid;
                const bool live = j < n_items;
                const uint32_t src = lo + (j >> 2), d = j & 3u;
                bool is_new = false;
                uint32_t qn = 0;
                if (live) {
                    const uint32_t q0 = (src - prev_lo) < R ? queue[src & RMASK] : slab[src];
                    bool won;
                    qn = successor(q0, d, won);
                    if (won) atomicOr(my_flag, WON);
                    // once this level has met the goal its successors are never read: skip the appends
                    if (qn != q0 && !(*(volatile uint32_t*)my_flag & WON)) {
                        const uint32_t idx = state_index<T>(lut, F, qn);
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
                        if (pos < q_cap) slab[pos] = qn;
                        else atomicOr(my_flag, OVER);
                    }
                }
            }
            __syncthreads();
            const uint32_t n_new = *my_cnt, flag = *my_flag;
            fwd += hi - lo;
            prev_lo = lo;
            lo = hi;
            hi += n_new;
            ++depth;
            if (tid == 0) lstart[depth] = lo;
            if (flag & WON) { dist = (int32_t)depth; break; }
            if (flag & OVER) { dist = TS_OPT_NOT_SEARCHED; break; }     // slab exhausted before the goal level
        }
        if (dist < 0) { no_solution(dist); continue; }

        // ---- 2. backward: mark the states of levels d-1 .. 1 that start a shortest solution ------
        const uint32_t D = (uint32_t)dist;
        if (D >= 2) {
            clear_bitmap(bitmap, words, tid);
            __syncthreads();                      // bitmap clear, lstart complete
            for (uint32_t k = D - 1u; k >= 1u; --k) {
                const uint32_t l0 = lstart[k], l1 = lstart[k + 1u];
                const uint32_t n_items = (l1 - l0) * 4u;
                for (uint32_t base = 0; base < n_items; base += SEARCH_THREADS) {
                    const uint32_t j = base + tid;
                    const bool live = j < n_items;
                    const uint32_t src = l0 + (j >> 2);
                    bool hit = false;
                    uint32_t q0 = 0;
                    if (live) {
                        q0 = slab[src];
                        bool won;
                        const uint32_t qn = successor(q0, j & 3u, won);
                        hit = k == D - 1u ? won : (qn != q0 && marked(qn));
                    }
                    // the four lanes of a state are lanes 4i .. 4i+3 of one warp
                    const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
                    if (live && (j & 3u) == 0u) {
                        const uint32_t hits = (m >> lane) & 0xFu;
                        slab[src] = hits ? state_index<T>(lut, F, q0) << KEY_SHIFT | (PLAN ? (uint32_t)(__ffs(hits) - 1) : 0u) : OPT_NONE;
                    }
                }
                __syncthreads();                  // every flag of level k computed
                for (uint32_t s = l0 + tid; s < l1; s += SEARCH_THREADS) {
                    const uint32_t e = slab[s];
                    if (e != OPT_NONE) atomicOr(&bitmap[e >> (5 + KEY_SHIFT)], 1u << ((e >> KEY_SHIFT) & 31u));
                }
                __syncthreads();                  // level k marked
                if (tid == 0) bwd += l1 - l0;
            }
        }

        // ---- 3. root: its optimal moves ---------------------------------------------------------
        if (tid < 32) {
            bool hit = false;
            if (lane < 4) {
                bool won;
                const uint32_t qn = successor(root, lane, won);
                hit = D == 1u ? won : (qn != root && marked(qn));
            }
            const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
            if (tid == 0) {
                a.d_distance[ticket] = dist;
                a.d_mask[ticket] = (uint8_t)(m & 0xFu);
                if constexpr (PLAN) s_move = (uint32_t)(__ffs(m) - 1);
            }
        }

        // ---- 4. plan: the lowest optimal move from each state of the solution --------------------
        if constexpr (PLAN) {
#pragma unroll 1
            for (uint32_t r = D + tid; r < (uint32_t)a.max_depth; r += SEARCH_THREADS) plan_at(r) = 0xFF;
            __syncthreads();                      // s_move of the root
            uint32_t q = root;
            for (uint32_t k = 0;;) {
                const uint32_t mv = s_move;
                if (tid == 0) plan_at(k) = (uint8_t)mv;
                if (++k == D) break;
                bool won;
                q = successor(q, mv, won);
                const uint32_t key = state_index<T>(lut, F, q);
                __syncthreads();                  // s_move read by every thread
                // q is good at level k, appended there once: exactly one entry of the range is its own
#pragma unroll 1
                for (uint32_t s = lstart[k] + tid; s < lstart[k + 1u]; s += SEARCH_THREADS) {
                    const uint32_t e = slab[s];
                    if (e >> 2 == key) s_move = e & 3u;
                }
                __syncthreads();                  // s_move of q
            }
        }
    }
    if (tid == 0) {
        atomicAdd((unsigned long long*)&a.d_counters[1], fwd);
        atomicAdd((unsigned long long*)&a.d_counters[2], bwd);
    }
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

static constexpr auto K9 = [](auto S, auto T, auto G) { return optimal_moves_kernel<decltype(S)::value, decltype(T)::value, false, decltype(G)::value>; };
static constexpr auto K9_PLAN = [](auto S, auto T, auto G) { return optimal_moves_kernel<decltype(S)::value, decltype(T)::value, true, decltype(G)::value>; };

}  // namespace ts

using namespace ts;

// the checks of a launch before its empty-query return
static int optimal_check_launch(const ts_optimal_moves_args* a) {
    if (int rc = check_item_plan(a)) return rc;
    if (int rc = check_item_table(a)) return rc;
    if (a->max_depth < 1 || a->max_depth > TS_OPT_MAX_DEPTH || a->spill_per_cta < 1 || a->spill_per_cta > 0xFFFFFFFFll)
        return TS_E_BAD_ARGUMENT;
    if (!a->d_spill || !a->d_counters || !a->d_distance || !a->d_mask) return TS_E_NULL_POINTER;
    return 0;
}

template <bool GMEM> static int optimal_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = check_item_plan(a)) return rc;
    return a->d_plan ? search_ctas_per_sm<GMEM>(K9_PLAN, *a, ctas_per_sm, n_sm) : search_ctas_per_sm<GMEM>(K9, *a, ctas_per_sm, n_sm);
}

template <bool GMEM> static int optimal_launch(const ts_optimal_moves_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = optimal_check_launch(a)) return rc;
    if constexpr (GMEM) {
        if (int rc = check_gmem(*a, d_bitmap)) return rc;
    }
    if (a->n_items == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)(a->d_plan ? search_kernel<GMEM>(K9_PLAN, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream)
                           : search_kernel<GMEM>(K9, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream));
}

extern "C" {

int ts_optimal_moves_smem_bytes(const ts_optimal_moves_args* a) {
    if (int rc = check_item_plan(a)) return rc;
    return (int)search_smem_bytes(*a);
}

int ts_optimal_moves_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) { return optimal_ctas_per_sm<false>(a, ctas_per_sm, n_sm); }

int ts_optimal_max_free_cells(const ts_optimal_moves_args* a, int32_t* d_max_free, void* stream) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;
    if (int rc = check_item_table(a)) return rc;
    if (!d_max_free) return TS_E_NULL_POINTER;
    if (a->n_items == 0) return 0;
    const long long blocks = (a->n_items + 255) / 256;
    return (int)dispatch_size(a->size, [&](auto S) {
        max_free_cells_kernel<decltype(S)::value><<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, (cudaStream_t)stream>>>(*a, d_max_free);
        return cudaGetLastError();
    });
}

int ts_optimal_moves(const ts_optimal_moves_args* a, int grid, void* stream) { return optimal_launch<false>(a, nullptr, grid, stream); }
int ts_optimal_moves_gmem_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) { return optimal_ctas_per_sm<true>(a, ctas_per_sm, n_sm); }
int ts_optimal_moves_gmem(const ts_optimal_moves_args* a, uint32_t* d_bitmap, int grid, void* stream) { return optimal_launch<true>(a, d_bitmap, grid, stream); }

}  // extern "C"
