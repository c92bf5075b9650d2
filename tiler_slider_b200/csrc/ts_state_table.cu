// ts_state_table.cu -- K10: the state table of many items (env id, positions): every state reachable
// from the item's root, each with its exact distance to the goal and its optimal moves (K9's
// definitions), one CTA per item, on chip.  K6/K9's machinery (ts_bfs_local.cuh): persistent CTAs
// drawing items from a ticket counter, the visited set a shared-memory bitmap over the perfect hash
// of a state among the free cells of its puzzle (or, in the device instances of 7x7 and 8x8 boards
// with four tiles, a device-memory one), the frontier ring, and the successor function, bitmap clear
// and plan and table checks written once there.
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

// FILL: the second launch (rows, order, sweep); otherwise the count pass.  GMEM: the device instance
// (7x7 and 8x8 boards with four tiles, ts_bfs_local.cuh)
template <int S, int T, bool FILL, bool GMEM>
__global__ void __launch_bounds__(SEARCH_THREADS) state_table_kernel(const ts_state_table_args a, uint32_t* const d_bitmap) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S), WARPS = SEARCH_THREADS / 32;
    static_assert(T >= 1 && T <= 4, "32-bit states");
    static_assert(!GMEM || gmem_shape(S, T), "device instances exist for 7x7 and 8x8 boards with four tiles only");
    extern __shared__ __align__(16) uint32_t dyn[];
    // GMEM: CTA b's bitmap is d_bitmap[b * bitmap_words ..], dynamic shared memory the ring alone.
    // __syncthreads orders the block's global accesses as it orders its shared ones, so the mark
    // phases of the sweep need no fence.  The order scan's index w * 32 + bit stays below
    // 64*63*62*61 = 15,249,024 (F = 64).
    uint32_t* const bitmap = GMEM ? d_bitmap + (size_t)blockIdx.x * (size_t)a.bitmap_words : dyn;
    uint32_t* const queue = GMEM ? dyn : dyn + a.bitmap_words;
    __shared__ uint8_t lut[128];                 // position byte -> rank among the free cells
    __shared__ uint8_t rank_byte[64];            // rank among the free cells -> position byte
    __shared__ uint32_t cnt[3];                  // entries appended during level L: cnt[L % 3]
    __shared__ uint32_t lflag[3];                // ... and whether the slab overflowed (count pass)
    __shared__ uint32_t s_won;                   // a successor met the goal
    __shared__ uint32_t s_progress[2];           // round r resolved a row: s_progress[r % 2]
    __shared__ uint32_t s_warp[WARPS];           // order: popcount sums per warp
    __shared__ long long s_ticket;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t R = (uint32_t)a.queue_smem, RMASK = R - 1u;
    uint32_t* const slab = a.d_spill + (FILL ? 0 : (size_t)blockIdx.x * (size_t)a.spill_per_cta);
    const size_t cap = (size_t)a.capacity;
    unsigned long long swept = 0;                // rows x rounds of the sweep (thread 0's count is added)

    for (;;) {
        __syncthreads();                         // the previous item is finished with shared memory
        if (tid == 0) s_ticket = (long long)atomicAdd((unsigned long long*)&a.d_counters[FILL ? 1 : 0], 1ull);
        __syncthreads();
        const long long ticket = s_ticket;
        if (ticket >= a.n_items) break;
        // count pass: the item is not enumerated (status `code`, no rows)
        auto no_table = [&](int32_t code) {
            if (tid == 0) { a.d_status[ticket] = code; a.d_count[ticket] = 0; }
        };
        if constexpr (FILL) {
            if (a.d_status[ticket] != 0) continue;
        }
        const long long env = a.d_env_ids ? (long long)a.d_env_ids[ticket] : ticket;
        if (env < 0 || env >= a.capacity) { if constexpr (!FILL) no_table(TS_OPT_NOT_SEARCHED); continue; }
        const size_t pid = (size_t)env;

        // ---- the item: walls, goal, root state, free-cell ranks (as K9) --------------------------
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, pid);
        const uint64_t free_cells = ~walls & cell_mask<S>();
        uint32_t root;
        if (!read_root<S, T>(a, ticket, pid, free_cells, root)) { if constexpr (!FILL) no_table(TS_OPT_BAD_STATE); continue; }
        uint64_t tboard = 0;
        uint32_t tq = 0;
        if (a.goal_mode == TS_GOAL_SET) tboard = load_board_elem<NB>(a.d_targets_packed, cap, pid);
        else static_for<0, T>([&](auto I) { constexpr int t = decltype(I)::value; tq |= (uint32_t)a.d_targets_packed[pid * PW + t] << (8 * t); });
        if (a.goal_mode == TS_GOAL_SET) sort_bytes4<T>(root);
        const uint32_t F = (uint32_t)__popcll(free_cells);
        fill_lut<S>(tid, free_cells, lut, FILL ? rank_byte : nullptr);
        unsigned long long bits = 1;
#pragma unroll
        for (int t = 0; t < T; ++t) bits *= (F > (uint32_t)t ? F - (uint32_t)t : 1u);
        const uint32_t words = (uint32_t)((bits + 31) / 32);
        if (words > (uint32_t)a.bitmap_words) { if constexpr (!FILL) no_table(TS_OPT_NOT_SEARCHED); continue; }
        clear_bitmap(bitmap, words, tid);
        if (tid == 0) { cnt[0] = cnt[1] = cnt[2] = 0; lflag[0] = lflag[1] = lflag[2] = 0; s_won = 0; }
        __syncthreads();

        // queue storage beyond the ring: the slab (count) or the item's rows (fill)
        const long long row0 = FILL ? a.d_offsets[ticket] : 0;
        const uint32_t n_rows = FILL ? (uint32_t)(a.d_offsets[ticket + 1] - row0) : 0u;
        uint8_t* const rows = FILL ? a.d_rows + (size_t)row0 * PW : nullptr;
        const uint32_t q_cap = FILL ? n_rows : (uint32_t)a.spill_per_cta;
        auto stored = [&](uint32_t p) { if constexpr (FILL) return load_row<PW>(rows + (size_t)p * PW); else return slab[p]; };
        auto store = [&](uint32_t p, uint32_t q) { if constexpr (FILL) store_row<PW>(rows + (size_t)p * PW, q); else slab[p] = q; };

        // state after move m (set goal: canonical); won = it meets the goal (ts_bfs_local.cuh)
        auto successor = [&](uint32_t q0, uint32_t m, bool& won) { return ts::successor<S, T>(q0, m, walls, a.goal_mode == TS_GOAL_SET, tboard, tq, won); };

        if (tid == 0) {
            const uint32_t idx = state_index<T>(lut, F, root);
            bitmap[idx >> 5] |= 1u << (idx & 31u);
            queue[0] = root;
        }
        __syncthreads();

        // ---- forward: BFS to exhaustion ---------------------------------------------------------
        // ring as K6/K9: entry p is in ring[p % R] when it was appended within R of the start of the
        // level being expanded, else in the queue storage (count: p >= spill_per_cta overflows)
        uint32_t lo = 0, hi = 1, depth = 0, prev_lo = 0;
        bool over = false;
        while (lo != hi) {
            uint32_t* const my_cnt = &cnt[depth % 3u];
            uint32_t* const my_flag = &lflag[depth % 3u];
            if (tid == 0) cnt[(depth + 1u) % 3u] = lflag[(depth + 1u) % 3u] = 0;
            const uint32_t n_work = (hi - lo) * 4u;
            for (uint32_t base = 0; base < n_work; base += SEARCH_THREADS) {
                const uint32_t j = base + tid;
                const bool live = j < n_work;
                const uint32_t src = lo + (j >> 2);
                bool is_new = false;
                uint32_t qn = 0;
                if (live) {
                    const uint32_t q0 = (src - prev_lo) < R ? queue[src & RMASK] : stored(src);
                    bool won;
                    qn = successor(q0, j & 3u, won);
                    if (FILL && won) *(volatile uint32_t*)&s_won = 1u;
                    if (qn != q0) {
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
                        if (pos >= q_cap) atomicOr(my_flag, TAB_OVER);           // count pass only
                        else if (pos - lo < R) queue[pos & RMASK] = qn;
                        else store(pos, qn);
                    }
                }
            }
            __syncthreads();
            const uint32_t n_new = *my_cnt;
            over = (*my_flag & TAB_OVER) != 0;
            prev_lo = lo;
            lo = hi;
            hi += n_new;
            ++depth;
            if (over) break;
        }

        if constexpr (!FILL) {
            if (tid == 0) {
                a.d_status[ticket] = over ? TS_OPT_NOT_SEARCHED : 0;
                a.d_count[ticket] = over ? 0 : (long long)hi;
            }
        } else {
            // ---- order: rows in ascending hash order, from the bitmap -------------------------------
            int32_t* const dist = a.d_distance + row0;
            uint8_t* const mask = a.d_mask + row0;
            uint32_t done = 0;                   // rows written by earlier chunks of words
            for (uint32_t base = 0; base < words; base += SEARCH_THREADS) {
                const uint32_t w = base + tid;
                const uint32_t word = w < words ? bitmap[w] : 0u;
                uint32_t incl = (uint32_t)__popc(word);
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (lane >= (uint32_t)o) incl += v;
                }
                if (lane == 31u) s_warp[warp] = incl;
                __syncthreads();
                uint32_t before = done, total = 0;
#pragma unroll
                for (int k = 0; k < WARPS; ++k) {
                    const uint32_t s = s_warp[k];
                    before += (uint32_t)k < warp ? s : 0u;
                    total += s;
                }
                uint32_t r = before + incl - (uint32_t)__popc(word);
#pragma unroll 1
                for (uint32_t b = word; b; b &= b - 1u, ++r) {
                    // index -> digits (least significant: tile 0, radix F) -> ranks -> bytes
                    uint32_t idx = w * 32u + (uint32_t)(__ffs(b) - 1), q = 0;
                    uint64_t taken = 0;
                    static_for<0, T>([&](auto I) {
                        constexpr int i = decltype(I)::value;
                        const uint32_t radix = F - (uint32_t)i;
                        const uint32_t d = i == T - 1 ? idx : idx % radix;
                        idx = i == T - 1 ? 0u : idx / radix;
                        // the d-th rank not taken by tiles 0 .. i-1: at most i corrections
                        uint32_t rk = d;
#pragma unroll
                        for (int k = 0; k < i; ++k) rk = d + (uint32_t)__popcll(taken & (~0ull >> (63u - rk)));
                        taken |= 1ull << rk;
                        q |= (uint32_t)rank_byte[rk] << (8 * i);
                    });
                    if (r < n_rows) {
                        store_row<PW>(rows + (size_t)r * PW, q);
                        dist[r] = TS_OPT_UNSOLVABLE;
                        mask[r] = 0;
                    }
                }
                done += total;
                __syncthreads();                 // s_warp read by every thread
            }

            // ---- sweep: retrograde rounds over the rows ----------------------------------------------
            if (s_won && !a.never_win) {
                clear_bitmap(bitmap, words, tid);
                if (tid == 0) s_progress[0] = s_progress[1] = 0;
                for (int32_t round = 1;; ++round) {
                    __syncthreads();             // bitmap clear / previous round marked; rows and dist visible
                    // the other slot was last read before this barrier
                    if (tid == 0) s_progress[(round + 1) & 1] = 0;
                    const uint32_t n_work = n_rows * 4u;
#pragma unroll 1
                    for (uint32_t base = 0; base < n_work; base += SEARCH_THREADS) {
                        const uint32_t j = base + tid, row = j >> 2;
                        const bool live = j < n_work && dist[row] == TS_OPT_UNSOLVABLE;
                        bool hit = false;
                        if (live) {
                            const uint32_t q0 = load_row<PW>(rows + (size_t)row * PW);
                            bool won;
                            const uint32_t qn = successor(q0, j & 3u, won);
                            if (round == 1) {
                                hit = won;
                            } else if (qn != q0) {
                                const uint32_t idx = state_index<T>(lut, F, qn);
                                hit = (bitmap[idx >> 5] >> (idx & 31u)) & 1u;
                            }
                        }
                        // the four lanes of a row are lanes 4i .. 4i+3 of one warp
                        const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
                        const uint32_t hits = (m >> (lane & ~3u)) & 0xFu;
                        if (live && (j & 3u) == 0u && hits) {
                            dist[row] = round;
                            mask[row] = (uint8_t)hits;
                            *(volatile uint32_t*)&s_progress[round & 1] = 1u;
                        }
                    }
                    __syncthreads();             // every row of round `round` decided
                    if (tid == 0) swept += n_rows;
                    if (!s_progress[round & 1]) break;
#pragma unroll 1
                    for (uint32_t row = tid; row < n_rows; row += SEARCH_THREADS) {
                        if (dist[row] != round) continue;
                        const uint32_t idx = state_index<T>(lut, F, load_row<PW>(rows + (size_t)row * PW));
                        atomicOr(&bitmap[idx >> 5], 1u << (idx & 31u));
                    }
                }
            }
        }
    }
    if (FILL && tid == 0) atomicAdd((unsigned long long*)&a.d_counters[2], swept);
}


// the count (FILL false) or fill pass
template <bool FILL>
static constexpr auto K10 = [](auto S, auto T, auto G) { return state_table_kernel<decltype(S)::value, decltype(T)::value, FILL, decltype(G)::value>; };

}  // namespace ts

using namespace ts;

// shape, shared-memory plan and the env table (the checks of ts_optimal_moves)
static int state_table_check(const ts_state_table_args* a, int grid) {
    if (int rc = check_item_plan(a)) return rc;
    if (int rc = check_item_table(a)) return rc;
    if (!a->d_counters || !a->d_status) return TS_E_NULL_POINTER;
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
template <bool GMEM> static int table_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = check_item_plan(a)) return rc;
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    int count = 0, fill = 0;
    if (int rc = search_ctas_per_sm<GMEM>(K10<false>, *a, &count, n_sm)) return rc;
    if (int rc = search_ctas_per_sm<GMEM>(K10<true>, *a, &fill, n_sm)) return rc;
    *ctas_per_sm = count < fill ? count : fill;
    return 0;
}

template <bool FILL, bool GMEM> static int table_pass(const ts_state_table_args* a, uint32_t* d_bitmap, int grid, void* stream) {
    if (int rc = FILL ? fill_check(a, grid) : count_check(a, grid)) return rc;
    if constexpr (GMEM) {
        if (int rc = check_gmem(*a, d_bitmap)) return rc;
    }
    if (a->n_items == 0) return 0;
    return (int)search_kernel<GMEM>(K10<FILL>, *a, d_bitmap, grid, nullptr, (cudaStream_t)stream);
}

extern "C" {

int ts_state_table_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) { return table_ctas_per_sm<false>(a, ctas_per_sm, n_sm); }
int ts_state_table_count(const ts_state_table_args* a, int grid, void* stream) { return table_pass<false, false>(a, nullptr, grid, stream); }
int ts_state_table_fill(const ts_state_table_args* a, int grid, void* stream) { return table_pass<true, false>(a, nullptr, grid, stream); }
int ts_state_table_gmem_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) { return table_ctas_per_sm<true>(a, ctas_per_sm, n_sm); }
int ts_state_table_count_gmem(const ts_state_table_args* a, uint32_t* d_bitmap, int grid, void* stream) { return table_pass<false, true>(a, d_bitmap, grid, stream); }
int ts_state_table_fill_gmem(const ts_state_table_args* a, uint32_t* d_bitmap, int grid, void* stream) { return table_pass<true, true>(a, d_bitmap, grid, stream); }

}  // extern "C"
