// ts_table_state_table.cu -- K12: K10's state tables (every state reachable from items, each with
// K9's distance and optimal-move mask) for 5 to 8 tiles, where a state is a 64-bit word and the
// perfect-hash bitmap outgrows even device memory.  K10's two passes (ts_state_table.cu) on K11's
// machinery (ts_table_search.cu): the CTA shape, the ticket counter, the per-CTA hash table with item
// epochs (ts_hash_table.cuh), a ring of 64-bit entries in shared memory and a slab of
// spill_per_cta entries per CTA in device memory.  Both passes take the same plan and grid.
//
//   count  root check (TS_OPT_BAD_STATE, K9's rule; never_win is enumerated all the same), then a
//          BFS to exhaustion; a new state is the one whose CAS claims an empty slot, and the ring
//          spills to the slab.  The item gets TS_OPT_NOT_SEARCHED at the first discovery index >=
//          spill_per_cta (K10's rule) or when the table is full (it holds 2 * spill_per_cta slots,
//          so only after that); else its number of states.
//   fill   (the caller has turned the counts into row offsets) the same BFS in a fresh epoch, the
//          queue beyond the ring in the item's own rows or its slab (below); then
//     order      the rows sorted ascending as little-endian 64-bit words: a stable LSD radix sort
//                inside the CTA, one pass per tile byte (T passes of 7-bit digits: every byte is
//                < 128, the padding bytes are 0), between the rows and the slab (the count pass
//                has checked that the item's rows fit it).  The BFS queue is the buffer the sort
//                starts from (the slab for odd T), so that its last pass writes the rows.  Per pass:
//                a digit histogram, and per tile of 256 rows each row's place = the digit's base +
//                the rows of that digit in lower warps of the tile (per-warp counts, scanned by one
//                thread per digit) + its rank among its warp's lanes of that digit
//                (__match_any_sync).  The counts live in the ring's shared memory, idle after the
//                BFS.  BFS order within a level depends on atomics; this order does not.
//     sweep      K10's retrograde rounds in place over the rows; a row's successor is marked when
//                the TAB_MARK bit of its slot is set (found by a probe as K11's backward pass), and
//                after each round's barrier the rows resolved in that round OR the mark into their
//                slots.  Skipped when no successor met the goal in the BFS (never_win included).
//   Rows hold pure keys (TAB_KEY), never flag bits.
#include "ts_hash_table.cuh"

namespace ts {

constexpr int SORT_DIGITS = 128;                        // a tile byte is < 128
constexpr int SORT_WARPS = SEARCH_THREADS / 32;
// the sort's shared memory, laid over the ring: per warp and digit the tile's count, then its
// place; the histogram of the pass
constexpr size_t TABLE_SORT_SMEM = (size_t)(SORT_WARPS + 1) * SORT_DIGITS * sizeof(uint32_t);

// FILL: the second launch (rows, order, sweep); otherwise the count pass.  Left to itself ptxas gives
// the fill pass 40 registers and spills in some instances; five CTAs per SM give it 48 and none
// (profiles/r12_table_state_table_ptxas.txt)
template <int S, int T, bool FILL>
__global__ void __launch_bounds__(SEARCH_THREADS, FILL ? 5 : 0) table_state_table_kernel(const ts_state_table_args a, uint64_t* const d_table, const uint64_t table_slots) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    static_assert(T >= 5 && T <= 8 && PW == 8, "64-bit states");
    extern __shared__ __align__(16) uint64_t ring[];
    uint32_t* const wcnt = reinterpret_cast<uint32_t*>(ring);    // sort: [SORT_WARPS][SORT_DIGITS]
    uint32_t* const hist = wcnt + SORT_WARPS * SORT_DIGITS;      // sort: [SORT_DIGITS]
    __shared__ uint32_t cnt[3];                  // entries appended during level L: cnt[L % 3]
    __shared__ uint32_t lflag[3];                // ... and whether the item overflowed (OVER, count pass)
    __shared__ uint32_t s_won;                   // a successor met the goal (fill pass)
    __shared__ uint32_t s_progress[2];           // round r resolved a row: s_progress[r % 2]
    __shared__ long long s_ticket;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t R = (uint32_t)a.queue_smem, RMASK = R - 1u;
    uint64_t* const slab = reinterpret_cast<uint64_t*>(a.d_spill) + (size_t)blockIdx.x * (size_t)a.spill_per_cta;
    uint64_t* const table = d_table + (size_t)blockIdx.x * table_slots;
    const uint64_t smask = table_slots - 1u;
    const size_t cap = (size_t)a.capacity;
    unsigned long long swept = 0;                // rows x rounds of the sweep (thread 0's count is added)
    uint32_t epoch = 0;                          // of the CTA's current item: 1 .. TAB_EPOCHS

    for (;;) {
        __syncthreads();                         // the previous item is finished with shared memory and the table
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

        // ---- the item: walls, goal, root state (as K11) -------------------------------------------
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, pid);
        const uint64_t free_cells = ~walls & cell_mask<S>();
        uint64_t root;
        if (!read_root64<S, T>(a, ticket, pid, free_cells, root)) { if constexpr (!FILL) no_table(TS_OPT_BAD_STATE); continue; }
        const bool set_goal = a.goal_mode == TS_GOAL_SET;
        uint64_t tboard = 0, tq = 0;
        if (set_goal) tboard = load_board_elem<NB>(a.d_targets_packed, cap, pid);
        else static_for<0, T>([&](auto I) { constexpr int t = decltype(I)::value; tq |= (uint64_t)a.d_targets_packed[pid * PW + t] << (8 * t); });
        if (set_goal) sort_bytes8<T>(root);

        // a new epoch; a wrapped one (the first item included) starts on a cleared slice
        epoch = epoch % TAB_EPOCHS + 1u;
        if (epoch == 1u) {
            for (uint64_t k = tid; k < table_slots; k += SEARCH_THREADS) table[k] = 0;
            __syncthreads();
        }
        const uint64_t ep = epoch_bits(epoch);

        // queue storage beyond the ring: the slab (count), or in the fill the buffer the sort starts
        // from, the item's rows for even T and the slab for odd T (its T passes then end in the rows)
        const long long row0 = FILL ? a.d_offsets[ticket] : 0;
        const uint32_t n_rows = FILL ? (uint32_t)(a.d_offsets[ticket + 1] - row0) : 0u;
        uint64_t* const rows = FILL ? reinterpret_cast<uint64_t*>(a.d_rows) + row0 : nullptr;
        uint64_t* const queue = FILL && !(T & 1) ? rows : slab;
        const uint32_t q_cap = FILL ? n_rows : (uint32_t)a.spill_per_cta;
        if (tid == 0) {
            cnt[0] = cnt[1] = cnt[2] = 0; lflag[0] = lflag[1] = lflag[2] = 0; s_won = 0;
            table_insert(table, smask, ep, root);
            ring[0] = root;
            if (FILL) queue[0] = root;
        }
        __syncthreads();

        auto successor = [&](uint64_t q0, uint32_t m, bool& won) { return successor64<S, T>(q0, m, walls, set_goal, tboard, tq, won); };

        // ---- forward: BFS to exhaustion ---------------------------------------------------------
        // ring as K10: entry p is in ring[p % R] when it was appended within R of the start of the
        // level being expanded; the count pass stores it in the slab otherwise (p >= spill_per_cta
        // overflows), the fill pass in the queue always (the sort reads every row from there)
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
                uint64_t qn = 0;
                if (live) {
                    const uint64_t q0 = (src - prev_lo) < R ? ring[src & RMASK] : queue[src];
                    bool won;
                    qn = successor(q0, j & 3u, won);
                    if (FILL && won) *(volatile uint32_t*)&s_won = 1u;
                    // once the item has overflowed its successors are never read (count pass)
                    if (qn != q0 && !(*(volatile uint32_t*)my_flag)) {
                        const int r = table_insert(table, smask, ep, qn);
                        is_new = r > 0;
                        if (r < 0) atomicOr(my_flag, TAB_OVER);
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
                        else {
                            const bool in_ring = pos - lo < R;
                            if (in_ring) ring[pos & RMASK] = qn;
                            if (FILL || !in_ring) queue[pos] = qn;
                        }
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
            // ---- order: a stable LSD radix sort on the tile bytes, queue -> other buffer -> ... -> rows
            for (uint32_t k = tid; k < SORT_WARPS * SORT_DIGITS; k += SEARCH_THREADS) wcnt[k] = 0;
            uint64_t* src = queue;
            uint64_t* dst = queue == rows ? slab : rows;
#pragma unroll 1
            for (uint32_t shift = 0; shift < 8u * T; shift += 8u) {
                if (tid < SORT_DIGITS) hist[tid] = 0;
                __syncthreads();                 // the ring / the previous pass is done; hist clear
                for (uint32_t i = tid; i < n_rows; i += SEARCH_THREADS) atomicAdd(&hist[(uint32_t)(src[i] >> shift) & 0x7Fu], 1u);
                __syncthreads();
                uint32_t next = 0;               // thread d < SORT_DIGITS: the place of the next row of digit d
                if (tid < SORT_DIGITS)
#pragma unroll 1
                    for (uint32_t k = 0; k < tid; ++k) next += hist[k];
#pragma unroll 1
                for (uint32_t t0 = 0; t0 < n_rows; t0 += SEARCH_THREADS) {
                    const uint32_t i = t0 + tid;
                    const bool live = i < n_rows;
                    const uint64_t key = live ? src[i] : 0ull;
                    const uint32_t d = live ? (uint32_t)(key >> shift) & 0x7Fu : (uint32_t)SORT_DIGITS;
                    const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
                    const uint32_t rank = (uint32_t)__popc(peers & ((1u << lane) - 1u));
                    uint32_t* const my = &wcnt[warp * SORT_DIGITS + (d & 0x7Fu)];
                    if (live && rank == 0u) *my = (uint32_t)__popc(peers);
                    __syncthreads();             // the tile's counts
                    if (tid < SORT_DIGITS) {     // counts -> places, warp by warp; absent ones stay 0
#pragma unroll
                        for (int w = 0; w < SORT_WARPS; ++w) {
                            const uint32_t c = wcnt[w * SORT_DIGITS + tid];
                            if (c) { wcnt[w * SORT_DIGITS + tid] = next; next += c; }
                        }
                    }
                    __syncthreads();             // the tile's places
                    if (live) dst[*my + rank] = key;
                    __syncwarp();                // only this warp's lanes read its entries
                    if (live && rank == 0u) *my = 0u;
                }
                uint64_t* const t = src; src = dst; dst = t;
            }
            // src == rows now; every row starts unresolved
            int32_t* const dist = a.d_distance + row0;
            uint8_t* const mask = a.d_mask + row0;
            for (uint32_t r = tid; r < n_rows; r += SEARCH_THREADS) { dist[r] = TS_OPT_UNSOLVABLE; mask[r] = 0; }

            // ---- sweep: retrograde rounds over the rows (K10), marks in the table -----------------------
            if (s_won && !a.never_win) {
                if (tid == 0) s_progress[0] = s_progress[1] = 0;
                for (int32_t round = 1;; ++round) {
                    __syncthreads();             // rows sorted, dist set / previous round marked
                    // the other slot was last read before this barrier
                    if (tid == 0) s_progress[(round + 1) & 1] = 0;
                    const uint32_t n_work = n_rows * 4u;
#pragma unroll 1
                    for (uint32_t base = 0; base < n_work; base += SEARCH_THREADS) {
                        const uint32_t j = base + tid, row = j >> 2;
                        const bool live = j < n_work && dist[row] == TS_OPT_UNSOLVABLE;
                        bool hit = false;
                        if (live) {
                            const uint64_t q0 = rows[row];
                            bool won;
                            const uint64_t qn = successor(q0, j & 3u, won);
                            if (round == 1) {
                                hit = won;
                            } else if (qn != q0) {
                                const long long h = table_find(table, smask, ep, qn);
                                hit = h >= 0 && (__ldcg(table + h) & TAB_MARK);
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
                        const long long h = table_find(table, smask, ep, rows[row]);
                        if (h >= 0) atomicOr((unsigned long long*)(table + h), (unsigned long long)TAB_MARK);
                    }
                }
            }
        }
    }
    if (FILL && tid == 0) atomicAdd((unsigned long long*)&a.d_counters[2], swept);
}

// the count (FILL false) or fill pass
template <bool FILL>
static constexpr auto K12 = [](auto S, auto T) { return table_state_table_kernel<decltype(S)::value, decltype(T)::value, FILL>; };

// dynamic shared memory of both passes: the ring, or the sort's counts when they need more
static size_t k12_smem(const ts_state_table_args& a) {
    const size_t ring = (size_t)a.queue_smem * sizeof(uint64_t);
    return ring > TABLE_SORT_SMEM ? ring : TABLE_SORT_SMEM;
}

}  // namespace ts

using namespace ts;

// the launch checks of each pass before its empty-query return: the table plan, the env table, K10's
// pass checks, the slab (both passes: the fill sorts through it), the table buffer, the rows' alignment
template <bool FILL> static int table_pass_check(const ts_state_table_args* a, const uint64_t* d_table, int64_t table_slots, int grid) {
    if (int rc = table_check_plan(a)) return rc;
    if (int rc = check_item_table(a)) return rc;
    if (!a->d_counters || !a->d_status) return TS_E_NULL_POINTER;
    if (a->n_items > 0 && grid < 1) return TS_E_BAD_ARGUMENT;
    if (FILL && (!a->d_offsets || !a->d_rows || !a->d_distance || !a->d_mask)) return TS_E_NULL_POINTER;
    if (a->spill_per_cta < 1 || a->spill_per_cta > 0xFFFFFFFFll) return TS_E_BAD_ARGUMENT;
    if (!a->d_spill || (!FILL && !a->d_count)) return TS_E_NULL_POINTER;
    if (int rc = table_check_buffer(a, d_table, table_slots)) return rc;
    if (FILL && reinterpret_cast<uintptr_t>(a->d_rows) % 8) return TS_E_MISALIGNED;
    return 0;
}

template <bool FILL> static int table_pass(const ts_state_table_args* a, uint64_t* d_table, int64_t table_slots, int grid, void* stream) {
    if (int rc = table_pass_check<FILL>(a, d_table, table_slots, grid)) return rc;
    if (a->n_items == 0) return 0;
    return (int)table_kernel(K12<FILL>, *a, k12_smem(*a), d_table, (uint64_t)table_slots, grid, nullptr, (cudaStream_t)stream);
}

extern "C" {

int ts_state_table_table_ctas_per_sm(const ts_state_table_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = table_check_plan(a)) return rc;
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    int dev = 0, count = 0, fill = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = table_kernel(K12<false>, *a, k12_smem(*a), nullptr, 0, 0, &count, nullptr);
    if (e == cudaSuccess) e = table_kernel(K12<true>, *a, k12_smem(*a), nullptr, 0, 0, &fill, nullptr);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    *ctas_per_sm = count < fill ? count : fill;
    return 0;
}

int ts_state_table_count_table(const ts_state_table_args* a, uint64_t* d_table, int64_t table_slots, int grid, void* stream) {
    return table_pass<false>(a, d_table, table_slots, grid, stream);
}
int ts_state_table_fill_table(const ts_state_table_args* a, uint64_t* d_table, int64_t table_slots, int grid, void* stream) {
    return table_pass<true>(a, d_table, table_slots, grid, stream);
}

}  // extern "C"
