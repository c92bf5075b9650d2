// ts_table_search.cu -- K11: K9's answers (exact distance to the goal, the set of optimal first moves
// and optionally a shortest solution of items) for 5 to 8 tiles, where a state is a 64-bit word and
// K9's perfect-hash bitmap (F!/(F-T)! bits) outgrows even device memory.  The CTA shape, the ticket
// counter, the forward level loop, the backward rule and the plan are K9's (ts_optimal.cu); the
// visited set is a hash table in device memory whose size follows the states an item reaches.
//
//   Table: the per-CTA hash table of ts_hash_table.cuh (keys, flag bits, item epochs).
//   Bound: the slab holds spill_per_cta states; the item stops with TS_OPT_NOT_SEARCHED once it has
//      discovered more (K9's rule), and table_slots >= 2 * spill_per_cta.  Inserts stop once the
//      level has met the goal or overflowed, so a table holds at most spill_per_cta + 255 keys of an
//      item; a probe is still bounded by table_slots, and a full table (more than spill_per_cta
//      keys) overflows the item like the slab does.
//   Forward: K9's level loop over 64-bit states (ring in shared memory, slab in device memory); a
//      new state is the one whose CAS claims an empty slot (looked at first, as K5 does).
//   Backward: K9's rule; the flags of level k are written into bit 7 / the move bits of the level's
//      slab entries, which keep their keys, and after a barrier ORed into the states' slots.
//   Plan: from the root, the move stored in the slot of each state reached.
#include "ts_hash_table.cuh"

namespace ts {

// PLAN as in K9: the instance that writes d_plan
template <int S, int T, bool PLAN>
__global__ void __launch_bounds__(SEARCH_THREADS) table_search_kernel(const ts_optimal_moves_args a, uint64_t* const d_table, const uint64_t table_slots) {
    constexpr int PW = pos_bytes(T), NB = board_bytes(S);
    static_assert(T >= 5 && T <= 8 && PW == 8, "64-bit states");
    extern __shared__ __align__(16) uint64_t ring[];
    __shared__ uint32_t lstart[SEARCH_LEVELS];   // level k = discovery indices [lstart[k], lstart[k+1])
    __shared__ uint32_t cnt[3];                  // entries appended during level L: cnt[L % 3]
    __shared__ uint32_t lflag[3];                // ... and whether a successor met the goal (WON) / the item overflowed (OVER)
    __shared__ long long s_ticket;

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t R = (uint32_t)a.queue_smem, RMASK = R - 1u;
    uint64_t* const slab = reinterpret_cast<uint64_t*>(a.d_spill) + (size_t)blockIdx.x * (size_t)a.spill_per_cta;
    uint64_t* const table = d_table + (size_t)blockIdx.x * table_slots;
    const uint64_t smask = table_slots - 1u;
    const uint32_t q_cap = (uint32_t)a.spill_per_cta;
    const size_t cap = (size_t)a.capacity;
    unsigned long long fwd = 0, bwd = 0;
    uint32_t epoch = 0;                          // of the CTA's current item: 1 .. TAB_EPOCHS

    for (;;) {
        __syncthreads();                         // the previous item is finished with shared memory and the table
        if (tid == 0) s_ticket = (long long)atomicAdd((unsigned long long*)&a.d_counters[0], 1ull);
        __syncthreads();
        const long long ticket = s_ticket;
        if (ticket >= a.n_items) break;
        auto plan_at = [&](uint32_t r) -> uint8_t& { return a.d_plan[(size_t)r * (size_t)a.n_items + (size_t)ticket]; };
        auto no_solution = [&](int32_t code) {
            if (tid == 0) { a.d_distance[ticket] = code; a.d_mask[ticket] = 0; }
            if constexpr (PLAN)
#pragma unroll 1
                for (uint32_t r = tid; r < (uint32_t)a.max_depth; r += SEARCH_THREADS) plan_at(r) = 0xFF;
        };
        const long long env = a.d_env_ids ? (long long)a.d_env_ids[ticket] : ticket;
        if (env < 0 || env >= a.capacity) { no_solution(TS_OPT_NOT_SEARCHED); continue; }
        const size_t pid = (size_t)env;

        // ---- the item: walls, goal, root state ----------------------------------------------------
        const uint64_t walls = load_board_elem<NB>(a.d_walls, cap, pid);
        const uint64_t free_cells = ~walls & cell_mask<S>();
        uint64_t root;
        if (!read_root64<S, T>(a, ticket, pid, free_cells, root)) { no_solution(TS_OPT_BAD_STATE); continue; }
        if (a.never_win) { no_solution(TS_OPT_UNSOLVABLE); continue; }
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
        if (tid == 0) {
            cnt[0] = cnt[1] = cnt[2] = 0; lflag[0] = lflag[1] = lflag[2] = 0;
            table_insert(table, smask, ep, root);
            ring[0] = root;
            slab[0] = root;
            lstart[0] = 0;
        }
        __syncthreads();

        auto successor = [&](uint64_t q0, uint32_t m, bool& won) { return successor64<S, T>(q0, m, walls, set_goal, tboard, tq, won); };
        auto marked = [&](uint64_t q) {
            const long long h = table_find(table, smask, ep, q);
            return h >= 0 && (__ldcg(table + h) & TAB_MARK);
        };

        // ---- 1. forward: BFS levels until a successor meets the goal (K9) ------------------------
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
                uint64_t qn = 0;
                if (live) {
                    const uint64_t q0 = (src - prev_lo) < R ? ring[src & RMASK] : slab[src];
                    bool won;
                    qn = successor(q0, d, won);
                    if (won) atomicOr(my_flag, TAB_WON);
                    // once this level has met the goal or overflowed its successors are never read
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
                        if (pos - lo < R) ring[pos & RMASK] = qn;
                        if (pos < q_cap) slab[pos] = qn;
                        else atomicOr(my_flag, TAB_OVER);
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
            if (flag & TAB_WON) { dist = (int32_t)depth; break; }
            if (flag & TAB_OVER) { dist = TS_OPT_NOT_SEARCHED; break; }
        }
        if (dist < 0) { no_solution(dist); continue; }

        // ---- 2. backward: mark the states of levels d-1 .. 1 that start a shortest solution ------
        const uint32_t D = (uint32_t)dist;
        if (D >= 2) {
            __syncthreads();                      // lstart complete
            for (uint32_t k = D - 1u; k >= 1u; --k) {
                const uint32_t l0 = lstart[k], l1 = lstart[k + 1u];
                const uint32_t n_items = (l1 - l0) * 4u;
                for (uint32_t base = 0; base < n_items; base += SEARCH_THREADS) {
                    const uint32_t j = base + tid;
                    const bool live = j < n_items;
                    const uint32_t src = l0 + (j >> 2);
                    bool hit = false;
                    uint64_t q0 = 0;
                    if (live) {
                        q0 = slab[src];
                        bool won;
                        const uint64_t qn = successor(q0, j & 3u, won);
                        hit = k == D - 1u ? won : (qn != q0 && marked(qn));
                    }
                    // the four lanes of a state are lanes 4i .. 4i+3 of one warp
                    const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
                    const uint32_t hits = (m >> lane) & 0xFu;
                    if (live && (j & 3u) == 0u && hits) slab[src] = q0 | TAB_MARK | move_bits((uint32_t)(__ffs(hits) - 1));
                }
                __syncthreads();                  // every flag of level k computed
                for (uint32_t s = l0 + tid; s < l1; s += SEARCH_THREADS) {
                    const uint64_t e = slab[s];
                    if (e & TAB_MARK) {
                        const long long h = table_find(table, smask, ep, e & TAB_KEY);
                        if (h >= 0) atomicOr((unsigned long long*)(table + h), (unsigned long long)(e & (TAB_MARK | TAB_MOVE)));
                    }
                }
                __syncthreads();                  // level k marked
                if (tid == 0) bwd += l1 - l0;
            }
        }

        // ---- 3. root: its optimal moves; 4. plan: the move stored with each state reached --------
        if (tid < 32) {
            bool hit = false;
            if (lane < 4) {
                bool won;
                const uint64_t qn = successor(root, lane, won);
                hit = D == 1u ? won : (qn != root && marked(qn));
            }
            const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
            if (tid == 0) {
                a.d_distance[ticket] = dist;
                a.d_mask[ticket] = (uint8_t)(m & 0xFu);
                if constexpr (PLAN) {
                    uint32_t mv = (uint32_t)(__ffs(m) - 1);
                    uint64_t q = root;
#pragma unroll 1
                    for (uint32_t k = 0;;) {
                        plan_at(k) = (uint8_t)mv;
                        if (++k == D) break;
                        bool won;
                        q = successor(q, mv, won);
                        // q is good at level k: in the table, its slot holds its lowest optimal move
                        const long long h = table_find(table, smask, ep, q);
                        mv = h >= 0 ? move_of(__ldcg(table + h)) : 0u;
                    }
                }
            }
        }
        if constexpr (PLAN)
#pragma unroll 1
            for (uint32_t r = D + tid; r < (uint32_t)a.max_depth; r += SEARCH_THREADS) plan_at(r) = 0xFF;
    }
    if (tid == 0) {
        atomicAdd((unsigned long long*)&a.d_counters[1], fwd);
        atomicAdd((unsigned long long*)&a.d_counters[2], bwd);
    }
}

static constexpr auto K11 = [](auto S, auto T) { return table_search_kernel<decltype(S)::value, decltype(T)::value, false>; };
static constexpr auto K11_PLAN = [](auto S, auto T) { return table_search_kernel<decltype(S)::value, decltype(T)::value, true>; };
// dynamic shared memory of K11: the ring alone
static size_t k11_smem(const ts_optimal_moves_args& a) { return (size_t)a.queue_smem * sizeof(uint64_t); }

}  // namespace ts

using namespace ts;

extern "C" {

int ts_optimal_moves_table_ctas_per_sm(const ts_optimal_moves_args* a, int* ctas_per_sm, int* n_sm) {
    if (int rc = table_check_plan(a)) return rc;
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = a->d_plan ? table_kernel(K11_PLAN, *a, k11_smem(*a), nullptr, 0, 0, ctas_per_sm, nullptr)
                                        : table_kernel(K11, *a, k11_smem(*a), nullptr, 0, 0, ctas_per_sm, nullptr);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    return 0;
}

int ts_optimal_moves_table(const ts_optimal_moves_args* a, uint64_t* d_table, int64_t table_slots, int grid, void* stream) {
    if (int rc = table_check_plan(a)) return rc;
    if (int rc = check_item_table(a)) return rc;
    if (a->max_depth < 1 || a->max_depth > TS_OPT_MAX_DEPTH || a->spill_per_cta < 1 || a->spill_per_cta > 0xFFFFFFFFll)
        return TS_E_BAD_ARGUMENT;
    if (!a->d_spill || !a->d_counters || !a->d_distance || !a->d_mask) return TS_E_NULL_POINTER;
    if (int rc = table_check_buffer(a, d_table, table_slots)) return rc;
    if (a->n_items == 0) return 0;
    if (grid < 1) return TS_E_BAD_ARGUMENT;
    return (int)(a->d_plan ? table_kernel(K11_PLAN, *a, k11_smem(*a), d_table, (uint64_t)table_slots, grid, nullptr, (cudaStream_t)stream)
                           : table_kernel(K11, *a, k11_smem(*a), d_table, (uint64_t)table_slots, grid, nullptr, (cudaStream_t)stream));
}

}  // extern "C"
