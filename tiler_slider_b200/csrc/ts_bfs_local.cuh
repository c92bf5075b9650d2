// ts_bfs_local.cuh -- what the on-chip searches, K6 (ts_bfs_local.cu, the batched BFS), K9
// (ts_optimal.cu, the optimal-move query) and K10 (ts_state_table.cu, the state tables), share: the
// CTA shape, canonical set-goal states, position byte -> bitboard bit, the perfect hash of a state
// over the free cells of its puzzle that keys the visited bitmap, the successor function, the lut
// fill, the bitmap clear and K9 and K10's root read (and their 64-bit siblings for K11 and K12's 5..8
// tiles, ts_table_search.cu and ts_table_state_table.cu); on the host the plan and env-table checks of K9 and K10, the plan check, the
// shared-memory size, the launch and the occupancy query, one each for the shared instances and the
// device-memory-bitmap instances (GMEM) of 7x7 and 8x8 boards with four tiles.
#pragma once
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

// threads of a search CTA, one (state, move) pair each (384 and 512 measured within noise: DESIGN.md)
constexpr int SEARCH_THREADS = 256;
// entries of a search's per-level buffers: K6 leaves a puzzle of more levels to the hash-partitioned
// search, K9 takes max_depth <= TS_OPT_MAX_DEPTH
constexpr int SEARCH_LEVELS = 256;
static_assert(TS_OPT_MAX_DEPTH + 2 <= SEARCH_LEVELS, "K9 keeps the start of levels 0 .. max_depth + 1");

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
// bitboard bit of position byte p as a mask, 0 when p is no cell of the board (so that a word of
// T tiles is well-formed iff its T masks are distinct free cells: popcount T, all inside free_cells)
template <int S> __device__ __forceinline__ uint64_t cell_bit(uint32_t p) {
    if constexpr (padded_board(S)) return p < 64u ? (1ull << p) & cell_mask<S>() : 0ull;
    else return (p >> 4) < (uint32_t)S && (p & 15u) < (uint32_t)S ? 1ull << pos_to_bit<S>(p) : 0ull;
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

// The successor function of the three searches: the state after move m from q0 on a board of these
// walls, through the step's slide_env (GameState.move, explainrl/environment/state.py:120-170); won =
// it meets the goal (is_won, state.py:172-186: set goal, occupancy tboard; ordered, word tq).  A
// set-goal state comes back canonical, its bytes sorted: tiles are interchangeable (state.py:185-186).
template <int S, int T>
__device__ __forceinline__ uint32_t successor(uint32_t q0, uint32_t m, uint64_t walls, bool set_goal, uint64_t tboard, uint32_t tq, bool& won) {
    uint32_t q[1] = {q0};
    slide_env<S, T>(q, walls, m >> 1, (m & 1u) ^ 1u);
    if (set_goal) {
        won = occupancy<S, T>(q) == tboard;
        sort_bytes4<T>(q[0]);
    } else {
        won = q[0] == tq;
    }
    return q[0];
}

// ---- 64-bit states (K11, 5..8 tiles): the 8 position bytes of a state as one word ----------------
// canonical form of a set-goal state of T <= 8 tiles: its T position bytes sorted ascending
template <int T> __device__ __forceinline__ void sort_bytes8(uint64_t& q) {
    uint32_t b[T];
    static_for<0, T>([&](auto I) { constexpr int i = decltype(I)::value; b[i] = (uint32_t)(q >> (8 * i)) & 0xFFu; });
#pragma unroll
    for (int round = 0; round < T; ++round)
#pragma unroll
        for (int i = round & 1; i + 1 < T; i += 2) {
            const uint32_t lo = min(b[i], b[i + 1]), hi = max(b[i], b[i + 1]);
            b[i] = lo; b[i + 1] = hi;
        }
    q = 0;
    static_for<0, T>([&](auto I) { constexpr int i = decltype(I)::value; q |= (uint64_t)b[i] << (8 * i); });
}

// successor<S,T> for 5..8 tiles: the same slide, goal test and canonicalisation on a 64-bit word
template <int S, int T>
__device__ __forceinline__ uint64_t successor64(uint64_t q0, uint32_t m, uint64_t walls, bool set_goal, uint64_t tboard, uint64_t tq, bool& won) {
    static_assert(T >= 5 && T <= 8, "two 32-bit position words");
    uint32_t q[2] = {(uint32_t)q0, (uint32_t)(q0 >> 32)};
    slide_env<S, T>(q, walls, m >> 1, (m & 1u) ^ 1u);
    uint64_t qn = (uint64_t)q[1] << 32 | q[0];
    if (set_goal) {
        won = occupancy<S, T>(q) == tboard;
        sort_bytes8<T>(qn);
    } else {
        won = qn == tq;
    }
    return qn;
}

// read_root<S,T> for 5..8 tiles: the root word of an item and whether it is a well-formed state
template <int S, int T, class A>
__device__ __forceinline__ bool read_root64(const A& a, long long ticket, size_t pid, uint64_t free_cells, uint64_t& root) {
    constexpr int PW = pos_bytes(T);
    const uint8_t* const root_pos = a.d_item_pos ? a.d_item_pos + (size_t)ticket * PW : a.d_pos + pid * PW;
    uint64_t occ = 0;
    root = 0;
    static_for<0, T>([&](auto I) {
        constexpr int t = decltype(I)::value;
        const uint32_t p = root_pos[t];
        root |= (uint64_t)p << (8 * t);
        occ |= cell_bit<S>(p);
    });
    return __popcll(occ) == T && !(occ & ~free_cells);
}

// position byte -> rank among the free cells (lut, 128 entries) and, given rank_byte, rank -> position
// byte, filled by the block; read after the caller's next __syncthreads.  tid as in clear_bitmap.
template <int S>
__device__ __forceinline__ void fill_lut(uint32_t tid, uint64_t free_cells, uint8_t* lut, uint8_t* rank_byte = nullptr) {
    if (tid < 128) {
        const uint32_t bit = pos_to_bit<S>(tid);
        const uint32_t rank = bit < 64 ? (uint32_t)__popcll(free_cells & ((1ull << bit) - 1ull)) : 0u;
        lut[tid] = (uint8_t)rank;
        if (rank_byte && (cell_bit<S>(tid) & free_cells)) rank_byte[rank] = (uint8_t)tid;
    }
}

// The root word of an item (K9, K10): row `ticket` of a.d_item_pos, else env pid's positions.  False
// when it is no state: each tile must stand on its own free cell (an off-board byte adds no bit, two
// tiles on one cell one), the states the hash is defined for.
template <int S, int T, class A>
__device__ __forceinline__ bool read_root(const A& a, long long ticket, size_t pid, uint64_t free_cells, uint32_t& root) {
    constexpr int PW = pos_bytes(T);
    const uint8_t* const root_pos = a.d_item_pos ? a.d_item_pos + (size_t)ticket * PW : a.d_pos + pid * PW;
    uint64_t occ = 0;
    root = 0;
    static_for<0, T>([&](auto I) {
        constexpr int t = decltype(I)::value;
        const uint32_t p = root_pos[t];
        root |= p << (8 * t);
        occ |= cell_bit<S>(p);
    });
    return __popcll(occ) == T && !(occ & ~free_cells);
}

// the first `words` words of a bitmap, rounded up to whole 16-byte units, cleared by the block.  tid
// is the kernel's thread index: a read of threadIdx.x outside the kernel's own body loses what
// __launch_bounds__ tells the compiler about it (tid < SEARCH_THREADS), and registers with it.
__device__ __forceinline__ void clear_bitmap(uint32_t* bitmap, uint32_t words, uint32_t tid) {
    for (uint32_t k = tid; k < (words + 3) / 4; k += SEARCH_THREADS) reinterpret_cast<uint4*>(bitmap)[k] = make_uint4(0u, 0u, 0u, 0u);
}

// ---- host side -------------------------------------------------------------------------------------
// tile count, goal mode and shared-memory plan of a search launch: a bitmap of whole 16-byte units,
// a power-of-two ring of at least 32 entries
template <class A> int check_search_plan(const A& a) {
    if (a.n_tiles < 1 || a.n_tiles > 4) return TS_E_UNSUPPORTED;            // 32-bit states
    if (a.goal_mode != TS_GOAL_ORDERED && a.goal_mode != TS_GOAL_SET) return TS_E_BAD_ARGUMENT;
    if (a.bitmap_words < 4 || a.bitmap_words % 4 || a.queue_smem < 32 || (a.queue_smem & (a.queue_smem - 1))) return TS_E_BAD_ARGUMENT;
    return 0;
}

// K9 and K10: shape and shared-memory plan
template <class A> int check_item_plan(const A* a) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;                                 // wide boards: no 64-bit board word
    return check_search_plan(*a);
}

// K9 and K10: the env table the items are read from
template <class A> int check_item_table(const A* a) {
    if (a->capacity <= 0 || a->capacity % TS_CAP_ALIGN) return TS_E_BAD_CAPACITY;
    if (a->n_items < 0 || (!a->d_env_ids && a->n_items > a->capacity)) return TS_E_BAD_RANGE;
    if (!a->d_walls || !a->d_targets_packed || !a->d_pos) return TS_E_NULL_POINTER;
    return 0;
}

template <class A> size_t search_smem_bytes(const A& a) { return ((size_t)a.bitmap_words + (size_t)a.queue_smem) * sizeof(uint32_t); }

// ---- device-memory bitmaps -------------------------------------------------------------------------
// With four tiles, a board of more than 38 free cells has a state space whose bitmap does not fit
// one CTA's shared memory; only 7x7 and 8x8 boards have that many.  Their device instances (GMEM)
// keep the bitmap in device memory instead, CTA b's at d_bitmap + b * bitmap_words, and dynamic
// shared memory holds the ring alone.  Every other shape fits shared memory at every wall count, so
// no other device instance is built.
__host__ __device__ constexpr bool gmem_shape(int size, int n_tiles) { return n_tiles == 4 && (size == 7 || size == 8); }

// the checks the device entry points add after their shared counterpart's: the shape, then the buffer
template <class A> int check_gmem(const A& a, const uint32_t* d_bitmap) {
    if (!gmem_shape(a.size, a.n_tiles)) return TS_E_UNSUPPORTED;
    if (!d_bitmap) return TS_E_NULL_POINTER;
    if (reinterpret_cast<uintptr_t>(d_bitmap) % 16) return TS_E_MISALIGNED;
    return 0;
}

// Instance <a.size, a.n_tiles, GMEM> of a search kernel (kernel_of(IC<S>, IC<T>, bool_constant<GMEM>)
// returns it; it takes a and the bitmap buffer d_bitmap[grid][bitmap_words], unused by the shared
// instances) with a's dynamic shared memory, the ring and, shared instances only, the bitmap:
// launched on `grid` CTAs, or, when ctas_per_sm is given, asked how many of its CTAs fit an SM.
// GMEM: a.size is 7 or 8 and a.n_tiles 4, checked by the caller.
template <bool GMEM, class KernelOf, class A>
cudaError_t search_kernel(KernelOf&& kernel_of, const A& a, uint32_t* d_bitmap, int grid, int* ctas_per_sm, cudaStream_t st) {
    const size_t smem = GMEM ? (size_t)a.queue_smem * sizeof(uint32_t) : search_smem_bytes(a);
    auto go = [&](auto S, auto T) {
        const auto kernel = kernel_of(S, T, std::bool_constant<GMEM>{});
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (ctas_per_sm) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, kernel, SEARCH_THREADS, smem);
        kernel<<<grid, SEARCH_THREADS, smem, st>>>(a, d_bitmap);
        return cudaGetLastError();
    };
    if constexpr (GMEM) return a.size == 7 ? go(IC<7>{}, IC<4>{}) : go(IC<8>{}, IC<4>{});
    else return dispatch_small(a.size, a.n_tiles, go);
}

// resident CTAs per SM of a's search kernel and the SM count of the current device
template <bool GMEM, class KernelOf, class A>
int search_ctas_per_sm(KernelOf&& kernel_of, const A& a, int* ctas_per_sm, int* n_sm) {
    if (!ctas_per_sm || !n_sm) return TS_E_NULL_POINTER;
    if (GMEM && !gmem_shape(a.size, a.n_tiles)) return TS_E_UNSUPPORTED;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = search_kernel<GMEM>(kernel_of, a, nullptr, 0, ctas_per_sm, nullptr);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    return 0;
}

}  // namespace ts
