// ts_hash_table.cuh -- what the hash-table searches for 5 to 8 tiles, K11 (ts_table_search.cu, the
// optimal-move query) and K12 (ts_table_state_table.cu, the state tables), share: the per-CTA visited
// table in device memory with its item epochs and flag bits, and on the host the plan check and the
// launch / occupancy query with the ring (and whatever else the kernel keeps there) alone in dynamic
// shared memory.
//
//   Table: CTA b owns d_table[b * table_slots ..], table_slots a power of two; open addressing with
//      linear probing from a 64-bit mix of the key.  A key is the state word; every position byte is
//      < 128, so bit 7 of each byte is free, and those eight bits hold:
//        bit 7             MARK: the state is good (K11's backward pass) / resolved (K12's sweep)
//        bits 15, 23       the lowest optimal move of a good state (K11's plan)
//        bits 31 .. 63     the item epoch of the slot (5 bits, 1 .. 31)
//      A slot whose epoch is not the current item's is empty, so an item starts on an empty table
//      without clearing it; the slice is cleared only when the epoch wraps (every 31 items of a CTA,
//      and before its first item, as the buffer's contents on entry are undefined).
#pragma once
#include "ts_bfs_local.cuh"

namespace ts {

constexpr uint64_t TAB_KEY = 0x7F7F7F7F7F7F7F7Full;        // the position bytes of a slot
constexpr uint64_t TAB_MARK = 1ull << 7;
constexpr uint64_t TAB_MOVE = 1ull << 15 | 1ull << 23;
constexpr uint64_t TAB_EPOCH = 0x8080808080000000ull;      // bits 31, 39, 47, 55, 63
constexpr uint32_t TAB_EPOCHS = 31;
constexpr uint32_t TAB_WON = 1u, TAB_OVER = 2u;

__device__ __forceinline__ uint64_t epoch_bits(uint32_t e) {
    uint64_t b = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) b |= (uint64_t)((e >> i) & 1u) << (31 + 8 * i);
    return b;
}
__device__ __forceinline__ uint64_t move_bits(uint32_t m) { return (uint64_t)(m & 1u) << 15 | (uint64_t)(m >> 1) << 23; }
__device__ __forceinline__ uint32_t move_of(uint64_t e) { return (uint32_t)((e >> 15) & 1u) | (uint32_t)((e >> 22) & 2u); }
// first slot of key q's probe sequence (the splitmix64 finaliser)
__device__ __forceinline__ uint64_t slot_of(uint64_t q, uint64_t smask) {
    q = (q ^ (q >> 30)) * 0xBF58476D1CE4E5B9ull;
    q = (q ^ (q >> 27)) * 0x94D049BB133111EBull;
    return (q ^ (q >> 31)) & smask;
}

// insert q: 1 new (this thread's CAS claimed an empty slot), 0 present, -1 the table is full.  Slots
// are read through L2 (ld.cg): other threads of the CTA claim them with atomics meanwhile.
__device__ __forceinline__ int table_insert(uint64_t* table, uint64_t smask, uint64_t ep, uint64_t q) {
    uint64_t h = slot_of(q, smask);
#pragma unroll 1
    for (uint64_t n = 0; n <= smask; ++n, h = (h + 1) & smask) {
        uint64_t v = __ldcg(table + h);
        if ((v & TAB_EPOCH) != ep) {
            const uint64_t old = atomicCAS((unsigned long long*)(table + h), (unsigned long long)v, (unsigned long long)(q | ep));
            if (old == v) return 1;
            v = old;                              // claimed meanwhile, in this epoch
        }
        if ((v & TAB_KEY) == q) return 0;
    }
    return -1;
}

// the slot holding q, or -1 when q is not in the table
__device__ __forceinline__ long long table_find(const uint64_t* table, uint64_t smask, uint64_t ep, uint64_t q) {
    uint64_t h = slot_of(q, smask);
#pragma unroll 1
    for (uint64_t n = 0; n <= smask; ++n, h = (h + 1) & smask) {
        const uint64_t v = __ldcg(table + h);
        if ((v & TAB_EPOCH) != ep) return -1;
        if ((v & TAB_KEY) == q) return (long long)h;
    }
    return -1;
}

// ---- host side -------------------------------------------------------------------------------------
// Instance kernel_of(IC<S>, IC<T>) (S = a.size, T = a.n_tiles) of a hash-table kernel taking (a,
// d_table, table_slots), with `smem` bytes of dynamic shared memory: launched on `grid` CTAs, or, when
// ctas_per_sm is given, asked how many of its CTAs fit an SM
template <class KernelOf, class A>
cudaError_t table_kernel(KernelOf&& kernel_of, const A& a, size_t smem, uint64_t* d_table, uint64_t table_slots,
                         int grid, int* ctas_per_sm, cudaStream_t st) {
    return dispatch_size(a.size, [&](auto S) {
        constexpr int SV = decltype(S)::value;
        if constexpr (SV < 3) return cudaErrorInvalidValue;                          // no smaller board holds five tiles
        else return dispatch_tiles<5, 8>(a.n_tiles, [&](auto T) {
            const auto kernel = kernel_of(S, T);
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            if (ctas_per_sm) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, kernel, SEARCH_THREADS, smem);
            kernel<<<grid, SEARCH_THREADS, smem, st>>>(a, d_table, table_slots);
            return cudaGetLastError();
        });
    });
}

// K9 / K10's plan checks (check_item_plan) for 5..8 tiles with no bitmap: shape, goal mode, ring
template <class A> int table_check_plan(const A* a) {
    if (!a) return TS_E_NULL_POINTER;
    if (a->size < 1 || a->size > TS_MAX_SIZE) return TS_E_BAD_SIZE;
    if (a->size > 8) return TS_E_UNSUPPORTED;
    if (a->n_tiles < 5 || a->n_tiles > 8) return TS_E_UNSUPPORTED;             // 64-bit states; 1..4 tiles: K9 / K10
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return TS_E_BAD_ARGUMENT;
    if (a->bitmap_words != 0 || a->queue_smem < 32 || (a->queue_smem & (a->queue_smem - 1))) return TS_E_BAD_ARGUMENT;
    return 0;
}

// the table buffer of a launch: a power of two >= 2 * spill_per_cta slots (TS_E_BAD_ARGUMENT), non-NULL
// (TS_E_NULL_POINTER), 8-byte aligned with the slab (TS_E_MISALIGNED)
template <class A> int table_check_buffer(const A* a, const uint64_t* d_table, int64_t table_slots) {
    if (table_slots < 2 * a->spill_per_cta || (table_slots & (table_slots - 1))) return TS_E_BAD_ARGUMENT;
    if (!d_table) return TS_E_NULL_POINTER;
    if (reinterpret_cast<uintptr_t>(d_table) % 8 || reinterpret_cast<uintptr_t>(a->d_spill) % 8) return TS_E_MISALIGNED;
    return 0;
}

}  // namespace ts
