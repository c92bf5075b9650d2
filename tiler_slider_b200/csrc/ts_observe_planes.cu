// ts_observe_planes.cu -- network-ready observation: [N][C][S][S] (channel first) of 0/1
// elements in the network's dtype (uint8, bfloat16, float16 or float32); format in
// include/tiler_slider.h.  Plane 0 blocked cells; ordered goal: plane 1+i tile i, plane 1+T+j
// target j; set goal: plane 1 the tile cells, plane 2 the target cells.
//
// A pure HBM writer like K3 (ts_observe.cu): C*S*S elements per env against ~14 bytes read,
// and only 1 + (#walls + T + NT) / (C*S*S) of them are non-zero.  The kernel never looks at the
// dtype beyond its width and the bit pattern of 1, so all four share one instantiation per S.
//
// The output of a call is one contiguous byte string of n_envs * C*S*S*width bytes; block b
// owns bytes [b*STAGE, (b+1)*STAGE) of it, whatever envs or planes that cuts through (an env of
// the largest shape, 16x16 with 32 tiles and 32 targets in fp32, is 66,560 bytes: more than one
// stage).  So every block starts 16-byte aligned, and only the last block of a call is short.
// A block zero-fills its stage in shared memory, drops in the non-zeros that fall inside it --
// one work item per (env, row) for the walls and the set-goal target rows, visiting the set bits
// only; one per (env, tile or target) for the one cell each of those planes has -- and hands
// the stage to the SM's copy engine (cp.async.bulk) in one piece.  A byte count that is not a
// multiple of 16 (the last block of an odd-sized call) streams its 16-byte multiple the same way
// and stores the remaining 1..15 bytes from threads.
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

namespace ts {

constexpr int PLANES_THREADS = 256;
constexpr int PLANES_STAGE = 28672;     // bytes per block, a multiple of 16 (K3's stage size)

struct PlanesParams {
    ts_observe_planes_args a;
    int32_t n_targets, wshift;          // n_targets: ordered targets present (0..32; set goal: 0); element = 1 << wshift bytes
    uint32_t one;                       // bit pattern of 1 in the element type
    int64_t env_bytes, total_bytes;     // C*S*S << wshift; n_envs * env_bytes
};

// ts_observe_planes_items: image e shows env ids[e] (NULL: e) with the tiles of item_pos[e] (NULL:
// that env's pos); a.first_env = 0 and a.n_envs = the item count
struct PlanesItemsParams : PlanesParams {
    const int32_t* ids;
    const uint8_t* item_pos;
};

__device__ __forceinline__ void put_one(uint8_t* stage, int off, int wshift, uint32_t one) {
    if (wshift == 0) stage[off] = (uint8_t)one;
    else if (wshift == 1) *reinterpret_cast<uint16_t*>(stage + off) = (uint16_t)one;
    else *reinterpret_cast<uint32_t*>(stage + off) = one;
}

// env shown by image `item` of an item call; false: its id lies outside [0, capacity) and the image stays zero
__device__ __forceinline__ bool item_env(const PlanesItemsParams& p, int64_t item, size_t& env) {
    const int64_t e = p.ids ? (int64_t)p.ids[item] : item;
    env = (size_t)e;
    return e >= 0 && e < p.a.capacity;
}

// PP = PlanesParams: images of the env range; PP = PlanesItemsParams: images of items (a compile-time
// variant, so the range instantiations are the kernels they were)
template <int S, class PP = PlanesParams>
__global__ void __launch_bounds__(PLANES_THREADS) observe_planes_kernel(const PP p) {
    constexpr bool ITEMS = std::is_same<PP, PlanesItemsParams>::value;
    constexpr int CELLS = S * S, NB = board_bytes(S), PS = pos_stride(S);
    __shared__ __align__(16) uint8_t stage[PLANES_STAGE];
    const ts_observe_planes_args& a = p.a;
    const int64_t start = (int64_t)blockIdx.x * PLANES_STAGE;
    const int len = (int)min((int64_t)PLANES_STAGE, p.total_bytes - start);
    const int64_t e_first = start / p.env_bytes;
    const int n_e = (int)((start + len - 1) / p.env_bytes - e_first) + 1;
    const int env_bytes = (int)p.env_bytes, ws = p.wshift;
    const int base = (int)(e_first * p.env_bytes - start);       // stage offset of env e_first's byte 0, in (-env_bytes, 0]
    const size_t cap = (size_t)a.capacity;
    const bool ordered = a.goal_mode == TS_GOAL_ORDERED;
    const int T = a.n_tiles, NT = p.n_targets, P = T + NT, pw = pos_bytes(T), tpw = pos_bytes(NT);
    const uint32_t one = p.one;

    for (int k = threadIdx.x; k < PLANES_STAGE / 16; k += PLANES_THREADS)
        reinterpret_cast<uint4*>(stage)[k] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();

    // walls (plane 0) and set-goal targets (plane 2): one work item per (env, row); a row whose
    // bytes lie outside the stage is not even loaded, and only the SET bits are visited
    constexpr uint32_t ROW = (1u << S) - 1u;      // drops the sentinels past column S-1
    for (int j = threadIdx.x; j < n_e * S; j += PLANES_THREADS) {
        const int e = j / S, r = j - e * S;
        size_t env;
        bool live = true;
        if constexpr (ITEMS) live = item_env(p, e_first + e, env);
        else env = (size_t)(a.first_env + e_first + e);
        const int o0 = base + e * env_bytes + ((r * S) << ws);              // plane 0, cell (r, 0)
        const int o2 = o0 + ((2 * CELLS) << ws);                            // plane 2, cell (r, 0)
        const bool in0 = live && o0 + (S << ws) > 0 && o0 < len;
        const bool in2 = live && !ordered && o2 + (S << ws) > 0 && o2 < len;
        uint32_t wrow = 0, trow = 0;
        if constexpr (wide_board(S)) {
            if (in0) wrow = (uint32_t)reinterpret_cast<const uint16_t*>(a.d_walls)[(cap + env) * (2 * wide_line_words(S)) + r] >> wide_line_lead(S);   // plane 1 = rows
            if (in2) trow = reinterpret_cast<const uint16_t*>(a.d_targets_packed)[env * WIDE_TARGET_WORDS + r];
        } else {
            if (in0) wrow = (uint32_t)(load_board_elem<NB>(a.d_walls, cap, env) >> (r * board_stride(S)));
            if (in2) trow = (uint32_t)(load_board_elem<NB>(a.d_targets_packed, cap, env) >> (r * board_stride(S)));
        }
        for (uint32_t m = wrow & ROW; m; m &= m - 1u) {
            const int o = o0 + ((__ffs(m) - 1) << ws);
            if (o >= 0 && o < len) put_one(stage, o, ws, one);
        }
        for (uint32_t m = trow & ROW; m; m &= m - 1u) {
            const int o = o2 + ((__ffs(m) - 1) << ws);
            if (o >= 0 && o < len) put_one(stage, o, ws, one);
        }
    }
    // tiles and ordered targets: one work item per (env, k), k < T a tile, T <= k < T+NT a target.
    // Every tile and target owns its plane (set goal: the tiles share plane 1, on distinct cells),
    // so the items are independent; duplicate targets each keep their own plane.
    for (int j = threadIdx.x; j < n_e * P; j += PLANES_THREADS) {
        const int e = j / P, k = j - e * P;
        size_t env;
        if constexpr (ITEMS) {
            if (!item_env(p, e_first + e, env)) continue;
        } else {
            env = (size_t)(a.first_env + e_first + e);
        }
        int plane, b;
        if (k < T) {
            plane = ordered ? 1 + k : 1;
            if constexpr (ITEMS) b = p.item_pos ? p.item_pos[(size_t)(e_first + e) * pw + k] : a.d_pos[env * pw + k];
            else b = a.d_pos[env * pw + k];
        } else {
            plane = 1 + k;
            b = a.d_targets_packed[env * tpw + (k - T)];
        }
        const int o = base + e * env_bytes + ((plane * CELLS + (b / PS) * S + b % PS) << ws);
        if (o >= 0 && o < len) put_one(stage, o, ws, one);
    }

    uint8_t* out = static_cast<uint8_t*>(a.d_out) + start;     // 16-byte aligned: PLANES_STAGE is a multiple of 16
    const int bulk = len & ~15;
    // Stream-out by the copy engine of the SM (TMA 1-D, SASS UBLKCP): the writers publish their
    // shared-memory stores to the async proxy, one elected thread issues the copy and stays until
    // the engine has read the stage.  The 1..15 bytes past the last 16-byte multiple of a short
    // block are plain stores of other threads (reads of the stage only, beside the engine's).
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0 && bulk > 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                     ::"l"(out), "r"((uint32_t)__cvta_generic_to_shared(stage)), "r"((uint32_t)bulk) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    const int t = bulk + (int)threadIdx.x - 32;                 // the tail from the second warp on
    if (threadIdx.x >= 32 && t < len) out[t] = stage[t];
}

template <int S, class PP> static void launch_observe_planes(const PP& p, cudaStream_t st) {
    const unsigned blocks = (unsigned)((p.total_bytes + PLANES_STAGE - 1) / PLANES_STAGE);
    observe_planes_kernel<S, PP><<<blocks, PLANES_THREADS, 0, st>>>(p);
}

// channels of the planes observation; the arguments have been checked (ts_api.cu)
int observe_planes_channels(const ts_observe_planes_args& a) {
    if (a.goal_mode != TS_GOAL_ORDERED) return 3;
    const int nt = a.n_targets == 0 ? a.n_tiles : (a.n_targets < 0 ? 0 : a.n_targets);
    return 1 + a.n_tiles + nt;
}

static void fill_planes_params(PlanesParams& p, const ts_observe_planes_args& a) {
    static const uint32_t ONE[4] = {1u, 0x3F80u, 0x3C00u, 0x3F800000u};    // u8, bf16, f16, f32
    static const int32_t SHIFT[4] = {0, 1, 1, 2};
    p.a = a;
    const int C = observe_planes_channels(a);
    p.n_targets = a.goal_mode == TS_GOAL_ORDERED ? C - 1 - a.n_tiles : 0;
    p.wshift = SHIFT[a.dtype];
    p.one = ONE[a.dtype];
    p.env_bytes = (int64_t)C * a.size * a.size << p.wshift;
    p.total_bytes = a.n_envs * p.env_bytes;
}

template <class PP> static cudaError_t launch_planes_size(const PP& p, cudaStream_t st) {
    switch (p.a.size) {
#define TS_OBSP(S) case S: launch_observe_planes<S>(p, st); break;
        TS_OBSP(1) TS_OBSP(2) TS_OBSP(3) TS_OBSP(4) TS_OBSP(5) TS_OBSP(6) TS_OBSP(7) TS_OBSP(8)
        TS_OBSP(9) TS_OBSP(10) TS_OBSP(11) TS_OBSP(12) TS_OBSP(13) TS_OBSP(14) TS_OBSP(15) TS_OBSP(16)
#undef TS_OBSP
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t observe_planes_dispatch(const ts_observe_planes_args& a, cudaStream_t st) {
    PlanesParams p;
    fill_planes_params(p, a);
    return launch_planes_size(p, st);
}

cudaError_t observe_planes_items_dispatch(const ts_observe_planes_args& a, const int32_t* ids, const uint8_t* item_pos,
                                          int64_t n_items, cudaStream_t st) {
    ts_observe_planes_args r = a;
    r.first_env = 0;
    r.n_envs = n_items;
    PlanesItemsParams p;
    fill_planes_params(p, r);
    p.ids = ids;
    p.item_pos = item_pos;
    return launch_planes_size(p, st);
}

}  // namespace ts
