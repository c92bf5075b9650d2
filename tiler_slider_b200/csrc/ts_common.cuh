// ts_common.cuh -- packed-state layout rules and the closed-form slide core shared by every
// sm_100a kernel of the Tiler-Slider step path.
//
// Results reproduced (reference paths relative to the reference checkout):
//   explainrl/environment/state.py:120-170  GameState.move   -> slide_env<S,T>()
//   explainrl/environment/state.py:172-186  GameState.is_won -> goal compare in the callers
//
// Layout in HBM (struct-of-arrays, environment index innermost; DESIGN.md section 3):
//   position word   one word of POS_BYTES(T) in {1,2,4,8} bytes per env; byte i = row*PS + col
//                   of tile i with PS = pos_stride(S); unused bytes are zero
//   board planes    a bitboard per env, bit row*BS + col with BS = board_stride(S), little
//                   endian, board_bytes(S) bytes, split into byte planes of width 16/8/4/2/1
//                   (widest first); plane k starts at byte offset plane_offset(k)*capacity of
//                   the buffer and is indexed by env
//   S <= 6 ("padded" boards): BS = PS = S+1.  Column S of every row of a WALL board and all
//                   bits past the last row are stored as 1 (sentinels): a slide toward higher
//                   indices stops there without any per-tile edge test.  Target boards (set
//                   goal) use the same stride without sentinels.
//   S = 7, 8 (compact boards): BS = S, PS = 16, no sentinels.
//   S >= 9 (wide boards): PS = 16; walls are two records of 4*ceil(S/2) bytes per env, rows and columns
//                   (walls[axis][env][line] u16), the set-goal target board 17 u16 words
//                   (tboard[env][16 rows + distinct-target count]); see ts_wide.cu.
//   capacity        allocation stride in envs, a multiple of 128 so that every plane start and
//                   every 4-env group is 16-byte aligned
// A thread owns GROUP=4 consecutive envs, so every stream is read with one 32/64/128-bit
// load per plane and a warp touches whole 128-byte lines.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace ts {

constexpr int GROUP = 4;           // envs per thread
constexpr int CAP_ALIGN = 128;     // capacity granularity (envs)
constexpr int MAX_SIZE = 16;
constexpr int MAX_TILES = 8;        // tile counts the register kernels are instantiated for
constexpr int MAX_TILES_ANY = 32;   // tile counts the library covers (9..32: per-env generic kernels, ts_generic.cu)

__host__ __device__ constexpr int pos_bytes(int T) { return T <= 1 ? 1 : T <= 2 ? 2 : T <= 4 ? 4 : T <= 8 ? 8 : T <= 16 ? 16 : 32; }   // T = 0: one (zero) byte
__host__ __device__ constexpr bool padded_board(int S) { return S <= 6; }
__host__ __device__ constexpr int board_stride(int S) { return padded_board(S) ? S + 1 : S; }
__host__ __device__ constexpr int pos_stride(int S) { return padded_board(S) ? S + 1 : 16; }
__host__ __device__ constexpr int board_bits(int S) { return S * board_stride(S); }
__host__ __device__ constexpr int board_bytes(int S) { return (board_bits(S) + 7) / 8; }
// wide boards (S >= 9) do not fit 64 bits: env-major sectors of sixteen 16-bit lines, see ts_wide.cu
__host__ __device__ constexpr bool wide_board(int S) { return S > 8; }
// wide WALL lines: 9 <= S <= 14 keep cell k at bit k+1, between edge sentinels at bit 0 and bit S+1;
// S = 15, 16 have no room: cell k at bit k, no sentinel
__host__ __device__ constexpr int wide_line_lead(int S) { return S <= 14 ? 1 : 0; }
// wide WALL records: ceil(S/2) pair words (two 16-bit lines each) per env and axis, two axis planes
__host__ __device__ constexpr int wide_line_words(int S) { return (S + 1) / 2; }
__host__ __device__ constexpr int walls_bytes(int S) { return wide_board(S) ? 8 * wide_line_words(S) : board_bytes(S); }   // per env
// wide set-goal target record: 16 row words + 1 word holding the number of DISTINCT target cells
// (the wide kernels test "every tile on a target cell", which is set equality exactly when that
// number equals the tile count; state.py:185-186)
constexpr int WIDE_TARGET_WORDS = 17;
__host__ __device__ constexpr int target_board_bytes(int S) { return wide_board(S) ? 2 * WIDE_TARGET_WORDS : board_bytes(S); }  // per env, set goal

// decomposition of nb bytes into planes of width 16 (repeated), 8, 4, 2, 1
__host__ __device__ constexpr int plane_count(int nb) {
    int k = nb / 16, rem = nb % 16;
    for (int w = 8; w >= 1; w >>= 1)
        if (rem >= w) { rem -= w; ++k; }
    return k;
}
__host__ __device__ constexpr int plane_width(int nb, int i) {
    int k = 0, rem = nb;
    while (rem >= 16) { if (k == i) return 16; rem -= 16; ++k; }
    for (int w = 8; w >= 1; w >>= 1)
        if (rem >= w) { if (k == i) return w; rem -= w; ++k; }
    return 0;
}
__host__ __device__ constexpr int plane_offset(int nb, int i) {
    int off = 0;
    for (int k = 0; k < i; ++k) off += plane_width(nb, k);
    return off;
}

// ---- compile-time loop -----------------------------------------------------------------
template <int I> struct IC { static constexpr int value = I; };
template <int B, int E, class F> __device__ __forceinline__ void static_for(F&& f) {
    if constexpr (B < E) { f(IC<B>{}); static_for<B + 1, E>(f); }
}

// host: f(IC<S>{}) for the board sizes of one 64-bit board, 1..8
template <class F> cudaError_t dispatch_size(int size, F&& f) {
    switch (size) {
        case 1: return f(IC<1>{});
        case 2: return f(IC<2>{});
        case 3: return f(IC<3>{});
        case 4: return f(IC<4>{});
        case 5: return f(IC<5>{});
        case 6: return f(IC<6>{});
        case 7: return f(IC<7>{});
        case 8: return f(IC<8>{});
        default: return cudaErrorInvalidValue;
    }
}
// host: f(IC<T>{}) for the tile counts T0..MAXT
template <int T0, int MAXT, class F> cudaError_t dispatch_tiles(int n_tiles, F&& f) {
    if constexpr (T0 > MAXT) return cudaErrorInvalidValue;
    else return n_tiles == T0 ? f(IC<T0>{}) : dispatch_tiles<T0 + 1, MAXT>(n_tiles, f);
}
// host: f(IC<S>{}, IC<T>{}) for those sizes and the tile counts 1..MAXT (default: those of one
// 32-bit state, 1..4; MAX_TILES: every tile count of the register kernels)
template <int MAXT = 4, class F> cudaError_t dispatch_small(int size, int n_tiles, F&& f) {
    static_assert(MAXT >= 1 && MAXT <= MAX_TILES, "register kernels hold 1..8 tiles");
    return dispatch_size(size, [&](auto S) { return dispatch_tiles<1, MAXT>(n_tiles, [&](auto T) { return f(S, T); }); });
}

// ---- streaming global access ---------------------------------------------------------------
// Every stream is touched once per step and the working set (>=400 MB at 16M envs) exceeds
// the 126 MB L2, so loads/stores carry the evict-first (.cs) policy.
template <int WORDS> __device__ __forceinline__ void ld_words(const void* p, uint32_t (&r)[WORDS]) {
    if constexpr (WORDS == 1) {
        r[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
    } else if constexpr (WORDS == 2) {
        uint2 v = __ldcs(reinterpret_cast<const uint2*>(p));
        r[0] = v.x; r[1] = v.y;
    } else {
        static_assert(WORDS % 4 == 0, "group loads are 4, 8 or 16*k bytes");
#pragma unroll
        for (int k = 0; k < WORDS / 4; ++k) {
            uint4 v = __ldcs(reinterpret_cast<const uint4*>(p) + k);
            r[4 * k] = v.x; r[4 * k + 1] = v.y; r[4 * k + 2] = v.z; r[4 * k + 3] = v.w;
        }
    }
}
template <int WORDS> __device__ __forceinline__ void st_words(void* p, const uint32_t (&r)[WORDS]) {
    if constexpr (WORDS == 1) {
        __stcs(reinterpret_cast<unsigned int*>(p), r[0]);
    } else if constexpr (WORDS == 2) {
        __stcs(reinterpret_cast<uint2*>(p), make_uint2(r[0], r[1]));
    } else {
#pragma unroll
        for (int k = 0; k < WORDS / 4; ++k)
            __stcs(reinterpret_cast<uint4*>(p) + k, make_uint4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]));
    }
}

// element e (0..3) of a 4-env group of W-byte elements held in raw[W] words -> out words
template <int W> __device__ __forceinline__ void group_elem(const uint32_t (&raw)[W], int e, uint32_t (&out)[(W + 3) / 4]) {
    if constexpr (W == 1) out[0] = (raw[0] >> (8 * e)) & 0xFFu;
    else if constexpr (W == 2) out[0] = (raw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
    else {
#pragma unroll
        for (int k = 0; k < W / 4; ++k) out[k] = raw[(W / 4) * e + k];
    }
}
template <int W> __device__ __forceinline__ void group_set(uint32_t (&raw)[W], int e, const uint32_t (&in)[(W + 3) / 4]) {
    if constexpr (W == 1) raw[0] = (raw[0] & ~(0xFFu << (8 * e))) | ((in[0] & 0xFFu) << (8 * e));
    else if constexpr (W == 2) raw[e >> 1] = (raw[e >> 1] & ~(0xFFFFu << (16 * (e & 1)))) | ((in[0] & 0xFFFFu) << (16 * (e & 1)));
    else {
#pragma unroll
        for (int k = 0; k < W / 4; ++k) raw[(W / 4) * e + k] = in[k];
    }
}

// ---- a 4-env group of bitboards held as its byte planes ------------------------------------
template <int NB> struct BoardGroup {
    static constexpr int NP = plane_count(NB);
    static constexpr int NWORDS = (NB + 3) / 4;
    uint32_t raw[NB];  // plane k occupies raw[plane_offset(k) .. +plane_width(k))

    __device__ __forceinline__ void load(const uint8_t* base, size_t capacity, size_t group) {
        static_for<0, NP>([&](auto I) {
            constexpr int k = decltype(I)::value;
            constexpr int w = plane_width(NB, k), off = plane_offset(NB, k);
            uint32_t tmp[w];
            ld_words<w>(base + (size_t)off * capacity + group * (size_t)(GROUP * w), tmp);
#pragma unroll
            for (int j = 0; j < w; ++j) raw[off + j] = tmp[j];
        });
    }
    __device__ __forceinline__ void store(uint8_t* base, size_t capacity, size_t group) const {
        static_for<0, NP>([&](auto I) {
            constexpr int k = decltype(I)::value;
            constexpr int w = plane_width(NB, k), off = plane_offset(NB, k);
            uint32_t tmp[w];
#pragma unroll
            for (int j = 0; j < w; ++j) tmp[j] = raw[off + j];
            st_words<w>(base + (size_t)off * capacity + group * (size_t)(GROUP * w), tmp);
        });
    }
    // board words of env e: word j holds bits 32j..32j+31
    __device__ __forceinline__ void get(int e, uint32_t (&bw)[NWORDS]) const {
#pragma unroll
        for (int j = 0; j < NWORDS; ++j) bw[j] = 0;
        static_for<0, NP>([&](auto I) {
            constexpr int k = decltype(I)::value;
            constexpr int w = plane_width(NB, k), off = plane_offset(NB, k);
            uint32_t tmp[w], el[(w + 3) / 4];
#pragma unroll
            for (int j = 0; j < w; ++j) tmp[j] = raw[off + j];
            group_elem<w>(tmp, e, el);
            if constexpr (w >= 4) {
#pragma unroll
                for (int j = 0; j < w / 4; ++j) bw[off / 4 + j] = el[j];
            } else {
                bw[off / 4] |= el[0] << (8 * (off % 4));
            }
        });
    }
    __device__ __forceinline__ void set(int e, const uint32_t (&bw)[NWORDS]) {
        static_for<0, NP>([&](auto I) {
            constexpr int k = decltype(I)::value;
            constexpr int w = plane_width(NB, k), off = plane_offset(NB, k);
            uint32_t tmp[w], el[(w + 3) / 4];
#pragma unroll
            for (int j = 0; j < w; ++j) tmp[j] = raw[off + j];
            if constexpr (w >= 4) {
#pragma unroll
                for (int j = 0; j < w / 4; ++j) el[j] = bw[off / 4 + j];
            } else {
                el[0] = bw[off / 4] >> (8 * (off % 4));
            }
            group_set<w>(tmp, e, el);
#pragma unroll
            for (int j = 0; j < w; ++j) raw[off + j] = tmp[j];
        });
    }
};

// byte `byte` of env `env`'s board inside a plane-layout buffer (runtime sizes: load-time and
// generic kernels only; the hot kernels use BoardGroup)
__host__ __device__ __forceinline__ size_t board_byte_addr(int nb, size_t cap, size_t env, int byte) {
    int off = 0;
    const int np = plane_count(nb);
    for (int k = 0; k < np; ++k) {
        const int w = plane_width(nb, k);
        if (byte < off + w) return (size_t)off * cap + env * (size_t)w + (size_t)(byte - off);
        off += w;
    }
    return 0;
}

// integer multiply-add pinned to the FMA pipe (IMAD), keeping it off the saturated ALU pipe
__device__ __forceinline__ uint32_t mad_u32(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// element `idx` of a plane-layout board buffer as a 64-bit board
template <int NB> __device__ __forceinline__ uint64_t load_board_elem(const uint8_t* base, size_t cap, size_t idx) {
    uint64_t b = 0;
    static_for<0, plane_count(NB)>([&](auto I) {
        constexpr int k = decltype(I)::value;
        constexpr int w = plane_width(NB, k), off = plane_offset(NB, k);
        const uint8_t* p = base + (size_t)off * cap + idx * w;
        uint64_t v;
        if constexpr (w == 8) v = *reinterpret_cast<const uint64_t*>(p);
        else if constexpr (w == 4) v = *reinterpret_cast<const uint32_t*>(p);
        else if constexpr (w == 2) v = *reinterpret_cast<const uint16_t*>(p);
        else v = *p;
        b |= v << (8 * off);
    });
    return b;
}

// position word `idx` of a packed position array (T <= 8: 1, 2, 4 or 8 bytes) into PR words, and back
template <int PW> __device__ __forceinline__ void ld_pos(const uint8_t* p, size_t idx, uint32_t (&q)[(PW + 3) / 4]) {
    if constexpr (PW == 1) q[0] = p[idx];
    else if constexpr (PW == 2) q[0] = reinterpret_cast<const uint16_t*>(p)[idx];
    else if constexpr (PW == 4) q[0] = reinterpret_cast<const uint32_t*>(p)[idx];
    else { const uint2 v = reinterpret_cast<const uint2*>(p)[idx]; q[0] = v.x; q[1] = v.y; }
}
template <int PW> __device__ __forceinline__ void st_pos(uint8_t* p, size_t idx, const uint32_t (&q)[(PW + 3) / 4]) {
    if constexpr (PW == 1) p[idx] = (uint8_t)q[0];
    else if constexpr (PW == 2) reinterpret_cast<uint16_t*>(p)[idx] = (uint16_t)q[0];
    else if constexpr (PW == 4) reinterpret_cast<uint32_t*>(p)[idx] = q[0];
    else reinterpret_cast<uint2*>(p)[idx] = make_uint2(q[0], q[1]);
}

// the four successor words s[move][word] of one item (ts_expand) to its 4*PW-byte output row, as
// vector stores: one u32 (T = 1), one u64 (T = 2), one 16-byte store (T = 3, 4), two (T = 5..8).
// The row is 16-byte aligned for PW >= 4 (the caller checks the buffer), 4*PW-aligned below.
template <int PW> __device__ __forceinline__ void st_succ4(uint8_t* row, const uint32_t (&s)[4][(PW + 3) / 4]) {
    if constexpr (PW == 1) __stcs(reinterpret_cast<unsigned int*>(row), s[0][0] | s[1][0] << 8 | s[2][0] << 16 | s[3][0] << 24);
    else if constexpr (PW == 2) __stcs(reinterpret_cast<uint2*>(row), make_uint2(s[0][0] | s[1][0] << 16, s[2][0] | s[3][0] << 16));
    else if constexpr (PW == 4) __stcs(reinterpret_cast<uint4*>(row), make_uint4(s[0][0], s[1][0], s[2][0], s[3][0]));
    else {
        __stcs(reinterpret_cast<uint4*>(row), make_uint4(s[0][0], s[0][1], s[1][0], s[1][1]));
        __stcs(reinterpret_cast<uint4*>(row) + 1, make_uint4(s[2][0], s[2][1], s[3][0], s[3][1]));
    }
}

// ---- SWAR helpers on 4 packed position bytes -------------------------------------------------
__device__ __forceinline__ uint32_t swap_nibbles(uint32_t x) {
    return ((x & 0x0F0F0F0Fu) << 4) | ((x >> 4) & 0x0F0F0F0Fu);
}
template <int I> __device__ __forceinline__ uint32_t byte_of(uint32_t x) {
    return __byte_perm(x, 0, 0x4440 + I);
}

// =============================================================================================
// slide_env<S,T>: one simultaneous slide of all T tiles of one env (state.py:137-170).
//
// Closed form (SURVEY 7.0, checked against the reference by the parity tests): inside every
// maximal wall-free run of a line, tiles keep their order and pack against the run's end in
// the move direction.  For a tile whose run ends before cell e (nearest wall past the tile,
// or the edge), the new position is  old + (#empty cells strictly between the tile and e).
// Every tile is independent of the others given the occupancy bitboard -- no ordering, no
// back-off loop.
//
// The four directions share one code path: UP/LEFT rotate the board and the positions by 180
// degrees so that every move goes "toward higher bit indices".
// =============================================================================================

// ---- padded boards (S <= 6): stride S+1, sentinel column + sentinel tail ---------------------
// In bit-index space a horizontal move has stride 1 and a vertical move stride BS = S+1.  For
// a tile at bit p the cells it can reach are bits p+st, p+2st, ... of (walls >> (p+st)),
// restricted to the line mask LM (all bits for a row, bits 0,BS,2BS,... for a column).  The
// sentinel column ends a row, the sentinel tail (all ones from bit S*BS-1 up) ends a column, so
//     t1 = (walls >> sh) & LM            first set bit = first non-enterable cell
//     run = (t1 - 1) & ~t1               cells before it
//     n   = popc(run & LM & ~(occ >> sh))
//     p  += st * n
// is the whole per-tile computation: no gather, no transposition, no edge test.
template <int S> struct Padded {
    static constexpr int BS = S + 1;
    static constexpr int NBITS = S * BS;                    // stored board bits incl. sentinel column
    static constexpr int KREV = NBITS - 2;                  // 180-degree rotation: bit i <-> KREV - i
    static constexpr uint32_t KREV4 = 0x01010101u * (uint32_t)KREV;
    static constexpr uint64_t TAIL = ~0ull << (NBITS - 1);  // sentinel of the last row + everything above
    static constexpr uint32_t col_mask() { uint32_t m = 0; for (int k = 0; k * BS < 32 && k < S; ++k) m |= 1u << (k * BS); return m; }
    static constexpr uint32_t COL = col_mask();
    static constexpr uint64_t sentinel_cols() { uint64_t m = 0; for (int r = 0; r < S; ++r) m |= 1ull << (r * BS + S); return m; }
    static constexpr uint64_t SENT = sentinel_cols() | (~0ull << NBITS);   // what a stored wall board has set
};

// Per-direction constants of the padded slide.  st: bit stride of the move; lm: line mask;
// fm / fk: positions are rotated as p' = p * fm + fk (fm = -1, fk = KREV per byte for UP/LEFT).
struct DirParams {
    uint32_t st, lm, fm, fk;
};
// h = 1 for LEFT/RIGHT, f = 1 for UP/LEFT (the directions that need the 180-degree rotation).
// Integer multiply-adds, not selects: the step is bound by instruction issue on the ALU pipe
// (LOP3/SHF/SEL/PRMT), IMAD runs on the FMA pipe.
template <int S> __device__ __forceinline__ DirParams dir_params(uint32_t h, uint32_t f) {
    using PD = Padded<S>;
    DirParams d;
    d.st = (uint32_t)PD::BS - h * (uint32_t)(PD::BS - 1);   // h ? 1 : BS
    d.lm = PD::COL + h * ~PD::COL;                           // h ? ~0 : COL
    d.fm = 1u - 2u * f;                                      // f ? -1 : +1
    d.fk = f * PD::KREV4;                                    // f ? KREV4 : 0
    return d;
}

template <int S, int T>
__device__ __forceinline__ bool slide_padded(uint32_t (&q)[(T + 3) / 4], uint64_t walls, const DirParams& dp) {
    using PD = Padded<S>;
    constexpr int PR = (T + 3) / 4;
    const uint32_t st = dp.st, lm = dp.lm, fm = dp.fm, fk = dp.fk;
    const bool f = (int32_t)fm < 0;
    // bytes past the stored board read as zero in the plane layout: (re)assert the sentinels
    const uint64_t w0 = walls | (~0ull << PD::NBITS);
    const uint64_t wr = (__brevll(walls) >> (63 - PD::KREV)) | PD::TAIL;
    const uint64_t wb = f ? wr : w0;

    uint32_t P[PR], ACC[PR], sh[T];
    uint64_t occ = 0;
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        P[w] = q[w] * fm + fk;                             // f ? KREV4 - q : q (bytewise, no borrow)
        ACC[w] = 0;
    }
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t p = byte_of<i % 4>(P[i / 4]);
        if constexpr (T > 1) occ |= 1ull << p;
        sh[i] = p + st;
    });
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t t1 = (uint32_t)(wb >> sh[i]) & lm;
        const uint32_t t2 = t1 - 1u;
        uint32_t empty;
        if constexpr (T > 1) {
            const uint32_t free_cells = ~(uint32_t)(occ >> sh[i]) & lm;
            empty = t2 & ~t1 & free_cells;
        } else {
            empty = t2 & ~t1 & lm;
        }
        ACC[i / 4] = mad_u32((uint32_t)__popc(empty), 1u << (8 * (i % 4)), ACC[i / 4]);
    });
    uint32_t any = 0;
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        const uint32_t pn = st * ACC[w] + P[w];
        q[w] = pn * fm + fk;
        any |= ACC[w];
    }
    // unused bytes of the last word stay zero: KREV4-(KREV4-0) = 0 and nothing is accumulated
    // into them (the flipped value KREV of an unused byte is never read as a tile).
    return any != 0;                                       // a tile moved iff some count is non-zero
}

template <int S, int T>
__device__ __forceinline__ uint64_t occupancy_padded(const uint32_t (&q)[(T + 3) / 4]) {
    uint64_t occ = 0;
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        occ |= 1ull << byte_of<i % 4>(q[i / 4]);
    });
    return occ;
}

// ---- compact boards (S = 7, 8): stride S, position byte (row<<4)|col ---------------------------
// Positions are nibble-swapped for vertical moves so that (line, offset) = (col, row); the wall
// bits of a vertical line are gathered from the row-major bitboard with one multiply (bits
// S*k -> GSHIFT+k; all partial products land on distinct bits, so there are no carries).
__host__ __device__ constexpr uint64_t make_col0(int S) { uint64_t m = 0; for (int k = 0; k < S; ++k) m |= 1ull << (S * k); return m; }
__host__ __device__ constexpr uint64_t make_magic(int S) { uint64_t m = 0; for (int j = 0; j < S; ++j) m |= 1ull << ((S - 1) * (S - 1) - (S - 1) * j); return m; }

template <int S> struct Compact {
    static constexpr uint64_t COL0 = make_col0(S);           // bits S*k, k < S: column 0
    static constexpr uint64_t MAGIC = make_magic(S);         // moves bit S*k to bit GSHIFT+k
    static constexpr int GSHIFT = (S - 1) * (S - 1);
};

template <int S, int T>
__device__ __forceinline__ void slide_compact(uint32_t (&q)[(T + 3) / 4], uint64_t walls, uint32_t h, uint32_t f) {
    using CT = Compact<S>;
    constexpr int PR = (T + 3) / 4;
    constexpr uint32_t KFLIP = 0x11111111u * (uint32_t)(S - 1);
    const bool horiz = h != 0;
    const bool flip = f != 0;
    const uint64_t wb = flip ? (__brevll(walls) >> (64 - S * S)) : walls;
    const uint32_t line_mul = horiz ? (uint32_t)S : 1u;   // vertical: shift by the column, then gather

    uint32_t Q[PR], LSo[PR], LSw[PR], OFF[PR];
    uint64_t occ = 0;
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        uint32_t x = horiz ? q[w] : swap_nibbles(q[w]);
        x = flip ? KFLIP - x : x;
        Q[w] = x;
        const uint32_t line = (x >> 4) & 0x0F0F0F0Fu;
        OFF[w] = x & 0x0F0F0F0Fu;
        LSo[w] = line * (uint32_t)S;
        LSw[w] = line * line_mul;
    }
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        occ |= 1ull << byte_of<i % 4>(LSo[i / 4] + OFF[i / 4]);
    });
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        const uint32_t shw = byte_of<i % 4>(LSw[i / 4]);
        const uint32_t sho = byte_of<i % 4>(LSo[i / 4]);
        const uint32_t o = byte_of<i % 4>(OFF[i / 4]);
        const uint64_t x = wb >> shw;
        const uint32_t g = (uint32_t)(((x & CT::COL0) * CT::MAGIC) >> CT::GSHIFT);
        const uint32_t wl = horiz ? (uint32_t)x : g;
        const uint32_t ol = (uint32_t)(occ >> sho);
        const uint32_t above = 0xFFFFFFFEu << o;           // offsets > o
        const uint32_t blk = (wl & above) | (1u << S);     // walls above o, edge sentinel at S
        const uint32_t run = (blk - 1u) & ~blk;            // offsets below the nearest wall
        Q[i / 4] += (uint32_t)__popc(run & above & ~ol) << (8 * (i % 4));
    });
#pragma unroll
    for (int w = 0; w < PR; ++w) {
        const uint32_t x = flip ? KFLIP - Q[w] : Q[w];
        q[w] = horiz ? x : swap_nibbles(x);
    }
}

template <int S, int T>
__device__ __forceinline__ uint64_t occupancy_compact(const uint32_t (&q)[(T + 3) / 4]) {
    uint64_t occ = 0;
    uint32_t P[(T + 3) / 4];
#pragma unroll
    for (int w = 0; w < (T + 3) / 4; ++w) P[w] = ((q[w] >> 4) & 0x0F0F0F0Fu) * (uint32_t)S + (q[w] & 0x0F0F0F0Fu);
    static_for<0, T>([&](auto I) {
        constexpr int i = decltype(I)::value;
        occ |= 1ull << byte_of<i % 4>(P[i / 4]);
    });
    return occ;
}

// ---- dispatch by board class (S*BS <= 64 bits) ---------------------------------------------------
// q[PR]: packed position words.  Updated in place.  action: 0 UP, 1 DOWN, 2 LEFT, 3 RIGHT
// (state.py:31-34).
template <int S, int T>
__device__ __forceinline__ void slide_env(uint32_t (&q)[(T + 3) / 4], uint64_t walls, uint32_t h, uint32_t f) {
    if constexpr (padded_board(S)) slide_padded<S, T>(q, walls, dir_params<S>(h, f));
    else slide_compact<S, T>(q, walls, h, f);
}
// the h / f bits of the four actions of a thread's envs, one per byte (SWAR decode)
__device__ __forceinline__ uint32_t actions_h4(uint32_t act4) { return (act4 >> 1) & 0x01010101u; }
__device__ __forceinline__ uint32_t actions_f4(uint32_t act4) { return ~act4 & 0x01010101u; }
template <int S, int T>
__device__ __forceinline__ uint64_t occupancy(const uint32_t (&q)[(T + 3) / 4]) {
    if constexpr (padded_board(S)) return occupancy_padded<S, T>(q);
    else return occupancy_compact<S, T>(q);
}
template <int NWORDS> __device__ __forceinline__ uint64_t board64(const uint32_t (&bw)[NWORDS]) {
    if constexpr (NWORDS >= 2) return (uint64_t)bw[0] | ((uint64_t)bw[1] << 32);
    else return bw[0];
}

// flag bits (mirrored in include/tiler_slider.h)
constexpr uint32_t F_DONE = 1, F_WON = 2, F_INVALID = 4, F_TIMEOUT = 8, F_STALE = 16;

// ---- programmatic dependent launch ----------------------------------------------------------------
// The step kernels are launched with the programmatic-stream-serialization attribute: the launch
// behind a step in the stream may place its CTAs while the step's last wave drains, which hides the
// launch latency of back-to-back steps (measured, Python loop without a CUDA graph: 73.9 -> 71.9 us
// per 16.7M-env step, 14.3 -> 12.6 us per 1M-env step; same as a graph replay).  The kernels execute
// griddepcontrol.wait before their first global access, so whatever ran ahead of them in the
// stream has completed and is visible.
__device__ __forceinline__ void dependent_launch_sync() {
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename K, typename A>
inline void launch_dependent(K kernel, unsigned blocks, unsigned threads, cudaStream_t stream, const A& args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(threads);
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, args);
}

}  // namespace ts
