// ts_api.cu -- C-ABI entry points (include/tiler_slider.h), argument validation, and the
// load-time kernels: K1 ts_encode, K0 ts_synth (K3 ts_observe lives in ts_observe.cu,
// ts_observe_planes in ts_observe_planes.cu, ts_expand in ts_expand.cu / ts_wide.cu / ts_generic.cu, ts_playout in
// ts_playout.cu / ts_wide.cu / ts_generic.cu).
//
// Reference map (paths relative to the reference checkout):
//   ts_encode   explainrl/environment/state.py:61-73        GameState.__init__ (is_blocked + lists)
//   ts_synth    explainrl/environment/environment.py:221-226 create_simple_env recipe
//   ts_observe  explainrl/environment/state.py:188-211      get_state_array (kernel in ts_observe.cu)
//   ts_step     see ts_step.cuh;  ts_valid_moves see ts_valid.cuh
#include <cstdarg>
#include <cstdio>
#include "ts_synth.cuh"

namespace ts {
#define TS_DECL(S)                                                              \
    cudaError_t step_dispatch_s##S(const ts_step_args&, cudaStream_t);          \
    cudaError_t valid_dispatch_s##S(const ts_valid_args&, cudaStream_t);        \
    cudaError_t goal_dispatch_s##S(const ts_goal_args&, cudaStream_t);
TS_DECL(1) TS_DECL(2) TS_DECL(3) TS_DECL(4) TS_DECL(5) TS_DECL(6) TS_DECL(7) TS_DECL(8)
#undef TS_DECL
cudaError_t observe_dispatch(const ts_observe_args&, cudaStream_t);
cudaError_t observe_planes_dispatch(const ts_observe_planes_args&, cudaStream_t);
cudaError_t observe_planes_items_dispatch(const ts_observe_planes_args&, const int32_t*, const uint8_t*, int64_t, cudaStream_t);
int observe_planes_channels(const ts_observe_planes_args&);
cudaError_t expand_dispatch(const ts_expand_args&, cudaStream_t);
cudaError_t wide_expand_dispatch(const ts_expand_args&, cudaStream_t);
cudaError_t generic_expand_dispatch(const ts_expand_args&, cudaStream_t);
cudaError_t playout_dispatch(const ts_playout_args&, cudaStream_t);
cudaError_t wide_playout_dispatch(const ts_playout_args&, cudaStream_t);
cudaError_t generic_playout_dispatch(const ts_playout_args&, cudaStream_t);
cudaError_t wide_step_dispatch(const ts_step_args&, cudaStream_t);
cudaError_t wide_valid_dispatch(const ts_valid_args&, cudaStream_t);
cudaError_t wide_goal_dispatch(const ts_goal_args&, cudaStream_t);
cudaError_t generic_step_dispatch(const ts_step_args&, cudaStream_t);
cudaError_t generic_goal_dispatch(const ts_goal_args&, cudaStream_t);
cudaError_t generic_valid_dispatch(const ts_valid_args&, cudaStream_t);
cudaError_t candidates_dispatch(const ts_synth_candidates_args&, cudaStream_t);
cudaError_t pool_reset_dispatch(const ts_pool_reset_args&, cudaStream_t);

static thread_local char g_err[256] = "ok";
static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
static int cuda_result(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int check_shape(int size, int n_tiles, int64_t first, int64_t n, int64_t cap) {
    if (size < 1 || size > MAX_SIZE) return fail(TS_E_BAD_SIZE, "size %d outside 1..%d", size, MAX_SIZE);
    if (n_tiles < 0 || n_tiles > MAX_TILES_ANY) return fail(TS_E_BAD_TILES, "n_tiles %d outside 0..%d", n_tiles, MAX_TILES_ANY);
    if (cap >= (int64_t)1 << 33) return fail(TS_E_BAD_CAPACITY, "capacity %lld too large (max 2^33 - 128 envs per call)", (long long)cap);
    if (cap <= 0 || cap % CAP_ALIGN != 0) return fail(TS_E_BAD_CAPACITY, "capacity %lld is not a positive multiple of %d", (long long)cap, CAP_ALIGN);
    if (first < 0 || n < 0 || first % GROUP != 0 || first + n > cap)
        return fail(TS_E_BAD_RANGE, "env range [%lld, %lld) invalid for capacity %lld (first_env must be a multiple of %d)",
                    (long long)first, (long long)(first + n), (long long)cap, GROUP);
    return 0;
}

// ---- K1 encode --------------------------------------------------------------------------------
__global__ void encode_kernel(const ts_encode_args a) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_envs) return;
    const size_t env = (size_t)(a.first_env + i), cap = (size_t)a.capacity;
    const int S = a.size, T = a.n_tiles, NT = a.n_targets, pw = pos_bytes(T), ps = pos_stride(S);
    store_walls(a.d_walls, cap, env, S, a.d_blocked + (size_t)i * S * S);
    const uint8_t* tl = a.d_tiles + (size_t)i * T * 2;
    for (int t = 0; t < pw; ++t) {
        const uint8_t v = t < T ? (uint8_t)(tl[2 * t] * ps + tl[2 * t + 1]) : 0;
        a.d_init[env * pw + t] = v;
        a.d_pos[env * pw + t] = v;
    }
    const uint8_t* tg = a.d_targets + (size_t)i * NT * 2;
    if (a.goal_mode == TS_GOAL_ORDERED) {
        for (int t = 0; t < pw; ++t)
            a.d_targets_packed[env * pw + t] = (t < NT && t < T) ? (uint8_t)(tg[2 * t] * ps + tg[2 * t + 1]) : 0;
    } else {
        int cells[MAX_SIZE * MAX_SIZE];
        const int n = NT < MAX_SIZE * MAX_SIZE ? NT : MAX_SIZE * MAX_SIZE;
        for (int t = 0; t < n; ++t) cells[t] = tg[2 * t] * S + tg[2 * t + 1];
        store_target_board(a.d_targets_packed, cap, env, S, T, cells, n);
    }
}

// ---- K0 synth -----------------------------------------------------------------------------------
__global__ void synth_kernel(const ts_synth_args a) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_envs) return;
    synth_env(a.size, a.n_tiles, a.n_walls, a.goal_mode, a.seed, (uint64_t)(a.env_index_base + i), (size_t)a.capacity,
              (size_t)(a.first_env + i), a.d_walls, a.d_targets_packed, a.d_init, a.d_pos);
}

}  // namespace ts

using namespace ts;

extern "C" {

int ts_version(void) { return TS_VERSION; }
const char* ts_last_error_string(void) { return g_err; }
int ts_pos_bytes(int n_tiles) { return pos_bytes(n_tiles); }
int ts_board_bytes(int size) { return board_bytes(size); }
int ts_board_stride(int size) { return board_stride(size); }
int ts_pos_stride(int size) { return pos_stride(size); }
int ts_plane_count(int n_bytes) { return plane_count(n_bytes); }
int ts_plane_width(int n_bytes, int k) { return plane_width(n_bytes, k); }
int ts_plane_offset(int n_bytes, int k) { return plane_offset(n_bytes, k); }
int ts_walls_bytes(int size) { return walls_bytes(size); }
int ts_target_board_bytes(int size) { return target_board_bytes(size); }
int ts_supported(int size, int n_tiles) { return size >= 1 && size <= MAX_SIZE && n_tiles >= 0 && n_tiles <= MAX_TILES_ANY; }

int ts_encode(const ts_encode_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->n_targets < 0 || a->n_targets > MAX_SIZE * MAX_SIZE) return fail(TS_E_BAD_TILES, "n_targets %d", a->n_targets);
    if (!a->d_blocked || (!a->d_tiles && a->n_tiles) || (!a->d_targets && a->n_targets) || !a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_pos)
        return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    const unsigned blocks = (unsigned)((a->n_envs + 127) / 128);
    encode_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(*a);
    return cuda_result(cudaGetLastError(), "ts_encode launch");
}

int ts_synth(const ts_synth_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->n_walls < 0 || a->n_walls + 2 * a->n_tiles > a->size * a->size)
        return fail(TS_E_BAD_ARGUMENT, "n_walls + 2*n_tiles = %d exceeds the %d cells", a->n_walls + 2 * a->n_tiles, a->size * a->size);
    if (!a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_pos) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    const unsigned blocks = (unsigned)((a->n_envs + 127) / 128);
    synth_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(*a);
    return cuda_result(cudaGetLastError(), "ts_synth launch");
}

// K7's checks and launch for the tile counts t_lo..t_hi of one entry point
static int synth_candidates(const ts_synth_candidates_args* a, void* stream, int t_lo, int t_hi) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, 0, 0, a->capacity)) return rc;
    if (a->size > 8 || a->n_tiles < t_lo || a->n_tiles > t_hi)
        return fail(TS_E_UNSUPPORTED, "candidates cover sizes up to 8 with %d to %d tiles (size %d, n_tiles %d)", t_lo, t_hi, a->size, a->n_tiles);
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->recipe != TS_RECIPE_UNIFORM && a->recipe != TS_RECIPE_WALK) return fail(TS_E_BAD_ARGUMENT, "recipe %d", a->recipe);
    if (a->walk_len < 0 || a->walk_len > TS_MAX_WALK) return fail(TS_E_BAD_ARGUMENT, "walk_len %d outside 0..%d", a->walk_len, TS_MAX_WALK);
    if (a->attempt < 0) return fail(TS_E_BAD_ARGUMENT, "attempt %d", a->attempt);
    const int need = a->n_walls + (a->recipe == TS_RECIPE_UNIFORM ? 2 : 1) * a->n_tiles;
    if (a->n_walls < 0 || need > a->size * a->size)
        return fail(TS_E_BAD_ARGUMENT, "the recipe needs %d distinct cells, the board has %d", need, a->size * a->size);
    if (a->env_index_base < 0) return fail(TS_E_BAD_RANGE, "env_index_base %lld", (long long)a->env_index_base);
    if (a->n_items < 0 || (!a->d_env_ids && a->n_items > a->capacity))
        return fail(TS_E_BAD_RANGE, "n_items %lld invalid for capacity %lld", (long long)a->n_items, (long long)a->capacity);
    if (!a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_pos) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_items == 0) return 0;
    return cuda_result(candidates_dispatch(*a, (cudaStream_t)stream), "ts_synth_candidates launch");
}
int ts_synth_candidates(const ts_synth_candidates_args* a, void* stream) { return synth_candidates(a, stream, 1, 4); }
int ts_synth_candidates_t8(const ts_synth_candidates_args* a, void* stream) { return synth_candidates(a, stream, 5, 8); }

int ts_pool_reset(const ts_pool_reset_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->count_bytes != 1 && a->count_bytes != 4) return fail(TS_E_BAD_ARGUMENT, "count_bytes %d (1 or 4)", a->count_bytes);
    if (a->n_pool < 1) return fail(TS_E_BAD_ARGUMENT, "n_pool %lld: the pool needs at least one puzzle", (long long)a->n_pool);
    if (a->pool_capacity <= 0 || a->pool_capacity % CAP_ALIGN != 0 || a->pool_capacity < a->n_pool || a->pool_capacity >= (int64_t)1 << 33)
        return fail(TS_E_BAD_CAPACITY, "pool_capacity %lld invalid for %lld puzzles (a positive multiple of %d)",
                    (long long)a->pool_capacity, (long long)a->n_pool, CAP_ALIGN);
    if (a->env_index_base < 0) return fail(TS_E_BAD_RANGE, "env_index_base %lld", (long long)a->env_index_base);
    if (!a->d_episode || !a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_pos || !a->d_step_count ||
        !a->d_pool_walls || !a->d_pool_targets || !a->d_pool_init)
        return fail(TS_E_NULL_POINTER, "null device pointer");
    const void* ptrs[] = {a->d_done, a->d_episode, a->d_walls, a->d_targets_packed, a->d_init, a->d_pos, a->d_step_count,
                          a->d_solve_depth, a->d_pool_walls, a->d_pool_targets, a->d_pool_init, a->d_pool_depth};
    for (const void* p : ptrs)
        if (p && !aligned16(p)) return fail(TS_E_MISALIGNED, "device pointer %p is not 16-byte aligned", p);
    if (a->n_envs == 0) return 0;
    return cuda_result(pool_reset_dispatch(*a, (cudaStream_t)stream), "ts_pool_reset launch");
}

int ts_step(const ts_step_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (!ts_supported(a->size, a->n_tiles)) return fail(TS_E_UNSUPPORTED, "no step kernel for size %d, n_tiles %d", a->size, a->n_tiles);
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->count_bytes != 1 && a->count_bytes != 4) return fail(TS_E_BAD_ARGUMENT, "count_bytes %d (1 or 4)", a->count_bytes);
    if (a->order != 0 && a->order != 1) return fail(TS_E_BAD_ARGUMENT, "order %d (0 ascending, 1 descending)", a->order);
    // 1-byte counters are bumped SWAR, four to a word: a frozen env (auto_reset = 0) resting at 255 would carry into its neighbour
    if (a->count_bytes == 1 && a->max_steps > (a->auto_reset ? 255 : 254)) return fail(TS_E_BAD_ARGUMENT, "max_steps %d needs count_bytes 4", a->max_steps);
    if (!a->d_walls || !a->d_targets_packed || !a->d_init || !a->d_pos || !a->d_step_count || !a->d_actions || !a->d_reward)
        return fail(TS_E_NULL_POINTER, "null device pointer");
    if (!a->d_done && !a->d_flags) return fail(TS_E_NULL_POINTER, "need d_done or d_flags");
    if (!a->auto_reset && !a->d_flags) return fail(TS_E_NULL_POINTER, "auto_reset=0 needs d_flags (done state is carried there)");
    const void* ptrs[] = {a->d_walls, a->d_targets_packed, a->d_init, a->d_pos, a->d_step_count, a->d_actions,
                          a->d_reward, a->d_done, a->d_flags, a->d_terminal_pos};
    for (const void* p : ptrs)
        if (p && !aligned16(p)) return fail(TS_E_MISALIGNED, "device pointer %p is not 16-byte aligned", p);
    // the wide kernel (S >= 9, 1..8 tiles) indexes envs with 32 bits (ts_wide.cu)
    if (wide_board(a->size) && a->n_tiles >= 1 && a->n_tiles <= MAX_TILES && a->first_env + a->n_envs >= ((int64_t)1 << 32))
        return fail(TS_E_BAD_RANGE, "env range [%lld, %lld) exceeds the 2^32-env limit of boards of size 9..16 with 1..%d tiles",
                    (long long)a->first_env, (long long)(a->first_env + a->n_envs), MAX_TILES);
    if (a->n_envs == 0) return 0;
    ts_step_args args = *a;
    if (args.max_steps < 1) args.max_steps = 1;   // step_count >= max_steps holds on the first step either way
    cudaStream_t st = (cudaStream_t)stream;
    if (a->n_tiles == 0 || a->n_tiles > MAX_TILES)      // nothing to slide / more tiles than the register kernels hold (ts_generic.cu)
        return cuda_result(generic_step_dispatch(args, st), "ts_step launch");
    // the bitboard kernels own whole 4-env groups: the ragged end of the range goes to the generic kernel
    const int64_t ragged = wide_board(a->size) ? 0 : a->n_envs % GROUP;
    args.n_envs -= ragged;
    cudaError_t e = cudaSuccess;
    if (args.n_envs > 0) {
        switch (a->size) {
            case 1: e = step_dispatch_s1(args, st); break;
            case 2: e = step_dispatch_s2(args, st); break;
            case 3: e = step_dispatch_s3(args, st); break;
            case 4: e = step_dispatch_s4(args, st); break;
            case 5: e = step_dispatch_s5(args, st); break;
            case 6: e = step_dispatch_s6(args, st); break;
            case 7: e = step_dispatch_s7(args, st); break;
            case 8: e = step_dispatch_s8(args, st); break;
            default: e = wide_step_dispatch(args, st); break;
        }
    }
    if (e == cudaSuccess && ragged) {
        args.first_env += args.n_envs;
        args.n_envs = ragged;
        e = generic_step_dispatch(args, st);
    }
    return cuda_result(e, "ts_step launch");
}

int ts_observe(const ts_observe_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    // ordered targets are read as a position word of ts_pos_bytes(n_targets) bytes, which holds at most 32
    if (a->goal_mode == TS_GOAL_ORDERED && (a->n_targets < -1 || a->n_targets > MAX_TILES_ANY))
        return fail(TS_E_BAD_TILES, "n_targets %d outside -1..%d", a->n_targets, MAX_TILES_ANY);
    if (!a->d_walls || !a->d_targets_packed || !a->d_pos || !a->d_obs) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    if (!aligned16(a->d_obs)) return fail(TS_E_MISALIGNED, "d_obs %p is not 16-byte aligned", (const void*)a->d_obs);
    return cuda_result(observe_dispatch(*a, (cudaStream_t)stream), "ts_observe launch");
}

// the checks of ts_observe_planes that do not involve the range or the buffers
static int check_planes_kind(const ts_observe_planes_args* a) {
    if (a->n_tiles < 0 || a->n_tiles > MAX_TILES_ANY) return fail(TS_E_BAD_TILES, "n_tiles %d outside 0..%d", a->n_tiles, MAX_TILES_ANY);
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->goal_mode == TS_GOAL_ORDERED && (a->n_targets < -1 || a->n_targets > MAX_TILES_ANY))
        return fail(TS_E_BAD_TILES, "n_targets %d outside -1..%d", a->n_targets, MAX_TILES_ANY);
    if (a->dtype < TS_OBS_U8 || a->dtype > TS_OBS_F32) return fail(TS_E_BAD_ARGUMENT, "dtype %d (TS_OBS_U8 .. TS_OBS_F32)", a->dtype);
    return 0;
}

int ts_observe_planes_channels(const ts_observe_planes_args* a) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_planes_kind(a)) return rc;
    return observe_planes_channels(*a);
}

int ts_observe_planes(const ts_observe_planes_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (int rc = check_planes_kind(a)) return rc;
    if (!a->d_walls || !a->d_targets_packed || !a->d_pos || !a->d_out) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    if (!aligned16(a->d_out)) return fail(TS_E_MISALIGNED, "d_out %p is not 16-byte aligned", a->d_out);
    return cuda_result(observe_planes_dispatch(*a, (cudaStream_t)stream), "ts_observe_planes launch");
}

// the item list of ts_observe_planes_items / ts_expand: n_items items, ids from d_env_ids or 0 .. n_items-1
static int check_items(int64_t n_items, const int32_t* d_env_ids, int64_t cap) {
    if (n_items < 0 || (!d_env_ids && n_items > cap))
        return fail(TS_E_BAD_RANGE, "n_items %lld invalid for capacity %lld (without env ids item i is env i)", (long long)n_items,
                    (long long)cap);
    return 0;
}

int ts_observe_planes_items(const ts_observe_planes_args* a, const int32_t* d_env_ids, const uint8_t* d_item_pos, int64_t n_items,
                            void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, 0, 0, a->capacity)) return rc;
    if (int rc = check_planes_kind(a)) return rc;
    if (int rc = check_items(n_items, d_env_ids, a->capacity)) return rc;
    if (!a->d_walls || !a->d_targets_packed || (!a->d_pos && !d_item_pos) || !a->d_out) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (n_items == 0) return 0;
    if (!aligned16(a->d_out)) return fail(TS_E_MISALIGNED, "d_out %p is not 16-byte aligned", a->d_out);
    if (d_item_pos && !aligned16(d_item_pos)) return fail(TS_E_MISALIGNED, "d_item_pos %p is not 16-byte aligned", (const void*)d_item_pos);
    return cuda_result(observe_planes_items_dispatch(*a, d_env_ids, d_item_pos, n_items, (cudaStream_t)stream), "ts_observe_planes_items launch");
}

int ts_expand(const ts_expand_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, 0, 0, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->never_win != 0 && a->never_win != 1) return fail(TS_E_BAD_ARGUMENT, "never_win %d (0 or 1)", a->never_win);
    if (int rc = check_items(a->n_items, a->d_env_ids, a->capacity)) return rc;
    if (!a->d_walls || !a->d_targets_packed || (!a->d_pos && !a->d_item_pos) || !a->d_succ)
        return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_items == 0) return 0;
    if (!aligned16(a->d_succ)) return fail(TS_E_MISALIGNED, "d_succ %p is not 16-byte aligned", (const void*)a->d_succ);
    if (a->d_item_pos && !aligned16(a->d_item_pos))
        return fail(TS_E_MISALIGNED, "d_item_pos %p is not 16-byte aligned", (const void*)a->d_item_pos);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (a->n_tiles == 0 || a->n_tiles > MAX_TILES) e = generic_expand_dispatch(*a, st);   // the kernel classes of ts_step
    else if (wide_board(a->size)) e = wide_expand_dispatch(*a, st);
    else e = expand_dispatch(*a, st);
    return cuda_result(e, "ts_expand launch");
}

int ts_playout(const ts_playout_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, 0, 0, a->capacity)) return rc;
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (a->never_win != 0 && a->never_win != 1) return fail(TS_E_BAD_ARGUMENT, "never_win %d (0 or 1)", a->never_win);
    if (a->policy != TS_PLAYOUT_PLAN && a->policy != TS_PLAYOUT_RANDOM)
        return fail(TS_E_BAD_ARGUMENT, "policy %d (TS_PLAYOUT_PLAN or TS_PLAYOUT_RANDOM)", a->policy);
    if (a->n_steps < 0) return fail(TS_E_BAD_ARGUMENT, "n_steps %d", a->n_steps);
    if (int rc = check_items(a->n_items, a->d_env_ids, a->capacity)) return rc;
    if (!a->d_walls || !a->d_targets_packed || (!a->d_pos && !a->d_item_pos) || !a->d_final || !a->d_steps || !a->d_won ||
        (a->policy == TS_PLAYOUT_PLAN && !a->d_plan))
        return fail(TS_E_NULL_POINTER, "null device pointer");
    // the step-major records hold n_steps * n_items elements, indexed with 64 bits
    const int64_t per_item = (int64_t)a->n_steps * pos_bytes(a->n_tiles);
    if (per_item > 0 && a->n_items > INT64_MAX / per_item)
        return fail(TS_E_BAD_RANGE, "n_steps %d x n_items %lld x pos_bytes overflows 64 bits", a->n_steps, (long long)a->n_items);
    // one launch of 128-thread blocks (the smallest of the three kernels) covers at most 2^31 - 1 blocks
    if (a->n_items > (int64_t)INT32_MAX * 128)
        return fail(TS_E_BAD_RANGE, "n_items %lld exceeds the %lld items of one launch", (long long)a->n_items,
                    (long long)INT32_MAX * 128);
    if (a->n_items == 0) return 0;
    if (!aligned16(a->d_final)) return fail(TS_E_MISALIGNED, "d_final %p is not 16-byte aligned", (const void*)a->d_final);
    if (a->d_item_pos && !aligned16(a->d_item_pos))
        return fail(TS_E_MISALIGNED, "d_item_pos %p is not 16-byte aligned", (const void*)a->d_item_pos);
    if (a->d_traj && !aligned16(a->d_traj)) return fail(TS_E_MISALIGNED, "d_traj %p is not 16-byte aligned", (const void*)a->d_traj);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (a->n_tiles == 0 || a->n_tiles > MAX_TILES) e = generic_playout_dispatch(*a, st);   // the kernel classes of ts_step
    else if (wide_board(a->size)) e = wide_playout_dispatch(*a, st);
    else e = playout_dispatch(*a, st);
    return cuda_result(e, "ts_playout launch");
}

int ts_valid_moves(const ts_valid_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (!ts_supported(a->size, a->n_tiles)) return fail(TS_E_UNSUPPORTED, "no kernel for size %d, n_tiles %d", a->size, a->n_tiles);
    if (!a->d_walls || !a->d_pos || !a->d_mask) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    cudaError_t e;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->n_tiles == 0)      // no tile, no move that changes anything
        return cuda_result(cudaMemsetAsync(a->d_mask + a->first_env, 0, (size_t)a->n_envs, st), "ts_valid_moves memset");
    if (a->n_tiles > MAX_TILES) return cuda_result(generic_valid_dispatch(*a, st), "ts_valid_moves launch");
    switch (a->size) {
        case 1: e = valid_dispatch_s1(*a, st); break;
        case 2: e = valid_dispatch_s2(*a, st); break;
        case 3: e = valid_dispatch_s3(*a, st); break;
        case 4: e = valid_dispatch_s4(*a, st); break;
        case 5: e = valid_dispatch_s5(*a, st); break;
        case 6: e = valid_dispatch_s6(*a, st); break;
        case 7: e = valid_dispatch_s7(*a, st); break;
        case 8: e = valid_dispatch_s8(*a, st); break;
        default: e = wide_valid_dispatch(*a, st); break;
    }
    return cuda_result(e, "ts_valid_moves launch");
}

int ts_goal_check(const ts_goal_args* a, void* stream) {
    if (!a) return fail(TS_E_NULL_POINTER, "null args");
    if (int rc = check_shape(a->size, a->n_tiles, a->first_env, a->n_envs, a->capacity)) return rc;
    if (!ts_supported(a->size, a->n_tiles)) return fail(TS_E_UNSUPPORTED, "no kernel for size %d, n_tiles %d", a->size, a->n_tiles);
    if (a->goal_mode != TS_GOAL_ORDERED && a->goal_mode != TS_GOAL_SET) return fail(TS_E_BAD_ARGUMENT, "goal_mode %d", a->goal_mode);
    if (!a->d_targets_packed || !a->d_pos || !a->d_won) return fail(TS_E_NULL_POINTER, "null device pointer");
    if (a->n_envs == 0) return 0;
    cudaError_t e;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->n_tiles == 0 || a->n_tiles > MAX_TILES) return cuda_result(generic_goal_dispatch(*a, st), "ts_goal_check launch");
    switch (a->size) {
        case 1: e = goal_dispatch_s1(*a, st); break;
        case 2: e = goal_dispatch_s2(*a, st); break;
        case 3: e = goal_dispatch_s3(*a, st); break;
        case 4: e = goal_dispatch_s4(*a, st); break;
        case 5: e = goal_dispatch_s5(*a, st); break;
        case 6: e = goal_dispatch_s6(*a, st); break;
        case 7: e = goal_dispatch_s7(*a, st); break;
        case 8: e = goal_dispatch_s8(*a, st); break;
        default: e = wide_goal_dispatch(*a, st); break;
    }
    return cuda_result(e, "ts_goal_check launch");
}

}  // extern "C"
