/*
 * tiler_slider.h -- C-ABI of libtiler_slider.so, the B200 (sm_100a) batched Tiler-Slider
 * step path.
 *
 * The reference (AnimeshSinha1309/tiler-slider) is pure Python and has no FFI boundary; the
 * path sits behind two classes, GameState (explainrl/environment/state.py:18-222) and
 * TilerSliderEnv (explainrl/environment/environment.py:14-194).  Each entry point below
 * names the reference code whose results it reproduces; INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *  - Every pointer named d_* (or inside a ts_*_args struct, unless marked host) is a DEVICE
 *    pointer into caller-owned memory (PyTorch tensors in this repo).  The library
 *    allocates nothing persistent except inside ts_host_ctx.
 *  - Calls are asynchronous on the given cudaStream_t (void*; 0 = legacy default stream),
 *    except ts_step_host which synchronises before it returns.
 *  - Return value: 0 = success; negative = argument error (TS_E_*); positive = cudaError_t
 *    from the launch.  ts_last_error_string() describes the last failure of the calling
 *    thread.  No global mutable state: re-entrant across streams and devices (the caller
 *    selects the device).
 *  - There is no CPU fallback anywhere in this library.
 *  - Domain: well-formed boards -- tiles on distinct cells, none on a blocked cell (what the
 *    reference's loaders produce; outside it the reference itself is erratic, SURVEY 7.0).  The
 *    kernels do not check this (tiler_slider_b200.Puzzle.validate does, on the host); a tile placed
 *    on a blocked cell slides out of it on boards up to 8x8 and 15x15 / 16x16, and stays put on
 *    9x9 .. 14x14 (the wide slide treats the own cell as wall-free).  GameState.move_to, which is
 *    defined for blocked start cells, therefore probes on a board whose start cell is open.
 *
 * Packed layout (struct-of-arrays, environment index innermost):
 *  - capacity: allocation stride in environments, a multiple of TS_CAP_ALIGN, below 2^33.  EVERY
 *    per-env array handed to the library (state, actions, reward, done, flags, ...) must hold
 *    `capacity` elements.  A call covers the env range [first_env, first_env + n_envs), first_env a
 *    multiple of 4; ts_step on boards of size 9..16 with 1..8 tiles needs first_env + n_envs < 2^32
 *    (32-bit env index; TS_E_BAD_RANGE otherwise).
 *  - write set of each entry point (everything else is left as it was, bit for bit):
 *      ts_encode, ts_synth, ts_step, ts_pool_reset: exactly the envs of the range (ts_step: whole
 *        4-env groups through the vectorised kernel, the ragged end, n_envs % 4 envs, through a
 *        per-env kernel);
 *      ts_observe: d_obs[0 .. n_envs) -- d_obs is RELATIVE to the range: env first_env + i is
 *        written to d_obs[i];
 *      ts_observe_planes: d_out[0 .. n_envs*C*size*size) elements, RELATIVE to the range as
 *        ts_observe's;
 *      ts_observe_planes_items: d_out[0 .. n_items*C*size*size) elements, in item order;
 *      ts_expand: d_succ[0 .. 4*n_items*pos_bytes) bytes, d_moved[0 .. n_items) and
 *        d_won[0 .. n_items) (when given), in item order -- no env buffer;
 *      ts_playout: d_final[0 .. n_items*pos_bytes) bytes, d_steps[0 .. n_items), d_won[0 .. n_items)
 *        and, when given, d_moves[0 .. n_steps*n_items) and d_traj[0 .. n_steps*n_items*pos_bytes)
 *        bytes, in item order (step-major for the last two) -- no env buffer;
 *      ts_valid_moves, ts_goal_check: d_mask / d_won are ABSOLUTE (env e at [e]); the range, and on
 *        boards up to 8x8 with 1..8 tiles also the (correct) result of the up-to-3 envs after the
 *        range that share its last 4-env group;
 *      ts_step_host: the device buffers as ts_step; the host buffers are RELATIVE to the range,
 *        elements [0, n_envs).
 *  - position word: ts_pos_bytes(T) in {1,2,4,8,16,32} bytes per env, byte i = row*PS + col of tile
 *    i (PS = ts_pos_stride(S)), unused bytes zero.  Arrays: pos (in/out), init, targets
 *    (ordered mode).
 *  - board: bitboard of ts_board_bytes(S) bytes per env, bit row*BS + col (BS =
 *    ts_board_stride(S)) set = blocked (walls) or target cell (targets, set mode), little
 *    endian, split into byte planes of width 16 (repeated), 8, 4, 2, 1 -- widest first; plane
 *    k of a buffer starts at byte offset ts_plane_offset(nb,k)*capacity and holds one element
 *    per env.  S <= 6: BS = PS = S+1 and a WALL board also has column S of every row and all
 *    bits past the last row set (sentinels that end a slide; ts_encode / ts_synth write
 *    them).  S = 7, 8: BS = S, PS = 16, no sentinels.
 *  - wide boards (S >= 9): walls = u16 [axis][capacity][L lines], L = S rounded up to even:
 *    plane 1 = rows (line r, one bit per column), used by LEFT/RIGHT, plane 0 = columns (line
 *    c, one bit per row), used by UP/DOWN; ts_walls_bytes(S) = 4*L bytes per env, of which a
 *    step reads the 2*L bytes of one axis.  S <= 14: cell k of a
 *    line is bit k+1, and bit 0 and bit S+1 of every line are set (edge sentinels); S = 15, 16:
 *    cell k is bit k, no sentinel.  Set-goal target record = u16 [capacity][17]: 16 rows, cell
 *    (r,c) = bit c of word r, then the number of distinct target cells (the step kernels test
 *    "every tile on a target cell" plus "that number == n_tiles", which is set equality).  PS = 16.
 */
#ifndef TILER_SLIDER_H
#define TILER_SLIDER_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TS_VERSION 201          /* 0.2.1 */
#define TS_CAP_ALIGN 128
#define TS_MAX_SIZE 16
#define TS_MAX_TILES 32         /* 0..8: register kernels; 9..32: per-env generic kernels (csrc/ts_generic.cu) */

/* flag bits of the per-env status byte */
#define TS_F_DONE 1u      /* environment.py:133-141  done = is_won or step_count >= max_steps */
#define TS_F_WON 2u       /* info['is_won'] / info['success']  (state.py:172-186)            */
#define TS_F_INVALID 4u   /* info['invalid_move']: no tile moved (environment.py:129)         */
#define TS_F_TIMEOUT 8u   /* info['timeout'] (environment.py:139-141)                         */
#define TS_F_STALE 16u    /* stepped while already done without auto_reset: frozen, no-op
                             (the reference raises RuntimeError, environment.py:113-114)      */

/* goal modes */
#define TS_GOAL_ORDERED 0 /* multi_color=True : tile i on target i (state.py:183-184); targets
                             are packed position words                                        */
#define TS_GOAL_SET 1     /* multi_color=False: occupancy == target set (state.py:185-186);
                             targets are a bitboard in the plane layout                       */

/* error codes */
#define TS_E_BAD_SIZE (-1)
#define TS_E_BAD_TILES (-2)
#define TS_E_BAD_CAPACITY (-3)
#define TS_E_NULL_POINTER (-4)
#define TS_E_MISALIGNED (-5)
#define TS_E_BAD_RANGE (-6)
#define TS_E_UNSUPPORTED (-7)
#define TS_E_BAD_ARGUMENT (-8)

int ts_version(void);
const char *ts_last_error_string(void);

/* layout queries (pure host arithmetic) */
int ts_pos_bytes(int n_tiles);   /* n_tiles = 0 (a board without tiles): 1, the byte is zero */
int ts_board_bytes(int size);
int ts_board_stride(int size);   /* BS: bit index of cell (r,c) in a board = r*BS + c */
int ts_pos_stride(int size);     /* PS: position byte of a tile at (r,c) = r*PS + c */
int ts_walls_bytes(int size);    /* bytes per env of the walls buffer (its size = this * capacity) */
int ts_target_board_bytes(int size); /* bytes per env of the set-goal target board buffer */
int ts_plane_count(int n_bytes);
int ts_plane_width(int n_bytes, int k);
int ts_plane_offset(int n_bytes, int k);
/* 1 if ts_step covers (size, n_tiles): 1 <= size <= 16, 0 <= n_tiles <= 32, else 0 */
int ts_supported(int size, int n_tiles);

/* ---------------------------------------------------------------------------------------
 * K1 ts_encode: dense per-env description -> packed layout.
 * Reproduces GameState.__init__ (state.py:61-73): is_blocked grid + location lists.
 *   d_blocked  u8 [n_envs][size*size]  nonzero = blocked cell
 *   d_tiles    u8 [n_envs][n_tiles][2] (row, col)
 *   d_targets  u8 [n_envs][n_targets][2]
 * Writes walls planes, init + pos position words, targets (ordered: position word of the first
 * min(n_targets, n_tiles) targets -- with n_targets != n_tiles the goal can never be met
 * (state.py:183-184) and the caller passes never_win = 1 to ts_step / ts_goal_check; set:
 * bitboard planes, any n_targets).  n_tiles may be 0 (d_tiles is then not read).
 * Environments are written at [first_env, first_env + n_envs).
 * ------------------------------------------------------------------------------------- */
typedef struct ts_encode_args {
    int32_t size, n_tiles, n_targets, goal_mode;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_blocked, *d_tiles, *d_targets;
    uint8_t *d_walls, *d_targets_packed, *d_init, *d_pos;
} ts_encode_args;
int ts_encode(const ts_encode_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * K0 ts_synth: synthetic puzzles generated on the device in the packed layout.
 * Same recipe as TilerSliderEnvFactory.create_simple_env (environment.py:221-226): a
 * uniformly random arrangement of distinct cells, the first n_walls blocked, the next
 * n_tiles tiles, the next n_tiles targets (always well formed).  The random stream is a
 * counter-based hash of (seed, global env index = env_index_base + local index), NOT
 * numpy's Mersenne Twister, so puzzles differ from create_simple_env(seed=...) but are
 * independent of how environments are sharded across GPUs.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_synth_args {
    int32_t size, n_tiles, n_walls, goal_mode;
    int64_t first_env, n_envs, capacity, env_index_base;
    uint64_t seed;
    uint8_t *d_walls, *d_targets_packed, *d_init, *d_pos;
} ts_synth_args;
int ts_synth(const ts_synth_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * K2 ts_step: one environment step for envs [first_env, first_env+n_envs) (first_env a
 * multiple of 4).  Fuses GameState.move (state.py:120-170), is_won (state.py:172-186) and
 * the bookkeeping of TilerSliderEnv.step (environment.py:119-143): invalid_move, win ->
 * done, step counter, timeout; plus (new in this repo) reward and optional auto-reset
 * (TilerSliderEnv.reset, environment.py:89-97: positions <- init, step_count <- 0).
 *
 *   reward  = won ? r_win : invalid_move ? r_invalid : r_step      (stale envs: 0)
 *   d_flags : TS_F_* bits.  With auto_reset = 0 it is read first: an env whose DONE bit is
 *             set is frozen and reports DONE|STALE.  With auto_reset = 1 it is write-only
 *             and may be NULL.
 *   d_done  : 0/1 byte per env (may be NULL if d_flags is given).
 *   d_terminal_pos : optional position words, written for a 4-env group whenever one of its
 *             envs finished this step: the positions after the move, before the reset.
 *   never_win: 1 when the goal can never be met (ordered mode with len(targets) !=
 *             len(tiles), state.py:183-184).
 *   n_tiles = 0: nothing moves (every step is INVALID); won iff the board has no targets either
 *             (ordered mode: the caller says so through never_win).
 *   count_bytes = 1 needs max_steps <= 255 with auto_reset, <= 254 without.
 *   order   : the order in which the launch walks the range; 0 = ascending, 1 = descending.
 *             Results do not depend on it.  Alternating it on back-to-back steps over one
 *             range makes each step start on the envs the previous one left in L2 (DESIGN
 *             section 3).  Other values: TS_E_BAD_ARGUMENT.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_step_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_walls, *d_targets_packed, *d_init;
    uint8_t *d_pos;
    void *d_step_count;
    int32_t count_bytes, max_steps, auto_reset, order;
    const uint8_t *d_actions;
    float r_win, r_step, r_invalid, reserved1;
    float *d_reward;
    uint8_t *d_done, *d_flags, *d_terminal_pos;
} ts_step_args;
int ts_step(const ts_step_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * K3 ts_observe: dense observation, GameState.get_state_array (state.py:188-211).
 *   d_obs f32 [n_envs][size][size][3] (HWC): ch0 blocked, ch1 tile index+1 (ordered mode) or
 *   1 (set mode), ch2 target index+1 or 1.  In set mode targets come from the bitboard.
 *   n_targets (ordered mode): 0 = as many targets as tiles, d_targets_packed as ts_step reads it;
 *   k > 0 = k targets in words of ts_pos_bytes(k) bytes per env (a board whose target count
 *   differs from its tile count, which ts_step's packed word cannot hold); -1 = no targets;
 *   outside -1..32: TS_E_BAD_TILES.  goal_mode other than TS_GOAL_ORDERED / TS_GOAL_SET:
 *   TS_E_BAD_ARGUMENT.  d_obs must be 16-byte aligned and hold n_envs*size*size*3 floats.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_observe_args {
    int32_t size, n_tiles, goal_mode, n_targets;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_walls, *d_targets_packed, *d_pos;
    float *d_obs;
} ts_observe_args;
int ts_observe(const ts_observe_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_observe_planes: the observation as a network input (csrc/ts_observe_planes.cu; no
 * reference counterpart).  d_out [n_envs][C][size][size], channel first, contiguous, every
 * element 0 or 1 in the type `dtype` names (TS_OBS_U8 / BF16 / F16 / F32: 1, 2, 2, 4 bytes).
 *   plane 0            blocked cells
 *   ordered goal       plane 1+i: tile i's cell (i < n_tiles); plane 1+n_tiles+j: target j's cell
 *                      (j < NT; NT from n_targets as in ts_observe: 0 = n_tiles, k > 0 = k, -1 = 0;
 *                      duplicate targets each keep their own plane);  C = 1 + n_tiles + NT
 *   set goal           plane 1: the tile cells; plane 2: the target cells (the bitboard);  C = 3
 * (single colour with one tile and one target gives the same 3 planes under either rule.)
 * Relation to ts_observe (channels last, HWC): set goal -- the planes are its three channels;
 * ordered goal -- ch0 = plane 0, ch1 = sum_i (i+1) plane(1+i), ch2 = max_j (j+1) plane(1+n_tiles+j).
 * ts_observe_planes_channels: C for these arguments (pure host arithmetic), or a negative
 * TS_E_* code when goal_mode, n_tiles or n_targets is out of range.  Argument errors as
 * ts_observe's, plus an unknown dtype (TS_E_BAD_ARGUMENT); d_out must be 16-byte aligned and hold
 * n_envs*C*size*size elements.
 * ------------------------------------------------------------------------------------- */
#define TS_OBS_U8 0
#define TS_OBS_BF16 1
#define TS_OBS_F16 2
#define TS_OBS_F32 3
typedef struct ts_observe_planes_args {
    int32_t size, n_tiles, goal_mode, n_targets;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_walls, *d_targets_packed, *d_pos;
    int32_t dtype, reserved0;
    void *d_out;
} ts_observe_planes_args;
int ts_observe_planes_channels(const ts_observe_planes_args *a);
int ts_observe_planes(const ts_observe_planes_args *a, void *stream);
/* ts_observe_planes_items: the same planes for n_items ITEMS instead of an env range (first_env and
 * n_envs of *a are not read).  Item i shows env e = d_env_ids[i] (NULL: e = i) -- its walls and
 * targets -- with the tiles of the position word d_item_pos[i] (NULL: d_pos[e]); d_out holds
 * n_items*C*size*size elements, item i at [i].  An e outside [0, capacity) gives an all-zero image and
 * nothing of it is read.  Argument errors as ts_observe_planes's, plus n_items < 0 or, without
 * d_env_ids, n_items > capacity (TS_E_BAD_RANGE); d_pos may be NULL when d_item_pos is given;
 * d_out and d_item_pos must be 16-byte aligned (checked only when n_items > 0). */
int ts_observe_planes_items(const ts_observe_planes_args *a, const int32_t *d_env_ids, const uint8_t *d_item_pos,
                            int64_t n_items, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_expand: the four successors of many states (csrc/ts_expand.cu, ts_wide.cu, ts_generic.cu;
 * GameState.move, state.py:120-170, and is_won, state.py:172-186, once per move), for search:
 * beam search, A* with a learned heuristic, MCTS expansion, value-iteration targets.  An ITEM is
 * a pair (env id, position word): the env supplies the puzzle (walls and targets), the word the
 * tiles.  For item i < n_items, env e = d_env_ids[i] (NULL: e = i), positions p = d_item_pos[i]
 * (NULL: d_pos[e]; words of ts_pos_bytes(n_tiles) bytes, unused bytes zero):
 *   d_succ[i][a]  [n_items][4][pos_bytes], item-major: the positions after move a from p (0 UP,
 *                 1 DOWN, 2 LEFT, 3 RIGHT) -- bit for bit what ts_step leaves in pos for that action
 *                 before any reset; tile order kept (no sorting in set mode), so d_succ read as
 *                 [4*n_items][pos_bytes] is the item list of the next level, with ids repeated 4 times
 *   d_moved[i]    optional: bit a set iff move a changes the positions (the step's !INVALID;
 *                 ts_valid_moves of p)
 *   d_won[i]      optional: bit a set iff the positions after move a meet the goal (the step's WON:
 *                 0 with never_win; n_tiles = 0: the rule of ts_step)
 * An e outside [0, capacity) gives zero successors and masks, and nothing of it is read.  No env
 * buffer is written.  Argument errors (all before the n_items = 0 return): size, n_tiles,
 * capacity, goal_mode, never_win outside 0/1 (TS_E_BAD_ARGUMENT), a NULL d_walls /
 * d_targets_packed / d_succ, or d_pos when d_item_pos is NULL (TS_E_NULL_POINTER), n_items < 0 or,
 * without d_env_ids, n_items > capacity (TS_E_BAD_RANGE); then, with n_items > 0, d_succ and
 * d_item_pos must be 16-byte aligned (TS_E_MISALIGNED).
 * ------------------------------------------------------------------------------------- */
typedef struct ts_expand_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t n_items, capacity;
    const int32_t *d_env_ids;
    const uint8_t *d_walls, *d_targets_packed, *d_pos, *d_item_pos;
    uint8_t *d_succ, *d_moved, *d_won;
} ts_expand_args;
int ts_expand(const ts_expand_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_playout: up to n_steps moves from many states in one launch (csrc/ts_playout.cu, ts_wide.cu,
 * ts_generic.cu; GameState.move, state.py:120-170, and is_won, state.py:172-186, once per move),
 * for MCTS simulation, replaying plans and recording trajectories.  Items as ts_expand's: item
 * i < n_items plays on env e = d_env_ids[i] (NULL: e = i) from positions d_item_pos[i] (NULL:
 * d_pos[e]).  The moves come from `policy`:
 *   TS_PLAYOUT_PLAN    d_plan u8 [n_steps][n_items], step-major: move k of item i is
 *                      d_plan[k*n_items + i] (0 UP, 1 DOWN, 2 LEFT, 3 RIGHT); a byte >= 4 ends the
 *                      plan (255: padding of ragged move strings).  A move that changes nothing is
 *                      still played and counted, as ts_step counts it.
 *   TS_PLAYOUT_RANDOM  each move drawn uniformly among the moves that change the positions (the
 *                      mask of ts_valid_moves), by K7's walk rule: item i's stream is K0's
 *                      synth_stream(seed, i), each move takes one draw r = splitmix64 >> 32 and is
 *                      the floor(r*n / 2^32)-th set bit, lowest first, of the n-bit mask; an empty
 *                      mask ends the playout.
 * The goal is checked after every move, as ts_step does: the playout stops after the first move that
 * meets it.  So a plan of moves 0..3 gives what n_steps ts_step calls with auto_reset = 0 and
 * max_steps > n_steps leave.  Outputs, for every item:
 *   d_final[i]      [n_items][pos_bytes]: the positions after the last move played (tile order kept)
 *   d_steps[i]      int32: moves played
 *   d_won[i]        1 iff the last move played met the goal (never 1 with never_win)
 *   d_moves[k][i]   optional u8 [n_steps][n_items]: the move played as move k; 255 for k >= steps
 *   d_traj[k][i]    optional [n_steps][n_items][pos_bytes]: the positions after move k; 0 for k >= steps
 * An e outside [0, capacity) reads nothing: zero positions, 0 moves, not won, 255 moves.
 * n_tiles = 0: nothing moves; a plan plays its moves as no-ops and the first one wins iff the board
 * has no targets (the rule of ts_step); a random playout plays none.  n_steps = 0: the start
 * positions, 0 moves, not won.  Argument errors (all before the n_items = 0 return): size, n_tiles,
 * capacity, goal_mode, never_win outside 0/1, an unknown policy, n_steps < 0 (TS_E_BAD_ARGUMENT);
 * n_items < 0 or, without d_env_ids, n_items > capacity (TS_E_BAD_RANGE); a NULL d_walls /
 * d_targets_packed / d_final / d_steps / d_won, d_pos when d_item_pos is NULL, or d_plan under
 * TS_PLAYOUT_PLAN (TS_E_NULL_POINTER); n_steps*n_items*pos_bytes beyond int64, or n_items beyond
 * (2^31 - 1) * 128, the items one launch covers (TS_E_BAD_RANGE);
 * then, with n_items > 0, d_final, d_item_pos and d_traj must be 16-byte aligned (TS_E_MISALIGNED).
 * ------------------------------------------------------------------------------------- */
#define TS_PLAYOUT_PLAN 0
#define TS_PLAYOUT_RANDOM 1
typedef struct ts_playout_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int32_t policy, n_steps;
    int64_t n_items, capacity;
    uint64_t seed;
    const int32_t *d_env_ids;
    const uint8_t *d_walls, *d_targets_packed, *d_pos, *d_item_pos, *d_plan;
    uint8_t *d_final;
    int32_t *d_steps;
    uint8_t *d_won, *d_moves, *d_traj;
} ts_playout_args;
int ts_playout(const ts_playout_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_valid_moves: bit d of d_mask[env] set when move d changes any tile position
 * (TilerSliderEnv.get_valid_moves, environment.py:149-171).
 * ------------------------------------------------------------------------------------- */
typedef struct ts_valid_args {
    int32_t size, n_tiles;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_walls, *d_pos;
    uint8_t *d_mask;
} ts_valid_args;
int ts_valid_moves(const ts_valid_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_goal_check: d_won[env] = 1 when the CURRENT positions meet the goal
 * (GameState.is_won, state.py:172-186), without moving.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_goal_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t first_env, n_envs, capacity;
    const uint8_t *d_targets_packed, *d_pos;
    uint8_t *d_won;
} ts_goal_args;
int ts_goal_check(const ts_goal_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * Breadth-first state-space expansion (BASELINE config 5; no reference counterpart -- the
 * successor function is GameState.move, state.py:120-170, the goal test is_won,
 * state.py:172-186; boards of size <= 8).
 *
 * State key (uint64): canonical position word in the low bits (ordered goal: the position
 * bytes; set goal: the bytes sorted ascending), puzzle id in bits 32..62 when n_tiles <= 4
 * (n_tiles > 4: one puzzle only), bit 63 = "meets the goal" (ignored by dedup).
 * TS_BFS_NONE marks a move that changed nothing.  The puzzle table is a packed batch
 * (walls / targets / init of `puzzle_capacity` stride, as written by ts_encode).
 *
 *   ts_bfs_seed              d_out_keys[i] = key of puzzle i's initial state, i < n_items
 *   ts_bfs_expand        K4  d_out_keys[4*i+d] = successor of d_in_keys[i] under move d
 *   ts_bfs_partition_count   d_counts[r] += #keys of d_in_keys owned by rank r = hash(key) % n_ranks
 *   ts_bfs_partition_scatter d_out_keys bucketed by owner; d_counts[r] = write cursor of bucket r
 *                            (initialise to the exclusive prefix sum of the counts)
 *   ts_bfs_hash_insert   K5  insert d_in_keys into the open-addressing table d_table
 *                            (table_capacity a power of two, empty = TS_BFS_NONE); keys not
 *                            seen before are appended to d_out_keys; d_counts[0] = append
 *                            cursor, d_counts[1] += #goal successors seen, d_counts[2] = 1 on
 *                            overflow of the table or of out_capacity
 *   ts_bfs_traceback         follow the recorded parents from a goal state back to the root and
 *                            emit the move string (the move between parent and child is found by
 *                            re-running the four slides on the parent)
 * The exchange between partition and insert is an NCCL all-to-all done by the caller.
 * ------------------------------------------------------------------------------------- */
#define TS_BFS_NONE 0xFFFFFFFFFFFFFFFFull
#define TS_BFS_WON_BIT 0x8000000000000000ull
typedef struct ts_bfs_args {
    int32_t size, n_tiles, goal_mode, never_win, n_ranks;
    int32_t rank;                       /* ts_bfs_trace_step: the caller's rank among n_ranks owners */
    int64_t n_items, puzzle_capacity, table_capacity, out_capacity;
    const uint8_t *d_walls, *d_targets_packed, *d_init;
    const uint64_t *d_in_keys;
    uint64_t *d_out_keys, *d_table, *d_counts;
    /* optional parent tracking: with d_table_parent given, ts_bfs_hash_insert records for every
     * new key the key it was expanded from; d_parent_keys = NULL marks roots.
     *   parent_per_item = 0 (single rank): d_in_keys must be exactly the output of ts_bfs_expand
     *     on d_parent_keys, so that the parent of d_in_keys[i] is d_parent_keys[i / 4];
     *   parent_per_item = 1 (several ranks): the parent of d_in_keys[i] is d_parent_keys[i] --
     *     the array ts_bfs_partition_scatter filled next to the keys (d_out_parents) and the
     *     caller exchanged with them. */
    const uint64_t *d_parent_keys;
    uint64_t *d_table_parent;
    /* ts_bfs_traceback: d_in_keys[i] = goal state of item i (TS_BFS_NONE: none), d_parent_keys[i]
     * = the state it was generated from (d_goal_parents of the inserts); writes the shortest move
     * string of item i to d_moves[i * max_moves ...] (0..3, root first) and its length to
     * d_lengths[i] (-1: no goal / longer than max_moves / broken chain) */
    uint8_t *d_moves;
    int32_t *d_lengths;
    int64_t max_moves;
    /* ts_bfs_hash_insert, optional: the first won_capacity goal successors seen (duplicates
     * included) are also copied to d_won_keys, in the order of d_counts[1] */
    uint64_t *d_won_keys;
    int64_t won_capacity;
    /* ts_bfs_hash_insert, optional per-puzzle tallies (puzzle id = key bits 32..62; 0 when
     * n_tiles > 4): d_states_per_puzzle[pid] += 1 for every new key; for every goal successor
     * d_solve_depth[pid] = min(itself, depth), and the first one to lower it also stores its key
     * in d_goal_keys[pid] (optional) -- a goal state at the smallest depth */
    int64_t *d_states_per_puzzle;
    int32_t *d_solve_depth;
    uint64_t *d_goal_keys;
    int32_t depth, reserved2;
    /* ts_bfs_expand_exchange (multi-GPU, peer memory): d_peer_bufs[r] = rank r's exchange buffer
     * as mapped into THIS process (NVLink peer mapping, e.g. torch symmetric memory):
     *   word 0, 1          arrival cursors of inbox 0 / inbox 1 (keys received so far)
     *   word 2             set to 1 when an inbox overflowed
     *   word TS_BFS_XHDR + p * inbox_capacity ...   inbox p (u64 keys)
     * The successors of d_in_keys are written straight into inbox `parity` of their owner rank
     * (hash(key) % n_ranks); d_counts[3] += number of keys sent. */
    uint64_t *const *d_peer_bufs;
    int64_t inbox_capacity;
    int32_t parity, parent_per_item;
    /* device-driven levels (ts_bfs_expand, ts_bfs_hash_insert), optional: the item count is read
     * on the DEVICE as min(n_items, *d_n_items * n_items_scale) -- n_items is then only the
     * bound the grid is sized for -- so consecutive levels can be launched back to back
     * without the host learning the frontier sizes in between: expand level d with
     * d_n_items = &new_count[d], insert with the same pointer, scale 4 and d_counts =
     * the counter block of level d+1. */
    const int64_t *d_n_items;
    int64_t n_items_scale;
    /* ts_bfs_partition_scatter, optional (with d_parent_keys = the frontier d_in_keys was expanded
     * from): d_out_parents[j] = parent of the key written to d_out_keys[j] */
    uint64_t *d_out_parents;
    /* ts_bfs_hash_insert, optional (with d_goal_keys and d_parent_keys): d_goal_parents[pid] = the
     * state the goal successor stored in d_goal_keys[pid] was generated from.  A shortest solution
     * is the chain root -> that state plus the move from it to the goal; the goal state's own
     * table entry must not be used for this, because a puzzle whose initial state already meets
     * the goal is won by its first step (a root is never a goal successor), and the root has no
     * parent. */
    uint64_t *d_goal_parents;
} ts_bfs_args;
#define TS_BFS_XHDR 16
int ts_bfs_seed(const ts_bfs_args *a, void *stream);
int ts_bfs_expand(const ts_bfs_args *a, void *stream);
int ts_bfs_partition_count(const ts_bfs_args *a, void *stream);
int ts_bfs_partition_scatter(const ts_bfs_args *a, void *stream);
int ts_bfs_hash_insert(const ts_bfs_args *a, void *stream);
/* expand + bucket + exchange in one kernel: no partition pass, no size exchange, no all-to-all;
 * the caller separates levels with any collective that orders the ranks' streams (an all-reduce
 * of the sent counts doubles as the termination test) and alternates `parity` level by level. */
int ts_bfs_expand_exchange(const ts_bfs_args *a, void *stream);
int ts_bfs_traceback(const ts_bfs_args *a, void *stream);
/* One step of a traceback over a visited set that is spread over n_ranks owners (hash-partitioned
 * search with parents): for every item i whose key d_in_keys[i] this rank owns, look the key up and
 * write its parent to d_out_keys[i] and the move that leads from the parent to it to d_moves[i]
 * (one byte per item).  Read as int64: parent >= 0; -1 (TS_BFS_NONE) the key is a root; -2 the chain
 * is broken (key or move not found); INT64_MIN (with move 0) for TS_BFS_NONE items and for keys of
 * other ranks -- so a MAX all-reduce of both arrays over the owners yields the step for every
 * item.  n_ranks = 1: every key is this rank's.  With d_parent_keys given (the last link of a
 * solution, d_goal_parents) nothing is looked up: the parent of item i is d_parent_keys[i], on
 * every rank. */
int ts_bfs_trace_step(const ts_bfs_args *a, void *stream);
/* n_levels device-driven BFS levels launched back to back (2 kernels per level, no host sync):
 * level d = first_depth .. first_depth + n_levels - 1 expands the lvl[4*d] keys of
 * front[d & 1] into succ (4 * frontier_capacity keys) and inserts them as level d+1 into
 * front[(d+1) & 1], counters in lvl[4*(d+1) ..] = (new keys, goal successors, overflow, -),
 * which must be zero on entry.  `a` supplies the puzzle tables, d_table / table_capacity, the
 * optional parent table (d_table_parent; parents are the frontier keys) and per-puzzle tallies.
 * known_frontier >= 0: the host knows the size of level first_depth (n_levels must be 1): that
 * level is launched with a grid of its own size instead of one persistent wave. */
int ts_bfs_levels(const ts_bfs_args *a, int32_t first_depth, int32_t n_levels, uint64_t *front0, uint64_t *front1,
                  uint64_t *succ, int64_t *lvl, int64_t frontier_capacity, int64_t known_frontier, void *stream);

/* ---------------------------------------------------------------------------------------
 * K6 ts_bfs_local: breadth-first search of many small puzzles, one CTA per puzzle, on chip
 * (csrc/ts_bfs_local.cu).  Same successor function, goal test, canonical states and result
 * definitions as the hash-partitioned search above; boards of size <= 8 with 1..4 tiles.
 * The visited set of a puzzle is a bitmap in shared memory over a perfect hash of the state (the
 * arrangement number of its T tiles among the F free cells of the puzzle: F!/(F-T)! bits,
 * bitmap_words u32 words, a multiple of 4); the frontier queue is a ring of `queue_smem` states
 * (a power of two >= 32) in shared memory -- the level being expanded and the one being appended --
 * and spills to d_spill[cta][spill_per_cta], indexed by discovery order.  Persistent grid: CTAs
 * draw puzzles from the ticket counter.
 *   d_puzzle_ids       optional: search puzzles d_puzzle_ids[0 .. n_puzzles) instead of 0 .. n_puzzles-1
 *   d_status[pid]      0 searched; 1 state space exceeds bitmap_words*32 bits; 2 spill slab exhausted; 3 deeper
 *                      than 255 levels -- for != 0 nothing else of the puzzle is valid (search it
 *                      with the hash-partitioned path)
 *   d_states_per_puzzle[pid], d_solve_depth[pid] (-1: no goal within max_depth)
 *   d_levels[d]        += new states at depth d over the searched puzzles (n_levels >= 256 entries)
 *   d_counters         [0] ticket (zero on entry), [1] += successors generated, [3] = max(depth reached)
 *   d_lengths / d_moves / d_parent_scratch  optional shortest move string per puzzle (0..3, root
 *                      first; length -1: unsolved or longer than max_moves); d_parent_scratch holds
 *                      grid * spill_per_cta words (spill_per_cta then bounds the states of a puzzle)
 * ts_bfs_local_smem_bytes: dynamic shared memory of a launch with these arguments;
 * ts_bfs_local_ctas_per_sm: resident CTAs per SM and the SM count, to size the grid.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_bfs_local_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t n_puzzles, puzzle_capacity;
    const uint8_t *d_walls, *d_targets_packed, *d_init;
    const int32_t *d_puzzle_ids;
    int32_t max_depth, bitmap_words, queue_smem, n_levels;
    uint32_t *d_spill;
    int64_t spill_per_cta;
    uint32_t *d_parent_scratch;
    int64_t *d_states_per_puzzle;
    int32_t *d_solve_depth, *d_status;
    int64_t *d_levels;
    uint64_t *d_counters;
    uint8_t *d_moves;
    int32_t *d_lengths;
    int64_t max_moves;
} ts_bfs_local_args;
int ts_bfs_local_smem_bytes(const ts_bfs_local_args *a);
int ts_bfs_local_ctas_per_sm(const ts_bfs_local_args *a, int *ctas_per_sm, int *n_sm);
int ts_bfs_local(const ts_bfs_local_args *a, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * Device-memory bitmaps (K6 here, K9 and K10 below).  With four tiles the bitmap of a board of
 * more than 38 free cells does not fit one CTA's shared memory; only 7x7 and 8x8 boards have that
 * many (up to 64*63*62*61 bits = 1.9 MB).  The *_gmem entry points run the same search with the
 * bitmap in device memory: CTA b's bitmap is d_bitmap[b * bitmap_words ..], so d_bitmap holds
 * grid * bitmap_words words and is 16-byte aligned; its contents on entry do not matter and are
 * left undefined.  Dynamic shared memory holds the ring alone (queue_smem * 4 bytes).  Same
 * arguments and results as the shared counterpart, as if shared memory were large enough.
 * Argument checks: every check of the shared counterpart with the same code, in the same order;
 * then TS_E_UNSUPPORTED unless (size, n_tiles) is (7, 4) or (8, 4), TS_E_NULL_POINTER for a NULL
 * d_bitmap, TS_E_MISALIGNED for a misaligned one; all before the empty-batch return.
 * *_gmem_ctas_per_sm: resident CTAs per SM of the device instance and the SM count (the shape is
 * checked after the shared query's checks).
 * ------------------------------------------------------------------------------------- */
int ts_bfs_local_gmem_ctas_per_sm(const ts_bfs_local_args *a, int *ctas_per_sm, int *n_sm);
int ts_bfs_local_gmem(const ts_bfs_local_args *a, uint32_t *d_bitmap, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * K7 ts_synth_candidates: candidate puzzles for a generator that keeps the ones K6 grades into a
 * band of shortest-solution lengths (csrc/ts_generate.cu; no reference counterpart).  One thread
 * per listed env: puzzle of env slot d_env_ids[i] (i < n_items; NULL: slot i; ids outside
 * [0, capacity) are skipped) written to walls / targets / init / pos.  The random stream is a
 * function of (seed, attempt, global env index = env_index_base + slot) only.
 *   recipe TS_RECIPE_UNIFORM: K0's draw.  attempt 0 writes exactly the puzzle ts_synth writes for
 *          that env; attempt a > 0 draws with the seed splitmix64(seed ^ a * 0xA0761D6478BD642F).
 *   recipe TS_RECIPE_WALK: walls and tiles as K0 (the first n_walls + n_tiles cells of the same
 *          permutation, same seed rule), then walk_len moves, each drawn uniformly among the moves
 *          that change the state (one 32-bit draw of the same stream per move: the k-th of the n
 *          such moves in UP, DOWN, LEFT, RIGHT order, k = draw * n >> 32); the walk stops early
 *          when no move changes the state.  Targets = the final positions (ordered goal: tile i's;
 *          set goal: the cells).  Every such puzzle is solvable.
 * Domain: size <= 8, 1 <= n_tiles <= 4 (what K6 grades).
 * ts_synth_candidates_t8: the same candidates, checks and stream rule for 5 <= n_tiles <= 8 (what
 * K11 grades); ts_synth_candidates returns TS_E_UNSUPPORTED for those tile counts.
 * ------------------------------------------------------------------------------------- */
#define TS_RECIPE_UNIFORM 0
#define TS_RECIPE_WALK 1
#define TS_MAX_WALK 65535
typedef struct ts_synth_candidates_args {
    int32_t size, n_tiles, n_walls, goal_mode;
    int32_t recipe, walk_len, attempt, reserved0;
    int64_t n_items, capacity, env_index_base;
    uint64_t seed;
    const int32_t *d_env_ids;
    uint8_t *d_walls, *d_targets_packed, *d_init, *d_pos;
} ts_synth_candidates_args;
int ts_synth_candidates(const ts_synth_candidates_args *a, void *stream);
int ts_synth_candidates_t8(const ts_synth_candidates_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * K8 ts_pool_reset: auto-reset into a pool of puzzles (csrc/ts_generate.cu; no reference
 * counterpart -- TilerSliderEnv.reset, environment.py:89-97, restarts the same puzzle).  For every
 * env of [first_env, first_env + n_envs) whose d_done byte is set (d_done = NULL: every env):
 *   j = H(seed, env_index_base + env, d_episode[env]) in [0, n_pool), d_episode[env] += 1,
 *   walls / targets / init <- pool puzzle j, pos <- init, step_count <- 0,
 *   d_solve_depth[env] <- d_pool_depth[j] (when both are given).
 * H(seed, g, e) = (mix(mix(seed ^ (g + 1) * 0xD1B54A32D192ED03) ^ (e + 1) * 0x9E3779B97F4A7C15) * n_pool) >> 64
 * with mix the splitmix64 finaliser (64x64 -> high 64 bits).  The pool is a packed batch of the
 * same size, tile count and goal mode (any board class, any tile count up to TS_MAX_TILES) with
 * stride pool_capacity.  Meant to run right after ts_step (it reads the done bytes the step wrote);
 * it is launched with programmatic dependent launch like the step.  Touches nothing outside the
 * range.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_pool_reset_args {
    int32_t size, n_tiles, goal_mode, count_bytes;
    int64_t first_env, n_envs, capacity, env_index_base;
    uint64_t seed;
    const uint8_t *d_done;
    uint32_t *d_episode;
    uint8_t *d_walls, *d_targets_packed, *d_init, *d_pos;
    void *d_step_count;
    int32_t *d_solve_depth;
    int64_t n_pool, pool_capacity;
    const uint8_t *d_pool_walls, *d_pool_targets, *d_pool_init;
    const int32_t *d_pool_depth;
} ts_pool_reset_args;
int ts_pool_reset(const ts_pool_reset_args *a, void *stream);

/* ---------------------------------------------------------------------------------------
 * K9 ts_optimal_moves: exact distance to the goal, the set of optimal first moves and optionally
 * a shortest solution of items (env id, positions), for the CURRENT positions of listed envs or
 * for any position words (csrc/ts_optimal.cu; no reference counterpart -- defined
 * through a BFS over GameState.move, state.py:120-170, with the goal test is_won,
 * state.py:172-186, checked after every move).  Boards of size <= 8 with 1..4 tiles.  For item
 * i < n_items, env e = d_env_ids[i] (NULL: e = i), positions s = d_item_pos[i * pos_bytes ..]
 * (d_item_pos NULL: s = d_pos[e]); the env gives the walls and the goal:
 *   d_distance[i]  the fewest moves that win from s (>= 1: a state already on the goal is at 1,
 *                  through any move that leaves the tiles on the goal, one that changes nothing
 *                  included); max_steps and step counters play no part.  Otherwise
 *                  TS_OPT_UNSOLVABLE (-1) no winning state reachable (never_win: always),
 *                  TS_OPT_CUTOFF (-2) none within max_depth moves, TS_OPT_NOT_SEARCHED (-3)
 *                  the state space exceeds bitmap_words*32 bits or the slab, or e is outside
 *                  [0, capacity), TS_OPT_BAD_STATE (-4) s is not a well-formed state of env e:
 *                  a tile byte on no in-board free cell (a wall, off the board, >= 128) or two
 *                  tiles on one cell (checked for every listed item, env positions included,
 *                  before never_win and the state-space size).
 *   d_mask[i]      bit m (UP=0, DOWN=1, LEFT=2, RIGHT=3, as ts_valid_moves) set iff move m starts
 *                  a shortest solution: distance 1: m wins; else distance(succ_m(s)) ==
 *                  distance(s) - 1.  0 whenever d_distance[i] < 0.
 *   d_plan         (NULL: no paths) uint8 [max_depth][n_items], step-major as ts_playout's plan:
 *                  d_plan[k * n_items + i] for k < d_distance[i] is move k of the
 *                  lexicographically smallest shortest solution from s (UP < DOWN < LEFT < RIGHT:
 *                  each move the lowest bit of the mask of the state it is played from); every
 *                  other entry, all rows of an item with d_distance[i] < 0 included, is 255.  The
 *                  kernel writes every entry.  d_distance and d_mask do not depend on d_plan.
 * All in item order, deterministic.  One CTA per item, persistent grid drawing items from the
 * ticket counter; visited set and optimal-state set: a shared-memory bitmap over the perfect hash
 * of K6; frontier: a ring of queue_smem states (a power of two >= 32) in shared memory, and every
 * state also in d_spill[cta][spill_per_cta] (it is read again by the backward pass), so
 * spill_per_cta bounds the states a search may reach.  1 <= max_depth <= TS_OPT_MAX_DEPTH.
 *   d_counters     [0] ticket (zero on entry), [1] += states expanded by the forward search,
 *                  [2] += states re-expanded by the backward pass
 * ts_optimal_moves_smem_bytes / ts_optimal_moves_ctas_per_sm: as for K6.
 * ts_optimal_max_free_cells: atomically raises *d_max_free (int32, device) to the most free cells
 * of any listed env (ids outside [0, capacity) skipped), which sizes bitmap_words; reads
 * size, n_items, capacity, d_env_ids and d_walls only (d_targets_packed and d_pos must be set).
 * ------------------------------------------------------------------------------------- */
#define TS_OPT_UNSOLVABLE (-1)
#define TS_OPT_CUTOFF (-2)
#define TS_OPT_NOT_SEARCHED (-3)
#define TS_OPT_BAD_STATE (-4)
#define TS_OPT_MAX_DEPTH 254
typedef struct ts_optimal_moves_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t n_items, capacity;
    const int32_t *d_env_ids;
    const uint8_t *d_walls, *d_targets_packed, *d_pos;
    int32_t max_depth, bitmap_words, queue_smem, reserved0;
    uint32_t *d_spill;
    int64_t spill_per_cta;
    uint64_t *d_counters;
    int32_t *d_distance;
    uint8_t *d_mask;
    const uint8_t *d_item_pos;      /* [n_items][pos_bytes] roots; NULL: the envs' positions */
    uint8_t *d_plan;                /* [max_depth][n_items] shortest solutions; NULL: none */
} ts_optimal_moves_args;
int ts_optimal_moves_smem_bytes(const ts_optimal_moves_args *a);
int ts_optimal_moves_ctas_per_sm(const ts_optimal_moves_args *a, int *ctas_per_sm, int *n_sm);
int ts_optimal_max_free_cells(const ts_optimal_moves_args *a, int32_t *d_max_free, void *stream);
int ts_optimal_moves(const ts_optimal_moves_args *a, int grid, void *stream);
/* device-memory bitmap (see ts_bfs_local_gmem): the instance with plans when d_plan is set */
int ts_optimal_moves_gmem_ctas_per_sm(const ts_optimal_moves_args *a, int *ctas_per_sm, int *n_sm);
int ts_optimal_moves_gmem(const ts_optimal_moves_args *a, uint32_t *d_bitmap, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * K11 ts_optimal_moves_table: K9 for boards of size 3..8 with 5..8 tiles (csrc/ts_table_search.cu),
 * the same struct, items, result definitions (d_distance, d_mask, d_plan) and counters, with the
 * visited set a per-CTA hash table in device memory instead of the perfect-hash bitmap: CTA b owns
 * d_table[b * table_slots ..] (uint64; contents on entry do not matter and are left undefined),
 * table_slots a power of two >= 2 * spill_per_cta.  States are 64-bit words (pos_bytes 8).
 *   d_spill        [grid][spill_per_cta] 64-bit entries (8-byte aligned); an item that discovers
 *                  more than spill_per_cta states gets TS_OPT_NOT_SEARCHED (-3): the bound depends
 *                  on the plan only, never on the other items of the launch.
 *   bitmap_words   unused, must be 0; queue_smem: ring entries (64-bit) in shared memory, a power
 *                  of two >= 32.
 * Argument checks: ts_optimal_moves' checks in the same order with the same codes, with n_tiles
 * outside 5..8 TS_E_UNSUPPORTED and bitmap_words != 0 TS_E_BAD_ARGUMENT; then table_slots not a
 * power of two >= 2 * spill_per_cta (TS_E_BAD_ARGUMENT), a NULL d_table (TS_E_NULL_POINTER), a
 * d_table or d_spill not 8-byte aligned (TS_E_MISALIGNED); all before the empty-query return.
 * ts_optimal_moves_table_ctas_per_sm: resident CTAs per SM with the ring alone in shared memory
 * (the instance with plans when d_plan is set) and the SM count.
 * ------------------------------------------------------------------------------------- */
int ts_optimal_moves_table_ctas_per_sm(const ts_optimal_moves_args *a, int *ctas_per_sm, int *n_sm);
int ts_optimal_moves_table(const ts_optimal_moves_args *a, uint64_t *d_table, int64_t table_slots, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * K10 ts_state_table: every state reachable from items (env id, positions), each with K9's
 * distance and optimal-move mask (csrc/ts_state_table.cu; no reference counterpart).  Items,
 * domain and root check as K9 (size <= 8, 1..4 tiles; env e = d_env_ids[i] (NULL: e = i), root
 * d_item_pos[i * pos_bytes ..] (NULL: d_pos[e])).  Two launches with the same arguments and grid:
 *   ts_state_table_count  forward BFS from each root to exhaustion:
 *     d_status[i]   0 enumerated; TS_OPT_NOT_SEARCHED (-3) the state space exceeds
 *                   bitmap_words*32 bits, the reachable set exceeds spill_per_cta states (the
 *                   slab the ring spills to), or e is outside [0, capacity); TS_OPT_BAD_STATE (-4)
 *                   the root is not a well-formed state (K9's rule)
 *     d_count[i]    int64: the states reachable from the root, the root included (0 if status != 0)
 *     d_counters    [0] ticket (zero on entry)
 *   the caller sets d_offsets (int64 [n_items + 1]) to the exclusive cumsum of d_count, then
 *   ts_state_table_fill   for each item with status 0 (the others are skipped), rows
 *     [d_offsets[i], d_offsets[i+1]) of:
 *     d_rows        uint8 [rows][pos_bytes]: each reachable state exactly once (set goal: canonical,
 *                   bytes ascending; padding bytes 0), in ascending order of the perfect hash
 *                   the bitmap is keyed by (deterministic); the rows also serve as the BFS queue
 *     d_distance    int32 [rows]: K9's distance of the row's state (>= 1), or -1 if no win is
 *                   reachable from it (never_win: every row)
 *     d_mask        uint8 [rows]: K9's mask of the row's state (0 where distance < 0)
 *     d_counters    [1] ticket (zero on entry), [2] += rows swept by the retrograde rounds
 * ts_state_table_ctas_per_sm: resident CTAs per SM of both kernels (the fewer) and the SM count.
 * ts_optimal_max_free_cells sizes bitmap_words for these launches as for K9.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_state_table_args {
    int32_t size, n_tiles, goal_mode, never_win;
    int64_t n_items, capacity;
    const int32_t *d_env_ids;
    const uint8_t *d_walls, *d_targets_packed, *d_pos;
    const uint8_t *d_item_pos;      /* [n_items][pos_bytes] roots; NULL: the envs' positions */
    int32_t bitmap_words, queue_smem;
    uint32_t *d_spill;              /* count pass: [grid][spill_per_cta] */
    int64_t spill_per_cta;
    uint64_t *d_counters;
    int64_t *d_count;               /* count pass output */
    int32_t *d_status;              /* count pass output, fill pass input */
    const int64_t *d_offsets;       /* fill pass input */
    uint8_t *d_rows;                /* fill pass outputs */
    int32_t *d_distance;
    uint8_t *d_mask;
} ts_state_table_args;
int ts_state_table_ctas_per_sm(const ts_state_table_args *a, int *ctas_per_sm, int *n_sm);
int ts_state_table_count(const ts_state_table_args *a, int grid, void *stream);
int ts_state_table_fill(const ts_state_table_args *a, int grid, void *stream);
/* device-memory bitmap (see ts_bfs_local_gmem): both passes of a table take the same plan, grid
 * and d_bitmap; ts_state_table_gmem_ctas_per_sm gives the fewer CTAs per SM of the two */
int ts_state_table_gmem_ctas_per_sm(const ts_state_table_args *a, int *ctas_per_sm, int *n_sm);
int ts_state_table_count_gmem(const ts_state_table_args *a, uint32_t *d_bitmap, int grid, void *stream);
int ts_state_table_fill_gmem(const ts_state_table_args *a, uint32_t *d_bitmap, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * K12 ts_state_table_*_table: K10 for boards of size 3..8 with 5..8 tiles
 * (csrc/ts_table_state_table.cu), the same struct, items, passes and result definitions, with
 * K11's visited set: CTA b owns d_table[b * table_slots ..] (uint64; contents on entry do not
 * matter and are left undefined), table_slots a power of two >= 2 * spill_per_cta.  States are
 * 64-bit words (pos_bytes 8).  Both passes take the same arguments, grid, d_spill and d_table.
 *   d_spill        [grid][spill_per_cta] 64-bit entries (8-byte aligned), used by BOTH passes: the
 *                  count pass's queue, and the fill pass's queue and sort buffer.
 *   bitmap_words   unused, must be 0; queue_smem: ring entries (64-bit) in shared memory, a power
 *                  of two >= 32.
 *   ts_state_table_count_table  forward BFS from each root to exhaustion (never_win included):
 *     d_status[i]   0 enumerated; TS_OPT_NOT_SEARCHED (-3) more than spill_per_cta states are
 *                   reachable, the root included (the bound depends on spill_per_cta alone, never on
 *                   the grid or the other items), or e is outside [0, capacity); TS_OPT_BAD_STATE
 *                   (-4) the root is not a well-formed state (K9's rule)
 *     d_count[i]    int64: the states reachable from the root, the root included (0 if status != 0)
 *     d_counters    [0] ticket (zero on entry)
 *   the caller sets d_offsets (int64 [n_items + 1]) to the exclusive cumsum of d_count, then
 *   ts_state_table_fill_table   for each item with status 0 (the others are skipped), rows
 *     [d_offsets[i], d_offsets[i+1]) of:
 *     d_rows        uint8 [rows][8] (8-byte aligned): each reachable state exactly once (set goal:
 *                   canonical, bytes ascending; padding bytes 0, never flag bits), in strictly
 *                   ascending order of the row's 8 bytes read as a little-endian 64-bit word
 *                   (deterministic: independent of the grid, the ring and the atomics)
 *     d_distance    int32 [rows]: K11's distance of the row's state (>= 1), or -1 if no win is
 *                   reachable from it (never_win: every row)
 *     d_mask        uint8 [rows]: K11's mask of the row's state (0 where distance < 0)
 *     d_counters    [1] ticket (zero on entry), [2] += rows swept by the retrograde rounds
 * Argument checks, all before the empty-query return: ts_optimal_moves_table's plan checks (size,
 * 5..8 tiles, goal mode, bitmap_words == 0, the ring), the env table, then K10's checks of the pass
 * (d_counters, d_status, grid < 1 with n_items > 0; count: spill_per_cta, d_spill, d_count; fill:
 * d_offsets, d_rows, d_distance, d_mask), then for both passes spill_per_cta outside 1..2^32-1
 * (TS_E_BAD_ARGUMENT) and a NULL d_spill (TS_E_NULL_POINTER), table_slots not a power of two >=
 * 2 * spill_per_cta (TS_E_BAD_ARGUMENT), a NULL d_table (TS_E_NULL_POINTER), a d_table, d_spill or
 * (fill) d_rows not 8-byte aligned (TS_E_MISALIGNED).
 * ts_state_table_table_ctas_per_sm: resident CTAs per SM of both kernels (the fewer) and the SM count.
 * ------------------------------------------------------------------------------------- */
int ts_state_table_table_ctas_per_sm(const ts_state_table_args *a, int *ctas_per_sm, int *n_sm); /* fewer of the two passes */
int ts_state_table_count_table(const ts_state_table_args *a, uint64_t *d_table, int64_t table_slots, int grid, void *stream);
int ts_state_table_fill_table(const ts_state_table_args *a, uint64_t *d_table, int64_t table_slots, int grid, void *stream);

/* ---------------------------------------------------------------------------------------
 * ts_step_host: the same step through HOST buffers (the call a host-side driver makes):
 * h_actions (pinned) -> device, ts_step, reward/done -> h_reward/h_done (pinned), pipelined in
 * chunks over the context's streams; returns after everything has landed.
 * a->d_actions/d_reward/d_done must still point at device staging of n_envs elements.
 * h_flags (optional, pinned): also download the TS_F_* status byte.  With h_reward = h_done =
 * NULL only that byte comes back (1 instead of 5 bytes per env over PCIe): it encodes done (bit
 * 0) and, since reward is a function of WON / INVALID, the reward.
 * ------------------------------------------------------------------------------------- */
typedef struct ts_host_ctx ts_host_ctx;
int ts_host_ctx_create(ts_host_ctx **out, int n_streams);
int ts_host_ctx_destroy(ts_host_ctx *ctx);
int ts_step_host(ts_host_ctx *ctx, const ts_step_args *a, const uint8_t *h_actions, float *h_reward,
                 uint8_t *h_done, uint8_t *h_flags, int64_t chunk_envs);

#ifdef __cplusplus
}
#endif
#endif /* TILER_SLIDER_H */
