/*
 * ts_oracle.c -- CPU restatement of the Tiler-Slider move path.  TEST INFRASTRUCTURE ONLY.
 *
 * This file is the parity checker for the CUDA product path.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * it.  Nothing under tiler_slider_b200/ imports, links or executes it.
 *
 * It restates, in plain C and deliberately in the reference's own sequential form
 * (slide table -> ordered processing -> back-off against a used set), the algorithm of
 *   explainrl/environment/state.py:47-73    GameState.__init__      -> tso_new
 *   explainrl/environment/state.py:75-118   _precompute_moves       -> build_slide_table
 *   explainrl/environment/state.py:120-170  GameState.move          -> tso_move
 *   explainrl/environment/state.py:172-186  GameState.is_won        -> tso_is_won
 *   explainrl/environment/state.py:188-211  get_state_array         -> tso_observe
 *   explainrl/environment/environment.py:82-98   reset              -> env_reset
 *   explainrl/environment/environment.py:100-143 step               -> env_step
 *   explainrl/environment/environment.py:149-171 get_valid_moves    -> tso_valid_moves
 * It shares no code and no formula with the CUDA kernels (which use a closed-form
 * bitboard compaction), so agreement between the two is meaningful.
 *
 * Parity pin: tests/test_oracle_golden.py checks this file against the reference's own
 * golden vectors (tests/test_user_scenarios.py, tests/test_state.py collision and
 * slide-table cases) and against the tests/golden fixtures, which were produced by importing the
 * unmodified Python reference (tests/golden/make_golden.py).
 *
 * Additions that do NOT exist in the reference (parity unpinned, defined by this repo):
 * reward, auto-reset, the "stale" freeze of finished environments, CPU BFS.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define TSO_UP 0
#define TSO_DOWN 1
#define TSO_LEFT 2
#define TSO_RIGHT 3

/* flag bits shared with include/tiler_slider.h */
#define TSO_F_DONE 1
#define TSO_F_WON 2
#define TSO_F_INVALID 4
#define TSO_F_TIMEOUT 8
#define TSO_F_STALE 16

#define TSO_STACK_TILES 32

typedef struct tso_state {
    int size;
    int n_tiles;
    int n_targets;
    int multi_color;
    uint8_t *is_blocked; /* [size*size] */
    int *move_to;        /* [size][size][4][2] */
    int *cur;            /* [n_tiles][2] */
    int *tgt;            /* [n_targets][2] */
} tso_state;

/* state.py:75-118 -- four directional sweeps, each cell inherits its neighbour's
 * destination when the neighbour is in bounds and not blocked. */
static void build_slide_table(tso_state *st) {
    const int S = st->size;
    int *mt = st->move_to;
#define MT(i, j, d, k) mt[((((i) * S) + (j)) * 4 + (d)) * 2 + (k)]
    for (int i = 0; i < S; ++i)
        for (int j = 0; j < S; ++j) {
            if (i > 0 && !st->is_blocked[(i - 1) * S + j]) {
                MT(i, j, TSO_UP, 0) = MT(i - 1, j, TSO_UP, 0);
                MT(i, j, TSO_UP, 1) = MT(i - 1, j, TSO_UP, 1);
            } else {
                MT(i, j, TSO_UP, 0) = i;
                MT(i, j, TSO_UP, 1) = j;
            }
        }
    for (int i = S - 1; i >= 0; --i)
        for (int j = 0; j < S; ++j) {
            if (i < S - 1 && !st->is_blocked[(i + 1) * S + j]) {
                MT(i, j, TSO_DOWN, 0) = MT(i + 1, j, TSO_DOWN, 0);
                MT(i, j, TSO_DOWN, 1) = MT(i + 1, j, TSO_DOWN, 1);
            } else {
                MT(i, j, TSO_DOWN, 0) = i;
                MT(i, j, TSO_DOWN, 1) = j;
            }
        }
    for (int i = 0; i < S; ++i)
        for (int j = 0; j < S; ++j) {
            if (j > 0 && !st->is_blocked[i * S + j - 1]) {
                MT(i, j, TSO_LEFT, 0) = MT(i, j - 1, TSO_LEFT, 0);
                MT(i, j, TSO_LEFT, 1) = MT(i, j - 1, TSO_LEFT, 1);
            } else {
                MT(i, j, TSO_LEFT, 0) = i;
                MT(i, j, TSO_LEFT, 1) = j;
            }
        }
    for (int i = 0; i < S; ++i)
        for (int j = S - 1; j >= 0; --j) {
            if (j < S - 1 && !st->is_blocked[i * S + j + 1]) {
                MT(i, j, TSO_RIGHT, 0) = MT(i, j + 1, TSO_RIGHT, 0);
                MT(i, j, TSO_RIGHT, 1) = MT(i, j + 1, TSO_RIGHT, 1);
            } else {
                MT(i, j, TSO_RIGHT, 0) = i;
                MT(i, j, TSO_RIGHT, 1) = j;
            }
        }
#undef MT
}

/* state.py:47-73 */
tso_state *tso_new(int size, int n_blocked, const int *blocked_rc, int n_tiles,
                   const int *init_rc, int n_targets, const int *tgt_rc, int multi_color) {
    tso_state *st = (tso_state *)calloc(1, sizeof(tso_state));
    st->size = size;
    st->n_tiles = n_tiles;
    st->n_targets = n_targets;
    st->multi_color = multi_color;
    st->is_blocked = (uint8_t *)calloc((size_t)size * size + 1, 1);
    st->move_to = (int *)malloc(sizeof(int) * ((size_t)size * size * 8 + 1));
    st->cur = (int *)malloc(sizeof(int) * (2 * (size_t)n_tiles + 1));
    st->tgt = (int *)malloc(sizeof(int) * (2 * (size_t)n_targets + 1));
    for (int b = 0; b < n_blocked; ++b)
        st->is_blocked[blocked_rc[2 * b] * size + blocked_rc[2 * b + 1]] = 1;
    memcpy(st->cur, init_rc, sizeof(int) * 2 * (size_t)n_tiles);
    memcpy(st->tgt, tgt_rc, sizeof(int) * 2 * (size_t)n_targets);
    build_slide_table(st);
    return st;
}

void tso_free(tso_state *st) {
    if (!st) return;
    free(st->is_blocked);
    free(st->move_to);
    free(st->cur);
    free(st->tgt);
    free(st);
}

/* state.py:172-186.  multi: ordered list equality (length mismatch => False).
 * single: set equality (duplicates collapse on both sides). */
int tso_is_won(const tso_state *st) {
    if (st->multi_color) {
        if (st->n_tiles != st->n_targets) return 0;
        for (int i = 0; i < 2 * st->n_tiles; ++i)
            if (st->cur[i] != st->tgt[i]) return 0;
        return 1;
    }
    for (int i = 0; i < st->n_tiles; ++i) {
        int hit = 0;
        for (int j = 0; j < st->n_targets && !hit; ++j)
            hit = st->cur[2 * i] == st->tgt[2 * j] && st->cur[2 * i + 1] == st->tgt[2 * j + 1];
        if (!hit) return 0;
    }
    for (int j = 0; j < st->n_targets; ++j) {
        int hit = 0;
        for (int i = 0; i < st->n_tiles && !hit; ++i)
            hit = st->cur[2 * i] == st->tgt[2 * j] && st->cur[2 * i + 1] == st->tgt[2 * j + 1];
        if (!hit) return 0;
    }
    return 1;
}

/* state.py:120-170.  Processing order = ascending key (stable insertion sort; the
 * reference's np.argsort tie order is irrelevant for well-formed states, SURVEY 7.0).
 * Each tile takes its wall-only destination from the slide table, then steps back one
 * cell at a time while that cell was already taken during this move. */
int tso_move(tso_state *st, int move) {
    const int S = st->size, T = st->n_tiles;
    int order_buf[TSO_STACK_TILES], key_buf[TSO_STACK_TILES], used_buf[2 * TSO_STACK_TILES];
    int *order = order_buf, *key = key_buf, *used = used_buf;
    if (T > TSO_STACK_TILES) {
        order = (int *)malloc(sizeof(int) * (size_t)T);
        key = (int *)malloc(sizeof(int) * (size_t)T);
        used = (int *)malloc(sizeof(int) * 2 * (size_t)T);
    }
    int n_used = 0;
    for (int i = 0; i < T; ++i) {
        int r = st->cur[2 * i], c = st->cur[2 * i + 1];
        key[i] = move == TSO_UP ? r : move == TSO_DOWN ? -r : move == TSO_LEFT ? c : -c;
        order[i] = i;
    }
    for (int a = 1; a < T; ++a) {
        int v = order[a], b = a - 1;
        while (b >= 0 && key[order[b]] > key[v]) {
            order[b + 1] = order[b];
            --b;
        }
        order[b + 1] = v;
    }
    for (int n = 0; n < T; ++n) {
        int i = order[n];
        int r = st->cur[2 * i], c = st->cur[2 * i + 1];
        const int *dst = &st->move_to[(((r * S) + c) * 4 + move) * 2];
        r = dst[0];
        c = dst[1];
        for (;;) {
            int taken = 0;
            for (int u = 0; u < n_used && !taken; ++u)
                taken = used[2 * u] == r && used[2 * u + 1] == c;
            if (!taken) break;
            if (move == TSO_UP) r += 1;
            else if (move == TSO_DOWN) r -= 1;
            else if (move == TSO_LEFT) c += 1;
            else c -= 1;
        }
        st->cur[2 * i] = r;
        st->cur[2 * i + 1] = c;
        used[2 * n_used] = r;
        used[2 * n_used + 1] = c;
        ++n_used;
    }
    if (T > TSO_STACK_TILES) {
        free(order);
        free(key);
        free(used);
    }
    return tso_is_won(st);
}

void tso_get_locations(const tso_state *st, int *out_rc) {
    memcpy(out_rc, st->cur, sizeof(int) * 2 * (size_t)st->n_tiles);
}

void tso_set_locations(tso_state *st, const int *rc) {
    memcpy(st->cur, rc, sizeof(int) * 2 * (size_t)st->n_tiles);
}

void tso_get_move_to(const tso_state *st, int *out) {
    memcpy(out, st->move_to, sizeof(int) * (size_t)st->size * st->size * 8);
}

/* state.py:188-211 -- float32 [S,S,3], HWC; later indices overwrite earlier ones. */
void tso_observe(const tso_state *st, float *out) {
    const int S = st->size;
    memset(out, 0, sizeof(float) * (size_t)S * S * 3);
    for (int i = 0; i < S * S; ++i) out[3 * i] = st->is_blocked[i] ? 1.0f : 0.0f;
    for (int i = 0; i < st->n_tiles; ++i)
        out[3 * (st->cur[2 * i] * S + st->cur[2 * i + 1]) + 1] = st->multi_color ? (float)(i + 1) : 1.0f;
    for (int i = 0; i < st->n_targets; ++i)
        out[3 * (st->tgt[2 * i] * S + st->tgt[2 * i + 1]) + 2] = st->multi_color ? (float)(i + 1) : 1.0f;
}

/* environment.py:149-171 -- bit d set when move d changes any tile position. */
int tso_valid_moves(const tso_state *st) {
    int mask = 0;
    int *save = (int *)malloc(sizeof(int) * (2 * (size_t)st->n_tiles + 1));
    tso_state tmp = *st;
    tmp.cur = (int *)malloc(sizeof(int) * (2 * (size_t)st->n_tiles + 1));
    memcpy(save, st->cur, sizeof(int) * 2 * (size_t)st->n_tiles);
    for (int d = 0; d < 4; ++d) {
        memcpy(tmp.cur, save, sizeof(int) * 2 * (size_t)st->n_tiles);
        tso_move(&tmp, d);
        if (memcmp(tmp.cur, save, sizeof(int) * 2 * (size_t)st->n_tiles) != 0) mask |= 1 << d;
    }
    free(tmp.cur);
    free(save);
    return mask;
}

/*
 * Batched scripted rollout: N independent environments, K steps each, driven by the
 * loop `obs, done, info = env.step(a); if done and auto_reset: env.reset()` of
 * environment.py:82-143.
 *
 *   blocked  u8 [N][S*S]      tiles/targets  u8 [N][T][2], [N][NT][2]   (row, col)
 *   actions  u8 [K][N]
 *   out_pos  i16[K][N][T][2]  positions after the move, BEFORE any auto-reset
 *   out_flags u8[K][N]        TSO_F_* bits
 *   out_count i32[K][N]       info['step_count'] (pre-increment, environment.py:128)
 *   out_reward f32[K][N]      repo-defined: won ? r_win : invalid ? r_invalid : r_step; stale => 0
 * Without auto_reset a finished environment is frozen and reports DONE|STALE.
 * Returns 0.
 */
int tso_rollout(int S, int T, int NT, int multi_color, long N, int K, const uint8_t *blocked,
                const uint8_t *tiles, const uint8_t *targets, const uint8_t *actions,
                int max_steps, int auto_reset, float r_win, float r_step, float r_invalid,
                int16_t *out_pos, uint8_t *out_flags, int32_t *out_count, float *out_reward,
                int16_t *final_pos, int32_t *final_count) {
    int *brc = (int *)malloc(sizeof(int) * (2 * (size_t)S * S + 2));
    int *irc = (int *)malloc(sizeof(int) * (2 * (size_t)T + 2));
    int *trc = (int *)malloc(sizeof(int) * (2 * (size_t)NT + 2));
    int *prev = (int *)malloc(sizeof(int) * (2 * (size_t)T + 2));
    for (long n = 0; n < N; ++n) {
        int nb = 0;
        for (int cell = 0; cell < S * S; ++cell)
            if (blocked[n * S * S + cell]) {
                brc[2 * nb] = cell / S;
                brc[2 * nb + 1] = cell % S;
                ++nb;
            }
        for (int i = 0; i < 2 * T; ++i) irc[i] = tiles[n * 2 * T + i];
        for (int i = 0; i < 2 * NT; ++i) trc[i] = targets[n * 2 * NT + i];
        /* reset(): environment.py:89-97 */
        tso_state *st = tso_new(S, nb, brc, T, irc, NT, trc, multi_color);
        int step_count = 0, done = 0;
        for (int k = 0; k < K; ++k) {
            const long o = (long)k * N + n;
            uint8_t flags = 0;
            float reward = 0.0f;
            int info_count = step_count;
            if (done) { /* environment.py:113-114 raises; the batch freezes instead */
                flags = TSO_F_DONE | TSO_F_STALE;
            } else {
                memcpy(prev, st->cur, sizeof(int) * 2 * (size_t)T);
                int won = tso_move(st, actions[o]);                       /* :123 */
                int invalid = memcmp(prev, st->cur, sizeof(int) * 2 * (size_t)T) == 0; /* :129 */
                if (won) { done = 1; flags |= TSO_F_WON; }                  /* :133-135 */
                if (invalid) flags |= TSO_F_INVALID;
                step_count += 1;                                           /* :138 */
                if (step_count >= max_steps) { done = 1; flags |= TSO_F_TIMEOUT; } /* :139-141 */
                if (done) flags |= TSO_F_DONE;
                reward = won ? r_win : (invalid ? r_invalid : r_step);
            }
            if (out_pos)
                for (int i = 0; i < 2 * T; ++i) out_pos[o * 2 * T + i] = (int16_t)st->cur[i];
            if (out_flags) out_flags[o] = flags;
            if (out_count) out_count[o] = info_count;
            if (out_reward) out_reward[o] = reward;
            if (done && auto_reset) { /* reset(): environment.py:89-97 */
                tso_set_locations(st, irc);
                step_count = 0;
                done = 0;
            }
        }
        if (final_pos)
            for (int i = 0; i < 2 * T; ++i) final_pos[n * 2 * T + i] = (int16_t)st->cur[i];
        if (final_count) final_count[n] = step_count;
        tso_free(st);
    }
    free(brc);
    free(irc);
    free(trc);
    free(prev);
    return 0;
}

/* ------------------------------------------------------------------------------------
 * CPU breadth-first search over tso_move (no reference counterpart: parity unpinned;
 * SURVEY 8(c) lists known answers obtained by running the reference move in a BFS).
 * Canonical key: ordered positions (multi) or sorted positions (single), cell index
 * r*S+c, 8 bits per tile (T <= 8).  Returns the number of reachable states; fills
 * level_counts[d] with the number of NEW states first seen at depth d and *solve_depth
 * with the first depth holding a won state reached by a move (-1 if none).  out_states
 * gets the visited keys sorted; out_by_level (optional) gets them level after level, so
 * the keys of depth d are the level_counts[d] that follow those of depths 0..d-1.
 * ---------------------------------------------------------------------------------- */
static uint64_t bfs_key(const tso_state *st) {
    int T = st->n_tiles, S = st->size;
    uint8_t cells[8];
    for (int i = 0; i < T; ++i) cells[i] = (uint8_t)(st->cur[2 * i] * S + st->cur[2 * i + 1]);
    if (!st->multi_color)
        for (int a = 1; a < T; ++a) {
            uint8_t v = cells[a];
            int b = a - 1;
            while (b >= 0 && cells[b] > v) { cells[b + 1] = cells[b]; --b; }
            cells[b + 1] = v;
        }
    uint64_t k = 0;
    for (int i = 0; i < T; ++i) k |= (uint64_t)cells[i] << (8 * i);
    return k;
}

static void bfs_unkey(tso_state *st, uint64_t k) {
    for (int i = 0; i < st->n_tiles; ++i) {
        int cell = (int)((k >> (8 * i)) & 0xFF);
        st->cur[2 * i] = cell / st->size;
        st->cur[2 * i + 1] = cell % st->size;
    }
}

static int cmp_u64(const void *a, const void *b) {
    uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : x > y;
}

long tso_bfs(tso_state *st, int max_depth, long max_states, long *level_counts, int *solve_depth,
             uint64_t *out_states, uint64_t *out_by_level) {
    if (st->n_tiles > 8) return -1;
    uint64_t *visited = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(max_states + 4));
    uint64_t *frontier = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(max_states + 4));
    uint64_t *next = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(4 * max_states + 4));
    long n_vis = 0, n_front = 0;
    *solve_depth = -1;
    frontier[n_front++] = bfs_key(st);
    visited[n_vis++] = frontier[0];
    if (out_by_level) out_by_level[0] = frontier[0];
    level_counts[0] = 1;
    int depth = 0;
    while (n_front > 0 && depth < max_depth) {
        long n_next = 0;
        ++depth;
        for (long f = 0; f < n_front; ++f)
            for (int d = 0; d < 4; ++d) {
                bfs_unkey(st, frontier[f]);
                int won = tso_move(st, d);
                if (won && *solve_depth < 0) *solve_depth = depth;
                next[n_next++] = bfs_key(st);
            }
        qsort(next, (size_t)n_next, sizeof(uint64_t), cmp_u64);
        /* visited is kept sorted; keep the successors that are new */
        long n_new = 0;
        for (long i = 0; i < n_next; ++i) {
            if (i > 0 && next[i] == next[i - 1]) continue;
            if (bsearch(&next[i], visited, (size_t)n_vis, sizeof(uint64_t), cmp_u64)) continue;
            if (n_vis + n_new >= max_states) { n_new = -1; break; }
            frontier[n_new++] = next[i];
        }
        if (n_new < 0) { n_vis = -2; break; }
        if (out_by_level) memcpy(out_by_level + n_vis, frontier, sizeof(uint64_t) * (size_t)n_new);
        memcpy(visited + n_vis, frontier, sizeof(uint64_t) * (size_t)n_new);
        n_vis += n_new;
        qsort(visited, (size_t)n_vis, sizeof(uint64_t), cmp_u64);
        n_front = n_new;
        level_counts[depth] = n_new;
    }
    if (out_states && n_vis > 0) memcpy(out_states, visited, sizeof(uint64_t) * (size_t)n_vis);
    free(visited);
    free(frontier);
    free(next);
    return n_vis;
}
