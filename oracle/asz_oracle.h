/*
 * asz_oracle.h -- CPU oracle for the AlphaSnake-Zero self-play hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This is a plain-C restatement of the reference's
 * algorithm (Fool-Yang/AlphaSnake-Zero, code/utils/{game,agent,mp_game_runner,
 * alpha_nnet}.py).  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load it, and only as the checker or
 * the timed CPU baseline -- never on the product path.
 *
 * Parity pin: the restatement is checked against the reference itself, executed
 * in the build container, through the golden fixtures in tests/golden/ (made by
 * tests/golden/make_golden.py, which imports /root/reference/code unmodified).
 * The value network has no runnable reference here (TensorFlow absent), so the
 * net restatement (oracle/net_oracle.py) is "parity unpinned" against TF.
 */
#ifndef ASZ_ORACLE_H
#define ASZ_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OG_MAX_SNAKES 8
#define OG_MAX_SIDE 19
#define OG_MAX_CELLS (OG_MAX_SIDE * OG_MAX_SIDE)
#define OG_MAX_SEG (OG_MAX_CELLS + 8)

typedef struct ogame ogame;

/* --- single game (game.py) ------------------------------------------------ */
ogame *og_new(int H, int W, int S, int health_dec);
void og_free(ogame *g);
ogame *og_clone(const ogame *g); /* Game.subgame, game.py:266-276 (no spawn in subgames is the caller's job) */
/* explicit layout (replay): start_yx[2*S], last_moves[S], food_yx[2*n_food] */
void og_init_explicit(ogame *g, const int *start_yx, const int *last_moves, const int *food_yx, int n_food);
/* native layout from the engine's counter-based RNG (Philox4x32-10) */
void og_init_native(ogame *g, uint64_t seed, uint32_t game_id, uint32_t episode);
/* spawn_mode: 0 = no spawn (sub-games), 1 = replay (spawn_cell = y*W+x or -1), 2 = native Philox.
 * moves[] has one entry per LIVE snake in live-list order (game.py:90-92).
 * returns 1 when the game ended (rewards final), else 0. */
int og_tic(ogame *g, const int *moves, int spawn_mode, int spawn_cell, uint32_t chance_thresh, uint64_t seed);
int og_n_live(const ogame *g);
void og_live_ids(const ogame *g, int *out);
/* plane for the k-th live snake: (2H-1)*(2W-1)*3 float32, C order NHWC (game.py:215-257) */
void og_make_state(const ogame *g, int k, float *out);
/* canonical dump, all int32:
 *  snake[S][6] = alive, health, length, last_move, head_cell(or -1 when off board / dead), reward(0 none, 1, -1)
 *  owner[H*W] (-1 none), dist[H*W] (max dist-from-tail of the segments on the cell; 0 none), food[H*W] 0/1
 *  counters[8] = wall, body, head, starve, food_eaten, game_length, episode, game_id */
void og_dump(const ogame *g, int32_t *snake, int32_t *owner, int32_t *dist, int32_t *food, int32_t *counters);
void og_load_dump(ogame *g, const int32_t *snake, const int32_t *owner, const int32_t *dist, const int32_t *food,
                  const int32_t *counters);
void og_set_ids(ogame *g, uint32_t game_id, uint32_t episode);

/* --- RNG / hashing shared by definition with the engine ------------------- */
void og_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t out[4]);
/* 128-bit key of a plane: order-free sum over pixels whose triple differs from the wall triple */
void og_plane_key(const float *plane, int n_pix, uint64_t key[2]);
/* deterministic stand-in for the value network (stub), includes no obstacle mask */
void og_stub_value(const uint64_t key[2], float v[3]);
/* AlphaNNet.v obstacle mask (alpha_nnet.py:63-76), numpy>=2 semantics (float32 compare) */
void og_obstacle_mask(const float *plane, int H, int W, float v[3]);

/* --- lockstep env batch (config 2 workload: random actions, encode, auto reset) */
typedef struct {
  uint64_t steps;          /* tics executed */
  uint64_t planes;         /* planes encoded */
  uint64_t episodes;       /* games finished */
  uint64_t plane_checksum; /* order-free sum of og_plane_key()[0] over every plane written */
  uint64_t counters[6];    /* wall, body, head, starve, food_eaten, game_length of finished games */
} oenv_stats;
/* runs G games for `tics` lockstep tics with n_threads OpenMP threads; games is an array of G ogame* (may be NULL to
 * allocate internally and discard).  encode != 0 => every live snake's plane is produced each tic. */
void oenv_run(ogame **games, int G, int H, int W, int S, int health_dec, uint32_t chance_thresh, uint64_t seed,
              int tics, int encode, int n_threads, oenv_stats *stats);
/* og_make_state of every live snake of G games, dense rows of (2H-1)*(2W-1)*3 floats in (game, snake id) order, with
 * ids[r] = game * 8 + snake id; games share one shape.  A NULL entry of games emits no rows (a finished game that was not
 * restarted).  Threads split the games.  planes / ids NULL: rows are only counted.  Returns the number of rows. */
int oenv_encode(ogame **games, int G, int n_threads, float *planes, int32_t *ids);

/* --- search (agent.py + mp_game_runner.py:79-115) -------------------------- */
typedef struct oagent oagent;
typedef void (*og_value_fn)(void *ctx, const float *planes, int n, int H, int W, float *v_out);
oagent *oa_new(double softmax_base, int training, int max_depth, int max_breadth, og_value_fn fn, void *ctx);
void oa_free(oagent *a);
void oa_clear(oagent *a);
void oa_set_rhat_mode(oagent *a, int before_backups);   /* 0 = reference order (default), 1 = all r-hat before the step's backups */
/* trace: one u8 per (epoch, step, subgame, snake id): in replay mode read, in native mode written.
 * Layout: moves[((epoch*max_steps + step)*n_sub_abs + abs_sub)*S + snake], 255 = no row.  root_moves[n_rows].
 * mode 0: sample with Philox(seed; root_turn, epoch, step, abs_sub, snake); mode 1: replay from the trace. */
typedef struct {
  int mode;
  uint64_t seed;
  uint32_t root_turn;
  int max_steps;
  int total_games;       /* G of the runner: sub-game slots are game_id*parallel + sibling, finished games keep theirs */
  uint8_t *tree_moves;   /* size epochs*max_steps*(total_games*parallel)*S */
  uint8_t *root_moves;   /* size n_rows */
} oa_trace;
/* games: n_games root games (ids = position).  Writes moves_out[n_rows] and q_out[n_rows*3] in ids order
 * (game order then live-list order, mp_game_runner.py:40-42).  Returns n_rows. */
int oa_make_moves(oagent *a, ogame **games, int n_games, oa_trace *tr, int *moves_out, float *q_out);
/* table inspection */
int oa_table_size(const oagent *a);
/* copies up to cap entries: key[2*i..], Q/W/N [3*i..], age[i]; returns count */
int oa_table_dump(const oagent *a, int cap, uint64_t *keys, float *Q, float *Wt, float *N, int32_t *age);
uint64_t oa_stat(const oagent *a, int which); /* 0 evals, 1 node visits, 2 hits, 3 subgames, 4 subgame tics */
/* training records (agent.py:93-97): planes and aliased Q rows */
int oa_n_records(const oagent *a);
void oa_get_record(const oagent *a, int i, float *plane, float *q);

void og_softermax(const float z[3], double base, float out[3]);
int og_argmax3(const float z[3]);
int og_choice3(const float p[3], double u);

#ifdef __cplusplus
}
#endif
#endif
