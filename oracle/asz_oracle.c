/*
 * asz_oracle.c -- CPU oracle (plain C restatement of the reference algorithm).
 * TEST INFRASTRUCTURE ONLY -- see asz_oracle.h.  Citations are file:line in
 * /root/reference/code/utils/.
 *
 * Representation note: the oracle keeps every snake as an explicit segment
 * list (head first), exactly like the reference's linked list, and derives the
 * board sets from it.  The CUDA engine uses a different representation (one
 * (owner, dist-from-tail) stamp per cell); agreement between the two is the
 * point of the parity tests.
 */
#include "asz_oracle.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>

/* ------------------------------------------------------------------------ */
/* Philox4x32-10 (Salmon et al. 2011), counter = (c0..c3), key = seed         */
/* ------------------------------------------------------------------------ */
void og_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t out[4]) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static inline uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }

/* stream ids of the engine's counter-based RNG (third counter word) */
enum { RS_INIT = 0, RS_SPAWN = 1, RS_ACT_LO = 2, RS_ACT_HI = 3, RS_TREE = 4, RS_ROOT = 5 };

/* ------------------------------------------------------------------------ */
/* Game                                                                      */
/* ------------------------------------------------------------------------ */
typedef struct {
  int alive;
  int health;
  int length;              /* == number of segments (game.py:307,361) */
  int sy[OG_MAX_SEG];      /* segment 0 = head ... length-1 = tail */
  int sx[OG_MAX_SEG];
} osnake;

struct ogame {
  int H, W, S, health_dec;
  uint32_t game_id, episode;
  int last_move[OG_MAX_SNAKES];
  osnake sn[OG_MAX_SNAKES];        /* indexed by snake id */
  int live[OG_MAX_SNAKES];         /* live list, ascending id (game.py:37,191) */
  int n_live;
  uint8_t food[OG_MAX_CELLS];
  int reward[OG_MAX_SNAKES];       /* 0 none, +1, -1 (game.py:20,192,201) */
  int wall, body, head, starve, food_eaten, game_length; /* game.py:56-61 */
};

ogame *og_new(int H, int W, int S, int health_dec) {
  if (H < 3 || W < 3 || H > OG_MAX_SIDE || W > OG_MAX_SIDE || S < 1 || S > OG_MAX_SNAKES) return NULL;
  ogame *g = (ogame *)calloc(1, sizeof(ogame));
  g->H = H; g->W = W; g->S = S; g->health_dec = health_dec;
  return g;
}
void og_free(ogame *g) { free(g); }
ogame *og_clone(const ogame *g) {
  ogame *c = (ogame *)malloc(sizeof(ogame));
  memcpy(c, g, sizeof(ogame));
  /* game.py:268 constructs a fresh Game => counters restart at 0; rewards are copied (:275) */
  c->wall = c->body = c->head = c->starve = c->food_eaten = c->game_length = 0;
  return c;
}
void og_set_ids(ogame *g, uint32_t game_id, uint32_t episode) { g->game_id = game_id; g->episode = episode; }

static void og_clear(ogame *g) {
  memset(g->food, 0, sizeof g->food);
  memset(g->reward, 0, sizeof g->reward);
  g->wall = g->body = g->head = g->starve = g->food_eaten = g->game_length = 0;
  g->n_live = g->S;
  for (int i = 0; i < g->S; ++i) g->live[i] = i;
}

/* game.py:25-47 with the random draws supplied by the caller */
void og_init_explicit(ogame *g, const int *start_yx, const int *last_moves, const int *food_yx, int n_food) {
  og_clear(g);
  for (int i = 0; i < g->S; ++i) {
    osnake *s = &g->sn[i];
    s->alive = 1; s->health = 100; s->length = 3;      /* game.py:37: three stacked segments */
    for (int k = 0; k < 3; ++k) { s->sy[k] = start_yx[2 * i]; s->sx[k] = start_yx[2 * i + 1]; }
    g->last_move[i] = last_moves[i];
  }
  for (int i = 0; i < n_food; ++i) g->food[food_yx[2 * i] * g->W + food_yx[2 * i + 1]] = 1;
}

static void start_cells(int H, int W, int out[16]) {
  /* game.py:25-28, same order */
  int c[16] = {1, 1, H - 2, W - 2, H - 2, 1, 1, W - 2, 1, W / 2, H / 2, W - 2, H - 2, W / 2, H / 2, 1};
  memcpy(out, c, sizeof c);
}

void og_init_native(ogame *g, uint64_t seed, uint32_t game_id, uint32_t episode) {
  g->game_id = game_id; g->episode = episode;
  uint32_t u[8], v[8], w[8];
  og_philox(game_id, episode, RS_INIT, 0, seed, u); og_philox(game_id, episode, RS_INIT, 1, seed, u + 4);
  og_philox(game_id, episode, RS_INIT, 2, seed, v); og_philox(game_id, episode, RS_INIT, 3, seed, v + 4);
  og_philox(game_id, episode, RS_INIT, 4, seed, w); og_philox(game_id, episode, RS_INIT, 5, seed, w + 4);
  int cells[16]; start_cells(g->H, g->W, cells);
  int perm[8] = {0, 1, 2, 3, 4, 5, 6, 7};
  int start[16], lm[8], food[2 * (OG_MAX_SNAKES + 1)];
  static const int dy[4] = {-1, -1, 1, 1}, dx[4] = {-1, 1, -1, 1}; /* game.py:46-47 list order */
  for (int i = 0; i < g->S; ++i) {
    int j = i + (int)mulhi32(u[i], (uint32_t)(8 - i));   /* sample without replacement (game.py:25-29) */
    int t = perm[i]; perm[i] = perm[j]; perm[j] = t;
    start[2 * i] = cells[2 * perm[i]]; start[2 * i + 1] = cells[2 * perm[i] + 1];
    lm[i] = (int)(v[i] & 3u);                            /* game.py:30 */
  }
  int nf = 0;
  food[0] = g->H / 2; food[1] = g->W / 2; nf = 1;        /* game.py:43 */
  for (int i = 0; i < g->S; ++i) {
    int d = (int)(w[i] & 3u);
    food[2 * nf] = start[2 * i] + dy[d]; food[2 * nf + 1] = start[2 * i + 1] + dx[d]; ++nf;
  }
  og_init_explicit(g, start, lm, food, nf);
}

/* load a canonical dump (the format og_dump writes); segment order is rebuilt from the dist map:
 * the segment at distance d sits on the cell stamped (owner, d), or, when no cell carries d, on the
 * cell of segment d+1 (stacked tail). */
void og_load_dump(ogame *g, const int32_t *snake, const int32_t *owner, const int32_t *dist, const int32_t *food,
                  const int32_t *counters) {
  const int C = g->H * g->W;
  og_clear(g);
  g->n_live = 0;
  for (int c = 0; c < C; ++c) g->food[c] = (uint8_t)(food[c] != 0);
  for (int i = 0; i < g->S; ++i) {
    const int32_t *o = snake + 6 * i;
    osnake *s = &g->sn[i];
    s->alive = o[0]; s->health = o[1]; s->length = o[2];
    g->last_move[i] = o[3]; g->reward[i] = o[5];
    if (!s->alive) continue;
    g->live[g->n_live++] = i;
    int cell_of = o[4];
    for (int d = s->length; d >= 1; --d) {
      for (int c = 0; c < C; ++c) if (owner[c] == i && dist[c] == d) { cell_of = c; break; }
      int q = s->length - d;               /* head is segment 0 */
      s->sy[q] = cell_of / g->W; s->sx[q] = cell_of % g->W;
    }
  }
  g->wall = counters[0]; g->body = counters[1]; g->head = counters[2]; g->starve = counters[3];
  g->food_eaten = counters[4]; g->game_length = counters[5];
  g->episode = (uint32_t)counters[6]; g->game_id = (uint32_t)counters[7];
}

int og_n_live(const ogame *g) { return g->n_live; }
void og_live_ids(const ogame *g, int *out) { for (int i = 0; i < g->n_live; ++i) out[i] = g->live[i]; }

static inline int on_board(const ogame *g, int y, int x) { return y >= 0 && y < g->H && x >= 0 && x < g->W; }

/* game.py:87-205 */
int og_tic(ogame *g, const int *moves, int spawn_mode, int spawn_cell, uint32_t chance_thresh, uint64_t seed) {
  const int H = g->H, W = g->W;
  static const int DY[4] = {-1, 0, 1, 0}, DX[4] = {0, 1, 0, -1}; /* game.py:330-342 */
  /* 1. move (game.py:90-114; Snake.move :329-358) */
  for (int i = 0; i < g->n_live; ++i) {
    int id = g->live[i];
    osnake *s = &g->sn[id];
    int mv = (moves[i] + g->last_move[id] - 1) % 4;
    if (mv < 0) mv += 4;                       /* Python % is non-negative */
    g->last_move[id] = mv;
    int ny = s->sy[0] + DY[mv], nx = s->sx[0] + DX[mv];
    /* push the new head, drop the last segment: length stays */
    memmove(s->sy + 1, s->sy, sizeof(int) * (size_t)(s->length - 1));
    memmove(s->sx + 1, s->sx, sizeof(int) * (size_t)(s->length - 1));
    s->sy[0] = ny; s->sx[0] = nx;
  }
  /* 2. health (game.py:117-118) */
  for (int i = 0; i < g->n_live; ++i) g->sn[g->live[i]].health -= g->health_dec;
  /* 3. eat, first come in list order (game.py:121-127; Snake.grow :360-365) */
  for (int i = 0; i < g->n_live; ++i) {
    osnake *s = &g->sn[g->live[i]];
    int y = s->sy[0], x = s->sx[0];
    if (on_board(g, y, x) && g->food[y * W + x]) {
      g->food[y * W + x] = 0;
      s->health = 100;
      s->sy[s->length] = s->sy[s->length - 1]; s->sx[s->length] = s->sx[s->length - 1];
      s->length += 1;
      g->food_eaten += 1;
    }
  }
  /* 4. spawn (game.py:130-138). empty = on board, no head (of any snake still listed), no body, no food */
  if (spawn_mode != 0) {
    uint8_t occ[OG_MAX_CELLS];
    memcpy(occ, g->food, (size_t)(H * W));
    int n_food = 0;
    for (int c = 0; c < H * W; ++c) n_food += g->food[c];
    for (int i = 0; i < g->n_live; ++i) {
      const osnake *s = &g->sn[g->live[i]];
      for (int k = 0; k < s->length; ++k)
        if (on_board(g, s->sy[k], s->sx[k])) occ[s->sy[k] * W + s->sx[k]] = 1;
    }
    if (spawn_mode == 1) {
      if (spawn_cell >= 0) {
        if (occ[spawn_cell]) fprintf(stderr, "og_tic: replayed food cell %d is not empty\n", spawn_cell);
        g->food[spawn_cell] = 1;
      }
    } else if (chance_thresh != 0u) {   /* game.py:130 `if self.food_spawn_chance > 0.0`: threshold 0 = chance 0 = never */
      uint32_t r[4];
      og_philox(g->game_id, g->episode, RS_SPAWN, (uint32_t)g->game_length, seed, r);
      if (n_food == 0 || r[0] <= chance_thresh) {
        int n_empty = 0;
        for (int c = 0; c < H * W; ++c) n_empty += !occ[c];
        if (n_empty > 0) {
          int k = (int)mulhi32(r[1], (uint32_t)n_empty);
          for (int c = 0; c < H * W; ++c)
            if (!occ[c] && k-- == 0) { g->food[c] = 1; break; }
        }
      }
    }
  }
  /* 5. kill decisions (game.py:144-165): wall > body > head-on > starvation, one cause each */
  int kill[OG_MAX_SNAKES] = {0};
  for (int i = 0; i < g->n_live; ++i) {
    const osnake *s = &g->sn[g->live[i]];
    int y = s->sy[0], x = s->sx[0];
    if (!on_board(g, y, x)) { kill[i] = 1; g->wall += 1; continue; }
    int in_body = 0, shared = 0, lose = 0;
    for (int j = 0; j < g->n_live; ++j) {
      const osnake *t = &g->sn[g->live[j]];
      for (int k = 1; k < t->length; ++k)           /* bodies = non-head segments of every listed snake */
        if (t->sy[k] == y && t->sx[k] == x) in_body = 1;
      if (j != i && t->sy[0] == y && t->sx[0] == x) {
        shared = 1;
        if (s->length <= t->length) lose = 1;       /* game.py:158 */
      }
    }
    if (in_body) { kill[i] = 1; g->body += 1; }
    else if (shared) { if (lose) { kill[i] = 1; g->head += 1; } }  /* elif chain: no starvation check here */
    else if (s->health <= 0) { kill[i] = 1; g->starve += 1; }
  }
  /* 6. remove (game.py:167-192) */
  int n = 0;
  for (int i = 0; i < g->n_live; ++i) {
    int id = g->live[i];
    if (kill[i]) { g->sn[id].alive = 0; g->reward[id] = -1; }
    else g->live[n++] = id;
  }
  g->n_live = n;
  /* 7. terminate (game.py:197-205) */
  g->game_length += 1;
  if (g->n_live <= 1) {
    if (g->n_live == 1) g->reward[g->live[0]] = 1;
    return 1;
  }
  return 0;
}

/* game.py:215-257.  All arithmetic in double, one rounding to float32 (:257). */
void og_make_state(const ogame *g, int k, float *out) {
  const int H = g->H, W = g->W, GH = 2 * H - 1, GW = 2 * W - 1;
  static _Thread_local double board[OG_MAX_CELLS][3];
  static _Thread_local double grid[(2 * OG_MAX_SIDE - 1) * (2 * OG_MAX_SIDE - 1)][3];
  const osnake *you = &g->sn[g->live[k]];
  const int last_move = g->last_move[g->live[k]];
  for (int i = 0; i < GH * GW; ++i) { grid[i][0] = 0.0; grid[i][1] = 1.0; grid[i][2] = 0.0; }  /* :219 */
  for (int i = 0; i < H * W; ++i) board[i][0] = board[i][1] = board[i][2] = 0.0;              /* :224 */
  double length_minus_half = you->length - 0.5;                                               /* :229 */
  for (int i = 0; i < g->n_live; ++i) {
    const osnake *s = &g->sn[g->live[i]];
    board[s->sy[0] * W + s->sx[0]][0] = (s->length - length_minus_half) * 0.04;               /* :232 */
    int dist = 1;
    for (int q = s->length - 1; q >= 0; --q) {                                                /* :236-241 tail -> head */
      board[s->sy[q] * W + s->sx[q]][1] = dist * 0.02;
      dist += 1;
    }
  }
  for (int c = 0; c < H * W; ++c)
    if (g->food[c]) board[c][2] = (101 - you->health) * 0.01;                                 /* :243-244 */
  int hy = you->sy[0], hx = you->sx[0];
  board[hy * W + hx][0] = board[hy * W + hx][1] = board[hy * W + hx][2] = -1.0;                /* :248 */
  int cy = GH / 2, cx = GW / 2;
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < W; ++x) {
      double *d = grid[(y - hy + cy) * GW + (x - hx + cx)];                                   /* :249-251 */
      d[0] = board[y * W + x][0]; d[1] = board[y * W + x][1]; d[2] = board[y * W + x][2];
    }
  /* numpy.rot90(grid, k) on axes (0,1) (:257); output shape (GH,GW) for even k, (GW,GH) for odd k */
  int OH = (last_move & 1) ? GW : GH, OW = (last_move & 1) ? GH : GW;
  for (int i = 0; i < OH; ++i)
    for (int j = 0; j < OW; ++j) {
      int gy, gx;
      switch (last_move) {
        case 0: gy = i; gx = j; break;
        case 1: gy = j; gx = GW - 1 - i; break;
        case 2: gy = GH - 1 - i; gx = GW - 1 - j; break;
        default: gy = GH - 1 - j; gx = i; break;
      }
      const double *s = grid[gy * GW + gx];
      float *o = out + ((size_t)i * OW + j) * 3;
      o[0] = (float)s[0]; o[1] = (float)s[1]; o[2] = (float)s[2];
    }
}

void og_dump(const ogame *g, int32_t *snake, int32_t *owner, int32_t *dist, int32_t *food, int32_t *counters) {
  const int C = g->H * g->W;
  for (int c = 0; c < C; ++c) { owner[c] = -1; dist[c] = 0; food[c] = g->food[c]; }
  for (int i = 0; i < g->S; ++i) {
    const osnake *s = &g->sn[i];
    int32_t *o = snake + 6 * i;
    o[0] = s->alive; o[1] = s->alive ? s->health : 0; o[2] = s->alive ? s->length : 0;
    o[3] = g->last_move[i];
    o[4] = -1; o[5] = g->reward[i];
    if (!s->alive) continue;
    if (on_board(g, s->sy[0], s->sx[0])) o[4] = s->sy[0] * g->W + s->sx[0];
    int d = 1;
    for (int q = s->length - 1; q >= 0; --q, ++d) {
      if (!on_board(g, s->sy[q], s->sx[q])) continue;
      int c = s->sy[q] * g->W + s->sx[q];
      owner[c] = i; dist[c] = d;   /* tail -> head: later (nearer the head) wins, as in make_state */
    }
  }
  counters[0] = g->wall; counters[1] = g->body; counters[2] = g->head; counters[3] = g->starve;
  counters[4] = g->food_eaten; counters[5] = g->game_length; counters[6] = (int32_t)g->episode;
  counters[7] = (int32_t)g->game_id;
}

/* ------------------------------------------------------------------------ */
/* plane key, stub value, obstacle mask                                       */
/* ------------------------------------------------------------------------ */
static inline uint64_t fmix64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
  return k;
}
void og_plane_key(const float *plane, int n_pix, uint64_t key[2]) {
  uint64_t k0 = 0, k1 = 0;
  for (int p = 0; p < n_pix; ++p) {
    uint32_t a, b, c;
    memcpy(&a, plane + 3 * p, 4); memcpy(&b, plane + 3 * p + 1, 4); memcpy(&c, plane + 3 * p + 2, 4);
    if (a == 0u && b == 0x3F800000u && c == 0u) continue;   /* wall-valued pixels contribute nothing */
    uint64_t x = ((uint64_t)a << 32) | b, y = ((uint64_t)c << 32) | (uint32_t)p;
    k0 += fmix64(fmix64(y ^ 0x9E3779B97F4A7C15ULL) ^ x);
    k1 += fmix64(fmix64(x ^ 0xC2B2AE3D27D4EB4FULL) + y);
  }
  if (k0 == 0) k0 = 1;   /* 0 is the engine's empty-slot tag */
  key[0] = k0; key[1] = k1;
}
void og_stub_value(const uint64_t key[2], float v[3]) {
  for (int i = 0; i < 3; ++i) {
    uint32_t x = (uint32_t)((key[1] >> (16 * i)) & 0xFFFFu);
    v[i] = ((float)x - 32767.5f) * (1.0f / 32768.0f);
  }
}
/* alpha_nnet.py:63-76; threshold compared in float32 (NumPy >= 2 semantics, SURVEY D-11) */
void og_obstacle_mask(const float *plane, int H, int W, float v[3]) {
  int GH = 2 * H - 1, GW = 2 * W - 1;   /* square boards only reach here rotated; cy/cx from the array shape */
  int cy = GH / 2, cx = GW / 2;
  const float thr = 0.04f;
  if (plane[((size_t)cy * GW + (cx - 1)) * 3 + 1] >= thr) v[0] = -1.0f;
  if (plane[((size_t)(cy - 1) * GW + cx) * 3 + 1] >= thr) v[1] = -1.0f;
  if (plane[((size_t)cy * GW + (cx + 1)) * 3 + 1] >= thr) v[2] = -1.0f;
}

/* ------------------------------------------------------------------------ */
/* lockstep env batch (config-2 workload)                                     */
/* ------------------------------------------------------------------------ */
typedef struct {
  ogame **games; int g0, g1, H, W, S, health_dec; uint32_t chance_thresh; uint64_t seed; int tics, encode;
  oenv_stats st;
} oenv_job;

static void *oenv_worker(void *arg) {
  oenv_job *jb = (oenv_job *)arg;
  const int H = jb->H, W = jb->W, S = jb->S;
  const int n_pix = (2 * H - 1) * (2 * W - 1);
  oenv_stats *st = &jb->st;
  memset(st, 0, sizeof *st);
  float *plane = jb->encode ? (float *)malloc(sizeof(float) * 3 * (size_t)n_pix) : NULL;
  for (int gi = jb->g0; gi < jb->g1; ++gi) {
    ogame *g = jb->games ? jb->games[gi] : NULL;
    int own = 0;
    if (!g) { g = og_new(H, W, S, jb->health_dec); og_init_native(g, jb->seed, (uint32_t)gi, 0); own = 1; }
    for (int t = 0; t < jb->tics; ++t) {
      int mv[OG_MAX_SNAKES];
      uint32_t r[8];
      og_philox(g->game_id, g->episode, RS_ACT_LO, (uint32_t)g->game_length, jb->seed, r);
      if (S > 4) og_philox(g->game_id, g->episode, RS_ACT_HI, (uint32_t)g->game_length, jb->seed, r + 4);
      for (int i = 0; i < g->n_live; ++i) mv[i] = (int)mulhi32(r[g->live[i]], 3u);
      int ended = og_tic(g, mv, 2, -1, jb->chance_thresh, jb->seed);
      st->steps += 1;
      if (ended) {
        st->episodes += 1;
        st->counters[0] += (uint64_t)g->wall; st->counters[1] += (uint64_t)g->body;
        st->counters[2] += (uint64_t)g->head; st->counters[3] += (uint64_t)g->starve;
        st->counters[4] += (uint64_t)g->food_eaten; st->counters[5] += (uint64_t)g->game_length;
        og_init_native(g, jb->seed, g->game_id, g->episode + 1);
      }
      if (jb->encode) {
        for (int k = 0; k < g->n_live; ++k) {
          uint64_t key[2];
          og_make_state(g, k, plane);
          og_plane_key(plane, n_pix, key);
          st->plane_checksum += key[0];
          st->planes += 1;
        }
      }
    }
    if (own) og_free(g);
  }
  free(plane);
  return NULL;
}

void oenv_run(ogame **games, int G, int H, int W, int S, int health_dec, uint32_t chance_thresh, uint64_t seed,
              int tics, int encode, int n_threads, oenv_stats *st) {
  memset(st, 0, sizeof *st);
  if (n_threads < 1) n_threads = 1;
  if (n_threads > G) n_threads = G > 0 ? G : 1;
  oenv_job *jobs = (oenv_job *)calloc((size_t)n_threads, sizeof(oenv_job));
  pthread_t *th = (pthread_t *)calloc((size_t)n_threads, sizeof(pthread_t));
  for (int t = 0; t < n_threads; ++t) {
    oenv_job *jb = &jobs[t];
    jb->games = games; jb->g0 = (int)((long long)G * t / n_threads); jb->g1 = (int)((long long)G * (t + 1) / n_threads);
    jb->H = H; jb->W = W; jb->S = S; jb->health_dec = health_dec; jb->chance_thresh = chance_thresh; jb->seed = seed;
    jb->tics = tics; jb->encode = encode;
    if (t > 0) pthread_create(&th[t], NULL, oenv_worker, jb);
  }
  oenv_worker(&jobs[0]);
  for (int t = 1; t < n_threads; ++t) pthread_join(th[t], NULL);
  for (int t = 0; t < n_threads; ++t) {
    st->steps += jobs[t].st.steps; st->planes += jobs[t].st.planes; st->episodes += jobs[t].st.episodes;
    st->plane_checksum += jobs[t].st.plane_checksum;
    for (int k = 0; k < 6; ++k) st->counters[k] += jobs[t].st.counters[k];
  }
  free(jobs); free(th);
}

/* batch encode: every live snake's og_make_state plane of G games, dense rows in (game, snake id) order */
typedef struct {
  ogame **games; int g0, g1; const int *row0; float *planes; int32_t *ids; size_t plen;
} oenc_job;

static void *oenc_worker(void *arg) {
  const oenc_job *jb = (const oenc_job *)arg;
  for (int gi = jb->g0; gi < jb->g1; ++gi) {
    const ogame *g = jb->games[gi];
    if (!g) continue;
    for (int k = 0; k < g->n_live; ++k) {   /* the live list is in ascending snake id */
      const size_t r = (size_t)jb->row0[gi] + (size_t)k;
      og_make_state(g, k, jb->planes + r * jb->plen);
      jb->ids[r] = (int32_t)(gi * 8 + g->live[k]);
    }
  }
  return NULL;
}

int oenv_encode(ogame **games, int G, int n_threads, float *planes, int32_t *ids) {
  int *row0 = (int *)malloc(sizeof(int) * (size_t)(G > 0 ? G : 1));
  int n = 0;
  size_t plen = 0;
  for (int gi = 0; gi < G; ++gi) {
    row0[gi] = n;
    if (!games[gi]) continue;
    n += games[gi]->n_live;
    plen = (size_t)3 * (2 * games[gi]->H - 1) * (2 * games[gi]->W - 1);
  }
  if (planes && ids && n > 0) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > G) n_threads = G;
    oenc_job *jobs = (oenc_job *)calloc((size_t)n_threads, sizeof(oenc_job));
    pthread_t *th = (pthread_t *)calloc((size_t)n_threads, sizeof(pthread_t));
    for (int t = 0; t < n_threads; ++t) {
      oenc_job *jb = &jobs[t];
      jb->games = games; jb->g0 = (int)((long long)G * t / n_threads); jb->g1 = (int)((long long)G * (t + 1) / n_threads);
      jb->row0 = row0; jb->planes = planes; jb->ids = ids; jb->plen = plen;
      if (t > 0) pthread_create(&th[t], NULL, oenc_worker, jb);
    }
    oenc_worker(&jobs[0]);
    for (int t = 1; t < n_threads; ++t) pthread_join(th[t], NULL);
    free(jobs); free(th);
  }
  free(row0);
  return n;
}

/* ------------------------------------------------------------------------ */
/* softermax / argmaxs / choice                                               */
/* ------------------------------------------------------------------------ */
/* agent.py:114-122, float32 throughout (NumPy >= 2 promotion), left-to-right sum */
void og_softermax(const float z[3], double base, float out[3]) {
  float n[3];
  const float b = (float)base;
  for (int i = 0; i < 3; ++i) n[i] = powf(b, atanhf(z[i]));
  float sigma = 0.0f;
  sigma = sigma + n[0]; sigma = sigma + n[1]; sigma = sigma + n[2];
  if (sigma == 0.0f) { out[0] = out[1] = out[2] = (float)(1.0 / 3.0); return; }
  for (int i = 0; i < 3; ++i) out[i] = n[i] / sigma;
}
/* agent.py:124-137: strict '>' ; ties fall toward the higher index */
int og_argmax3(const float z[3]) {
  if (z[0] > z[1]) return (z[0] > z[2]) ? 0 : 2;
  return (z[1] > z[2]) ? 1 : 2;
}
/* numpy.random.choice(3, p): cdf = cumsum(float64 p); cdf /= cdf[-1]; searchsorted(cdf, u, 'right') */
int og_choice3(const float p[3], double u) {
  double c0 = (double)p[0], c1 = c0 + (double)p[1], c2 = c1 + (double)p[2];
  c0 /= c2; c1 /= c2;
  int idx = 0;
  if (c0 <= u) idx = 1;
  if (c1 <= u) idx = 2;
  return idx;   /* cdf[2] == 1.0 > u always */
}

/* ------------------------------------------------------------------------ */
/* Search: Agent.make_moves + MCTSAgent.make_moves + MCTSMPGameRunner.run     */
/* ------------------------------------------------------------------------ */
typedef struct {
  uint64_t key[2];
  float Q[3], Wt[3], N[3];
  int32_t age;
  int pending;       /* cached_values[key] is None (agent.py:184) */
  int used;
  float *plane;      /* exact bytes, kept to detect 128-bit key aliasing */
} oentry;

struct oagent {
  double base;
  int training, D, breadth;
  og_value_fn fn; void *ctx;
  oentry **tab; size_t cap, n;   /* open addressing over pointers: entries never move */
  uint64_t stats[8];
  uint64_t alias_errors;
  int rhat_before_backups;   /* 0 = reference (agent.py:214: Q_row is a live alias), 1 = every r-hat of a step from the values before the
                                step's backups (what a parallel implementation computes); see oa_set_rhat_mode */
  /* records */
  float *rec_planes; float *rec_q; int n_rec, cap_rec, plane_len;
};

static void stub_value_fn(void *ctx, const float *planes, int n, int H, int W, float *v) {
  (void)ctx;
  const int n_pix = (2 * H - 1) * (2 * W - 1);
  for (int i = 0; i < n; ++i) {
    uint64_t key[2];
    og_plane_key(planes + (size_t)i * n_pix * 3, n_pix, key);
    og_stub_value(key, v + 3 * i);
    og_obstacle_mask(planes + (size_t)i * n_pix * 3, H, W, v + 3 * i);
  }
}

oagent *oa_new(double base, int training, int D, int breadth, og_value_fn fn, void *ctx) {
  oagent *a = (oagent *)calloc(1, sizeof(oagent));
  a->base = base; a->training = training; a->D = D; a->breadth = breadth;
  a->fn = fn ? fn : stub_value_fn; a->ctx = ctx;
  a->cap = 1u << 12; a->tab = (oentry **)calloc(a->cap, sizeof(oentry *));
  return a;
}
static void tab_free_entries(oagent *a) {
  for (size_t i = 0; i < a->cap; ++i) if (a->tab[i]) { free(a->tab[i]->plane); free(a->tab[i]); a->tab[i] = NULL; }
}
void oa_clear(oagent *a) {   /* agent.py:140-147 */
  tab_free_entries(a);
  a->n = 0; a->n_rec = 0;
}
void oa_free(oagent *a) {
  if (!a) return;
  tab_free_entries(a); free(a->tab); free(a->rec_planes); free(a->rec_q); free(a);
}
static void tab_place(oagent *a, oentry *e) {
  size_t h = (size_t)(e->key[0] ^ e->key[1]) & (a->cap - 1);
  while (a->tab[h]) h = (h + 1) & (a->cap - 1);
  a->tab[h] = e;
}
static oentry *tab_find(oagent *a, const uint64_t key[2], int insert) {
  if (insert && (a->n + 1) * 2 > a->cap) {   /* grow + rehash (pointers stay valid) */
    size_t ocap = a->cap; oentry **old = a->tab;
    a->cap = ocap * 2; a->tab = (oentry **)calloc(a->cap, sizeof(oentry *));
    for (size_t i = 0; i < ocap; ++i) if (old[i]) tab_place(a, old[i]);
    free(old);
  }
  size_t h = (size_t)(key[0] ^ key[1]) & (a->cap - 1);
  while (a->tab[h]) {
    if (a->tab[h]->key[0] == key[0] && a->tab[h]->key[1] == key[1]) return a->tab[h];
    h = (h + 1) & (a->cap - 1);
  }
  if (!insert) return NULL;
  oentry *e = (oentry *)calloc(1, sizeof(oentry));
  e->used = 1; e->key[0] = key[0]; e->key[1] = key[1];
  a->tab[h] = e; a->n += 1;
  return e;
}
static void tab_evict(oagent *a) {   /* agent.py:101-110: delete keys with age > D */
  size_t ocap = a->cap; oentry **old = a->tab;
  a->tab = (oentry **)calloc(a->cap, sizeof(oentry *)); a->n = 0;
  for (size_t i = 0; i < ocap; ++i) if (old[i]) {
    if (old[i]->age > a->D) { free(old[i]->plane); free(old[i]); continue; }
    tab_place(a, old[i]); a->n += 1;
  }
  free(old);
}

int oa_table_size(const oagent *a) { return (int)a->n; }
int oa_table_dump(const oagent *a, int cap, uint64_t *keys, float *Q, float *Wt, float *N, int32_t *age) {
  int n = 0;
  for (size_t i = 0; i < a->cap && n < cap; ++i) if (a->tab[i]) {
    const oentry *e = a->tab[i];
    keys[2 * n] = e->key[0]; keys[2 * n + 1] = e->key[1];
    for (int k = 0; k < 3; ++k) { Q[3 * n + k] = e->Q[k]; Wt[3 * n + k] = e->Wt[k]; N[3 * n + k] = e->N[k]; }
    age[n] = e->age; ++n;
  }
  return n;
}
/* The reference computes r-hat = pmf . Q_row row by row inside the backup loop, and Q_row aliases the live table entry
 * (agent.py:180,214): when a row's current state is an ancestor on the path of an EARLIER row of the same step, it sees that
 * row's backup.  mode 1 computes every r-hat of a step before any backup of the step (the order-free definition the CUDA
 * kernels implement); it exists so that tests can separate this one documented deviation from everything else. */
void oa_set_rhat_mode(oagent *a, int before_backups) { a->rhat_before_backups = before_backups ? 1 : 0; }

uint64_t oa_stat(const oagent *a, int which) { return which == 7 ? a->alias_errors : a->stats[which & 7]; }
int oa_n_records(const oagent *a) { return a->n_rec; }
void oa_get_record(const oagent *a, int i, float *plane, float *q) {
  memcpy(plane, a->rec_planes + (size_t)i * a->plane_len, sizeof(float) * (size_t)a->plane_len);
  memcpy(q, a->rec_q + 3 * (size_t)i, sizeof(float) * 3);
}

typedef struct { oentry **e; int *mv; int n; } opath;   /* MCTSAgent.keys / .moves (agent.py:158-159) */

/* back one value up every (key, move) of a path, last to first (agent.py:67-72, :215-220) */
static void backup(opath *p, float r) {
  for (int j = p->n - 1; j >= 0; --j) {
    oentry *e = p->e[j]; int m = p->mv[j];
    e->N[m] += 1.0f; e->Wt[m] += r; e->Q[m] = e->Wt[m] / e->N[m];
  }
}

int oa_make_moves(oagent *a, ogame **games, int n_games, oa_trace *tr, int *moves_out, float *q_out) {
  if (n_games <= 0) return 0;
  const int H = games[0]->H, W = games[0]->W, S = games[0]->S;
  const int n_pix = (2 * H - 1) * (2 * W - 1), plen = 3 * n_pix;
  a->plane_len = plen;
  /* agent.py:30-31 */
  for (size_t i = 0; i < a->cap; ++i) if (a->tab[i]) a->tab[i]->age += 1;
  int parallel = 8;
  if (a->breadth < parallel) parallel = a->breadth;          /* agent.py:32-34 */
  const int epochs = a->breadth / parallel;                   /* agent.py:37 */
  const int n_sub = n_games * parallel;
  ogame **sub = (ogame **)calloc((size_t)n_sub, sizeof(ogame *));
  int *depth = (int *)malloc(sizeof(int) * (size_t)n_sub);
  int *alive_sub = (int *)malloc(sizeof(int) * (size_t)n_sub);
  opath *paths = (opath *)calloc((size_t)n_sub * S, sizeof(opath));
  int *created = (int *)calloc((size_t)n_sub * S, sizeof(int));   /* snake alive at sub-game creation */
  const int max_path = 64;
  for (int i = 0; i < n_sub * S; ++i) {
    paths[i].e = (oentry **)malloc(sizeof(oentry *) * max_path);
    paths[i].mv = (int *)malloc(sizeof(int) * max_path);
  }
  const int max_rows = n_sub * S;
  float *planes = (float *)malloc(sizeof(float) * (size_t)plen * max_rows);
  float *miss_planes = (float *)malloc(sizeof(float) * (size_t)plen * max_rows);
  float *miss_v = (float *)malloc(sizeof(float) * 3 * (size_t)max_rows);
  oentry **row_e = (oentry **)malloc(sizeof(oentry *) * (size_t)max_rows);
  int *row_sub = (int *)malloc(sizeof(int) * (size_t)max_rows), *row_snake = (int *)malloc(sizeof(int) * (size_t)max_rows);
  int *row_new = (int *)malloc(sizeof(int) * (size_t)max_rows);
  float *row_pmf = (float *)malloc(sizeof(float) * 3 * (size_t)max_rows);
  int *row_mv = (int *)malloc(sizeof(int) * (size_t)max_rows);

  for (int ep = 0; ep < epochs; ++ep) {
    /* agent.py:39-50 */
    for (int gi = 0; gi < n_games; ++gi) {
      int d = a->D - 2 * (games[gi]->n_live - 2);             /* agent.py:45 */
      for (int p = 0; p < parallel; ++p) {
        int sid = gi * parallel + p;
        if (sub[sid]) og_free(sub[sid]);
        sub[sid] = og_clone(games[gi]);
        depth[sid] = d; alive_sub[sid] = 1;
        for (int s = 0; s < S; ++s) { paths[sid * S + s].n = 0; created[sid * S + s] = games[gi]->sn[s].alive; }
      }
    }
    a->stats[3] += (uint64_t)n_sub;
    /* MCTSMPGameRunner.run (mp_game_runner.py:85-115) */
    int remaining = n_sub, turn = 0;
    while (remaining > 0) {
      turn += 1;
      /* --- MCTSAgent.make_moves (agent.py:161-223) --- */
      int n_rows = 0, n_miss = 0;
      for (int sid = 0; sid < n_sub; ++sid) {
        if (!alive_sub[sid]) continue;
        ogame *g = sub[sid];
        for (int k = 0; k < g->n_live; ++k) {
          float *pl = planes + (size_t)n_rows * plen;
          og_make_state(g, k, pl);
          uint64_t key[2]; og_plane_key(pl, n_pix, key);
          oentry *e = tab_find(a, key, 0);
          row_new[n_rows] = 0;
          if (e) {                                             /* agent.py:178-180 */
            if (memcmp(e->plane, pl, sizeof(float) * (size_t)plen) != 0) a->alias_errors += 1;
            if (!e->pending) a->stats[2] += 1;
          } else {                                             /* agent.py:181-184 */
            e = tab_find(a, key, 1);
            e->pending = 1;
            e->plane = (float *)malloc(sizeof(float) * (size_t)plen);
            memcpy(e->plane, pl, sizeof(float) * (size_t)plen);
            memcpy(miss_planes + (size_t)n_miss * plen, pl, sizeof(float) * (size_t)plen);
            row_new[n_rows] = 1; n_miss += 1;
          }
          e->age = 0;                                          /* agent.py:185 */
          row_e[n_rows] = e; row_sub[n_rows] = sid; row_snake[n_rows] = g->live[k];
          n_rows += 1;
        }
      }
      a->stats[1] += (uint64_t)n_rows; a->stats[0] += (uint64_t)n_miss;
      if (n_miss > 0) {                                        /* agent.py:189-201 */
        a->fn(a->ctx, miss_planes, n_miss, H, W, miss_v);
        int j = 0;
        for (int r = 0; r < n_rows; ++r) if (row_new[r]) {
          oentry *e = row_e[r];
          for (int k = 0; k < 3; ++k) { e->Wt[k] = miss_v[3 * j + k]; e->N[k] = 1.0f; e->Q[k] = e->Wt[k] / e->N[k]; }
          e->pending = 0; ++j;
        }
      }
      /* agent.py:204-205: all pmfs first, then all draws, in row order */
      for (int r = 0; r < n_rows; ++r) og_softermax(row_e[r]->Q, a->base, row_pmf + 3 * r);
      for (int r = 0; r < n_rows; ++r) {
        /* absolute sub-game id = root game id * parallel + sibling: finished root games keep their slots */
        const uint32_t abs_sub = games[row_sub[r] / parallel]->game_id * (uint32_t)parallel + (uint32_t)(row_sub[r] % parallel);
        size_t ti = (((size_t)ep * (size_t)tr->max_steps + (size_t)(turn - 1)) * ((size_t)tr->total_games * (size_t)parallel) + (size_t)abs_sub) * (size_t)S + (size_t)row_snake[r];
        if (tr->mode == 1) row_mv[r] = tr->tree_moves[ti];
        else {
          uint32_t rr[4];
          og_philox(abs_sub * (uint32_t)S + (uint32_t)row_snake[r], tr->root_turn, RS_TREE,
                    (uint32_t)ep * 256u + (uint32_t)(turn - 1), tr->seed, rr);
          double u = (double)rr[0] * (1.0 / 4294967296.0);
          row_mv[r] = og_choice3(row_pmf + 3 * r, u);
          if (tr->tree_moves) tr->tree_moves[ti] = (uint8_t)row_mv[r];
        }
      }
      /* agent.py:208-222 */
      if (a->rhat_before_backups) {     /* not the reference: all estimates first (row_pmf[3r] is reused to carry r-hat) */
        for (int r = 0; r < n_rows; ++r) {
          float *pm = row_pmf + 3 * r; const float *q = row_e[r]->Q;
          float est = pm[0] * q[0]; est = est + pm[1] * q[1]; est = est + pm[2] * q[2];
          pm[0] = est;
        }
      }
      for (int r = 0; r < n_rows; ++r) {
        opath *p = &paths[row_sub[r] * S + row_snake[r]];
        const float *pm = row_pmf + 3 * r; const float *q = row_e[r]->Q;   /* live alias (agent.py:180,214) */
        float est = pm[0] * q[0]; est = est + pm[1] * q[1]; est = est + pm[2] * q[2];
        if (a->rhat_before_backups) est = pm[0];
        backup(p, est);
        if (p->n >= max_path) { fprintf(stderr, "oa_make_moves: path overflow\n"); abort(); }
        p->e[p->n] = row_e[r]; p->mv[p->n] = row_mv[r]; p->n += 1;
      }
      /* tic every sub-game (mp_game_runner.py:103-113) */
      int r0 = 0;
      for (int sid = 0; sid < n_sub; ++sid) {
        if (!alive_sub[sid]) continue;
        ogame *g = sub[sid];
        int nl = g->n_live;
        int ended = og_tic(g, row_mv + r0, 0, -1, 0, 0);
        r0 += nl;
        a->stats[4] += 1;
        if (ended || turn >= depth[sid]) { alive_sub[sid] = 0; remaining -= 1; }
      }
    }
    /* terminal backup (agent.py:60-72) */
    for (int sid = 0; sid < n_sub; ++sid)
      for (int s = 0; s < S; ++s) {
        if (!created[sid * S + s]) continue;
        int rw = sub[sid]->reward[s];
        if (rw != 0) backup(&paths[sid * S + s], (float)rw);
      }
  }
  /* root read-out (agent.py:74-87): first key of the last epoch's paths */
  int n_rows = 0;
  for (int gi = 0; gi < n_games; ++gi)
    for (int k = 0; k < games[gi]->n_live; ++k) {
      int s = games[gi]->live[k];
      opath *p = &paths[(gi * parallel) * S + s];
      const float *q = p->e[0]->Q;
      q_out[3 * n_rows] = q[0]; q_out[3 * n_rows + 1] = q[1]; q_out[3 * n_rows + 2] = q[2];
      if (a->training) {                                       /* agent.py:90-97 */
        float pmf[3]; og_softermax(q, a->base, pmf);
        if (tr->mode == 1) moves_out[n_rows] = tr->root_moves[n_rows];
        else {
          uint32_t rr[4];
          og_philox(games[gi]->game_id * (uint32_t)S + (uint32_t)s, tr->root_turn, RS_ROOT, 0, tr->seed, rr);
          moves_out[n_rows] = og_choice3(pmf, (double)rr[0] * (1.0 / 4294967296.0));
          if (tr->root_moves) tr->root_moves[n_rows] = (uint8_t)moves_out[n_rows];
        }
        if (a->n_rec == a->cap_rec) {
          a->cap_rec = a->cap_rec ? a->cap_rec * 2 : 256;
          a->rec_planes = (float *)realloc(a->rec_planes, sizeof(float) * (size_t)plen * (size_t)a->cap_rec);
          a->rec_q = (float *)realloc(a->rec_q, sizeof(float) * 3 * (size_t)a->cap_rec);
        }
        og_make_state(games[gi], k, a->rec_planes + (size_t)a->n_rec * plen);
        memcpy(a->rec_q + 3 * (size_t)a->n_rec, q, sizeof(float) * 3);   /* snapshot (SURVEY D-17) */
        a->n_rec += 1;
      } else {
        moves_out[n_rows] = og_argmax3(q);                     /* agent.py:98-99 */
      }
      n_rows += 1;
    }
  tab_evict(a);                                                /* agent.py:101-110 */

  for (int i = 0; i < n_sub; ++i) if (sub[i]) og_free(sub[i]);
  for (int i = 0; i < n_sub * S; ++i) { free(paths[i].e); free(paths[i].mv); }
  free(sub); free(depth); free(alive_sub); free(paths); free(created); free(planes); free(miss_planes); free(miss_v);
  free(row_e); free(row_sub); free(row_snake); free(row_new); free(row_pmf); free(row_mv);
  return n_rows;
}
