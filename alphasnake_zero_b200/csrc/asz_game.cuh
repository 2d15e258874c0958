// asz_game.cuh -- one warp = one Battlesnake game.  Warp-level restatement of Game.__init__, Game.tic and
// Game.make_state (reference: code/utils/game.py:13-61, 87-205, 215-257) over the cell-stamp board of asz_common.cuh.
//
// Thread mapping: lane s (< S <= 8) owns snake s; every lane owns CPL consecutive cells of the board, so that
// row-major cell order equals (lane, slot) order (used by the k-th-empty-cell food spawn).
// The board lives in shared memory while a game is being stepped (random access by head cells), the per-snake and
// per-game scalars live in registers.
#pragma once
#include "asz_common.cuh"

namespace asz {

template <int SIDE_>
struct Geo {
  static constexpr int SIDE = SIDE_;
  static constexpr int CELLS = SIDE * SIDE;
  static constexpr int CPL = (CELLS + 31) / 32;  // cells per lane
  static constexpr int PC = CPL * 32;            // padded cell count (state stride, u16 units)
  static constexpr int N = 2 * SIDE - 1;         // side of the egocentric plane (game.py:217-218)
  static constexpr int NPIX = N * N;
  static constexpr int PLANE = NPIX * 3;         // floats per plane, NHWC
  static constexpr int STAGE = ((PLANE + 3 + 3) / 4) * 4;  // staging floats (plane + up to 3 of misalignment)
};

// ---- packed records in HBM ---------------------------------------------------------------------------------------
// The one definition of the record format, for the kernels and for the host's state interchange alike.
// snake: head:16 | len:16 | health low byte:8 | last_move:2 | alive:1 | reward:2 (0 none, 1 = +1, 2 = -1) | pad:3 |
// health high byte:8.  Health is a SIGNED 16-bit value split over bits 32..39 and 48..55: the kill chain of game.py:156-165
// is an elif chain, so the winner of a head-on collision skips the starvation check and can end a tic alive with
// health <= 0 (down to 1 - 7*health_dec after seven wins in a row); it starves on the next tic it does not eat.
struct Snake {
  int head;    // cell index, kNoHead = none
  int len;
  int health;
  int last;
  int alive;
  int reward;
};
constexpr int kNoHead = 0xFFFF;
constexpr uint64_t kEmptySnake = (uint64_t)kNoHead;   // record of a slot without a snake: unpack_snake gives head kNoHead, all else 0
__host__ __device__ __forceinline__ uint64_t pack_snake(const Snake& s) {
  return (uint64_t)(s.head & 0xFFFF) | ((uint64_t)(s.len & 0xFFFF) << 16) | ((uint64_t)(s.health & 0xFF) << 32) |
         ((uint64_t)(s.last & 3) << 40) | ((uint64_t)(s.alive & 1) << 42) | ((uint64_t)(s.reward & 3) << 43) |
         ((uint64_t)((s.health >> 8) & 0xFF) << 48);
}
__host__ __device__ __forceinline__ Snake unpack_snake(uint64_t v) {
  Snake s;
  s.head = (int)(v & 0xFFFF); s.len = (int)((v >> 16) & 0xFFFF); s.health = (int)(int16_t)(uint16_t)(((v >> 32) & 0xFF) | (((v >> 48) & 0xFF) << 8));
  s.last = (int)((v >> 40) & 3); s.alive = (int)((v >> 42) & 1); s.reward = (int)((v >> 43) & 3);
  return s;
}
__host__ __device__ __forceinline__ bool snake_alive(uint64_t v) { return (v >> 42) & 1ull; }

// game meta: 8 x u32, one per slot; flags bit 0 = done
enum MetaSlot : int { META_TURN = 0, META_EPISODE, META_WALL, META_BODY, META_HEAD, META_STARVE, META_EATEN, META_FLAGS };
constexpr uint32_t kMetaDone = 1u;
struct Meta {
  uint32_t turn, episode, wall, body, headc, starve, eaten, flags;
};
// the word of slot `slot` (lane `slot` of a warp writes slot `slot` of the record)
__device__ __forceinline__ uint32_t meta_word(const Meta& m, int slot) {
  return slot == META_TURN ? m.turn : slot == META_EPISODE ? m.episode : slot == META_WALL ? m.wall : slot == META_BODY ? m.body
       : slot == META_HEAD ? m.headc : slot == META_STARVE ? m.starve : slot == META_EATEN ? m.eaten : m.flags;
}
// the record from the warp's lanes: lane k holds slot k
__device__ __forceinline__ Meta meta_from_lanes(uint32_t v) {
  Meta m;
  m.turn = __shfl_sync(kFull, v, META_TURN); m.episode = __shfl_sync(kFull, v, META_EPISODE); m.wall = __shfl_sync(kFull, v, META_WALL);
  m.body = __shfl_sync(kFull, v, META_BODY); m.headc = __shfl_sync(kFull, v, META_HEAD); m.starve = __shfl_sync(kFull, v, META_STARVE);
  m.eaten = __shfl_sync(kFull, v, META_EATEN); m.flags = __shfl_sync(kFull, v, META_FLAGS);
  return m;
}

struct TicResult {
  unsigned live_mask;   // snakes alive after the tic
  unsigned dead_mask;   // snakes that died this tic
  bool ended;           // <= 1 snake left (game.py:199)
};

// ---- Game.__init__ (game.py:13-61) with the engine's Philox streams -------------------------------------------
template <class G>
__device__ __forceinline__ void warp_init_native(uint16_t* sb, Snake& sn, Meta& m, int S, uint64_t seed, uint32_t game_id,
                                                 uint32_t episode) {
  const int lane = lane_id();
  uint32_t u[8], v[8], w[8];
  philox4x32_10(game_id, episode, RS_INIT, 0, seed, u); philox4x32_10(game_id, episode, RS_INIT, 1, seed, u + 4);
  philox4x32_10(game_id, episode, RS_INIT, 2, seed, v); philox4x32_10(game_id, episode, RS_INIT, 3, seed, v + 4);
  philox4x32_10(game_id, episode, RS_INIT, 4, seed, w); philox4x32_10(game_id, episode, RS_INIT, 5, seed, w + 4);
  constexpr int H = G::SIDE, W = G::SIDE;
  // the 8 standard start cells in the reference's order (game.py:25-28), as cell indices
  int perm[8] = {1 * W + 1, (H - 2) * W + (W - 2), (H - 2) * W + 1, 1 * W + (W - 2),
                 1 * W + W / 2, (H / 2) * W + (W - 2), (H - 2) * W + W / 2, (H / 2) * W + 1};
  int my_start = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {   // partial Fisher-Yates == sample without replacement (game.py:25-29)
    if (i < S) {
      const int j = i + (int)mulhi32(u[i], (uint32_t)(8 - i));
      int pj = perm[0];
#pragma unroll
      for (int q = 1; q < 8; ++q) if (q == j) pj = perm[q];
      const int pi = perm[i];
#pragma unroll
      for (int q = 0; q < 8; ++q) if (q == j) perm[q] = pi;
      perm[i] = pj;
      if (lane == i) my_start = pj;
    }
  }
#pragma unroll
  for (int q = 0; q < G::CPL; ++q) sb[lane * G::CPL + q] = 0;
  __syncwarp();
  sn = unpack_snake(kEmptySnake);
  if (lane == 0) sb[(H / 2) * W + W / 2] = kFood;                     // game.py:43
  if (lane < S) {
    uint32_t vv = v[0], ww = w[0];
#pragma unroll
    for (int q = 1; q < 8; ++q) if (q == lane) { vv = v[q]; ww = w[q]; }
    sn.head = my_start; sn.len = 3; sn.health = 100; sn.last = (int)(vv & 3u); sn.alive = 1;   // game.py:30,37
    const int d = (int)(ww & 3u);                                      // game.py:46-47 list order
    const int fy = my_start / W + ((d & 2) ? 1 : -1), fx = my_start % W + ((d & 1) ? 1 : -1);
    sb[fy * W + fx] = kFood;
  }
  __syncwarp();
  if (lane < S) sb[my_start] = (uint16_t)((lane << 12) | 3);          // three stacked segments: topmost has dist 3
  __syncwarp();
  m.turn = 0; m.episode = episode; m.wall = m.body = m.headc = m.starve = m.eaten = 0; m.flags = 0;
}

// ---- Game.tic (game.py:87-205) -----------------------------------------------------------------------------------
// move: this lane's relative move (0 left, 1 straight, 2 right), read only where sn.alive.
// spawn_mode 0: none (sub-games, game.py:268), 1: replay (spawn_cell or -1), 2: native Philox (never when chance_thresh == 0).
template <class G>
// spawn_r (optional): the two RS_SPAWN draws of this tic when the caller already has them (the env kernel computes them
// in the same SIMT pass as the random actions); nullptr = drawn here.
__device__ __forceinline__ TicResult warp_tic(uint16_t* sb, Snake& sn, Meta& m, int move, int health_dec, int spawn_mode,
                                              int spawn_cell, uint32_t chance_thresh, uint64_t seed, uint32_t game_id,
                                              int S = kMaxSnakes, const uint32_t* spawn_r = nullptr) {
  constexpr int SIDE = G::SIDE, CPL = G::CPL, CELLS = G::CELLS;
  const int lane = lane_id();
  const bool was_alive = sn.alive != 0;
  // 1. move (game.py:90-114, Snake.move :329-358) and 2. health (:117-118)
  int nh = -1;
  bool off = false;
  if (was_alive) {
    const int dir = (move + sn.last + 3) & 3;                 // (m + last - 1) mod 4, game.py:92
    sn.last = dir;
    int y = sn.head / SIDE, x = sn.head - y * SIDE;
    y += (dir == 0) ? -1 : (dir == 2) ? 1 : 0;                // 0 up, 1 right, 2 down, 3 left (game.py:330-342)
    x += (dir == 1) ? 1 : (dir == 3) ? -1 : 0;
    off = ((unsigned)y >= (unsigned)SIDE) || ((unsigned)x >= (unsigned)SIDE);
    nh = off ? -1 : y * SIDE + x;
    sn.health -= health_dec;
  }
  // 3. eat, first come in list order (game.py:121-127).  One __match_any_sync groups the snakes by the cell they move to (a dead
  // or off-board snake gets a key of its own): the lower lanes of a group are the snakes that come first in list order, the other
  // members are the head-on opponents of step 5.
  const bool onfood = was_alive && !off && sb[nh < 0 ? 0 : nh] == kFood;
  const unsigned same_cell = __match_any_sync(kFull, (was_alive && nh >= 0) ? nh : -1 - lane);
  const bool earlier = (same_cell & ((1u << lane) - 1u)) != 0u;
  bool shared = false, lose = false;
  // head cells among this lane's cells (for the spawn's empty set): every live snake's new head, gathered lane by lane
  unsigned blocked = 0;
  {
    unsigned movers = __ballot_sync(kFull, was_alive && nh >= 0);
    while (movers) {                                           // warp-uniform: one trip per live snake
      const int s2 = __ffs(movers) - 1;
      movers &= movers - 1;
      const int nh2 = __shfl_sync(kFull, nh, s2);
      if (nh2 / CPL == lane) blocked |= 1u << (nh2 - lane * CPL);
    }
  }
  const bool eat = onfood && !earlier;
  const unsigned ate_mask = __ballot_sync(kFull, eat);
  if (eat) { sb[nh] = 0; sn.health = 100; sn.len += 1; }       // Snake.grow, game.py:360-365
  m.eaten += (uint32_t)__popc(ate_mask);
  __syncwarp();
  // every stamp ages by one; growers get it back (tail duplicated); a stamp reaching 0 vacates the cell
  int n_food = 0, n_empty = 0;
  unsigned empty_bits = 0;
#pragma unroll 1   // rolled on purpose: the hot loop of env_step_kernel is larger than the 32 KB L1.5 instruction cache (DESIGN.md 4.1)
  for (int q = 0; q < CPL; ++q) {
    const int c = lane * CPL + q;
    uint32_t v = sb[c];
    if (cell_is_body(v)) {
      const int o = cell_owner(v);
      int d = cell_dist(v) - 1;
      if (d == 0) v = 0;
      else { if ((ate_mask >> o) & 1u) d += 1; v = (uint32_t)((o << 12) | d); }
      sb[c] = (uint16_t)v;
    }
    n_food += (v == kFood);
    if (v == 0 && c < CELLS && !((blocked >> q) & 1u)) { n_empty += 1; empty_bits |= 1u << q; }
  }
  __syncwarp();
  // 4. spawn (game.py:130-138): before the kill decision, so about-to-die snakes still block their cells
  if (spawn_mode == 1) {
    if (lane == 0 && spawn_cell >= 0) sb[spawn_cell] = kFood;
    __syncwarp();
  } else if (spawn_mode == 2 && chance_thresh != 0u) {   // game.py:130 `if self.food_spawn_chance > 0.0` (threshold 0 = chance 0)
    uint32_t r[4];
    if (spawn_r != nullptr) { r[0] = spawn_r[0]; r[1] = spawn_r[1]; }
    else philox4x32_10(game_id, m.episode, RS_SPAWN, m.turn, seed, r);
    const bool no_food = !__any_sync(kFull, n_food > 0);
    if (no_food || r[0] <= chance_thresh) {
      const int pre = warp_excl_scan_i32(n_empty, lane);
      const int tot_empty = __shfl_sync(kFull, pre + n_empty, 31);
      if (tot_empty > 0) {
        int k = (int)mulhi32(r[1], (uint32_t)tot_empty) - pre;
        if (k >= 0 && k < n_empty) {
#pragma unroll
          for (int q = 0; q < CPL; ++q)
            if ((empty_bits >> q) & 1u) { if (k == 0) sb[lane * CPL + q] = kFood; --k; }
        }
      }
    }
    __syncwarp();
  }
  // 5. kill decision (game.py:144-165): wall > body > head-on > starvation, first matching rule only
  int cause = 0;
  if (was_alive) {
    if (off) cause = 1;
    else if (cell_is_body(sb[nh])) cause = 2;
  }
  // head-on (game.py:156-163): another snake moved to the same cell; the shorter or equal one loses.  Rare, so the lengths are
  // only compared when some group has more than one member (warp-uniform branch)
  shared = was_alive && !off && (same_cell & ~(1u << lane)) != 0u;
  if (__any_sync(kFull, shared)) {
#pragma unroll 1
    for (int s2 = 0; s2 < kMaxSnakes; ++s2) {
      if (s2 >= S) break;
      const int len2 = __shfl_sync(kFull, sn.len, s2);
      if (shared && s2 != lane && ((same_cell >> s2) & 1u) && sn.len <= len2) lose = true;
    }
  }
  if (was_alive && cause == 0) {
    if (shared) { if (lose) cause = 3; }
    else if (sn.health <= 0) cause = 4;
  }
  const unsigned dead_mask = __ballot_sync(kFull, cause != 0);
  // 6. remove (game.py:167-192): the dead snake's stamps are cleared, its head was never stamped
  if (dead_mask) {
    m.wall += (uint32_t)__popc(__ballot_sync(kFull, cause == 1));
    m.body += (uint32_t)__popc(__ballot_sync(kFull, cause == 2));
    m.headc += (uint32_t)__popc(__ballot_sync(kFull, cause == 3));
    m.starve += (uint32_t)__popc(__ballot_sync(kFull, cause == 4));
#pragma unroll 1   // rolled on purpose: the hot loop of env_step_kernel is larger than the 32 KB L1.5 instruction cache (DESIGN.md 4.1)
    for (int q = 0; q < CPL; ++q) {
      const uint32_t v = sb[lane * CPL + q];
      if (cell_is_body(v) && ((dead_mask >> cell_owner(v)) & 1u)) sb[lane * CPL + q] = 0;
    }
    __syncwarp();
  }
  if (cause != 0) { sn.alive = 0; sn.reward = 2; sn.head = kNoHead; sn.len = 0; sn.health = 0; }
  else if (was_alive) { sb[nh] = (uint16_t)((lane << 12) | sn.len); sn.head = nh; }
  __syncwarp();
  // 7. terminate (game.py:197-205)
  m.turn += 1;
  TicResult r;
  r.live_mask = __ballot_sync(kFull, sn.alive != 0);
  r.dead_mask = dead_mask;
  r.ended = __popc(r.live_mask) <= 1;
  if (r.ended) { m.flags |= kMetaDone; if (sn.alive) sn.reward = 1; }
  return r;
}

// ---- Game.make_state (game.py:215-257) ---------------------------------------------------------------------------
// Per-game, viewer independent part, computed once from this lane's cells:
//   f1   = ch1 value  dist*0.02 in double, rounded once to float (game.py:239,257)
//   hs   = id of the snake whose head is on the cell, or -1 (the head is the stamp with dist == length)
//   food = cell holds food
template <class G>
struct CellView {
  float f1[G::CPL];
  int8_t hs[G::CPL];
  bool food[G::CPL];
  int8_t cy[G::CPL], cx[G::CPL];   // (y, x) of this lane's cells: constants of the thread
};
// body_lut (optional, shared memory): body_lut[d] = float(double(d) * 0.02) for d < G::PC + 8
template <class G>
__device__ __forceinline__ void warp_cell_view(const uint16_t* sb, const Snake& sn, CellView<G>& cv, const float* body_lut = nullptr) {
  const int lane = lane_id();
#pragma unroll
  for (int q = 0; q < G::CPL; ++q) {
    const uint32_t v = sb[lane * G::CPL + q];
    const bool body = cell_is_body(v);
    const int o = body ? cell_owner(v) : 0;
    const int len_o = __shfl_sync(kFull, sn.len, o);
    const int d = cell_dist(v);
    cv.f1[q] = !body ? 0.0f : (body_lut != nullptr ? body_lut[d] : (float)((double)d * 0.02));
    cv.hs[q] = (int8_t)((body && d == len_o) ? o : -1);
    cv.food[q] = (v == kFood);
    const int c = lane * G::CPL + q;
    cv.cy[q] = (int8_t)(c / G::SIDE); cv.cx[q] = (int8_t)(c - (c / G::SIDE) * G::SIDE);
  }
}

// Encode the plane of viewer `vs` (warp-uniform snake id).  Cell-centric: the staging buffer is filled with the wall
// background [0,1,0] (game.py:219), then each lane scatters its CPL board cells to their rotated, recentred pixel
// (game.py:247-257), then the warp streams the plane to HBM with 16-byte stores.  `stage` holds the plane at float
// offset a = (gidx0 & 3) so that shared and global addresses share their 16-byte phase.
// gidx0 = float index of the plane's first element in the output buffer (planes are only 4-byte aligned: 1323 floats).
// When out == nullptr nothing is written (key only).  When key != nullptr the 128-bit plane key is accumulated.
template <class G, bool kWantKey>
__device__ __forceinline__ void warp_encode(const CellView<G>& cv, const Snake& sn, int vs, float* stage, float* out,
                                            size_t gidx0, uint64_t* key0, uint64_t* key1) {
  constexpr int SIDE = G::SIDE, CPL = G::CPL, CELLS = G::CELLS, N = G::N, PLANE = G::PLANE;
  const int lane = lane_id();
  const int vhead = __shfl_sync(kFull, sn.head, vs);
  const int vlen = __shfl_sync(kFull, sn.len, vs);
  const int vhp = __shfl_sync(kFull, sn.health, vs);
  const int vrot = __shfl_sync(kFull, sn.last, vs);
  const int hy = vhead / SIDE, hx = vhead - hy * SIDE;
  // ch0 of a head of snake `lane` as seen by the viewer (game.py:229,232), ch2 of food (game.py:244): double math
  const float my_hv = (float)(((double)sn.len - ((double)vlen - 0.5)) * 0.04);
  const float foodv = (float)((double)(101 - vhp) * 0.01);
  const int a = (int)(gidx0 & 3);
  if (out != nullptr) {
    // background: element e of the plane is 1.0 iff e % 3 == 1; stage index = a + e
    for (int q4 = lane; q4 < G::STAGE / 4; q4 += 32) {
      const int e0 = q4 * 4 - a;               // may be negative for the first vector: harmless filler
      const int r = ((e0 % 3) + 3) % 3;
      float4 v;
      v.x = (r == 1) ? 1.0f : 0.0f; v.y = (r == 0) ? 1.0f : 0.0f; v.z = (r == 2) ? 1.0f : 0.0f; v.w = v.x;
      reinterpret_cast<float4*>(stage)[q4] = v;
    }
    __syncwarp();
  }
  uint64_t k0 = 0, k1 = 0;
#pragma unroll
  for (int q = 0; q < CPL; ++q) {
    const int c = lane * CPL + q;
    const int hsq = cv.hs[q];
    const float hv = __shfl_sync(kFull, my_hv, hsq < 0 ? 0 : hsq);
    if (c < CELLS) {
      const int y = c / SIDE, x = c - y * SIDE;
      const int gy = y - hy + (SIDE - 1), gx = x - hx + (SIDE - 1);       // game.py:249-251
      int i, j;                                                           // numpy.rot90(grid, k), game.py:257
      if (vrot == 0) { i = gy; j = gx; }
      else if (vrot == 1) { i = N - 1 - gx; j = gy; }
      else if (vrot == 2) { i = N - 1 - gy; j = N - 1 - gx; }
      else { i = gx; j = N - 1 - gy; }
      const int p = i * N + j;
      float t0, t1, t2;
      if (c == vhead) { t0 = t1 = t2 = -1.0f; }                           // game.py:248
      else { t0 = (hsq >= 0) ? hv : 0.0f; t1 = cv.f1[q]; t2 = cv.food[q] ? foodv : 0.0f; }
      if (out != nullptr) { float* d = stage + a + 3 * p; d[0] = t0; d[1] = t1; d[2] = t2; }
      if (kWantKey) key_accumulate((uint32_t)p, __float_as_uint(t0), __float_as_uint(t1), __float_as_uint(t2), k0, k1);
    }
  }
  if (kWantKey) {
    k0 = warp_sum_u64(k0); k1 = warp_sum_u64(k1);
    if (k0 == 0) k0 = 1;
    *key0 = k0; *key1 = k1;
  }
  if (out != nullptr) {
    __syncwarp();
    const size_t gbase = gidx0 - (size_t)a;                 // 16-byte aligned float index (buffer base is aligned)
    const size_t gA = (gidx0 + 3) & ~(size_t)3, gend = gidx0 + PLANE, gE = gend & ~(size_t)3;
    const int nvec = (int)((gE - gA) >> 2), v0 = (int)((gA - gbase) >> 2);
    const float4* s4 = reinterpret_cast<const float4*>(stage) + v0;
    float4* o4 = reinterpret_cast<float4*>(out + gA);
    for (int v = lane; v < nvec; v += 32) st_stream_f4(o4 + v, s4[v]);
    const int nhead = (int)(gA - gidx0), ntail = (int)(gend - gE);
    if (lane < nhead) out[gidx0 + lane] = stage[a + lane];
    if (lane < ntail) out[gE + lane] = stage[(int)(gE - gbase) + lane];
    __syncwarp();                                            // stage is reused by the next plane
  }
}

// ---- plane encode of the env kernel: pitched rows, one emission per game -------------------------------------------
// A plane at 11x11 is 21x21x3 floats of which only the 11 rows that intersect the board window are not pure wall background.  Those
// rows (one contiguous element range [W0, W0 + WIN) of the plane) are staged in a per-warp buffer whose background is written
// once per kernel (stage[s] = 1 iff s % 3 == 1); per plane the warp scatters its board cells into it, hands it to the bulk-copy
// engine (cp.async.bulk shared -> global) and later restores the touched pixels.  Two staging buffers per warp alternate, so the
// scatter of one plane overlaps the copy of the previous one.
// The engine's plane buffers (the network's input batch, the record store) keep consecutive planes PITCH floats apart,
// PITCH = PLANE rounded up to 8 floats (5,312 B instead of 5,292 B at 11x11): every plane starts on a 32-byte sector of HBM,
// every copy starts and ends on one, and no sector is assembled from two different copies.  The planes of one game are
// consecutive rows, so the game is emitted as ONE sequence of bulk copies: wall before the first window, then per plane its
// window (from the staging buffer) and the wall run up to the next window -- the wall after plane k and the wall before plane
// k+1 are one contiguous range, copied from a per-CTA constant "seam" buffer that holds a plane end, the pad floats and a plane
// start.
__device__ __forceinline__ void fill_wall_pattern(float* dst, int n_floats, int tid, int nthreads) {
  for (int q4 = tid; q4 < n_floats / 4; q4 += nthreads) {
    const int r = q4 % 3;   // element 4*q4 has phase (4*q4) % 3 == q4 % 3
    float4 v;
    v.x = (r == 1) ? 1.0f : 0.0f; v.y = (r == 0) ? 1.0f : 0.0f; v.z = (r == 2) ? 1.0f : 0.0f; v.w = v.x;
    reinterpret_cast<float4*>(dst)[q4] = v;
  }
}
// L2 policy of the plane stores: planes are written once and read much later by another kernel (the batch is larger than
// L2), so they should leave L2 first and not push the game records (read and rewritten every launch) out of it
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_s2g(float* gdst, const float* ssrc, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <class G>
struct PitchGeo {
  static constexpr int PITCH = ((G::PLANE + 7) / 8) * 8;
  static constexpr int WIN = G::SIDE * 3 * G::N;                       // floats of the window rows
  static constexpr int MAX_OFF = 15;                                   // largest staging offset of stage_off()
  static constexpr int WSTAGE = ((MAX_OFF + WIN + 8 + 3) / 4) * 4;     // staging floats per buffer
  static constexpr int HEAD_MAX = ((G::SIDE - 1) * 3 * G::N) & ~7;     // longest wall before a window (window on the last rows)
  static constexpr int TAIL_MAX = PITCH - ((WIN + 7) & ~7);            // longest wall + pad after a window (window on the first rows)
  static constexpr int SEAM_AT = (TAIL_MAX + 7) & ~7;                  // index of the plane boundary inside the seam buffer
  static constexpr int SEAMLEN = SEAM_AT + ((HEAD_MAX + 7) & ~7) + 8;
};
// staging offset of a window whose first float sits a (0..7) floats past a 32-byte boundary of the output:
// off % 4 == a % 4 (shared and global addresses agree modulo 16 bytes), off % 3 == 0 (pixel phase of the background), off >= a
__device__ __forceinline__ int stage_off(int a) { return (int)((0xF69C3690u >> (4 * a)) & 15u); }

__device__ __forceinline__ void fill_seam_pattern(float* seam, int seam_at, int seamlen, int pitch, int plane, int tid, int nthreads) {
  for (int j = tid; j < seamlen; j += nthreads) {
    const int e = j >= seam_at ? j - seam_at : pitch - (seam_at - j);    // element of the plane this float belongs to
    seam[j] = (e < plane && e % 3 == 1) ? 1.0f : 0.0f;                   // wall [0,1,0]; pad floats are 0
  }
}

// Per plane the encode is table driven and keeps no per-lane bookkeeping: per staging buffer only the (rotation, base) pair of
// the plane it holds is kept -- warp-uniform -- and the rotation-dependent linear term of a cell, 3 * (A*y + B*x), is read from
// a 1 KB table in shared memory, so the restore pass recomputes its indices instead of remembering them per lane (such
// per-lane arrays would cost registers that the kernel's occupancy does not have); head and food values come from tables (the
// same float64 products, evaluated once per CTA); the viewer's own head is patched by the one lane that owns the cell.
template <class G>
struct PitchLut {
  static constexpr int LIN = 4 * G::PC;                 // int16 [4 rotations][PC cells]: 3 * (A*y + B*x)
  static constexpr int HV = 2 * G::CELLS + 2;           // float [len_s - len_viewer + CELLS]: ((d + 0.5) * 0.04), game.py:229,232
  static constexpr int FOOD = 128;                      // float [101 - health] for 0 <= 101 - health < 128, game.py:244
  static constexpr int BYTES = ((LIN * 2 + (HV + FOOD) * 4 + 15) / 16) * 16;
};
template <class G>
struct EncodeCtxP {
  float* cur;                    // staging buffer of the next plane
  float* oth;                    // the other buffer (its bulk store may still be in flight)
  const float* seam;
  uint64_t policy;
  const int16_t* lin; const float* hv; const float* food;
  int cur_rot, cur_base, oth_rot, oth_base;     // plane each buffer still holds (rot < 0: background only)
};
template <class G>
__device__ __forceinline__ void fill_pitch_luts(unsigned char* raw, int tid, int nthreads) {
  using L = PitchLut<G>;
  int16_t* lin = reinterpret_cast<int16_t*>(raw);
  float* hv = reinterpret_cast<float*>(raw + L::LIN * 2);
  float* food = hv + L::HV;
  constexpr int SIDE = G::SIDE, N = G::N;
  for (int i = tid; i < L::LIN; i += nthreads) {
    const int rot = i / G::PC, c = i - rot * G::PC;
    const int cc = c < G::CELLS ? c : 0;                 // padding cells alias cell 0 (only ever used by the restore pass)
    const int y = cc / SIDE, x = cc - y * SIDE;
    const int v = rot == 0 ? N * y + x : rot == 1 ? y - N * x : rot == 2 ? -(N * y + x) : -(y - N * x);
    lin[i] = (int16_t)(3 * v);
  }
  for (int i = tid; i < L::HV; i += nthreads) hv[i] = (float)(((double)(i - G::CELLS) + 0.5) * 0.04);
  for (int i = tid; i < L::FOOD; i += nthreads) food[i] = (float)((double)i * 0.01);
}
template <class G>
__device__ __forceinline__ void load_lin(const int16_t* lin, int rot, int lane, int (&out)[G::CPL]) {
  const int16_t* p = lin + rot * G::PC + lane * G::CPL;
  if constexpr (G::CPL % 4 == 0) {
#pragma unroll
    for (int q4 = 0; q4 < G::CPL / 4; ++q4) {
      const uint2 v = reinterpret_cast<const uint2*>(p)[q4];
      out[4 * q4] = (int)(int16_t)(v.x & 0xFFFFu); out[4 * q4 + 1] = (int)v.x >> 16;
      out[4 * q4 + 2] = (int)(int16_t)(v.y & 0xFFFFu); out[4 * q4 + 3] = (int)v.y >> 16;
    }
  } else {
#pragma unroll
    for (int q2 = 0; q2 < G::CPL / 2; ++q2) {
      const uint32_t v = reinterpret_cast<const uint32_t*>(p)[q2];
      out[2 * q2] = (int)(int16_t)(v & 0xFFFFu); out[2 * q2 + 1] = (int)v >> 16;
    }
  }
}

// Encodes the planes of the first n_emit live snakes of one game to gbase (the game's first row: rows are PITCH apart).
// keys (optional, when kWantKey): 2 words per row; row_ids (optional): game*8 + snake per row.
template <class G, bool kWantKey>
__device__ __forceinline__ void warp_encode_game_v3b(const CellView<G>& cv, const Snake& sn, unsigned live_mask, int n_emit,
                                                     EncodeCtxP<G>& ctx, float* gbase, uint64_t* keys, int32_t* row_ids, int gid8) {
  constexpr int SIDE = G::SIDE, CPL = G::CPL, CELLS = G::CELLS, N = G::N, U = G::SIDE - 1;
  using P = PitchGeo<G>;
  const int lane = lane_id();
  int prev_end = 0;
  unsigned rest = live_mask;
  for (int k = 0; k < n_emit; ++k) {
    const int vs = __ffs(rest) - 1;
    rest &= rest - 1;
    const int vhead = __shfl_sync(kFull, sn.head, vs);
    const int vlen = __shfl_sync(kFull, sn.len, vs);
    const int vhp = __shfl_sync(kFull, sn.health, vs);
    const int vrot = __shfl_sync(kFull, sn.last, vs);
    const int hy = vhead / SIDE, hx = vhead - hy * SIDE;
    const float my_hv = ctx.hv[sn.len - vlen + CELLS];                                 // game.py:229,232
    const int fi = 101 - vhp;
    const float foodv = (unsigned)fi < (unsigned)PitchLut<G>::FOOD ? ctx.food[fi] : (float)((double)fi * 0.01);   // game.py:244
    // recentring + rot90 (game.py:249-257) are one affine map of the cell (y, x) to the output pixel A*y + B*x + Cc with
    // warp-uniform A, B, Cc; i0 = first output row of the board window, D = 3*Cc - W0 in closed form per rotation
    const int t = (vrot & 1) ? hy : hx;                      // rot0: hx, rot1: hy, rot2: hx, rot3: hy
    const int r = (vrot & 1) ? hx : hy;                      // rot0: hy, rot1: hx, rot2: hy, rot3: hx
    const bool flip_t = (vrot == 0) || (vrot == 1);          // D uses (U - t) for rot 0, 1 and (U + t) for rot 2, 3
    const bool far = (vrot == 1) || (vrot == 2);             // ... plus U*N for rot 1, 2
    const int D = 3 * ((flip_t ? U - t : U + t) + (far ? U * N : 0));
    const int i0 = (vrot == 0 || vrot == 3) ? U - r : r;     // rot0: U-hy, rot1: hx, rot2: hy, rot3: U-hx
    const int W0 = i0 * 3 * N;
    const int a = W0 & 7;
    const int off = stage_off(a);
    const int base3 = D + off;
    float* stage = ctx.cur;
    if (lane == 0) bulk_wait_read<1>();      // the store that read this buffer two planes ago has finished reading it
    __syncwarp();
    if (ctx.cur_rot >= 0) {                  // warp-uniform: put the background back where that plane's cells were scattered
      int lin[CPL];
      load_lin<G>(ctx.lin, ctx.cur_rot, lane, lin);
      const int b = ctx.cur_base;
#pragma unroll
      for (int q = 0; q < CPL; ++q) { float* d = stage + (b + lin[q]); d[0] = 0.0f; d[1] = 1.0f; d[2] = 0.0f; }
      __syncwarp();
    }
    int lin[CPL];
    load_lin<G>(ctx.lin, vrot, lane, lin);
    uint64_t k0 = 0, k1 = 0;
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
      const int c = lane * CPL + q;
      const int hsq = cv.hs[q];
      const float hv = __shfl_sync(kFull, my_hv, hsq < 0 ? 0 : hsq);
      if (c < CELLS) {
        float t0 = (hsq >= 0) ? hv : 0.0f, t1 = cv.f1[q], t2 = cv.food[q] ? foodv : 0.0f;
        if (kWantKey) {
          if (c == vhead) { t0 = t1 = t2 = -1.0f; }
          const int Cc = (D + W0) / 3;
          key_accumulate((uint32_t)(lin[q] / 3 + Cc), __float_as_uint(t0), __float_as_uint(t1), __float_as_uint(t2), k0, k1);
        }
        float* d = stage + (base3 + lin[q]);
        d[0] = t0; d[1] = t1; d[2] = t2;
      }
    }
    if (lane == vhead / CPL) {               // game.py:248: the viewer's own head is -1 in all channels (same lane wrote the cell above)
      float* d = stage + (base3 + (int)ctx.lin[vrot * G::PC + vhead]);
      d[0] = -1.0f; d[1] = -1.0f; d[2] = -1.0f;
    }
    if (kWantKey) {
      k0 = warp_sum_u64(k0); k1 = warp_sum_u64(k1);
      if (k0 == 0) k0 = 1;
    }
    fence_proxy_async_smem();
    __syncwarp();
    const int EA = W0 - a, EE = (W0 + P::WIN + 7) & ~7;
    const int plane_off = k * P::PITCH;
    if (lane == 0) {
      const int run = plane_off + EA - prev_end;
      if (run > 0) bulk_s2g(gbase + prev_end, ctx.seam + P::SEAM_AT - (plane_off - prev_end), (uint32_t)(run * 4), ctx.policy);
      bulk_s2g(gbase + plane_off + EA, stage + (off - a), (uint32_t)((EE - EA) * 4), ctx.policy);
      if (k == n_emit - 1 && EE < P::PITCH)
        bulk_s2g(gbase + plane_off + EE, ctx.seam + P::SEAM_AT - (P::PITCH - EE), (uint32_t)((P::PITCH - EE) * 4), ctx.policy);
      bulk_commit();
      if (row_ids != nullptr) row_ids[k] = gid8 + vs;
      if (kWantKey) { keys[2 * k] = k0; keys[2 * k + 1] = k1; }
    }
    prev_end = plane_off + EE;
    ctx.cur = ctx.oth; ctx.oth = stage;
    const int orot = ctx.oth_rot, obase = ctx.oth_base;
    ctx.oth_rot = vrot; ctx.oth_base = base3;
    ctx.cur_rot = orot; ctx.cur_base = obase;
  }
}

}  // namespace asz
