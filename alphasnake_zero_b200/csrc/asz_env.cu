// asz_env.cu -- lockstep Battlesnake tic with the plane encoding fused in, plus the env part of the C ABI.
//
// Kernel (env_step_kernel): persistent, 3 CTAs x 8 warps per SM, one warp = one game at a time, two games per scheduling ticket.
// A warp loads a game record (cells + snakes + meta, ~350 B at 11x11x4; prefetched one game ahead), steps it in shared memory
// (asz_game.cuh: warp_tic) and writes the record back -- for both games of its ticket -- then takes the ticket's rows of the
// batch AND its next ticket with ONE 64-bit atomicAdd, and encodes the plane of every surviving snake (5,292 B each at 11x11)
// into the network's input batch: the cells are scattered into a staged window in shared memory and the copy engine
// (cp.async.bulk shared -> global) writes the plane, wall runs from a constant buffer.  Rows are asz_plane_pitch() floats apart:
// planes start on 32-byte sectors and a game's planes are one sequence of bulk copies (warp_encode_game_v3b).
// Roofline: HBM write bandwidth (planes are > 95 % of the bytes; SURVEY.md 8(d)).  What the kernel must NOT be bound by is the
// rate at which one L2 slice serves atomics on one address (2.3 - 3.6 ns each): with one atomic per game that was the
// bound, and the two values were the "two timing regimes" of rounds 1 and 2 (DESIGN.md 4.1).
#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>

#include "asz_engine.hpp"
#include "asz_game.cuh"

namespace asz {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
bool cuda_ok(cudaError_t err, const char* what) {
  if (err == cudaSuccess) return true;
  g_err = std::string(what) + ": " + cudaGetErrorString(err);
  return false;
}

struct EnvParams {
  uint16_t* cells; uint64_t* snakes; uint32_t* meta;
  int G, S, health_dec;
  uint32_t flags; int spawn_mode; uint32_t chance_thresh; uint64_t seed;
  const uint8_t* actions; const int32_t* spawn_cells;
  float* planes; int32_t* row_ids; uint64_t* keys; int max_rows; int32_t* row_count;
  uint8_t* ended; int8_t* rewards; unsigned long long* totals;
  unsigned long long* sched;   // ONE 64-bit word, zero when the launch starts: low half = rows handed out so far (the batch's row
                               // allocator), high half = tickets handed out beyond the warps' static first ticket (the persistent
                               // kernel's dynamic scheduler).  A ticket takes both with a single returning atomicAdd; an L2 slice
                               // serves such atomics on one word one after the other (2.3 - 3.6 ns each), which is why there is
                               // one per ticket of two games and not one (or two, round 1) per game
  unsigned long long* sched_next;   // the word the NEXT launch uses: zeroed by this one (the engine alternates between two words, so no
                                    // memset node sits between two launches)
  unsigned long long* prof;   // ASZ_ENV_PROFILE builds only: per-phase cycle sums (tools/env_profile.py)
  int device, n_sm;    // the engine's device and its multiprocessor count (grid size of the persistent kernel)
  int row_base;        // rows of this launch are written at [row_base, row_base + n) of planes / row_ids / keys (max_rows is absolute)
  int pair_tickets, n_tickets;   // scheduling tickets of the launch (set by EnvLaunch::launch): the first pair_tickets are two games each
};

// Phase timers for the measurement build (nvcc -DASZ_ENV_PROFILE, tools/env_profile.py); they compile to nothing otherwise.
#ifdef ASZ_ENV_PROFILE
#define ASZ_PROF_DECL long long prof_t = clock64();
#define ASZ_PROF(k) do { const long long prof_n = clock64(); if (lane == 0) s_prof[warp][k] += (unsigned long long)(prof_n - prof_t); prof_t = prof_n; } while (0)
#else
#define ASZ_PROF_DECL
#define ASZ_PROF(k) do { } while (0)
#endif

// ---- the fused step kernel ----------------------------------------------------------------------------------------
// Persistent: MINB CTAs per SM, every warp loops over games g = warp_global, warp_global + n_warps, ... so that the
// staging buffers' wall background is written once per warp and bulk stores of one game overlap the tic of the next.
// L2 policies: plane stores carry evict_first and the game records (read and rewritten by every launch, 21 MB at 65,536
// games) evict_last.
// ACTS: the caller supplies the actions (p.actions); false = none are read (in-kernel random actions, or no tic at all).
template <int SIDE>
struct EnvSmem {
  using G = Geo<SIDE>;
  static constexpr int BG = PitchGeo<G>::SEAMLEN;          // per-CTA constant wall buffer (floats)
  static constexpr int WSTAGE = PitchGeo<G>::WSTAGE;       // floats per staging buffer
  static constexpr int LUT_BYTES = PitchLut<G>::BYTES;     // index / value tables of warp_encode_game_v3b
};

template <int SIDE, int WARPS, int MINB, bool ACTS>
__global__ void __launch_bounds__(WARPS * 32, MINB) env_step_kernel(const EnvParams p) {
  using G = Geo<SIDE>;
  using SM = EnvSmem<SIDE>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = (int)(threadIdx.x >> 5), lane = lane_id();
  // smem: [per-CTA wall pattern][per warp: 2 staging buffers][per warp: 2 boards][per-CTA body-value table]
  float* s_bg = reinterpret_cast<float*>(smem_raw);
  float* stage0 = s_bg + SM::BG + warp * 2 * SM::WSTAGE;
  uint16_t* sb = reinterpret_cast<uint16_t*>(s_bg + SM::BG + WARPS * 2 * SM::WSTAGE) + warp * 2 * G::PC;   // the ticket's two games
  float* s_lut = reinterpret_cast<float*>(reinterpret_cast<uint16_t*>(s_bg + SM::BG + WARPS * 2 * SM::WSTAGE) + WARPS * 2 * G::PC);
  for (int d = (int)threadIdx.x; d < G::PC + 8; d += WARPS * 32) s_lut[d] = (float)((double)d * 0.02);   // game.py:239, float64 product
  unsigned char* s_plut = reinterpret_cast<unsigned char*>(s_lut + G::PC + 8);
  fill_pitch_luts<G>(s_plut, (int)threadIdx.x, WARPS * 32);
  const bool enc = (p.flags & ASZ_STEP_ENCODE) != 0;
  if (enc) {
    fill_seam_pattern(s_bg, PitchGeo<G>::SEAM_AT, PitchGeo<G>::SEAMLEN, PitchGeo<G>::PITCH, G::PLANE, (int)threadIdx.x, WARPS * 32);
    fill_wall_pattern(stage0, SM::WSTAGE, lane, 32);
    fill_wall_pattern(stage0 + SM::WSTAGE, SM::WSTAGE, lane, 32);
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) *p.sched_next = 0ull;
  EncodeCtxP<G> ctxp;
  ctxp.cur = stage0; ctxp.oth = stage0 + SM::WSTAGE; ctxp.seam = s_bg;
  ctxp.policy = l2_policy_evict_first();
  ctxp.lin = reinterpret_cast<const int16_t*>(s_plut);
  ctxp.hv = reinterpret_cast<const float*>(s_plut + PitchLut<G>::LIN * 2);
  ctxp.food = ctxp.hv + PitchLut<G>::HV;
  ctxp.cur_rot = ctxp.oth_rot = -1; ctxp.cur_base = ctxp.oth_base = 0;
  __shared__ uint32_t s_wtot[WARPS][12];         // per-warp totals (only lane 0 of the warp touches its row)
  if (lane < 12) s_wtot[warp][lane] = 0u;
#ifdef ASZ_ENV_PROFILE
  __shared__ unsigned long long s_prof[WARPS][8];
  if (lane < 8) s_prof[warp][lane] = 0ull;
#endif
  __syncwarp();

  // Dynamic scheduling in TICKETS of (mostly) two consecutive games.  The first ticket of a warp is static, later
  // ones come from the kernel's scheduling word, which also hands out the batch rows: ONE atomicAdd per ticket takes the rows of
  // both games and the warp's next ticket.  Why pairs: every one of these atomics hits the same 8-byte word, and an L2 slice
  // serves same-address atomics one after the other at 2.3 - 3.6 ns each (which of the two depends on the slice the word is homed
  // in and on the state of the L2, neither under the kernel's control): with one atomic per game, 65,536 games took 150 us or
  // 236 us per launch -- exactly that serialisation -- whatever the rest of the kernel did; with two per game 360 us
  // (profiles/r02_env_hot_word_scan.txt).  Flow per ticket: tic A, tic B, the atomic, then the planes of B (its snakes are still
  // in registers) and of A (the boards stay in the warp's two board buffers, A's snake records in a 64-byte stash); the next
  // ticket's first record is prefetched into registers while the planes are encoded, B's record while A is stepped.
  const int n_warps = (int)gridDim.x * WARPS;
  constexpr int BW = G::CPL / 2;                 // 32-bit words of board per lane
  uint32_t pf_board[BW];
  uint64_t pf_snake = 0;
  uint32_t pf_meta = 0;
  // the caller's actions of a game travel with its record (cp.async into a per-warp slot: no register held across
  // the encode), instead of being an exposed load inside the tic
  __shared__ __align__(8) uint8_t s_act[WARPS][2][8];
  __shared__ uint64_t s_stash[WARPS][8];         // game A's snake records between its tic and its encode (game B's stay in registers)
  constexpr bool given_actions = ACTS;
  int pf_slot = 0, act_slot = 0;                 // slot the next prefetch writes / slot of the game being stepped
  const uint64_t keep = l2_policy_evict_last();
  auto prefetch = [&](int gi) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.cells + (size_t)gi * G::PC);
#pragma unroll
    for (int q = 0; q < BW; ++q) pf_board[q] = ld_hint_u32(src + lane * BW + q, keep);
    if (lane < 8) { pf_snake = ld_hint_u64(p.snakes + (size_t)gi * 8 + lane, keep); pf_meta = ld_hint_u32(p.meta + (size_t)gi * 8 + lane, keep); }
    if constexpr (given_actions) if (lane == 0) {
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\ncp.async.commit_group;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_act[warp][pf_slot][0])),
                   "l"(p.actions + (size_t)gi * 8)
                   : "memory");
    }
  };
  // the prefetched record -> the board buffer `board`, the lanes' snake registers and the game counters
  auto unpack = [&](uint16_t* board, Snake& sn, Meta& m) {
    uint32_t* dst = reinterpret_cast<uint32_t*>(board);
#pragma unroll
    for (int q = 0; q < BW; ++q) dst[lane * BW + q] = pf_board[q];
    sn = unpack_snake(kEmptySnake);
    if (lane < 8) sn = unpack_snake(pf_snake);
    m = meta_from_lanes(pf_meta);
    act_slot = pf_slot; pf_slot ^= 1;
    __syncwarp();
  };
  // one game: tic (results, in-place reset, record write-back) and its live snakes = the rows it needs
  // `stash` (game A of a pair): where the lanes' packed snake records wait for the encode; `pf_rec`: the record as unpacked
  // `last` (the ticket's last game): the ticket's atomic -- rows of its games, next ticket -- is issued as soon as this game's rows are
  // known, BEFORE its record is written back, so that the write-back covers part of the atomic's latency; `n_before` = rows of the
  // ticket's earlier game
  auto step_game = [&](int g, uint16_t* board, Snake& sn, Meta& m, unsigned& live_mask, int& n_rows, uint64_t* stash, uint64_t pf_rec,
                       bool last, int n_before, int& row, int& nxt) {
    live_mask = 0u; n_rows = 0;
    auto rows_and_ticket = [&]() {
      if (enc && !(m.flags & kMetaDone)) {
        live_mask = __ballot_sync(kFull, sn.alive != 0);
        n_rows = __popc(live_mask);
      }
      if (last && lane == 0) {
        const unsigned long long v = atomicAdd(p.sched, (1ull << 32) | (unsigned long long)(unsigned)(n_before + n_rows));
        row = (int)(uint32_t)v; nxt = n_warps + (int)(v >> 32);
        s_wtot[warp][8] += (uint32_t)(n_before + n_rows);
      }
    };
    if ((p.flags & ASZ_STEP_TIC) && !(m.flags & kMetaDone)) {
      int move = 1;
      uint32_t spawn_r[2] = {0u, 0u};
      const bool merged_rng = (p.flags & ASZ_STEP_RANDOM_ACT) && p.spawn_mode == ASZ_SPAWN_NATIVE;
      if (p.flags & ASZ_STEP_RANDOM_ACT) {
        // one SIMT pass draws the action streams (lanes 0..3 RS_ACT_LO, 4..7 RS_ACT_HI) and, in lanes >= 8, this tic's
        // RS_SPAWN block: same streams and counters as separate calls, one Philox instead of two per game
        uint32_t r[4];
        const uint32_t stream = lane >= 8 ? (uint32_t)RS_SPAWN : (lane & 4) ? (uint32_t)RS_ACT_HI : (uint32_t)RS_ACT_LO;
        philox4x32_10((uint32_t)g, m.episode, stream, m.turn, p.seed, r);
        const uint32_t rv = (lane & 3) == 0 ? r[0] : (lane & 3) == 1 ? r[1] : (lane & 3) == 2 ? r[2] : r[3];
        move = (int)mulhi32(rv, 3u);
        spawn_r[0] = __shfl_sync(kFull, r[0], 8); spawn_r[1] = __shfl_sync(kFull, r[1], 8);
      } else if constexpr (given_actions) {
        if (lane == 0) asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
        if (lane < 8) move = (int)s_act[warp][act_slot][lane];
      }
      const int spawn_cell = (p.spawn_mode == ASZ_SPAWN_REPLAY) ? p.spawn_cells[g] : -1;
      const TicResult r = warp_tic<G>(board, sn, m, move, p.health_dec, p.spawn_mode, spawn_cell, p.chance_thresh, p.seed,
                                      (uint32_t)g, p.S, merged_rng ? spawn_r : nullptr);
      if (p.rewards != nullptr && lane < 8)
        p.rewards[(size_t)g * 8 + lane] = (int8_t)(sn.reward == 1 ? 1 : sn.reward == 2 ? -1 : 0);
      if (lane == 0) {
        if (p.ended != nullptr) p.ended[g] = r.ended ? 1 : 0;
        s_wtot[warp][7] += 1u;
        if (r.ended) {   // mp_game_runner.py:56-61
          s_wtot[warp][0] += m.wall; s_wtot[warp][1] += m.body; s_wtot[warp][2] += m.headc; s_wtot[warp][3] += m.starve;
          s_wtot[warp][4] += m.eaten; s_wtot[warp][5] += m.turn; s_wtot[warp][6] += 1u;
        }
      }
      if (r.ended && (p.flags & ASZ_STEP_AUTO_RESET)) warp_init_native<G>(board, sn, m, p.S, p.seed, (uint32_t)g, m.episode + 1);
      rows_and_ticket();
      // write the record back
      {
        uint32_t* gc = reinterpret_cast<uint32_t*>(p.cells + (size_t)g * G::PC);
        const uint32_t* src = reinterpret_cast<const uint32_t*>(board);
        if constexpr (BW % 2 == 0) {
#pragma unroll
          for (int q = 0; q < BW / 2; ++q) {
            const uint2 v = reinterpret_cast<const uint2*>(src)[lane * (BW / 2) + q];
            st_hint_v2u32(gc + 2 * (lane * (BW / 2) + q), v.x, v.y, keep);
          }
        } else {
#pragma unroll
          for (int q = 0; q < BW; ++q) st_hint_u32(gc + lane * BW + q, src[lane * BW + q], keep);
        }
      }
      if (lane < 8) {
        const uint32_t mv = meta_word(m, lane);
        const uint64_t rec = pack_snake(sn);
        if (stash != nullptr) stash[lane] = rec;
        st_hint_u64(p.snakes + (size_t)g * 8 + lane, rec, keep);
        st_hint_u32(p.meta + (size_t)g * 8 + lane, mv, keep);
      }
    } else {
      if (p.flags & ASZ_STEP_TIC) {     // a finished game is not stepped: its results of this tic are "nothing happened"
        if (lane == 0 && p.ended != nullptr) p.ended[g] = 0;
        if (lane < 8 && p.rewards != nullptr) p.rewards[(size_t)g * 8 + lane] = 0;
      }
      if (stash != nullptr && lane < 8) stash[lane] = pf_rec;      // not stepped: the record as it was loaded
      rows_and_ticket();
    }
  };
  // planes of one game into rows [row, row + n_rows) (rows of a game stay contiguous, ascending snake id); rows at or past
  // p.max_rows are not written
  auto encode_game = [&](int g, const uint16_t* board, const Snake& sn, unsigned live_mask, int n_rows, int row) {
    if (n_rows <= 0) return;
    CellView<G> cv;
    warp_cell_view<G>(board, sn, cv, s_lut);
    const int n_emit = min(n_rows, p.max_rows - row);
    if (n_emit > 0) {
      float* gbase = p.planes + (size_t)row * PitchGeo<G>::PITCH;
      if (p.flags & ASZ_STEP_KEYS) warp_encode_game_v3b<G, true>(cv, sn, live_mask, n_emit, ctxp, gbase, p.keys + 2 * (size_t)row, p.row_ids + row, g * 8);
      else warp_encode_game_v3b<G, false>(cv, sn, live_mask, n_emit, ctxp, gbase, nullptr, p.row_ids + row, g * 8);
    }
  };

  // tickets [0, T1) are pairs (games 2t, 2t + 1), tickets [T1, NT) the last games one by one: a warp that draws its last ticket
  // late holds up the launch by one ticket, so the end of the launch is handed out in single games
  const int T1 = p.pair_tickets, NT = p.n_tickets;
  auto first_game = [&](int tk) { return tk < T1 ? 2 * tk : tk + T1; };
  int t = (int)blockIdx.x * WARPS + warp;
  if (t < NT) prefetch(first_game(t));
  while (t < NT) {
    ASZ_PROF_DECL
    const int gA = first_game(t);
    const int cnt = t < T1 ? 2 : 1;
    Snake sn; Meta m;
    unsigned maskA = 0u, maskB = 0u;
    int nA = 0, nB = 0;
    int row = 0, nxt = 0;
    // one copy of the tic and of the encode in the instruction stream, two trips each: the loop body is ~40 KB of SASS already,
    // beyond the 32 KB L1.5 instruction cache; unrolling either loop costs 20 - 45 % (218 / 197 / 240 us, measured)
#pragma unroll 1
    for (int h = 0; h < cnt; ++h) {
      uint16_t* board = sb + h * G::PC;
      const uint64_t rec0 = pf_snake;
      unpack(board, sn, m);
      if (h == 0) { ASZ_PROF(0); }                // waiting for the prefetched record
      if (h + 1 < cnt) prefetch(gA + 1);          // B's record streams in while A is stepped
      unsigned mk; int nk;
      step_game(gA + h, board, sn, m, mk, nk, (h + 1 < cnt) ? &s_stash[warp][0] : nullptr, rec0, h + 1 == cnt, nA, row, nxt);
      if (h == 0) { maskA = mk; nA = nk; } else { maskB = mk; nB = nk; }
    }
    ASZ_PROF(1);   // draws, tics, results, the ticket's atomic, record write-backs
    // the next ticket's first record streams in while this ticket's planes are encoded
    nxt = __shfl_sync(kFull, nxt, 0);
    ASZ_PROF(2);   // waiting for the scheduling word
    if (nxt < NT) prefetch(first_game(nxt));
    ASZ_PROF(3);   // issuing the prefetch
    row = __shfl_sync(kFull, row, 0) + p.row_base;
    // the last game stepped is still in the snake registers: its planes first, then game A's from the stash
#pragma unroll 1
    for (int h = cnt - 1; h >= 0; --h) {
      if (h + 1 < cnt) {
        __syncwarp();
        if (lane < 8) sn = unpack_snake(s_stash[warp][lane]);
      }
      encode_game(gA + h, sb + h * G::PC, sn, h ? maskB : maskA, h ? nB : nA, (h + 1 < cnt) ? row + nB : row);
    }
    __syncwarp();   // the board buffers are reused by the next ticket
    ASZ_PROF(5);   // plane encode
    t = nxt;
  }
  if (lane == 0) {
    bulk_wait_read<0>();   // shared memory must stay valid until the copy engine has read it
  }
  __syncwarp();
  if (lane < 9 && s_wtot[warp][lane] != 0u) atomicAdd(&p.totals[lane], (unsigned long long)s_wtot[warp][lane]);
#ifdef ASZ_ENV_PROFILE
  if (p.prof != nullptr && lane < 8) atomicAdd(&p.prof[lane], s_prof[warp][lane]);
#endif
}

// ---- reset kernel ---------------------------------------------------------------------------------------------------
template <int SIDE, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) env_reset_kernel(uint16_t* cells, uint64_t* snakes, uint32_t* meta, int Gn,
                                                               int S, uint64_t seed) {
  using G = Geo<SIDE>;
  __shared__ __align__(16) uint16_t s_board[WARPS][G::PC];
  const int warp = (int)(threadIdx.x >> 5), lane = lane_id();
  const int g = (int)blockIdx.x * WARPS + warp;
  if (g >= Gn) return;
  uint16_t* sb = s_board[warp];
  Snake sn; Meta m;
  warp_init_native<G>(sb, sn, m, S, seed, (uint32_t)g, 0);
#pragma unroll
  for (int q = 0; q < G::CPL; ++q) cells[(size_t)g * G::PC + lane * G::CPL + q] = sb[lane * G::CPL + q];
  if (lane < 8) snakes[(size_t)g * 8 + lane] = pack_snake(sn);
  uint32_t* gm = meta + (size_t)g * 8;
  if (lane < 8) gm[lane] = meta_word(m, lane);
}

template <int SIDE>
struct EnvLaunch {
  // 3 CTAs x 8 warps per SM at 80 registers (2 x 4 at 19x19).  Measured alternatives at 11x11 (tools/env_sustain.py, us per
  // launch of 65,536 games): 8 warps x 3 CTAs 176.8 | 12 x 2 176.8 | 10 x 2 177.3 | 8 x 2 196.2 (too few warps) |
  // 7 x 4 206.6, 5 x 5 211.1, 6 x 5 227.2, 8 x 4 233 (register spills)
  static constexpr int WARPS = SIDE >= 19 ? 4 : 8;
  static constexpr int MINB = SIDE >= 19 ? 2 : 3;
  // the last kTailRounds games of every warp are handed out one by one, everything before in pairs (2: +2.5 us, 4 and 6: the
  // same as 3)
  static constexpr int kTailRounds = 3;
  using G = Geo<SIDE>;
  using SM = EnvSmem<SIDE>;
  static constexpr size_t kSmemBytes = (size_t)(SM::BG + WARPS * 2 * SM::WSTAGE) * sizeof(float) + (size_t)WARPS * 2 * G::PC * sizeof(uint16_t) +
                                       (size_t)(G::PC + 8) * sizeof(float) + (size_t)SM::LUT_BYTES;
  template <bool ACTS>
  static int launch(const EnvParams& p, cudaStream_t st) {
    // function attributes are per device: one flag per device and kernel instantiation (the caller holds a DeviceGuard)
    static bool configured[kMaxDevices] = {false};
    const int dev = p.device;
    if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
      if (!cuda_ok(cudaFuncSetAttribute(env_step_kernel<SIDE, WARPS, MINB, ACTS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kSmemBytes), "cudaFuncSetAttribute(env_step_kernel)"))
        return ASZ_ERR_CUDA;
      if (!cuda_ok(cudaFuncSetAttribute(env_step_kernel<SIDE, WARPS, MINB, ACTS>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                        cudaSharedmemCarveoutMaxShared), "cudaFuncSetAttribute(carveout)"))
        return ASZ_ERR_CUDA;
      if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
    }
    const int blocks = std::min((p.G + WARPS - 1) / WARPS, p.n_sm * MINB);
    EnvParams q = p;
    q.pair_tickets = std::max(0, p.G - kTailRounds * blocks * WARPS) / 2;
    q.n_tickets = p.G - q.pair_tickets;
    env_step_kernel<SIDE, WARPS, MINB, ACTS><<<blocks, WARPS * 32, kSmemBytes, st>>>(q);
    return cuda_ok(cudaGetLastError(), "env_step_kernel launch") ? ASZ_OK : ASZ_ERR_CUDA;
  }
  static int step(const EnvParams& p, cudaStream_t st) {
    const bool acts = (p.flags & ASZ_STEP_TIC) && !(p.flags & ASZ_STEP_RANDOM_ACT);
    return acts ? launch<true>(p, st) : launch<false>(p, st);
  }
  static int reset(const GameSet& gs, int S, uint64_t seed, cudaStream_t st) {
    const int blocks = (gs.n + WARPS - 1) / WARPS;
    env_reset_kernel<SIDE, WARPS><<<blocks, WARPS * 32, 0, st>>>(gs.cells, gs.snakes, gs.meta, gs.n, S, seed);
    return cuda_ok(cudaGetLastError(), "env_reset_kernel launch") ? ASZ_OK : ASZ_ERR_CUDA;
  }
};

int gameset_alloc(GameSet& gs, int n, int pc) {
  gs.n = n;
  ASZ_CUDA(cudaMalloc(&gs.cells, (size_t)n * pc * sizeof(uint16_t)));
  ASZ_CUDA(cudaMalloc(&gs.snakes, (size_t)n * 8 * sizeof(uint64_t)));
  ASZ_CUDA(cudaMalloc(&gs.meta, (size_t)n * 8 * sizeof(uint32_t)));
  ASZ_CUDA(cudaMemset(gs.cells, 0, (size_t)n * pc * sizeof(uint16_t)));
  ASZ_CUDA(cudaMemset(gs.snakes, 0, (size_t)n * 8 * sizeof(uint64_t)));
  ASZ_CUDA(cudaMemset(gs.meta, 0, (size_t)n * 8 * sizeof(uint32_t)));
  return ASZ_OK;
}
void gameset_free(GameSet& gs) {
  cudaFree(gs.cells); cudaFree(gs.snakes); cudaFree(gs.meta);
  gs = GameSet();
}

// cells, plane floats and plane pitch of the engine's buffers: the kernels' own geometry
template <int SIDE>
static void engine_geometry(asz_engine* e) {
  using G = Geo<SIDE>;
  e->pc = G::PC; e->plane = G::PLANE; e->pitch = PitchGeo<G>::PITCH;
}

}  // namespace asz

using namespace asz;

extern "C" {

const char* asz_last_error(void) { return g_err.c_str(); }
int asz_version(void) { return ASZ_VERSION; }

// allocations of asz_engine_create; on failure the caller destroys the partially built engine (cudaFree(nullptr) is a no-op)
static int engine_alloc(asz_engine* e, const asz_config* cfg) {
  e->cfg = *cfg;
  ASZ_CUDA(cudaGetDevice(&e->device));
  ASZ_CUDA(cudaDeviceGetAttribute(&e->n_sm, cudaDevAttrMultiProcessorCount, e->device));
  switch (cfg->side) {
    case 7: engine_geometry<7>(e); break;
    case 11: engine_geometry<11>(e); break;
    default: engine_geometry<19>(e); break;
  }
  double th = (double)cfg->food_chance * 4294967296.0;
  // 0 = the reference's `food_spawn_chance > 0.0` guard is false (game.py:130): no spawning at all, not even on a board without food
  e->chance_thresh = cfg->food_chance <= 0.0f ? 0u : th >= 4294967295.0 ? 4294967295u : th < 1.0 ? 1u : (uint32_t)th;
  const size_t G = (size_t)cfg->games, rows = G * (size_t)cfg->snakes;
  int rc = gameset_alloc(e->root, cfg->games, e->pc);
  if (rc != ASZ_OK) return rc;
  ASZ_CUDA(cudaMalloc(&e->planes, rows * (size_t)e->pitch * sizeof(float) + 32));
  ASZ_CUDA(cudaMalloc(&e->row_ids, rows * sizeof(int32_t)));
  // the kernel's scheduling word (low half: rows of the step, high half: tickets handed out) and its alternate, 64 bytes apart
  ASZ_CUDA(cudaMalloc(&e->row_count, kSchedBytes));
  ASZ_CUDA(cudaMemset(e->row_count, 0, kSchedBytes));
  ASZ_CUDA(cudaMalloc(&e->totals, 32 * sizeof(unsigned long long)));   // [0..15] totals, [16..23] profile build's cycle sums
  ASZ_CUDA(cudaMemset(e->totals, 0, 32 * sizeof(unsigned long long)));
  if (cfg->max_breadth > 0) {
    rc = search_create(e);
    if (rc != ASZ_OK) return rc;
  }
  return ASZ_OK;
}


int asz_engine_create(asz_engine** out, const asz_config* cfg) {
  if (!out || !cfg) { set_error("asz_engine_create: null argument"); return ASZ_ERR_ARG; }
  if (cfg->side != 7 && cfg->side != 11 && cfg->side != 19) { set_error("side must be 7, 11 or 19"); return ASZ_ERR_ARG; }
  if (cfg->snakes < 1 || cfg->snakes > ASZ_MAX_SNAKES) { set_error("snakes must be in 1..8"); return ASZ_ERR_ARG; }
  if (cfg->games < 1) { set_error("games must be >= 1"); return ASZ_ERR_ARG; }
  if (cfg->health_dec < 0 || cfg->health_dec > 100) { set_error("health_dec out of range"); return ASZ_ERR_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("no CUDA device: this engine has no CPU fallback");
    return ASZ_ERR_CUDA;
  }
  asz_engine* e = new asz_engine();
  const int rc = engine_alloc(e, cfg);
  if (rc != ASZ_OK) { asz_engine_destroy(e); return rc; }
  *out = e;
  return ASZ_OK;
}

int asz_engine_destroy(asz_engine* e) {
  if (!e) return ASZ_OK;
  DeviceGuard guard(e->device);
  cudaDeviceSynchronize();   // launches and copies still in flight (asz_env_submit_host never waited for) use the buffers freed below
  search_destroy(e);
  records_destroy(e);
  pit_destroy(e);
  host_pipe_destroy(e);
  gameset_free(e->root);
  cudaFree(e->planes); cudaFree(e->row_ids); cudaFree(e->row_count); cudaFree(e->totals);
  delete e;
  return ASZ_OK;
}

static int reset_games(asz_engine* e, cudaStream_t st) {
  ASZ_CUDA(cudaMemsetAsync(e->totals, 0, 32 * sizeof(unsigned long long), st));
  switch (e->cfg.side) {
    case 7: return EnvLaunch<7>::reset(e->root, e->cfg.snakes, e->cfg.seed, st);
    case 11: return EnvLaunch<11>::reset(e->root, e->cfg.snakes, e->cfg.seed, st);
    default: return EnvLaunch<19>::reset(e->root, e->cfg.snakes, e->cfg.seed, st);
  }
}

int asz_reset(asz_engine* e, void* stream) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  return reset_games(e, (cudaStream_t)stream);
}

int asz_env_step(asz_engine* e, const asz_step_args* a, void* stream) {
  if (!e || !a) { set_error("null argument"); return ASZ_ERR_ARG; }
  if ((a->flags & ASZ_STEP_ENCODE) && (!a->d_planes || !a->d_row_ids || !a->d_row_count || a->max_rows <= 0)) {
    set_error("ASZ_STEP_ENCODE needs d_planes, d_row_ids, d_row_count and max_rows"); return ASZ_ERR_ARG;
  }
  if ((a->flags & ASZ_STEP_ENCODE) && ((uintptr_t)a->d_planes & 31u)) { set_error("d_planes must be 32-byte aligned"); return ASZ_ERR_ARG; }
  // the encode writes whole rows of plane_pitch floats (pad included): a buffer sized for rows of any other length would be
  // written past its end
  if ((a->flags & ASZ_STEP_ENCODE) && a->plane_pitch != e->pitch) {
    set_error("plane_pitch is " + std::to_string(a->plane_pitch) + ": it must equal asz_plane_pitch() = " + std::to_string(e->pitch));
    return ASZ_ERR_ARG;
  }
  if ((a->flags & ASZ_STEP_KEYS) && !a->d_keys) { set_error("ASZ_STEP_KEYS needs d_keys"); return ASZ_ERR_ARG; }
  if ((a->flags & ASZ_STEP_TIC) && !(a->flags & ASZ_STEP_RANDOM_ACT) && !a->d_actions) { set_error("d_actions is null"); return ASZ_ERR_ARG; }
  if ((a->flags & ASZ_STEP_TIC) && !(a->flags & ASZ_STEP_RANDOM_ACT) && ((uintptr_t)a->d_actions & 7u)) { set_error("d_actions must be 8-byte aligned"); return ASZ_ERR_ARG; }
  if ((a->flags & ASZ_STEP_TIC) && a->spawn_mode == ASZ_SPAWN_REPLAY && !a->d_spawn_cells) { set_error("d_spawn_cells is null"); return ASZ_ERR_ARG; }
  if (a->spawn_mode < 0 || a->spawn_mode > 2) { set_error("bad spawn_mode"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:env_step (tic + encode)");
  cudaStream_t st = (cudaStream_t)stream;
  EnvParams p;
  p.device = e->device; p.n_sm = e->n_sm;
  p.cells = e->root.cells; p.snakes = e->root.snakes; p.meta = e->root.meta;
  p.G = e->cfg.games; p.S = e->cfg.snakes; p.health_dec = e->cfg.health_dec;
  p.flags = a->flags; p.spawn_mode = a->spawn_mode; p.chance_thresh = e->chance_thresh; p.seed = e->cfg.seed;
  p.actions = a->d_actions; p.spawn_cells = a->d_spawn_cells;
  if (a->row_base < 0 || ((a->flags & ASZ_STEP_ENCODE) && a->row_base > a->max_rows)) { set_error("row_base out of range"); return ASZ_ERR_ARG; }
  p.planes = a->d_planes; p.row_ids = a->d_row_ids; p.keys = a->d_keys; p.max_rows = a->max_rows; p.row_base = a->row_base;
  // Rows are always counted in the engine's own scheduling word and copied to the caller's d_row_count after the launch.  The
  // engine alternates between two words: this launch uses the one the previous launch zeroed and zeroes the other one (whose row
  // count every stream-ordered reader of the previous launch has consumed by the time this kernel runs), so there is no memset
  // node between two launches.
  const bool own_count = a->d_row_count != nullptr && reinterpret_cast<const char*>(a->d_row_count) >= reinterpret_cast<const char*>(e->row_count) &&
                         reinterpret_cast<const char*>(a->d_row_count) < reinterpret_cast<const char*>(e->row_count) + kSchedBytes;
  const int flip = e->sched_flip ^ 1;                                // committed when the launch has been enqueued
  char* const pair = reinterpret_cast<char*>(e->row_count);
  p.sched = reinterpret_cast<unsigned long long*>(pair + (flip ? 64 : 0));       // low word = the row count the callers read
  p.sched_next = reinterpret_cast<unsigned long long*>(pair + (flip ? 0 : 64));
  p.row_count = reinterpret_cast<int32_t*>(p.sched);
  p.ended = a->d_ended; p.rewards = a->d_rewards; p.totals = e->totals; p.prof = e->totals + 16;
  int rc;
  switch (e->cfg.side) {
    case 7: rc = EnvLaunch<7>::step(p, st); break;
    case 11: rc = EnvLaunch<11>::step(p, st); break;
    default: rc = EnvLaunch<19>::step(p, st); break;
  }
  if (rc != ASZ_OK) return rc;
  e->sched_flip = flip;
  if (a->d_row_count && !own_count)
    ASZ_CUDA(cudaMemcpyAsync(a->d_row_count, e->rows_ptr(), sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return ASZ_OK;
}

// ---- host-buffer path: submit / wait, two steps in flight ------------------------------------------------------------------------
// The step's inputs go host -> device on the engine's own copy stream, so that the copy of step k+1 runs under the kernel of
// step k; the kernel waits for its copy through an event.  The per-game results are written by the kernel itself into the
// caller's pinned buffers (posted PCIe writes while the launch runs); the row count follows as one 4-byte copy into a pinned word
// of the slot, then the slot's event.  asz_env_wait_host blocks on that event only.
static int host_pipe_create(asz_engine* e) {
  asz_engine::HostPipe& hp = e->hostpipe;
  if (hp.ready) return ASZ_OK;
  const size_t G = (size_t)e->cfg.games;
  ASZ_CUDA(cudaStreamCreateWithFlags(&hp.copy, cudaStreamNonBlocking));
  ASZ_CUDA(cudaStreamCreateWithFlags(&hp.copy_out, cudaStreamNonBlocking));
  ASZ_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&hp.h_rows), 2 * 16 * sizeof(int32_t), cudaHostAllocDefault));
  for (int i = 0; i < 2; ++i) {
    ASZ_CUDA(cudaEventCreateWithFlags(&hp.copied[i], cudaEventDisableTiming));
    ASZ_CUDA(cudaEventCreateWithFlags(&hp.done[i], cudaEventDisableTiming));
    ASZ_CUDA(cudaEventCreateWithFlags(&hp.stepped[i], cudaEventDisableTiming));
    ASZ_CUDA(cudaMalloc(&hp.actions[i], G * 8));
    ASZ_CUDA(cudaMalloc(&hp.spawn[i], G * sizeof(int32_t)));
    ASZ_CUDA(cudaMalloc(&hp.d_ended[i], G));
    ASZ_CUDA(cudaMalloc(&hp.d_rewards[i], G * 8));
    ASZ_CUDA(cudaMalloc(&hp.d_rows[i], 64));
  }
  hp.ready = true;
  return ASZ_OK;
}

}  // extern "C"
namespace asz {
void host_pipe_destroy(asz_engine* e) {
  asz_engine::HostPipe& hp = e->hostpipe;
  for (int i = 0; i < 2; ++i) {
    if (hp.copied[i]) cudaEventDestroy(hp.copied[i]);
    if (hp.done[i]) cudaEventDestroy(hp.done[i]);
    if (hp.stepped[i]) cudaEventDestroy(hp.stepped[i]);
    cudaFree(hp.actions[i]); cudaFree(hp.spawn[i]); cudaFree(hp.d_ended[i]); cudaFree(hp.d_rewards[i]); cudaFree(hp.d_rows[i]);
  }
  if (hp.h_rows) cudaFreeHost(hp.h_rows);
  if (hp.copy) cudaStreamDestroy(hp.copy);
  if (hp.copy_out) cudaStreamDestroy(hp.copy_out);
  hp = asz_engine::HostPipe();
}
}  // namespace asz
extern "C" {

// device-visible alias of a pinned host buffer (nullptr for pageable memory).  Asked every step on purpose: an address may be
// unpinned and reused between two steps.
static void* pinned_alias(void* h) {
  if (!h) return nullptr;
  cudaPointerAttributes at;
  void* d = nullptr;
  if (cudaPointerGetAttributes(&at, h) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) d = at.devicePointer;
  cudaGetLastError();   // a pageable pointer makes cudaPointerGetAttributes report an error on old drivers: not ours
  return d;
}

// results_by_copy: the kernel writes the per-game results into the slot's device buffers and the engine's second copy stream
// brings them to the host under the NEXT step's kernel (the pipelined calls); otherwise pinned result buffers are written by the
// kernel itself over PCIe while it runs, which costs the kernel ~10 % but leaves nothing to do after it (the blocking call)
static int host_submit(asz_engine* e, uint32_t flags, int32_t spawn_mode, const uint8_t* h_actions, const int32_t* h_spawn_cells,
                       uint8_t* h_ended, int8_t* h_rewards, void* stream, int32_t* ticket, bool results_by_copy) {
  if (!e || !ticket) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:env_submit_host");
  { const int rc0 = host_pipe_create(e); if (rc0 != ASZ_OK) return rc0; }
  asz_engine::HostPipe& hp = e->hostpipe;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t G = (size_t)e->cfg.games;
  const int slot = hp.next;
  if (hp.busy[slot]) { set_error("asz_env_submit_host: two steps are in flight already; asz_env_wait_host the oldest first"); return ASZ_ERR_ARG; }
  const bool need_actions = (flags & ASZ_STEP_TIC) && !(flags & ASZ_STEP_RANDOM_ACT);
  const bool need_spawn = (flags & ASZ_STEP_TIC) && spawn_mode == ASZ_SPAWN_REPLAY;
  if (need_actions && !h_actions) { set_error("h_actions is null"); return ASZ_ERR_ARG; }
  if (need_spawn && !h_spawn_cells) { set_error("h_spawn_cells is null"); return ASZ_ERR_ARG; }
  if (need_actions || need_spawn) {
    // the slot's device buffers were last read by the step waited for two submissions ago: free to overwrite
    if (need_actions) ASZ_CUDA(cudaMemcpyAsync(hp.actions[slot], h_actions, G * 8, cudaMemcpyHostToDevice, hp.copy));
    if (need_spawn) ASZ_CUDA(cudaMemcpyAsync(hp.spawn[slot], h_spawn_cells, G * sizeof(int32_t), cudaMemcpyHostToDevice, hp.copy));
    ASZ_CUDA(cudaEventRecord(hp.copied[slot], hp.copy));
    ASZ_CUDA(cudaStreamWaitEvent(st, hp.copied[slot], 0));
  }
  asz_step_args a;
  memset(&a, 0, sizeof a);
  a.flags = flags; a.spawn_mode = spawn_mode; a.d_actions = hp.actions[slot]; a.d_spawn_cells = hp.spawn[slot];
  a.d_planes = e->planes; a.d_row_ids = e->row_ids; a.max_rows = (int32_t)(G * (size_t)e->cfg.snakes); a.plane_pitch = e->pitch;
  a.d_row_count = e->rows_ptr(); a.d_ended = hp.d_ended[slot]; a.d_rewards = hp.d_rewards[slot];
  // Result buffers in pinned (page-locked, UVA-mapped) host memory can be written by the kernel itself, one posted PCIe write
  // per game while the launch runs, instead of by two device->host copies after it.
  bool zc_ended = false, zc_rewards = false;
  if (!results_by_copy && (flags & ASZ_STEP_TIC)) {
    if (void* d = pinned_alias(h_ended)) { a.d_ended = static_cast<uint8_t*>(d); zc_ended = true; }
    if (void* d = pinned_alias(h_rewards)) { a.d_rewards = static_cast<int8_t*>(d); zc_rewards = true; }
  }
  const int rc = asz_env_step(e, &a, stream);
  if (rc != ASZ_OK) return rc;
  if (results_by_copy) {
    // the row count leaves the hot word before the next launch zeroes it; everything else waits for the kernel on the out stream
    ASZ_CUDA(cudaMemcpyAsync(hp.d_rows[slot], e->rows_ptr(), sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    ASZ_CUDA(cudaEventRecord(hp.stepped[slot], st));
    ASZ_CUDA(cudaStreamWaitEvent(hp.copy_out, hp.stepped[slot], 0));
    if (h_ended) ASZ_CUDA(cudaMemcpyAsync(h_ended, hp.d_ended[slot], G, cudaMemcpyDeviceToHost, hp.copy_out));
    if (h_rewards) ASZ_CUDA(cudaMemcpyAsync(h_rewards, hp.d_rewards[slot], G * 8, cudaMemcpyDeviceToHost, hp.copy_out));
    ASZ_CUDA(cudaMemcpyAsync(hp.h_rows + 16 * slot, hp.d_rows[slot], sizeof(int32_t), cudaMemcpyDeviceToHost, hp.copy_out));
    ASZ_CUDA(cudaEventRecord(hp.done[slot], hp.copy_out));
  } else {
    if (h_ended && !zc_ended) ASZ_CUDA(cudaMemcpyAsync(h_ended, hp.d_ended[slot], G, cudaMemcpyDeviceToHost, st));
    if (h_rewards && !zc_rewards) ASZ_CUDA(cudaMemcpyAsync(h_rewards, hp.d_rewards[slot], G * 8, cudaMemcpyDeviceToHost, st));
    ASZ_CUDA(cudaMemcpyAsync(hp.h_rows + 16 * slot, e->rows_ptr(), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASZ_CUDA(cudaEventRecord(hp.done[slot], st));
  }
  hp.busy[slot] = true;
  hp.next = slot ^ 1;
  *ticket = slot;
  return ASZ_OK;
}

int asz_env_submit_host(asz_engine* e, uint32_t flags, int32_t spawn_mode, const uint8_t* h_actions,
                        const int32_t* h_spawn_cells, uint8_t* h_ended, int8_t* h_rewards, void* stream, int32_t* ticket) {
  return host_submit(e, flags, spawn_mode, h_actions, h_spawn_cells, h_ended, h_rewards, stream, ticket, true);
}

int asz_env_wait_host(asz_engine* e, int32_t ticket, int32_t* h_row_count) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  asz_engine::HostPipe& hp = e->hostpipe;
  if (ticket < 0 || ticket > 1 || !hp.ready || !hp.busy[ticket]) { set_error("asz_env_wait_host: no step in flight under this ticket"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  hp.busy[ticket] = false;
  ASZ_CUDA(cudaEventSynchronize(hp.done[ticket]));
  if (h_row_count) *h_row_count = hp.h_rows[16 * ticket];
  return ASZ_OK;
}

int asz_env_step_host(asz_engine* e, uint32_t flags, int32_t spawn_mode, const uint8_t* h_actions,
                      const int32_t* h_spawn_cells, uint8_t* h_ended, int8_t* h_rewards, int32_t* h_row_count,
                      float* h_planes, int32_t* h_row_ids, void* stream) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:env_step_host");
  cudaStream_t st = (cudaStream_t)stream;
  int32_t ticket = -1, rows = 0;
  int rc = host_submit(e, flags, spawn_mode, h_actions, h_spawn_cells, h_ended, h_rewards, stream, &ticket, false);
  if (rc != ASZ_OK) return rc;
  rc = asz_env_wait_host(e, ticket, &rows);
  if (rc != ASZ_OK) return rc;
  if (h_row_count) *h_row_count = rows;
  if ((h_planes || h_row_ids) && rows > 0) {
    // the engine's buffer is pitched, the caller's rows are dense: one strided copy
    if (h_planes) ASZ_CUDA(cudaMemcpy2DAsync(h_planes, (size_t)e->plane * sizeof(float), e->planes, (size_t)e->pitch * sizeof(float),
                                             (size_t)e->plane * sizeof(float), (size_t)rows, cudaMemcpyDeviceToHost, st));
    if (h_row_ids) ASZ_CUDA(cudaMemcpyAsync(h_row_ids, e->row_ids, (size_t)rows * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASZ_CUDA(cudaStreamSynchronize(st));
  }
  return ASZ_OK;
}

int asz_get_totals(asz_engine* e, uint64_t* h_totals) {
  if (!e || !h_totals) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  ASZ_CUDA(cudaDeviceSynchronize());
  ASZ_CUDA(cudaMemcpy(h_totals, e->totals, 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return ASZ_OK;
}

int asz_internal_profile(asz_engine* e, uint64_t* h_cycles) {
  if (!e || !h_cycles) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  ASZ_CUDA(cudaDeviceSynchronize());
  ASZ_CUDA(cudaMemcpy(h_cycles, e->totals + 16, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  ASZ_CUDA(cudaMemset(e->totals + 16, 0, 8 * sizeof(uint64_t)));
  return ASZ_OK;
}

int asz_internal_state(asz_engine* e, void** d_ptrs) {
  if (!e || !d_ptrs) { set_error("null argument"); return ASZ_ERR_ARG; }
  d_ptrs[0] = e->root.cells; d_ptrs[1] = e->root.snakes; d_ptrs[2] = e->root.meta;
  return ASZ_OK;
}
float* asz_internal_planes(asz_engine* e) { return e ? e->planes : nullptr; }
int32_t* asz_internal_row_ids(asz_engine* e) { return e ? e->row_ids : nullptr; }
size_t asz_plane_floats(const asz_engine* e) { return e ? (size_t)e->plane : 0; }
size_t asz_plane_pitch(const asz_engine* e) { return e ? (size_t)e->pitch : 0; }

// ---- state interchange (host side conversion between the canonical dump and the packed records) ----------------
static int gs_get_state(const asz_config& cfg, int pc, const GameSet& gs, int32_t game, int32_t* h_snake, int32_t* h_owner,
                        int32_t* h_dist, int32_t* h_food, int32_t* h_counters) {
  if (game < 0 || game >= gs.n) { set_error("game index out of range"); return ASZ_ERR_ARG; }
  const int C = cfg.side * cfg.side;
  std::vector<uint16_t> cells(pc);
  uint64_t sn[8]; uint32_t meta[8];
  ASZ_CUDA(cudaDeviceSynchronize());
  ASZ_CUDA(cudaMemcpy(cells.data(), gs.cells + (size_t)game * pc, pc * sizeof(uint16_t), cudaMemcpyDeviceToHost));
  ASZ_CUDA(cudaMemcpy(sn, gs.snakes + (size_t)game * 8, sizeof sn, cudaMemcpyDeviceToHost));
  ASZ_CUDA(cudaMemcpy(meta, gs.meta + (size_t)game * 8, sizeof meta, cudaMemcpyDeviceToHost));
  for (int c = 0; c < C; ++c) {
    const uint16_t v = cells[c];
    h_food[c] = v == kFood; h_owner[c] = -1; h_dist[c] = 0;
    if (cell_is_body(v)) { h_owner[c] = cell_owner(v); h_dist[c] = cell_dist(v); }
  }
  for (int s = 0; s < cfg.snakes; ++s) {
    const Snake v = unpack_snake(sn[s]);
    int32_t* o = h_snake + 6 * s;
    o[0] = v.alive; o[1] = v.health; o[2] = v.len;
    o[3] = v.last; o[4] = v.head == kNoHead ? -1 : v.head; o[5] = v.reward == 1 ? 1 : v.reward == 2 ? -1 : 0;
  }
  for (int k = 0; k < 5; ++k) h_counters[k] = (int32_t)meta[META_WALL + k];
  h_counters[5] = (int32_t)meta[META_TURN]; h_counters[6] = (int32_t)meta[META_EPISODE]; h_counters[7] = (int32_t)(meta[META_FLAGS] & kMetaDone);
  return ASZ_OK;
}

static int gs_set_state(const asz_config& cfg, int pc, GameSet& gs, int32_t game, const int32_t* h_snake,
                        const int32_t* h_owner, const int32_t* h_dist, const int32_t* h_food, const int32_t* h_counters) {
  if (game < 0 || game >= gs.n) { set_error("game index out of range"); return ASZ_ERR_ARG; }
  const int C = cfg.side * cfg.side;
  std::vector<uint16_t> cells(pc, 0);
  uint64_t sn[8] = {0}; uint32_t meta[8] = {0};
  for (int c = 0; c < C; ++c) {
    if (h_food[c]) cells[c] = kFood;
    else if (h_owner[c] >= 0) {
      if (h_owner[c] >= cfg.snakes || h_dist[c] <= 0 || h_dist[c] > kDistMask) { set_error("bad cell stamp"); return ASZ_ERR_ARG; }
      cells[c] = (uint16_t)((h_owner[c] << 12) | h_dist[c]);
    }
  }
  int live = 0;
  for (int s = 0; s < 8; ++s) {
    uint64_t v = kEmptySnake;
    if (s < cfg.snakes) {
      const int32_t* o = h_snake + 6 * s;
      const int alive = o[0] != 0, hp = alive ? o[1] : 0;
      live += alive;
      if (hp < -32768 || hp > 32767) { set_error("health out of range"); return ASZ_ERR_ARG; }
      Snake r;
      r.head = (alive && o[4] >= 0) ? o[4] : kNoHead; r.len = alive ? o[2] : 0; r.health = hp;
      r.last = o[3]; r.alive = alive; r.reward = o[5] > 0 ? 1 : o[5] < 0 ? 2 : 0;
      v = pack_snake(r);
    }
    sn[s] = v;
  }
  meta[META_TURN] = (uint32_t)h_counters[5]; meta[META_EPISODE] = (uint32_t)h_counters[6];
  for (int k = 0; k < 5; ++k) meta[META_WALL + k] = (uint32_t)h_counters[k];
  meta[META_FLAGS] = (h_counters[7] != 0 || live <= 1) ? kMetaDone : 0u;
  ASZ_CUDA(cudaDeviceSynchronize());
  ASZ_CUDA(cudaMemcpy(gs.cells + (size_t)game * pc, cells.data(), pc * sizeof(uint16_t), cudaMemcpyHostToDevice));
  ASZ_CUDA(cudaMemcpy(gs.snakes + (size_t)game * 8, sn, sizeof sn, cudaMemcpyHostToDevice));
  ASZ_CUDA(cudaMemcpy(gs.meta + (size_t)game * 8, meta, sizeof meta, cudaMemcpyHostToDevice));
  return ASZ_OK;
}

int asz_get_state(asz_engine* e, int32_t game, int32_t* h_snake, int32_t* h_owner, int32_t* h_dist, int32_t* h_food,
                  int32_t* h_counters) {
  if (!e || !h_snake || !h_owner || !h_dist || !h_food || !h_counters) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  return gs_get_state(e->cfg, e->pc, e->root, game, h_snake, h_owner, h_dist, h_food, h_counters);
}
int asz_set_state(asz_engine* e, int32_t game, const int32_t* h_snake, const int32_t* h_owner, const int32_t* h_dist,
                  const int32_t* h_food, const int32_t* h_counters) {
  if (!e || !h_snake || !h_owner || !h_dist || !h_food || !h_counters) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  return gs_set_state(e->cfg, e->pc, e->root, game, h_snake, h_owner, h_dist, h_food, h_counters);
}

}  // extern "C"
