// asz_pit.cu -- the pit (pit_mp_game_runner.py:14-63 with pit_agent.py:10-28 on both sides) as a device-resident match over
// the engine's root games.  Per turn, where the reference's loop runs on the host:
//   pit_mp_game_runner.py:27-34  team split of the live rows          pit_slot_map_kernel + pit_partition_kernel + pit_gather_kernel
//   pit_agent.py:11 AlphaNNet.v   network forward per side            asz_net_forward_pitched on the team buffer (asz_net.cu)
//   alpha_nnet.py:63-76, pit_agent.py:16-23  obstacle mask + argmaxs  pit_policy_kernel
//   pit_mp_game_runner.py:39-42  actions (np.ones), Game.tic          asz_env_step (TIC | ENCODE)
//   pit_mp_game_runner.py:44-60  winner bookkeeping, early exit       pit_referee_kernel
// The host waits once per turn, for one 12-byte line: the row counts of the two teams (they size the forwards) and the number of
// games still running.
// A side with a searcher engine attached (asz_pit_set_search) plays the search Agent instead (agent.py:25-111, training=False):
//   asz_copy_root_games                 the running games into the searcher (the others arrive finished)   copy_root_games_kernel
//   Agent.make_moves                    root-turn search with the side's network or stand-in              asz_search_run_net / _stub
//   agent.py:98-99 argmaxs of root Q    the side's moves from the searcher's root moves                   pit_policy_kernel
// A search waits on the host once per search step (asz_search_run_net), on top of the turn's one wait.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <string>

#include "asz_engine.hpp"
#include "asz_game.cuh"

namespace asz {

struct PitState {
  int G = 0, S = 0, rows = 0;          // rows = G*S: capacity of every per-row buffer
  uint8_t* running = nullptr;          // [G]
  int32_t* winner = nullptr;           // [G] snake id, -1 = draw or undecided
  int32_t* decided = nullptr;          // [G] tics played when decided, -1 = running
  uint8_t* actions = nullptr;          // [G*8] moves of the step
  int32_t* spawn = nullptr;            // [G] the caller's spawn trace, clamped
  uint8_t* ended = nullptr;            // [G] results of the step
  int8_t* rewards = nullptr;           // [G*8]
  int32_t* row_count = nullptr;        // [1] rows of the last encode
  int32_t* row_of_slot = nullptr;      // [G*8] encode row of (game, snake), -1 = none
  int32_t* src_of_dst = nullptr;       // [rows] encode row of each team-buffer row
  int32_t* slot_of_dst = nullptr;      // [rows] game*8 + snake of each team-buffer row
  float* team = nullptr;               // [rows][pitch] Alice's rows at [0, nA), Bob's at [nA, nA + nB)
  float* values = nullptr;             // [rows][3] raw network outputs
  uint64_t* keys = nullptr;            // [rows*2] plane keys of the encode (allocated when a stand-in plays)
  int32_t* line = nullptr;             // device [4]: nA, nB, running
  int32_t* h_line = nullptr;           // pinned copy
  cudaEvent_t fwd_begin = nullptr, fwd_end = nullptr;
  asz_net* net[2] = {nullptr, nullptr};
  int word[2] = {-1, -1};              // stand-in key word per side, -1 = network
  asz_engine* searcher[2] = {nullptr, nullptr};   // the match's searcher per side (asz_pit_set_search at asz_pit_begin)
  int alice = 0;
  bool open = false;
  int turn = 0;
  double n_net_rows = 0.0, n_stub_rows = 0.0, fwd_ms = 0.0;
  double n_search_rows = 0.0, search_ms = 0.0;
};

struct PitParams {
  int G, S, rows, alice, side, pitch, numpy1_mask, nA, turn;
  int word_a, word_b;
  const uint8_t* root_moves_a; const uint8_t* root_moves_b;   // a searched side's moves by slot, null = argmax of its values
  const uint64_t* snakes; const uint32_t* meta;
  uint8_t* running; int32_t* winner; int32_t* decided;
  uint8_t* actions; uint8_t* moves;
  const uint8_t* ended; const int8_t* rewards;
  const int32_t* row_ids; const int32_t* row_count; int32_t* row_of_slot;
  int32_t* src_of_dst; int32_t* slot_of_dst;
  const float* planes; float* team; const float* values; const uint64_t* keys;
  int32_t* line;
};

constexpr int kPartThreads = 1024;   // one block: 32 warps, one warp sum each

// Match start: running = not finished; a game finished before the match is decided at turn 0 with no winner.
__global__ void pit_begin_kernel(const PitParams p) {
  const int g = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  bool run = false;
  if (g < p.G) {
    run = !(p.meta[(size_t)g * 8 + META_FLAGS] & kMetaDone);
    p.running[g] = run ? 1 : 0;
    p.winner[g] = -1;
    p.decided[g] = run ? -1 : 0;
  }
  const unsigned b = __ballot_sync(kFull, run);   // one atomic per warp, not per game (same-address atomics serialise, DESIGN.md 4.1)
  if (lane_id() == 0 && b) atomicAdd(&p.line[2], __popc(b));
}

// encode row of every (game, snake) slot: the encode hands rows out in unspecified game order
__global__ void pit_slot_map_kernel(const PitParams p) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= p.rows || i >= *p.row_count) return;
  p.row_of_slot[p.row_ids[i]] = i;
}

__device__ __forceinline__ int block_excl_scan(int v, int* warp_sums, int* total) {
  const int lane = lane_id(), warp = (int)(threadIdx.x >> 5);
  const int incl = warp_excl_scan_i32(v, lane) + v;
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int w = warp_sums[lane];
    const int ex = warp_excl_scan_i32(w, lane);
    warp_sums[lane] = ex;
    if (lane == 31) *total = ex + w;
  }
  __syncthreads();
  const int r = warp_sums[warp] + incl - v;
  __syncthreads();   // warp_sums is reused by the next scan
  return r;
}

// pit_mp_game_runner.py:30-33: the rows of running games, Alice's (snake id < alice) first, then Bob's, each team in (game, snake)
// order.  One block; thread t owns a contiguous range of games, so thread order is game order.  Each thread walks ceil(G / 1024)
// games twice, serially: 16 at 16,384 games, 64 at the 65,536 games of the engine's largest workloads.  The kernel's time grows
// linearly with G beyond that (tools/bench_pit.py reports what the non-forward part of a turn costs); a multi-block scan is
// the change to make if pits of ~10^6 games are ever played.
__global__ void __launch_bounds__(kPartThreads) pit_partition_kernel(const PitParams p) {
  __shared__ int warp_sums[32];
  __shared__ int totals[2];
  const int per = (p.G + kPartThreads - 1) / kPartThreads;
  const int g0 = (int)threadIdx.x * per, g1 = min(p.G, g0 + per);
  int ca = 0, cb = 0;
  for (int g = g0; g < g1; ++g) {
    if (!p.running[g]) continue;
    for (int s = 0; s < p.S; ++s)
      if (p.row_of_slot[g * 8 + s] >= 0) { if (s < p.alice) ++ca; else ++cb; }
  }
  int oa = block_excl_scan(ca, warp_sums, &totals[0]);
  int ob = block_excl_scan(cb, warp_sums, &totals[1]);
  ob += totals[0];
  for (int g = g0; g < g1; ++g) {
    if (!p.running[g]) continue;
    for (int s = 0; s < p.S; ++s) {
      const int r = p.row_of_slot[g * 8 + s];
      if (r < 0) continue;
      const int d = s < p.alice ? oa++ : ob++;
      p.src_of_dst[d] = r;
      p.slot_of_dst[d] = g * 8 + s;
    }
  }
  if (threadIdx.x == 0) { p.line[0] = totals[0]; p.line[1] = totals[1]; }
}

// one warp per team-buffer row of [first, first + n): copy the plane (pitch floats, 16-byte aligned rows)
__global__ void pit_gather_kernel(const PitParams p, int first, int n) {
  const int k = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (k >= n) return;
  const int w = first + k;
  const float4* src = reinterpret_cast<const float4*>(p.planes + (size_t)p.src_of_dst[w] * p.pitch);
  float4* dst = reinterpret_cast<float4*>(p.team + (size_t)w * p.pitch);
  for (int i = lane_id(); i < p.pitch / 4; i += 32) dst[i] = src[i];
}

// one thread per team-buffer row: the side's values (network outputs or the stand-in's key bits), AlphaNNet.v's obstacle mask
// (alpha_nnet.py:63-76), Agent.argmaxs (pit_agent.py:16-23), the move into its slot.  A searched side's row takes its searcher's
// root move instead; a row the search dropped (Q table overflow, reported as ASZ_ERR_CAPACITY) plays straight, as it does in the
// search's own sub-games.
__global__ void pit_policy_kernel(const PitParams p, int n) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const int slot = p.slot_of_dst[i];
  const uint8_t* root_moves = i < p.nA ? p.root_moves_a : p.root_moves_b;
  uint8_t mv;
  if (root_moves) {
    mv = root_moves[slot];
    if (mv > 2) mv = 1;
  } else {
    const int word = i < p.nA ? p.word_a : p.word_b;
    float v[3];
    if (word < 0) {
      v[0] = p.values[3 * (size_t)i]; v[1] = p.values[3 * (size_t)i + 1]; v[2] = p.values[3 * (size_t)i + 2];
    } else {
      stub_value3(p.keys[2 * (size_t)p.src_of_dst[i] + word], v);
    }
    obstacle_mask3(p.team + (size_t)i * p.pitch, p.side, p.numpy1_mask, v);
    mv = (uint8_t)argmax3(v);
  }
  p.actions[slot] = mv;
  if (p.moves) p.moves[slot] = mv;
}

// asz_copy_root_games: block g copies game g's packed record (cells, snakes, meta), the block copy of search_epoch_begin_kernel.  A
// game whose flag byte reads `skip_if_set` (nonzero / zero) arrives finished (kMetaDone), so a search on the copy leaves it alone.
__global__ void copy_root_games_kernel(const uint16_t* __restrict__ src_cells, const uint64_t* __restrict__ src_snakes,
                                       const uint32_t* __restrict__ src_meta, uint16_t* cells, uint64_t* snakes, uint32_t* meta, int pc,
                                       const uint8_t* flags, int skip_if_set) {
  const int g = (int)blockIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(src_cells + (size_t)g * pc);   // pc is a multiple of 32 cells: 64-byte records
  uint4* dst = reinterpret_cast<uint4*>(cells + (size_t)g * pc);
  for (int i = (int)threadIdx.x; i < pc / 8; i += (int)blockDim.x) dst[i] = src[i];
  if (threadIdx.x < 8) {
    const size_t k = (size_t)g * 8 + threadIdx.x;
    snakes[k] = src_snakes[k];
    uint32_t m = src_meta[k];
    if (threadIdx.x == META_FLAGS && flags && ((flags[g] != 0) == (skip_if_set != 0))) m |= kMetaDone;
    meta[k] = m;
  }
}

// the loop replays np.maximum(spawn_trace[turn], -1)
__global__ void pit_spawn_clamp_kernel(const int32_t* in, int G, int32_t* out) {
  const int g = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (g < G) out[g] = max(in[g], -1);
}

// pit_mp_game_runner.py:44-60, one thread per game, after the tic
__global__ void pit_referee_kernel(const PitParams p) {
  const int g = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  bool still = false;
  if (g < p.G && p.running[g]) {
    int w = -1;
    bool done = false;
    if (p.ended[g]) {                      // :44-48 the lowest id with reward +1, else a draw
      for (int s = p.S - 1; s >= 0; --s)
        if (p.rewards[(size_t)g * 8 + s] == 1) w = s;
      done = true;
    } else {                               // :49-60 a team without live snakes: the lowest live id wins
      unsigned live = 0;
      for (int s = 0; s < p.S; ++s)
        if (snake_alive(p.snakes[(size_t)g * 8 + s])) live |= 1u << s;
      const unsigned amask = (1u << p.alice) - 1u;
      if (!(live & amask) || !(live & ~amask)) { done = true; w = live ? __ffs(live) - 1 : -1; }
    }
    if (done) { p.winner[g] = w; p.decided[g] = p.turn; p.running[g] = 0; }
    still = !done;
  }
  const unsigned b = __ballot_sync(kFull, still);
  if (lane_id() == 0 && b) atomicAdd(&p.line[2], __popc(b));
}

static int pit_create(asz_engine* e) {
  if (e->pit) return ASZ_OK;
  PitState* s = new PitState();
  e->pit = s;
  s->G = e->cfg.games; s->S = e->cfg.snakes; s->rows = s->G * s->S;
  const size_t G = (size_t)s->G, rows = (size_t)s->rows;
  ASZ_CUDA(cudaMalloc(&s->running, G));
  ASZ_CUDA(cudaMalloc(&s->winner, G * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->decided, G * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->actions, G * 8));
  ASZ_CUDA(cudaMalloc(&s->spawn, G * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->ended, G));
  ASZ_CUDA(cudaMalloc(&s->rewards, G * 8));
  ASZ_CUDA(cudaMalloc(&s->row_count, sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->row_of_slot, G * 8 * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->src_of_dst, rows * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->slot_of_dst, rows * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->team, rows * (size_t)e->pitch * sizeof(float) + 32));
  ASZ_CUDA(cudaMalloc(&s->values, rows * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&s->line, 4 * sizeof(int32_t)));
  ASZ_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&s->h_line), 16 * sizeof(int32_t), cudaHostAllocDefault));
  ASZ_CUDA(cudaEventCreate(&s->fwd_begin));
  ASZ_CUDA(cudaEventCreate(&s->fwd_end));
  return ASZ_OK;
}

void pit_destroy(asz_engine* e) {
  PitState* s = e->pit;
  if (!s) return;
  cudaFree(s->running); cudaFree(s->winner); cudaFree(s->decided); cudaFree(s->actions); cudaFree(s->spawn); cudaFree(s->ended);
  cudaFree(s->rewards); cudaFree(s->row_count); cudaFree(s->row_of_slot); cudaFree(s->src_of_dst); cudaFree(s->slot_of_dst);
  cudaFree(s->team); cudaFree(s->values); cudaFree(s->keys); cudaFree(s->line);
  if (s->h_line) cudaFreeHost(s->h_line);
  if (s->fwd_begin) cudaEventDestroy(s->fwd_begin);
  if (s->fwd_end) cudaEventDestroy(s->fwd_end);
  delete s;
  e->pit = nullptr;
}

static PitParams make_params(asz_engine* e) {
  PitState* s = e->pit;
  PitParams p;
  memset(&p, 0, sizeof p);
  p.G = s->G; p.S = s->S; p.rows = s->rows; p.alice = s->alice; p.side = e->cfg.side; p.pitch = e->pitch; p.numpy1_mask = e->cfg.numpy1_mask;
  p.turn = s->turn; p.word_a = s->word[0]; p.word_b = s->word[1];
  p.snakes = e->root.snakes; p.meta = e->root.meta;
  p.running = s->running; p.winner = s->winner; p.decided = s->decided;
  p.actions = s->actions; p.ended = s->ended; p.rewards = s->rewards;
  p.row_ids = e->row_ids; p.row_count = s->row_count; p.row_of_slot = s->row_of_slot;
  p.src_of_dst = s->src_of_dst; p.slot_of_dst = s->slot_of_dst;
  p.planes = e->planes; p.team = s->team; p.values = s->values; p.keys = s->keys;
  p.line = s->line;
  return p;
}

// a stand-in side without a searcher values the engine's own encode: the encode writes plane keys
static bool stub_plays(const PitState* s) {
  return (s->word[0] >= 0 && !s->searcher[0]) || (s->word[1] >= 0 && !s->searcher[1]);
}

static int copy_root_games(asz_engine* dst, const asz_engine* src, const uint8_t* flags, int skip_if_set, cudaStream_t st) {
  copy_root_games_kernel<<<src->cfg.games, 64, 0, st>>>(src->root.cells, src->root.snakes, src->root.meta, dst->root.cells,
                                                         dst->root.snakes, dst->root.meta, src->pc, flags, skip_if_set);
  return cuda_ok(cudaGetLastError(), "copy_root_games_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

// one searched side's turn: the running games into its searcher, the root-turn search with the side's network (or stand-in with
// the side's key word), the root moves left in the searcher's buffer for pit_policy_kernel
static int pit_search_side(asz_engine* e, int side, cudaStream_t st) {
  PitState* s = e->pit;
  asz_engine* q = s->searcher[side];
  const auto t0 = std::chrono::steady_clock::now();
  int rc = copy_root_games(q, e, s->running, 0, st);
  if (rc != ASZ_OK) return rc;
  if (s->net[side]) {
    rc = asz_search_run_net(q, s->net[side], nullptr, 0, nullptr, st);
  } else {
    search_set_stub_word(q, s->word[side]);
    rc = asz_search_run_stub(q, nullptr, 0, nullptr, st);
    search_set_stub_word(q, 1);
  }
  // every search ends in a host synchronisation (asz_search_finish), so the host clock spans the device work
  s->search_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

// Game.tic of every unfinished game (tic) and the planes of every live snake into the engine's plane buffer
static int pit_step(asz_engine* e, bool tic, int32_t spawn_mode, const int32_t* spawn, cudaStream_t st) {
  PitState* s = e->pit;
  asz_step_args a;
  memset(&a, 0, sizeof a);
  a.flags = (tic ? ASZ_STEP_TIC : 0u) | ASZ_STEP_ENCODE | (stub_plays(s) ? ASZ_STEP_KEYS : 0u);
  a.spawn_mode = spawn_mode;
  a.d_actions = s->actions; a.d_spawn_cells = spawn;
  a.d_planes = e->planes; a.d_row_ids = e->row_ids; a.d_keys = stub_plays(s) ? s->keys : nullptr; a.max_rows = s->rows;
  a.d_row_count = s->row_count; a.d_ended = s->ended; a.d_rewards = s->rewards;
  a.plane_pitch = e->pitch;
  return asz_env_step(e, &a, st);
}

// after an encode and the referee: the team buffer's row lists, then the host's one wait of the turn
static int pit_partition(asz_engine* e, cudaStream_t st) {
  PitState* s = e->pit;
  const PitParams p = make_params(e);
  ASZ_CUDA(cudaMemsetAsync(s->row_of_slot, 0xFF, (size_t)s->G * 8 * sizeof(int32_t), st));
  pit_slot_map_kernel<<<(s->rows + 255) / 256, 256, 0, st>>>(p);
  if (!cuda_ok(cudaGetLastError(), "pit_slot_map_kernel")) return ASZ_ERR_CUDA;
  pit_partition_kernel<<<1, kPartThreads, 0, st>>>(p);
  if (!cuda_ok(cudaGetLastError(), "pit_partition_kernel")) return ASZ_ERR_CUDA;
  ASZ_CUDA(cudaMemcpyAsync(s->h_line, s->line, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  ASZ_CUDA(cudaStreamSynchronize(st));
  return ASZ_OK;
}

static int check_player(const asz_engine* e, const asz_pit_player* pl, const char* who) {
  char msg[160];
  if (!pl) { snprintf(msg, sizeof msg, "asz_pit_begin: %s is null", who); set_error(msg); return ASZ_ERR_ARG; }
  if (pl->net) {
    if (net_side(pl->net) != e->cfg.side) {
      snprintf(msg, sizeof msg, "asz_pit_begin: %s's network is for side %d, the engine's boards have side %d", who,
               net_side(pl->net), e->cfg.side);
      set_error(msg); return ASZ_ERR_ARG;
    }
    if (net_device(pl->net) != e->device) {
      snprintf(msg, sizeof msg, "asz_pit_begin: %s's network is on device %d, the engine on device %d", who, net_device(pl->net),
               e->device);
      set_error(msg); return ASZ_ERR_ARG;
    }
  } else if (pl->stub_word != 0 && pl->stub_word != 1) {
    snprintf(msg, sizeof msg, "asz_pit_begin: %s's stub_word must be 0 or 1", who); set_error(msg); return ASZ_ERR_ARG;
  }
  return ASZ_OK;
}

// games of the same shape on the same device: the packed records of one engine are records of the other
static bool same_games(const asz_engine* a, const asz_engine* b) {
  return a->cfg.side == b->cfg.side && a->cfg.snakes == b->cfg.snakes && a->cfg.games == b->cfg.games && a->device == b->device;
}

static int check_searcher(const asz_engine* e, const asz_engine* q, const char* who) {
  if (!q) return ASZ_OK;
  char msg[200];
  const char* why = nullptr;
  if (q == e) why = "is the match's own engine";
  else if (!q->search) why = "has no search configured (max_breadth 0)";
  else if (q->cfg.training) why = "is a training search (a pit plays with training = 0)";
  else if (!same_games(e, q)) why = "differs from the engine in board side, snake count, game count or device";
  else if (q->cfg.health_dec != e->cfg.health_dec || q->cfg.numpy1_mask != e->cfg.numpy1_mask)
    why = "differs from the engine in health_dec or numpy1_mask (its sub-games would not be the match's games)";
  if (!why) return ASZ_OK;
  snprintf(msg, sizeof msg, "asz_pit_begin: %s's searcher %s", who, why);
  set_error(msg);
  return ASZ_ERR_ARG;
}

}  // namespace asz

using namespace asz;

extern "C" {

int asz_pit_begin(asz_engine* e, const asz_pit_player* alice, const asz_pit_player* bob, int32_t alice_snakes, int32_t* h_running,
                  void* stream) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  if (e->pit) e->pit->open = false;   // a new begin abandons the match in progress, whether or not it starts a new one
  int rc;
  if ((rc = check_player(e, alice, "Alice")) != ASZ_OK || (rc = check_player(e, bob, "Bob")) != ASZ_OK) return rc;
  if (alice_snakes < 0 || alice_snakes > e->cfg.snakes) { set_error("asz_pit_begin: alice_snakes must be in 0..S"); return ASZ_ERR_ARG; }
  if ((rc = check_searcher(e, e->pit_searcher[0], "Alice")) != ASZ_OK || (rc = check_searcher(e, e->pit_searcher[1], "Bob")) != ASZ_OK)
    return rc;
  if (e->pit_searcher[0] && e->pit_searcher[0] == e->pit_searcher[1]) {
    set_error("asz_pit_begin: one searcher is attached to both sides (each side needs its own Q table)");
    return ASZ_ERR_ARG;
  }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:pit begin");
  if ((rc = pit_create(e)) != ASZ_OK) { pit_destroy(e); return rc; }   // a later begin allocates afresh
  PitState* s = e->pit;
  s->net[0] = alice->net; s->net[1] = bob->net;
  s->word[0] = alice->net ? -1 : alice->stub_word; s->word[1] = bob->net ? -1 : bob->stub_word;
  s->searcher[0] = e->pit_searcher[0]; s->searcher[1] = e->pit_searcher[1];
  s->alice = alice_snakes;
  s->turn = 0;
  s->n_net_rows = s->n_stub_rows = s->fwd_ms = 0.0;
  s->n_search_rows = s->search_ms = 0.0;
  if (stub_plays(s) && !s->keys) ASZ_CUDA(cudaMalloc(&s->keys, (size_t)s->rows * 2 * sizeof(uint64_t)));
  cudaStream_t st = (cudaStream_t)stream;
  for (int side = 0; side < 2; ++side)   // Agent.clear (agent.py:140-147): a match does not depend on earlier matches
    if (s->searcher[side] && (rc = asz_search_clear(s->searcher[side], stream)) != ASZ_OK) return rc;
  ASZ_CUDA(cudaMemsetAsync(s->line, 0, 4 * sizeof(int32_t), st));
  const PitParams p = make_params(e);
  pit_begin_kernel<<<(s->G + 255) / 256, 256, 0, st>>>(p);
  if (!cuda_ok(cudaGetLastError(), "pit_begin_kernel")) return ASZ_ERR_CUDA;
  if ((rc = pit_step(e, false, ASZ_SPAWN_NATIVE, nullptr, st)) != ASZ_OK) return rc;   // pit_mp_game_runner.py:27
  if ((rc = pit_partition(e, st)) != ASZ_OK) return rc;
  s->open = true;
  if (h_running) *h_running = s->h_line[2];
  return ASZ_OK;
}

int asz_pit_turn(asz_engine* e, int32_t spawn_mode, const int32_t* d_spawn_cells, uint8_t* d_moves, int32_t* h_running, void* stream) {
  if (!e || !e->pit || !e->pit->open) { set_error("asz_pit_turn: no match begun (asz_pit_begin)"); return ASZ_ERR_STATE; }
  if (spawn_mode < ASZ_SPAWN_NONE || spawn_mode > ASZ_SPAWN_NATIVE) { set_error("asz_pit_turn: bad spawn_mode"); return ASZ_ERR_ARG; }
  if (spawn_mode == ASZ_SPAWN_REPLAY && !d_spawn_cells) { set_error("asz_pit_turn: ASZ_SPAWN_REPLAY needs d_spawn_cells"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:pit turn");
  PitState* s = e->pit;
  cudaStream_t st = (cudaStream_t)stream;
  if (d_moves) ASZ_CUDA(cudaMemsetAsync(d_moves, 255, (size_t)s->G * 8, st));
  if (s->h_line[2] == 0) {
    if (h_running) *h_running = 0;
    return ASZ_OK;
  }
  const int nA = s->h_line[0], nB = s->h_line[1], n = nA + nB;
  ASZ_CUDA(cudaMemsetAsync(s->actions, 1, (size_t)s->G * 8, st));   // pit_mp_game_runner.py:39 np.ones((G, 8))
  PitParams p = make_params(e);
  p.nA = nA; p.moves = d_moves;
  int rc;
  int overflow = ASZ_OK;           // a searcher's Q table overflowed: the turn is played out, then reported
  std::string overflow_msg;
  bool timed = false;
  if (n > 0) {
    const int seg_begin[2] = {0, nA}, seg_len[2] = {nA, nB};
    const bool searched[2] = {s->searcher[0] != nullptr, s->searcher[1] != nullptr};
    for (int side = 0; side < 2; ++side) {
      if (!searched[side] || seg_len[side] == 0) continue;   // a side with no snake to move does not search
      rc = pit_search_side(e, side, st);
      if (rc == ASZ_ERR_CAPACITY) { overflow = rc; overflow_msg = asz_last_error(); }
      else if (rc != ASZ_OK) return rc;
      (side == 0 ? p.root_moves_a : p.root_moves_b) = asz_search_root_moves(s->searcher[side]);
      s->n_search_rows += seg_len[side];
    }
    // the rows the sides without a searcher value: Alice's segment, Bob's, or both (contiguous either way)
    const int g0 = searched[0] ? nA : 0, g1 = searched[1] ? nA : n;
    if (g1 > g0) {
      pit_gather_kernel<<<(g1 - g0 + 7) / 8, 256, 0, st>>>(p, g0, g1 - g0);
      if (!cuda_ok(cudaGetLastError(), "pit_gather_kernel")) return ASZ_ERR_CUDA;
    }
    // pit_agent.py:11 nnet.v(states): one forward per side, or one over both segments when the sides share a network
    const bool shared = s->net[0] && s->net[0] == s->net[1] && !searched[0] && !searched[1];
    timed = (s->net[0] && !searched[0] && nA > 0) || (s->net[1] && !searched[1] && nB > 0);
    if (timed) ASZ_CUDA(cudaEventRecord(s->fwd_begin, st));
    for (int side = 0; side < (shared ? 1 : 2); ++side) {
      const int begin = seg_begin[side], len = shared ? n : seg_len[side];
      if (!s->net[side] || searched[side] || len == 0) continue;
      if ((rc = asz_net_forward_pitched(s->net[side], s->team + (size_t)begin * e->pitch, e->pitch, len, s->values + (size_t)begin * 3,
                                        stream)) != ASZ_OK)
        return rc;
    }
    if (timed) ASZ_CUDA(cudaEventRecord(s->fwd_end, st));
    for (int side = 0; side < 2; ++side)
      if (!searched[side]) (s->net[side] ? s->n_net_rows : s->n_stub_rows) += seg_len[side];
    pit_policy_kernel<<<(n + 127) / 128, 128, 0, st>>>(p, n);
    if (!cuda_ok(cudaGetLastError(), "pit_policy_kernel")) return ASZ_ERR_CUDA;
  }
  const int32_t* spawn = nullptr;
  if (spawn_mode == ASZ_SPAWN_REPLAY) {
    pit_spawn_clamp_kernel<<<(s->G + 255) / 256, 256, 0, st>>>(d_spawn_cells, s->G, s->spawn);
    if (!cuda_ok(cudaGetLastError(), "pit_spawn_clamp_kernel")) return ASZ_ERR_CUDA;
    spawn = s->spawn;
  }
  if ((rc = pit_step(e, true, spawn_mode, spawn, st)) != ASZ_OK) return rc;   // pit_mp_game_runner.py:42
  s->turn += 1;
  p.turn = s->turn;
  ASZ_CUDA(cudaMemsetAsync(s->line, 0, 4 * sizeof(int32_t), st));
  pit_referee_kernel<<<(s->G + 255) / 256, 256, 0, st>>>(p);
  if (!cuda_ok(cudaGetLastError(), "pit_referee_kernel")) return ASZ_ERR_CUDA;
  if ((rc = pit_partition(e, st)) != ASZ_OK) return rc;   // the turn's one host wait
  if (timed) {
    float ms = 0.0f;
    ASZ_CUDA(cudaEventElapsedTime(&ms, s->fwd_begin, s->fwd_end));
    s->fwd_ms += ms;
  }
  if (h_running) *h_running = s->h_line[2];
  if (overflow != ASZ_OK) set_error(overflow_msg);
  return overflow;
}

int asz_pit_finish(asz_engine* e, int32_t* d_winners, int32_t* d_decided_turn, int32_t* h_turns, void* stream) {
  if (!e || !e->pit || !e->pit->open) { set_error("asz_pit_finish: no match begun (asz_pit_begin)"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  PitState* s = e->pit;
  cudaStream_t st = (cudaStream_t)stream;
  if (d_winners) ASZ_CUDA(cudaMemcpyAsync(d_winners, s->winner, (size_t)s->G * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  if (d_decided_turn) ASZ_CUDA(cudaMemcpyAsync(d_decided_turn, s->decided, (size_t)s->G * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  ASZ_CUDA(cudaStreamSynchronize(st));
  if (h_turns) *h_turns = s->turn;
  s->open = false;
  if (s->h_line[2] > 0) {
    char msg[160];
    snprintf(msg, sizeof msg, "pit match ended after %d turns with %d games still running (results so far written)", s->turn,
             s->h_line[2]);
    set_error(msg);
    return ASZ_ERR_STATE;
  }
  return ASZ_OK;
}

int asz_pit_run(asz_engine* e, const asz_pit_player* alice, const asz_pit_player* bob, int32_t alice_snakes, int32_t max_turns,
                int32_t* d_winners, int32_t* d_decided_turn, int32_t* h_turns, void* stream) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  if (e->pit) e->pit->open = false;   // abandons a match in progress even when this one cannot start
  if (max_turns < 0) { set_error("asz_pit_run: max_turns must be >= 0"); return ASZ_ERR_ARG; }
  int32_t running = 0;
  int rc = asz_pit_begin(e, alice, bob, alice_snakes, &running, stream);
  if (rc != ASZ_OK) return rc;
  for (int t = 0; running > 0 && (max_turns == 0 || t < max_turns); ++t) {
    rc = asz_pit_turn(e, ASZ_SPAWN_NATIVE, nullptr, nullptr, &running, stream);
    if (rc == ASZ_ERR_CAPACITY) {     // a searcher's table overflowed: the match stops with the results so far written
      const std::string msg = asz_last_error();
      const int frc = asz_pit_finish(e, d_winners, d_decided_turn, h_turns, stream);
      if (frc != ASZ_OK && frc != ASZ_ERR_STATE) return frc;
      set_error(msg);
      return rc;
    }
    if (rc != ASZ_OK) {
      e->pit->open = false;           // the match is over either way; ASZ_ERR_STATE stays reserved for "results written"
      return rc;
    }
  }
  return asz_pit_finish(e, d_winners, d_decided_turn, h_turns, stream);
}

int asz_pit_stats(asz_engine* e, double* h_stats) {
  if (!e || !h_stats) { set_error("null argument"); return ASZ_ERR_ARG; }
  const PitState* s = e->pit;
  h_stats[0] = s ? s->turn : 0; h_stats[1] = s ? s->n_net_rows : 0.0; h_stats[2] = s ? s->n_stub_rows : 0.0;
  h_stats[3] = s ? s->fwd_ms : 0.0;
  return ASZ_OK;
}

int asz_pit_search_stats(asz_engine* e, double* h_stats) {
  if (!e || !h_stats) { set_error("null argument"); return ASZ_ERR_ARG; }
  const PitState* s = e->pit;
  h_stats[0] = s ? s->n_search_rows : 0.0; h_stats[1] = s ? s->search_ms : 0.0;
  return ASZ_OK;
}

int asz_pit_set_search(asz_engine* e, int32_t side, asz_engine* searcher) {
  if (!e) { set_error("null engine"); return ASZ_ERR_ARG; }
  if (side != 0 && side != 1) { set_error("asz_pit_set_search: side must be 0 (Alice) or 1 (Bob)"); return ASZ_ERR_ARG; }
  e->pit_searcher[side] = searcher;   // checked against the engine by asz_pit_begin
  return ASZ_OK;
}

int asz_copy_root_games(asz_engine* dst, const asz_engine* src, const uint8_t* d_skip, void* stream) {
  if (!dst || !src) { set_error("null engine"); return ASZ_ERR_ARG; }
  if (!same_games(dst, src)) {
    set_error("asz_copy_root_games: the engines differ in board side, snake count, game count or device");
    return ASZ_ERR_ARG;
  }
  if (dst == src) { set_error("asz_copy_root_games: an engine cannot be copied onto itself"); return ASZ_ERR_ARG; }
  DeviceGuard guard(dst->device);
  return copy_root_games(dst, src, d_skip, 1, (cudaStream_t)stream);
}

}  // extern "C"
