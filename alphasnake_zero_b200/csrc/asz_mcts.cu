// asz_mcts.cu -- the reference's randomized synchronous parallel MCTS (code/utils/agent.py, mp_game_runner.py:79-115)
// as warp-cooperative kernels over device-resident sub-games and a GPU hash table.
//
// Reference loop (SURVEY.md Appendix C) and where it runs here:
//   Agent.make_moves        epoch loop            host loop in asz_search_* calls (sequentially dependent by definition)
//   Game.subgame x 8        agent.py:43-50        search_epoch_begin_kernel  (block copy of the packed records)
//   MCTSAgent.make_moves    agent.py:161-223      search_step_kernel   : tic of the previous step's moves, leave check,
//                                                                        terminal backup, plane key, table probe / insert,
//                                                                        planes of the misses into the eval batch
//                                                 <value network on the eval batch, outside this file>
//                                                 search_sample_kernel : new-node priors, softermax, sample, r-hat
//   path backup             agent.py:208-222      deferred into the next search_step_kernel (atomics on N, W)
//   terminal backup         agent.py:60-72        search_step_kernel when a sub-game leaves
//   root read-out / move    agent.py:74-99        search_root_kernel
//   ageing / eviction       agent.py:30-31,101-110  last-touch stamps, expiry on probe, periodic compaction
//
// Table entry: tag = key0 (0 = empty), check word = key1, W[3], N[3] (float like the reference; Q is W/N on read:
// agent.py:72,220 recompute it after every update so it is never independent state), last-touch root turn, and the
// eval-batch index while the value is pending (agent.py:184 stores None for the same purpose).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "asz_engine.hpp"
#include "asz_game.cuh"

namespace asz {

constexpr uint32_t kNoRow = 0xFFFFFFFFu;
constexpr uint32_t kTouchInvalid = 0xFFFFFFFFu;   // touch stamp of a slot whose insert has not been published yet

struct Table {
  int log2cap = 0;
  uint64_t cap = 0;
  uint64_t* key = nullptr;    // [cap]
  uint64_t* chk = nullptr;    // [cap]
  float4* w = nullptr;        // [cap] W0..2, pad
  float4* n = nullptr;        // [cap] N0..2, pad
  uint32_t* touch = nullptr;  // [cap] root turn of the last touch
  int32_t* eval = nullptr;    // [cap] eval-batch index while pending, -1 when the value is in w/n
};

enum Stat { ST_EVALS = 0, ST_VISITS = 1, ST_HITS = 2, ST_SUBGAMES = 3, ST_SUBTICS = 4, ST_COLLISIONS = 5, ST_INSERTS = 6,
            ST_EXPIRED = 7, ST_OCCUPIED = 8, ST_OVERFLOW = 9, ST_COUNT = 16 };

struct SearchState {
  int P = 0, E = 0, Dmax = 0, n_sub = 0, max_rows = 0;
  GameSet sub;
  int32_t* sub_depth = nullptr;   // [n_sub]
  uint8_t* sub_left = nullptr;    // [n_sub]
  uint8_t* created = nullptr;     // [n_sub] mask of snakes alive at creation (agent.py:158)
  uint32_t* path_slot = nullptr;  // [n_sub*8*Dmax]
  uint8_t* path_move = nullptr;   // [n_sub*8*Dmax]
  uint8_t* path_len = nullptr;    // [n_sub*8]
  uint32_t* row_slot = nullptr;   // [n_sub*8]
  uint8_t* row_new = nullptr;     // [n_sub*8]
  uint8_t* row_move = nullptr;    // [n_sub*8]
  float* row_rhat = nullptr;      // [n_sub*8]
  Table tab, tab_alt;
  float* eval_planes = nullptr;   // [max_rows][plane]
  uint32_t* eval_slot = nullptr;  // [max_rows]
  uint64_t* eval_keys = nullptr;  // [max_rows*2]
  float* eval_values = nullptr;   // [max_rows*3]
  int32_t* n_miss = nullptr;      // [1]
  unsigned long long* stats = nullptr;  // [ST_COUNT]
  float* root_q = nullptr;        // [G*8*3]
  uint8_t* root_moves = nullptr;  // [G*8]
  uint32_t root_turn = 0;         // current root turn (1-based while a search is open)
  int stub_word = 1;              // word of the plane key the stand-in value function reads (a pit's stand-in side may pick 0)
  int epoch = -1, step = 0;
  bool open = false;
  // host copies of stats[ST_OCCUPIED], stats[ST_OVERFLOW] (refreshed wherever the host synchronises anyway)
  unsigned long long h_occ_ovf[2] = {0, 0};
  unsigned long long overflow_reported = 0;   // overflow count already turned into an error
  unsigned long long n_compactions = 0, n_mid_compactions = 0;   // table compactions: all / between two epochs of a turn
};

// ---- table ------------------------------------------------------------------------------------------------------
struct ProbeResult { uint32_t slot; bool is_new; };

// expiry (agent.py:30-31,101-110): an entry untouched for more than D root turns at the END of an earlier turn is gone.
__device__ __forceinline__ bool expired(uint32_t touch, uint32_t cur_turn, int D) {
  return (int)(cur_turn - 1u - touch) > D;
}

// One thread probes; concurrent probes of the same key from other warps are resolved by the CAS on the tag
// (insert) or on the touch stamp (re-creation of an expired entry).
__device__ __forceinline__ ProbeResult table_probe(const Table& t, uint64_t k0, uint64_t k1, uint32_t cur_turn, int D,
                                                   unsigned long long* stats) {
  const uint64_t mask = t.cap - 1;
  uint64_t h = fmix64(k1 ^ (k0 >> 7)) & mask;
  ProbeResult r; r.slot = kNoRow; r.is_new = false;
  for (uint64_t it = 0; it < t.cap; ++it, h = (h + 1) & mask) {
    uint64_t tag = t.key[h];
    if (tag == 0ull) {
      const uint64_t old = atomicCAS(reinterpret_cast<unsigned long long*>(&t.key[h]), 0ull, (unsigned long long)k0);
      if (old == 0ull) {
        t.chk[h] = k1;
        __threadfence();                                                       // publish: check word before the stamp
        *reinterpret_cast<volatile uint32_t*>(&t.touch[h]) = cur_turn;
        atomicAdd(&stats[ST_INSERTS], 1ull); atomicAdd(&stats[ST_OCCUPIED], 1ull);
        r.slot = (uint32_t)h; r.is_new = true;
        return r;
      }
      tag = old;
    }
    if (tag == k0) {
      // a concurrent insert claims the tag first and publishes the stamp last: wait for it (another warp, a few cycles)
      uint32_t seen;
      while ((seen = *reinterpret_cast<volatile uint32_t*>(&t.touch[h])) == kTouchInvalid) __nanosleep(32);
      __threadfence();
      if (seen != cur_turn) {
        if (t.chk[h] != k1) atomicAdd(&stats[ST_COLLISIONS], 1ull);   // same 64-bit tag, different check word
        if (expired(seen, cur_turn, D)) {
          if (atomicCAS(&t.touch[h], seen, cur_turn) == seen) {   // this thread re-creates the evicted entry
            t.chk[h] = k1;
            atomicAdd(&stats[ST_EXPIRED], 1ull);
            r.slot = (uint32_t)h; r.is_new = true;
            return r;
          }
        } else {
          t.touch[h] = cur_turn;                                   // agent.py:185 cache_hit[key] = 0
        }
      }
      r.slot = (uint32_t)h;
      return r;
    }
  }
  atomicAdd(&stats[ST_OVERFLOW], 1ull);
  return r;
}

// ---- kernels ------------------------------------------------------------------------------------------------------
struct SearchParams {
  // root
  const uint16_t* r_cells; const uint64_t* r_snakes; const uint32_t* r_meta; int G, S, health_dec;
  // sub-games
  uint16_t* cells; uint64_t* snakes; uint32_t* meta; int n_sub, P, D, Dmax;
  int32_t* sub_depth; uint8_t* sub_left; uint8_t* created;
  uint32_t* path_slot; uint8_t* path_move; uint8_t* path_len;
  uint32_t* row_slot; uint8_t* row_new; uint8_t* row_move; float* row_rhat;
  Table tab;
  float* eval_planes; uint32_t* eval_slot; uint64_t* eval_keys; const float* eval_values; int32_t* n_miss; int max_rows;
  unsigned long long* stats;
  uint32_t root_turn; int epoch, step;
  float base; int training; uint64_t seed;
  // trace (device, may be null): [E][Dmax][n_sub][S] u8
  uint8_t* trace; int trace_mode;   // 0 none, 1 replay (read), 2 record (write)
  float* root_q; uint8_t* root_moves; const uint8_t* root_trace;  // root_trace [G*8] for replay
};

// Game.subgame x P (game.py:266-276, agent.py:39-50): one thread block row copies the packed records.
template <int SIDE>
__global__ void search_epoch_begin_kernel(const SearchParams p) {
  using G = Geo<SIDE>;
  const int sub = (int)blockIdx.x;
  const int g = sub / p.P;
  const uint16_t* src = p.r_cells + (size_t)g * G::PC;
  uint16_t* dst = p.cells + (size_t)sub * G::PC;
  for (int i = (int)threadIdx.x; i < G::PC / 2; i += (int)blockDim.x)
    reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(src)[i];
  if (threadIdx.x < 8) {
    const uint64_t sv = p.r_snakes[(size_t)g * 8 + threadIdx.x];
    p.snakes[(size_t)sub * 8 + threadIdx.x] = sv;
    const unsigned alive = __ballot_sync(0xffu, snake_alive(sv));
    // meta: sub-game counters restart (game.py:268 builds a fresh Game); done flag is inherited
    const uint32_t rflags = p.r_meta[(size_t)g * 8 + META_FLAGS];
    const uint32_t repi = p.r_meta[(size_t)g * 8 + META_EPISODE];
    p.meta[(size_t)sub * 8 + threadIdx.x] = threadIdx.x == META_EPISODE ? repi : threadIdx.x == META_FLAGS ? (rflags & kMetaDone) : 0u;
    p.path_len[(size_t)sub * 8 + threadIdx.x] = 0;
    p.row_slot[(size_t)sub * 8 + threadIdx.x] = kNoRow;
    if (threadIdx.x == 0) {
      p.sub_depth[sub] = p.D - 2 * (__popc(alive) - 2);   // agent.py:45
      p.sub_left[sub] = (uint8_t)(rflags & kMetaDone);
      p.created[sub] = (uint8_t)alive;
      if (!(rflags & kMetaDone) && sub % p.P == 0) atomicAdd(&p.stats[ST_SUBGAMES], (unsigned long long)p.P);
    }
  }
}

// back one value up every (slot, move) of a path (agent.py:67-72, 215-220): N += 1, W += r
__device__ __forceinline__ void backup_path(const SearchParams& p, size_t i, int len, float r) {
  for (int j = len - 1; j >= 0; --j) {
    const uint32_t s = p.path_slot[i * p.Dmax + j];
    const int m = p.path_move[i * p.Dmax + j];
    atomicAdd(reinterpret_cast<float*>(&p.tab.n[s]) + m, 1.0f);
    atomicAdd(reinterpret_cast<float*>(&p.tab.w[s]) + m, r);
  }
}

template <int SIDE, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) search_step_kernel(const SearchParams p) {
  using G = Geo<SIDE>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = (int)(threadIdx.x >> 5), lane = lane_id();
  float* stage = reinterpret_cast<float*>(smem_raw) + warp * G::STAGE;
  uint16_t* sb = reinterpret_cast<uint16_t*>(smem_raw + (size_t)WARPS * G::STAGE * sizeof(float)) + warp * G::PC;
  const int sub = (int)blockIdx.x * WARPS + warp;
  if (sub >= p.n_sub) return;
  if (p.sub_left[sub]) return;
  // load the record
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.cells + (size_t)sub * G::PC);
    uint32_t* dst = reinterpret_cast<uint32_t*>(sb);
#pragma unroll
    for (int q = 0; q < G::CPL / 2; ++q) dst[q * 32 + lane] = src[q * 32 + lane];
  }
  Snake sn = unpack_snake(kEmptySnake);
  if (lane < 8) sn = unpack_snake(p.snakes[(size_t)sub * 8 + lane]);
  Meta m = meta_from_lanes((lane < 8) ? p.meta[(size_t)sub * 8 + lane] : 0u);
  __syncwarp();
  const size_t ri = (size_t)sub * 8 + lane;   // (sub-game, snake) index of this lane, valid for lane < 8
  bool left = false;
  if (p.step > 1) {
    // deferred from the previous step (agent.py:208-222): back r-hat up the path, then push (slot, move)
    int move = 1;
    if (lane < 8) {
      const uint32_t rs = p.row_slot[ri];
      if (rs != kNoRow) {
        const int len = p.path_len[ri];
        move = p.row_move[ri];
        backup_path(p, ri, len, p.row_rhat[ri]);
        if (len < p.Dmax) { p.path_slot[ri * p.Dmax + len] = rs; p.path_move[ri * p.Dmax + len] = (uint8_t)move; p.path_len[ri] = (uint8_t)(len + 1); }
      }
    }
    // mp_game_runner.py:103-113: tic, then leave when the game ended or the depth is reached
    const TicResult r = warp_tic<G>(sb, sn, m, move, p.health_dec, ASZ_SPAWN_NONE, -1, 0u, 0ull, 0u, p.S);
    left = r.ended || (int)m.turn >= p.sub_depth[sub];
    if (lane == 0) atomicAdd(&p.stats[ST_SUBTICS], 1ull);
    // write the record back
    {
      uint32_t* dst = reinterpret_cast<uint32_t*>(p.cells + (size_t)sub * G::PC);
      const uint32_t* src = reinterpret_cast<const uint32_t*>(sb);
#pragma unroll
      for (int q = 0; q < G::CPL / 2; ++q) dst[q * 32 + lane] = src[q * 32 + lane];
      if (lane < 8) {
        p.snakes[ri] = pack_snake(sn);
        p.meta[ri] = meta_word(m, lane);
      }
    }
    if (left) {
      // terminal backup (agent.py:60-72): snakes alive at creation whose reward is known
      if (lane < 8 && ((p.created[sub] >> lane) & 1) && sn.reward != 0)
        backup_path(p, ri, p.path_len[ri], sn.reward == 1 ? 1.0f : -1.0f);
      if (lane < 8) p.row_slot[ri] = kNoRow;
      if (lane == 0) p.sub_left[sub] = 1;
      return;
    }
  }
  // ---- this step's rows: key, probe / insert, plane of a miss into the eval batch (agent.py:170-186) ----
  const unsigned live_mask = __ballot_sync(kFull, sn.alive != 0);
  if (lane < 8 && !sn.alive) p.row_slot[ri] = kNoRow;
  CellView<G> cv;
  warp_cell_view<G>(sb, sn, cv);
  // Pass 1: key and probe of every live snake (lane 0 probes, one snake after the other: parallel lanes on diverged probe paths
  // were measured slower); lane vs keeps its snake's result.  Then ONE returning atomic for the sub-game's rows of the eval batch
  // instead of one per miss (same-address returning atomics are served one after the other by their L2 slice, DESIGN.md 4.1).
  // Pass 2: the planes of the misses.
  unsigned rest = live_mask;
  int n_rows = 0, n_new = 0;
  uint32_t my_slot = kNoRow; int my_new = 0;
  uint64_t my_k0 = 0ull, my_k1 = 0ull;
  while (rest) {
    const int vs = __ffs(rest) - 1;
    rest &= rest - 1;
    uint64_t k0, k1;
    warp_encode<G, true>(cv, sn, vs, stage, nullptr, 0, &k0, &k1);
    uint32_t slot = kNoRow; int is_new = 0;
    if (lane == 0) {
      const ProbeResult pr = table_probe(p.tab, k0, k1, p.root_turn, p.D, p.stats);
      slot = pr.slot; is_new = pr.is_new ? 1 : 0;
    }
    slot = __shfl_sync(kFull, slot, 0); is_new = __shfl_sync(kFull, is_new, 0);
    if (lane == vs) { my_slot = slot; my_new = is_new; my_k0 = k0; my_k1 = k1; }
    ++n_rows;
  }
  const unsigned new_mask = __ballot_sync(kFull, my_new != 0);
  int eidx = -1;
  if (new_mask) {
    int base = 0;
    if (lane == 0) base = atomicAdd(p.n_miss, __popc(new_mask));
    base = __shfl_sync(kFull, base, 0);
    if (my_new) {
      eidx = base + __popc(new_mask & ((1u << lane) - 1u));
      if (eidx < p.max_rows) {
        p.eval_slot[eidx] = my_slot; p.eval_keys[2 * (size_t)eidx] = my_k0; p.eval_keys[2 * (size_t)eidx + 1] = my_k1;
        p.tab.eval[my_slot] = eidx;
      } else { eidx = -1; }
    }
  }
  if (lane < 8 && sn.alive) { p.row_slot[ri] = my_slot; p.row_new[ri] = (uint8_t)my_new; }
  unsigned todo = __ballot_sync(kFull, eidx >= 0);
  n_new = __popc(todo);
  while (todo) {
    const int vs = __ffs(todo) - 1;
    todo &= todo - 1;
    const int e = __shfl_sync(kFull, eidx, vs);
    warp_encode<G, false>(cv, sn, vs, stage, p.eval_planes, (size_t)e * G::PLANE, nullptr, nullptr);
  }
  if (lane == 0) {
    atomicAdd(&p.stats[ST_VISITS], (unsigned long long)n_rows);
    atomicAdd(&p.stats[ST_EVALS], (unsigned long long)n_new);
  }
}

// agent.py:114-122 (float32 throughout, left-to-right sum, all-masked => uniform)
__device__ __forceinline__ void softermax3(const float q[3], float base, float pmf[3]) {
  float n[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) n[k] = powf(base, atanhf(q[k]));
  float sigma = 0.0f;
  sigma = __fadd_rn(sigma, n[0]); sigma = __fadd_rn(sigma, n[1]); sigma = __fadd_rn(sigma, n[2]);
  if (sigma == 0.0f) { pmf[0] = pmf[1] = pmf[2] = (float)(1.0 / 3.0); return; }
#pragma unroll
  for (int k = 0; k < 3; ++k) pmf[k] = __fdiv_rn(n[k], sigma);
  // reference: Q == +1 gives inf/inf = NaN and numpy.random.choice raises; here the +inf weight takes all the mass
#pragma unroll
  for (int k = 0; k < 3; ++k) if (isinf(n[k])) { pmf[0] = pmf[1] = pmf[2] = 0.0f; pmf[k] = 1.0f; }
}
// numpy.random.choice(3, p=pmf): cdf = cumsum(float64 p) / last; searchsorted(cdf, u, 'right')
__device__ __forceinline__ int choice3(const float pmf[3], double u) {
  const double c0 = (double)pmf[0], c1 = c0 + (double)pmf[1], c2 = c1 + (double)pmf[2];
  int idx = 0;
  if (c0 / c2 <= u) idx = 1;
  if (c1 / c2 <= u) idx = 2;
  return idx;
}
__device__ __forceinline__ void read_q(const Table& t, uint32_t slot, float q[3]) {
  const float4 w = t.w[slot], n = t.n[slot];
  q[0] = __fdiv_rn(w.x, n.x); q[1] = __fdiv_rn(w.y, n.y); q[2] = __fdiv_rn(w.z, n.z);
}

// One thread per (sub-game, snake) row: new-node priors (agent.py:193-201), softermax + sample (:204-205),
// estimated reward (:214).  The path backup itself is deferred to the next search_step_kernel.
__global__ void search_sample_kernel(const SearchParams p) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)p.n_sub * 8) return;
  const uint32_t slot = p.row_slot[i];
  if (slot == kNoRow) return;
  float q[3];
  const int e = *reinterpret_cast<volatile int32_t*>(&p.tab.eval[slot]);
  if (e >= 0) {
    const float v0 = p.eval_values[3 * (size_t)e], v1 = p.eval_values[3 * (size_t)e + 1], v2 = p.eval_values[3 * (size_t)e + 2];
    q[0] = v0; q[1] = v1; q[2] = v2;   // W = V, N = 1, Q = W / N
    if (p.row_new[i]) {
      p.tab.w[slot] = make_float4(v0, v1, v2, 0.0f);
      p.tab.n[slot] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
      __threadfence();
      *reinterpret_cast<volatile int32_t*>(&p.tab.eval[slot]) = -1;
    }
  } else {
    __threadfence();
    read_q(p.tab, slot, q);
  }
  float pmf[3];
  softermax3(q, p.base, pmf);
  const int sub = (int)(i >> 3), snake = (int)(i & 7);
  int mv;
  const size_t ti = (((size_t)p.epoch * p.Dmax + (size_t)(p.step - 1)) * (size_t)p.n_sub + (size_t)sub) * (size_t)p.S + (size_t)snake;
  if (p.trace_mode == 1) {
    mv = p.trace[ti];
  } else {
    uint32_t r[4];
    philox4x32_10((uint32_t)sub * (uint32_t)p.S + (uint32_t)snake, p.root_turn - 1u, RS_TREE,
                  (uint32_t)p.epoch * 256u + (uint32_t)(p.step - 1), p.seed, r);
    mv = choice3(pmf, (double)r[0] * (1.0 / 4294967296.0));
    if (p.trace_mode == 2) p.trace[ti] = (uint8_t)mv;
  }
  float est = __fmul_rn(pmf[0], q[0]);
  est = __fadd_rn(est, __fmul_rn(pmf[1], q[1]));
  est = __fadd_rn(est, __fmul_rn(pmf[2], q[2]));
  p.row_move[i] = (uint8_t)mv;
  p.row_rhat[i] = est;
}

// agent.py:74-99: root Q = table entry of the first key on the snake's path in the last epoch; root move.
__global__ void search_root_kernel(const SearchParams p) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= p.G * 8) return;
  const int g = i >> 3, s = i & 7;
  p.root_moves[i] = 255;
  if (s >= p.S) return;
  if (p.r_meta[(size_t)g * 8 + META_FLAGS] & kMetaDone) return;
  if (!snake_alive(p.r_snakes[(size_t)g * 8 + s])) return;
  const size_t pi = ((size_t)g * p.P) * 8 + s;
  if (p.path_len[pi] == 0) return;
  const uint32_t slot = p.path_slot[pi * p.Dmax];
  float q[3];
  read_q(p.tab, slot, q);
  p.root_q[3 * (size_t)i] = q[0]; p.root_q[3 * (size_t)i + 1] = q[1]; p.root_q[3 * (size_t)i + 2] = q[2];
  int mv;
  if (p.training) {
    if (p.root_trace != nullptr) mv = p.root_trace[i];
    else {
      float pmf[3];
      softermax3(q, p.base, pmf);
      uint32_t r[4];
      philox4x32_10((uint32_t)g * (uint32_t)p.S + (uint32_t)s, p.root_turn - 1u, RS_ROOT, 0u, p.seed, r);
      mv = choice3(pmf, (double)r[0] * (1.0 / 4294967296.0));
    }
  } else {
    mv = argmax3(q);
  }
  p.root_moves[i] = (uint8_t)mv;
}

// deterministic stand-in for the value network: value from the plane key, then AlphaNNet.v's obstacle mask
// (alpha_nnet.py:63-76).  Used by the parity tests and the search-only throughput measurement.
__global__ void stub_value_kernel(const uint64_t* keys, int word, const float* planes, const int32_t* n_ptr, int side, int numpy1_mask,
                                  float* out) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= *n_ptr) return;
  const int N = 2 * side - 1;
  float v[3];
  stub_value3(keys[2 * (size_t)i + word], v);
  obstacle_mask3(planes + (size_t)i * N * N * 3, side, numpy1_mask, v);
  out[3 * (size_t)i] = v[0]; out[3 * (size_t)i + 1] = v[1]; out[3 * (size_t)i + 2] = v[2];
}

// obstacle mask alone (applied to a network's raw outputs)
__global__ void obstacle_mask_kernel(const float* planes, int n, int side, int numpy1_mask, float* v) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const int N = 2 * side - 1;
  obstacle_mask3(planes + (size_t)i * N * N * 3, side, numpy1_mask, v + 3 * (size_t)i);
}

// test hook: softermax + inverse-CDF draw + argmaxs on arbitrary rows (agent.py:114-137, numpy.random.choice)
__global__ void policy_debug_kernel(const float* z, const double* u, int n, float base, float* pmf, int32_t* choice, int32_t* amax) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const float q[3] = {z[3 * i], z[3 * i + 1], z[3 * i + 2]};
  float p[3];
  softermax3(q, base, p);
  pmf[3 * i] = p[0]; pmf[3 * i + 1] = p[1]; pmf[3 * i + 2] = p[2];
  choice[i] = choice3(p, u[i]);
  amax[i] = argmax3(q);
}

// ---- table maintenance --------------------------------------------------------------------------------------------
// ref_turn: the root turn whose END decides eviction (agent.py:101-110): the current turn when called from asz_search_finish, the
// previous one when the table is compacted between two epochs of a turn (entries touched in this turn have age 0 either way)
__global__ void table_rebuild_kernel(const Table src, Table dst, uint32_t ref_turn, int D, unsigned long long* occupied) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= src.cap) return;
  const uint64_t k0 = src.key[i];
  if (k0 == 0ull) return;
  if ((int)(ref_turn - src.touch[i]) > D) return;   // evicted (agent.py:101-110)
  const uint64_t k1 = src.chk[i];
  const uint64_t mask = dst.cap - 1;
  uint64_t h = fmix64(k1 ^ (k0 >> 7)) & mask;
  for (;; h = (h + 1) & mask) {
    if (atomicCAS(reinterpret_cast<unsigned long long*>(&dst.key[h]), 0ull, (unsigned long long)k0) == 0ull) break;
  }
  dst.chk[h] = k1; dst.w[h] = src.w[i]; dst.n[h] = src.n[i]; dst.touch[h] = src.touch[i]; dst.eval[h] = -1;
  atomicAdd(occupied, 1ull);
}

// live (non-evicted) entries as of the end of root turn cur_turn, compacted
__global__ void table_dump_kernel(const Table t, uint32_t cur_turn, int D, int cap_out, int* count, uint64_t* keys, float* Wt,
                                  float* Nn, int32_t* age) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.cap) return;
  const uint64_t k0 = t.key[i];
  if (k0 == 0ull) return;
  const int a = (int)(cur_turn - t.touch[i]);
  if (a > D) return;
  const int o = atomicAdd(count, 1);
  if (o >= cap_out) return;
  keys[2 * (size_t)o] = k0; keys[2 * (size_t)o + 1] = t.chk[i];
  const float4 w = t.w[i], n = t.n[i];
  Wt[3 * (size_t)o] = w.x; Wt[3 * (size_t)o + 1] = w.y; Wt[3 * (size_t)o + 2] = w.z;
  Nn[3 * (size_t)o] = n.x; Nn[3 * (size_t)o + 1] = n.y; Nn[3 * (size_t)o + 2] = n.z;
  age[o] = a;
}

static int table_alloc(Table& t, int log2cap) {
  t.log2cap = log2cap; t.cap = 1ull << log2cap;
  ASZ_CUDA(cudaMalloc(&t.key, t.cap * sizeof(uint64_t)));
  ASZ_CUDA(cudaMalloc(&t.chk, t.cap * sizeof(uint64_t)));
  ASZ_CUDA(cudaMalloc(&t.w, t.cap * sizeof(float4)));
  ASZ_CUDA(cudaMalloc(&t.n, t.cap * sizeof(float4)));
  ASZ_CUDA(cudaMalloc(&t.touch, t.cap * sizeof(uint32_t)));
  ASZ_CUDA(cudaMalloc(&t.eval, t.cap * sizeof(int32_t)));
  ASZ_CUDA(cudaMemset(t.key, 0, t.cap * sizeof(uint64_t)));
  ASZ_CUDA(cudaMemset(t.touch, 0xFF, t.cap * sizeof(uint32_t)));
  return ASZ_OK;
}
static void table_free(Table& t) {
  cudaFree(t.key); cudaFree(t.chk); cudaFree(t.w); cudaFree(t.n); cudaFree(t.touch); cudaFree(t.eval);
  t = Table();
}

int search_create(asz_engine* e) {
  const asz_config& c = e->cfg;
  if (c.max_depth < 1 || c.max_depth > 64) { set_error("max_depth must be in 1..64"); return ASZ_ERR_ARG; }
  SearchState* s = new SearchState();
  e->search = s;
  s->P = std::min(8, c.max_breadth);                  // agent.py:32-34
  s->E = c.max_breadth / s->P;                        // agent.py:37
  s->Dmax = std::max(1, c.max_depth);
  s->n_sub = c.games * s->P;
  s->max_rows = s->n_sub * c.snakes;
  int rc = gameset_alloc(s->sub, s->n_sub, e->pc);
  if (rc != ASZ_OK) return rc;
  const size_t ns = (size_t)s->n_sub;
  ASZ_CUDA(cudaMalloc(&s->sub_depth, ns * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->sub_left, ns));
  ASZ_CUDA(cudaMalloc(&s->created, ns));
  ASZ_CUDA(cudaMalloc(&s->path_slot, ns * 8 * s->Dmax * sizeof(uint32_t)));
  ASZ_CUDA(cudaMalloc(&s->path_move, ns * 8 * s->Dmax));
  ASZ_CUDA(cudaMalloc(&s->path_len, ns * 8));
  ASZ_CUDA(cudaMalloc(&s->row_slot, ns * 8 * sizeof(uint32_t)));
  ASZ_CUDA(cudaMalloc(&s->row_new, ns * 8));
  ASZ_CUDA(cudaMalloc(&s->row_move, ns * 8));
  ASZ_CUDA(cudaMalloc(&s->row_rhat, ns * 8 * sizeof(float)));
  ASZ_CUDA(cudaMemset(s->path_len, 0, ns * 8));
  ASZ_CUDA(cudaMemset(s->sub_left, 1, ns));
  int lg = c.table_log2;
  if (lg <= 0) {
    const double est = 2.0 * (double)c.games * c.max_breadth * c.snakes * 2.5 * (c.max_depth + 2);
    lg = 16;
    while (lg < 28 && (double)(1ull << lg) < est) ++lg;
  }
  if (lg < 10 || lg > 31) { set_error("table_log2 must be in 10..31"); return ASZ_ERR_ARG; }
  rc = table_alloc(s->tab, lg);
  if (rc != ASZ_OK) return rc;
  ASZ_CUDA(cudaMalloc(&s->eval_planes, (size_t)s->max_rows * e->plane * sizeof(float) + 16));
  ASZ_CUDA(cudaMalloc(&s->eval_slot, (size_t)s->max_rows * sizeof(uint32_t)));
  ASZ_CUDA(cudaMalloc(&s->eval_keys, (size_t)s->max_rows * 2 * sizeof(uint64_t)));
  ASZ_CUDA(cudaMalloc(&s->eval_values, (size_t)s->max_rows * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&s->n_miss, sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&s->stats, ST_COUNT * sizeof(unsigned long long)));
  ASZ_CUDA(cudaMemset(s->stats, 0, ST_COUNT * sizeof(unsigned long long)));
  ASZ_CUDA(cudaMalloc(&s->root_q, (size_t)c.games * 8 * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&s->root_moves, (size_t)c.games * 8));
  ASZ_CUDA(cudaMemset(s->root_q, 0, (size_t)c.games * 8 * 3 * sizeof(float)));
  return ASZ_OK;
}

void search_set_stub_word(asz_engine* e, int word) { e->search->stub_word = word; }

void search_destroy(asz_engine* e) {
  SearchState* s = e->search;
  if (!s) return;
  gameset_free(s->sub);
  cudaFree(s->sub_depth); cudaFree(s->sub_left); cudaFree(s->created); cudaFree(s->path_slot); cudaFree(s->path_move);
  cudaFree(s->path_len); cudaFree(s->row_slot); cudaFree(s->row_new); cudaFree(s->row_move); cudaFree(s->row_rhat);
  table_free(s->tab); table_free(s->tab_alt);
  cudaFree(s->eval_planes); cudaFree(s->eval_slot); cudaFree(s->eval_keys); cudaFree(s->eval_values); cudaFree(s->n_miss);
  cudaFree(s->stats); cudaFree(s->root_q); cudaFree(s->root_moves);
  delete s;
  e->search = nullptr;
}

static SearchParams make_params(asz_engine* e) {
  SearchState* s = e->search;
  SearchParams p;
  memset(&p, 0, sizeof p);
  p.r_cells = e->root.cells; p.r_snakes = e->root.snakes; p.r_meta = e->root.meta;
  p.G = e->cfg.games; p.S = e->cfg.snakes; p.health_dec = e->cfg.health_dec;
  p.cells = s->sub.cells; p.snakes = s->sub.snakes; p.meta = s->sub.meta;
  p.n_sub = s->n_sub; p.P = s->P; p.D = e->cfg.max_depth; p.Dmax = s->Dmax;
  p.sub_depth = s->sub_depth; p.sub_left = s->sub_left; p.created = s->created;
  p.path_slot = s->path_slot; p.path_move = s->path_move; p.path_len = s->path_len;
  p.row_slot = s->row_slot; p.row_new = s->row_new; p.row_move = s->row_move; p.row_rhat = s->row_rhat;
  p.tab = s->tab;
  p.eval_planes = s->eval_planes; p.eval_slot = s->eval_slot; p.eval_keys = s->eval_keys; p.eval_values = s->eval_values;
  p.n_miss = s->n_miss; p.max_rows = s->max_rows; p.stats = s->stats;
  p.root_turn = s->root_turn; p.epoch = s->epoch; p.step = s->step;
  p.base = e->cfg.softmax_base; p.training = e->cfg.training; p.seed = e->cfg.seed;
  p.root_q = s->root_q; p.root_moves = s->root_moves;
  return p;
}

// Copies the live entries into the spare table and swaps (slots held by evicted entries are given back).
static int table_compact(asz_engine* e, uint32_t ref_turn, cudaStream_t st) {
  SearchState* s = e->search;
  if (!s->tab_alt.key) { int rc = table_alloc(s->tab_alt, s->tab.log2cap); if (rc != ASZ_OK) return rc; }
  ASZ_CUDA(cudaMemsetAsync(s->tab_alt.key, 0, s->tab_alt.cap * sizeof(uint64_t), st));
  ASZ_CUDA(cudaMemsetAsync(s->tab_alt.touch, 0xFF, s->tab_alt.cap * sizeof(uint32_t), st));
  ASZ_CUDA(cudaMemsetAsync(&s->stats[ST_OCCUPIED], 0, sizeof(unsigned long long), st));
  table_rebuild_kernel<<<(unsigned)((s->tab.cap + 255) / 256), 256, 0, st>>>(s->tab, s->tab_alt, ref_turn, e->cfg.max_depth,
                                                                            &s->stats[ST_OCCUPIED]);
  if (!cuda_ok(cudaGetLastError(), "table_rebuild_kernel")) return ASZ_ERR_CUDA;
  std::swap(s->tab, s->tab_alt);
  s->h_occ_ovf[0] = 0;
  s->n_compactions += 1;
  if (ref_turn != s->root_turn) s->n_mid_compactions += 1;
  return ASZ_OK;
}

template <int SIDE>
struct SearchLaunch {
  static constexpr int WARPS = (SIDE >= 19) ? 4 : 8;
  using G = Geo<SIDE>;
  static size_t smem_bytes() { return (size_t)WARPS * (G::STAGE * sizeof(float) + G::PC * sizeof(uint16_t)); }
  static int epoch_begin(const SearchParams& p, cudaStream_t st) {
    search_epoch_begin_kernel<SIDE><<<p.n_sub, 64, 0, st>>>(p);
    return cuda_ok(cudaGetLastError(), "search_epoch_begin_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
  }
  static int step(const SearchParams& p, int dev, cudaStream_t st) {
    static bool configured[kMaxDevices] = {false};   // function attributes are per device
    if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
      if (!cuda_ok(cudaFuncSetAttribute(search_step_kernel<SIDE, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem_bytes()), "cudaFuncSetAttribute(search_step_kernel)"))
        return ASZ_ERR_CUDA;
      if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
    }
    const int blocks = (p.n_sub + WARPS - 1) / WARPS;
    search_step_kernel<SIDE, WARPS><<<blocks, WARPS * 32, smem_bytes(), st>>>(p);
    return cuda_ok(cudaGetLastError(), "search_step_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
  }
};

}  // namespace asz

using namespace asz;

extern "C" {

int asz_search_begin(asz_engine* e, void* stream) {
  if (!e || !e->search) { set_error("search is not configured (max_breadth == 0)"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  SearchState* s = e->search;
  if (s->open) { set_error("asz_search_begin: a search is already open"); return ASZ_ERR_STATE; }
  (void)stream;
  s->root_turn += 1;   // agent.py:30-31: every entry ages by one
  s->epoch = -1; s->step = 0; s->open = true;
  return ASZ_OK;
}

int asz_search_epoch_begin(asz_engine* e, void* stream) {
  if (!e || !e->search || !e->search->open) { set_error("no open search"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:search epoch_begin (subgame x8)");
  SearchState* s = e->search;
  if (s->epoch + 1 >= s->E) { set_error("all epochs of this root turn are done"); return ASZ_ERR_STATE; }
  s->epoch += 1; s->step = 0;
  cudaStream_t st = (cudaStream_t)stream;
  // Evicted entries keep their slots until a compaction, so a long root turn could fill the table on its own: between two
  // epochs no path, row or pending evaluation refers to a slot, and a table more than 3/4 full (as of the last host
  // synchronisation) is compacted right here
  if (s->h_occ_ovf[0] * 4 > s->tab.cap * 3) {
    const int rc = table_compact(e, s->root_turn - 1u, st);
    if (rc != ASZ_OK) return rc;
  }
  const SearchParams p = make_params(e);
  int rc;
  switch (e->cfg.side) {
    case 7: rc = SearchLaunch<7>::epoch_begin(p, st); break;
    case 11: rc = SearchLaunch<11>::epoch_begin(p, st); break;
    default: rc = SearchLaunch<19>::epoch_begin(p, st); break;
  }
  if (rc != ASZ_OK) return rc;
  // stats: sub-games of live root games are counted on the host side by the caller if needed
  return ASZ_OK;
}

int asz_search_step_probe(asz_engine* e, int32_t* h_n_miss, void* stream) {
  if (!e || !e->search || !e->search->open || e->search->epoch < 0) { set_error("no open epoch"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:search step_probe (tic, backup, key, probe)");
  SearchState* s = e->search;
  if (s->step > s->Dmax) { set_error("epoch already finished"); return ASZ_ERR_STATE; }
  s->step += 1;
  cudaStream_t st = (cudaStream_t)stream;
  ASZ_CUDA(cudaMemsetAsync(s->n_miss, 0, sizeof(int32_t), st));
  const SearchParams p = make_params(e);
  int rc;
  switch (e->cfg.side) {
    case 7: rc = SearchLaunch<7>::step(p, e->device, st); break;
    case 11: rc = SearchLaunch<11>::step(p, e->device, st); break;
    default: rc = SearchLaunch<19>::step(p, e->device, st); break;
  }
  if (rc != ASZ_OK) return rc;
  if (h_n_miss) {
    ASZ_CUDA(cudaMemcpyAsync(h_n_miss, s->n_miss, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    ASZ_CUDA(cudaMemcpyAsync(s->h_occ_ovf, &s->stats[ST_OCCUPIED], sizeof s->h_occ_ovf, cudaMemcpyDeviceToHost, st));
    ASZ_CUDA(cudaStreamSynchronize(st));
    if (*h_n_miss > s->max_rows) *h_n_miss = s->max_rows;
  }
  return ASZ_OK;
}

int asz_search_step_sample(asz_engine* e, const float* d_values, uint8_t* d_trace, int32_t trace_mode, void* stream) {
  if (!e || !e->search || !e->search->open || e->search->step < 1) { set_error("no probed step"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:search step_sample (priors, softermax, sample)");
  SearchState* s = e->search;
  if (s->step > s->Dmax) return ASZ_OK;   // the closing probe of an epoch has no rows
  if (trace_mode != 0 && !d_trace) { set_error("trace_mode set but d_trace is null"); return ASZ_ERR_ARG; }
  SearchParams p = make_params(e);
  if (d_values) p.eval_values = d_values;
  p.trace = d_trace; p.trace_mode = trace_mode;
  const size_t n = (size_t)s->n_sub * 8;
  search_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
  return cuda_ok(cudaGetLastError(), "search_sample_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

int asz_search_stub_values(asz_engine* e, void* stream) {
  if (!e || !e->search) { set_error("search is not configured"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  SearchState* s = e->search;
  const int n = s->max_rows;   // the kernel reads the live count from device memory: no host sync
  stub_value_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(s->eval_keys, s->stub_word, s->eval_planes, s->n_miss,
                                                                      e->cfg.side, e->cfg.numpy1_mask, s->eval_values);
  return cuda_ok(cudaGetLastError(), "stub_value_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

int asz_obstacle_mask(asz_engine* e, const float* d_planes, int32_t n, float* d_values, void* stream) {
  if (!e || !d_planes || !d_values) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:obstacle_mask");
  if (n <= 0) return ASZ_OK;
  obstacle_mask_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_planes, n, e->cfg.side, e->cfg.numpy1_mask, d_values);
  return cuda_ok(cudaGetLastError(), "obstacle_mask_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

int asz_debug_policy(const float* d_z, const double* d_u, int32_t n, float base, float* d_pmf, int32_t* d_choice, int32_t* d_argmax,
                     void* stream) {
  if (!d_z || !d_u || !d_pmf || !d_choice || !d_argmax) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (n <= 0) return ASZ_OK;
  policy_debug_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_z, d_u, n, base, d_pmf, d_choice, d_argmax);
  return cuda_ok(cudaGetLastError(), "policy_debug_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

int asz_search_finish(asz_engine* e, const uint8_t* d_root_trace, float* d_root_q, uint8_t* d_root_moves, void* stream) {
  if (!e || !e->search || !e->search->open) { set_error("no open search"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:search finish (root Q, moves, eviction)");
  SearchState* s = e->search;
  cudaStream_t st = (cudaStream_t)stream;
  SearchParams p = make_params(e);
  p.root_trace = d_root_trace;
  if (d_root_q) p.root_q = d_root_q;
  if (d_root_moves) p.root_moves = d_root_moves;
  const int n = e->cfg.games * 8;
  search_root_kernel<<<(n + 127) / 128, 128, 0, st>>>(p);
  if (!cuda_ok(cudaGetLastError(), "search_root_kernel")) return ASZ_ERR_CUDA;
  s->open = false;
  // compaction when the table is more than half full of (mostly evicted) entries
  static_assert(ST_OVERFLOW == ST_OCCUPIED + 1, "occupied and overflow are read with one copy");
  ASZ_CUDA(cudaMemcpyAsync(s->h_occ_ovf, &s->stats[ST_OCCUPIED], sizeof s->h_occ_ovf, cudaMemcpyDeviceToHost, st));
  ASZ_CUDA(cudaStreamSynchronize(st));
  if (s->h_occ_ovf[0] * 2 > s->tab.cap) {
    const int rc = table_compact(e, s->root_turn, st);
    if (rc != ASZ_OK) return rc;
  }
  // A probe that found no slot dropped its row: that snake then played "straight" in its sub-game and the search result is
  // not the reference's.  Never silent: the turn's outputs are written, but the call fails.
  if (s->h_occ_ovf[1] > s->overflow_reported) {
    char msg[160];
    snprintf(msg, sizeof msg, "Q table overflow: %llu probes found no free slot in 2^%d slots this root turn (raise table_log2)",
             s->h_occ_ovf[1] - s->overflow_reported, s->tab.log2cap);
    s->overflow_reported = s->h_occ_ovf[1];
    set_error(msg);
    return ASZ_ERR_CAPACITY;
  }
  return ASZ_OK;
}

// Whole root-turn search: the epoch / step loops of Agent.make_moves (agent.py:37-58) in native code.  net == nullptr: the stub
// value function, with no host synchronisation inside the loops.  Otherwise the hand-written value network; the only host
// synchronisation is the miss count of each step (it sizes the network batch).
static int search_run(asz_engine* e, asz_net* net, uint8_t* d_trace, int32_t trace_mode, const uint8_t* d_root_trace, void* stream) {
  int rc = asz_search_begin(e, stream);
  if (rc != ASZ_OK) return rc;
  SearchState* s = e->search;
  for (int ep = 0; ep < s->E; ++ep) {
    if ((rc = asz_search_epoch_begin(e, stream)) != ASZ_OK) return rc;
    for (int st = 1; st <= s->Dmax + 1; ++st) {
      int32_t n_miss = 0;
      if ((rc = asz_search_step_probe(e, net ? &n_miss : nullptr, stream)) != ASZ_OK) return rc;
      if (st <= s->Dmax) {
        if (!net) {
          if ((rc = asz_search_stub_values(e, stream)) != ASZ_OK) return rc;
        } else if (n_miss > 0) {
          if ((rc = asz_net_forward(net, s->eval_planes, n_miss, s->eval_values, stream)) != ASZ_OK) return rc;   // alpha_nnet.py:62
          if ((rc = asz_obstacle_mask(e, s->eval_planes, n_miss, s->eval_values, stream)) != ASZ_OK) return rc;   // alpha_nnet.py:63-76
        }
        if ((rc = asz_search_step_sample(e, nullptr, d_trace, trace_mode, stream)) != ASZ_OK) return rc;
      }
    }
  }
  return asz_search_finish(e, d_root_trace, nullptr, nullptr, stream);
}

int asz_search_run_stub(asz_engine* e, uint8_t* d_trace, int32_t trace_mode, const uint8_t* d_root_trace, void* stream) {
  return search_run(e, nullptr, d_trace, trace_mode, d_root_trace, stream);
}

int asz_search_run_net(asz_engine* e, asz_net* net, uint8_t* d_trace, int32_t trace_mode, const uint8_t* d_root_trace, void* stream) {
  if (!net) { set_error("asz_search_run_net: null network"); return ASZ_ERR_ARG; }
  return search_run(e, net, d_trace, trace_mode, d_root_trace, stream);
}

int asz_search_clear(asz_engine* e, void* stream) {
  if (!e || !e->search) { set_error("search is not configured"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  SearchState* s = e->search;
  cudaStream_t st = (cudaStream_t)stream;
  ASZ_CUDA(cudaMemsetAsync(s->tab.key, 0, s->tab.cap * sizeof(uint64_t), st));
  ASZ_CUDA(cudaMemsetAsync(s->tab.touch, 0xFF, s->tab.cap * sizeof(uint32_t), st));
  ASZ_CUDA(cudaMemsetAsync(s->stats, 0, ST_COUNT * sizeof(unsigned long long), st));
  s->root_turn = 0; s->open = false; s->epoch = -1; s->step = 0;
  s->h_occ_ovf[0] = s->h_occ_ovf[1] = 0; s->overflow_reported = 0; s->n_compactions = s->n_mid_compactions = 0;
  return ASZ_OK;
}

int asz_search_info(asz_engine* e, int32_t* h_info) {
  if (!e || !e->search || !h_info) { set_error("search is not configured"); return ASZ_ERR_STATE; }
  SearchState* s = e->search;
  h_info[0] = s->P; h_info[1] = s->E; h_info[2] = s->Dmax; h_info[3] = s->n_sub; h_info[4] = s->max_rows;
  h_info[5] = s->tab.log2cap; h_info[6] = (int32_t)s->root_turn; h_info[7] = s->epoch;
  return ASZ_OK;
}

float* asz_search_eval_planes(asz_engine* e) { return (e && e->search) ? e->search->eval_planes : nullptr; }
float* asz_search_eval_values(asz_engine* e) { return (e && e->search) ? e->search->eval_values : nullptr; }
float* asz_search_root_q(asz_engine* e) { return (e && e->search) ? e->search->root_q : nullptr; }
uint8_t* asz_search_root_moves(asz_engine* e) { return (e && e->search) ? e->search->root_moves : nullptr; }

int asz_search_stats(asz_engine* e, uint64_t* h_stats) {
  if (!e || !e->search || !h_stats) { set_error("search is not configured"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  ASZ_CUDA(cudaDeviceSynchronize());
  ASZ_CUDA(cudaMemcpy(h_stats, e->search->stats, ST_COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  h_stats[10] = e->search->n_compactions; h_stats[11] = e->search->n_mid_compactions;   // host-side counts
  return ASZ_OK;
}

int asz_search_table_dump(asz_engine* e, int32_t cap, uint64_t* h_keys, float* h_w, float* h_n, int32_t* h_age, int32_t* h_count) {
  if (!e || !e->search || !h_count) { set_error("search is not configured"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  SearchState* s = e->search;
  int* d_count; uint64_t* d_keys; float *d_w, *d_n; int32_t* d_age;
  const size_t c = (size_t)std::max(cap, 1);
  ASZ_CUDA(cudaMalloc(&d_count, sizeof(int))); ASZ_CUDA(cudaMemset(d_count, 0, sizeof(int)));
  ASZ_CUDA(cudaMalloc(&d_keys, c * 2 * sizeof(uint64_t))); ASZ_CUDA(cudaMalloc(&d_w, c * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&d_n, c * 3 * sizeof(float))); ASZ_CUDA(cudaMalloc(&d_age, c * sizeof(int32_t)));
  table_dump_kernel<<<(unsigned)((s->tab.cap + 255) / 256), 256>>>(s->tab, s->root_turn, e->cfg.max_depth, cap, d_count, d_keys, d_w,
                                                                    d_n, d_age);
  ASZ_CUDA(cudaDeviceSynchronize());
  int count = 0;
  ASZ_CUDA(cudaMemcpy(&count, d_count, sizeof(int), cudaMemcpyDeviceToHost));
  *h_count = count;
  const size_t m = (size_t)std::min(count, cap);
  if (m > 0 && h_keys && h_w && h_n && h_age) {
    ASZ_CUDA(cudaMemcpy(h_keys, d_keys, m * 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    ASZ_CUDA(cudaMemcpy(h_w, d_w, m * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    ASZ_CUDA(cudaMemcpy(h_n, d_n, m * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    ASZ_CUDA(cudaMemcpy(h_age, d_age, m * sizeof(int32_t), cudaMemcpyDeviceToHost));
  }
  cudaFree(d_count); cudaFree(d_keys); cudaFree(d_w); cudaFree(d_n); cudaFree(d_age);
  return ASZ_OK;
}

}  // extern "C"
