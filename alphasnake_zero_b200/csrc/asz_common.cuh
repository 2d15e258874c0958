// asz_common.cuh -- shared device helpers of the B200 self-play engine (sm_100a).
//
// Counter-based RNG, plane-key hashing, the cell-stamp encoding of the board and small warp utilities.
// Nothing here comes from the CPU oracle: the definitions (Philox streams, key function) are the engine's own and the
// oracle restates them independently so that seeded full-size runs can be compared bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace asz {

constexpr int kMaxSnakes = 8;
constexpr unsigned kFull = 0xffffffffu;

// ---- board cell stamps ------------------------------------------------------------------------------------------
// One u16 per cell: 0 = empty, kFood = food, else (owner << 12) | dist, dist = distance from the tail of the topmost
// segment on the cell (tail = 1, head = length).  game.py keeps linked lists + three sets (game.py:32-53, 302-386);
// every quantity the rules and the plane encoding need is a function of these stamps:
//   * all live snakes move every tic, so every stamp loses 1 per tic and a cell is vacated when it reaches 0
//     (Snake.move pops the tail, game.py:348-356; a stacked tail keeps the cell because its top segment has dist 2)
//   * growing duplicates the tail (game.py:360-365): every stamp of that snake gains 1
//   * make_state writes dist*0.02 tail->head so the topmost segment wins (game.py:236-241): exactly the stamp.
constexpr uint16_t kFood = 0x8000u;
constexpr uint16_t kDistMask = 0x0fffu;
__host__ __device__ __forceinline__ bool cell_is_body(uint32_t v) { return v != 0u && v != kFood; }
__host__ __device__ __forceinline__ int cell_owner(uint32_t v) { return (int)((v >> 12) & 7u); }
__host__ __device__ __forceinline__ int cell_dist(uint32_t v) { return (int)(v & kDistMask); }

// ---- Philox4x32-10 ----------------------------------------------------------------------------------------------
enum RngStream : uint32_t { RS_INIT = 0, RS_SPAWN = 1, RS_ACT_LO = 2, RS_ACT_HI = 3, RS_TREE = 4, RS_ROOT = 5 };

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed,
                                                       uint32_t out[4]) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll 2   // not 10: code size (instruction cache) matters more than the loop overhead in the kernels that inline this
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
  return (uint32_t)(((uint64_t)a * b) >> 32);
}

// ---- plane key --------------------------------------------------------------------------------------------------
// agent.py:175 keys the Q cache by the raw bytes of the encoded plane.  The engine keys it by a 128-bit order-free sum
// over the plane's pixels whose (ch0,ch1,ch2) bit triple differs from the wall triple (0, 1.0f, 0): a pure function of
// the plane bytes (so it induces the same equivalence classes up to hash collisions) that can be evaluated from the
// board cells without materialising the plane.
__host__ __device__ __forceinline__ uint64_t fmix64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
  return k;
}
__host__ __device__ __forceinline__ void key_accumulate(uint32_t pix, uint32_t a, uint32_t b, uint32_t c, uint64_t& k0,
                                                        uint64_t& k1) {
  if (a == 0u && b == 0x3F800000u && c == 0u) return;
  const uint64_t x = ((uint64_t)a << 32) | b, y = ((uint64_t)c << 32) | pix;
  k0 += fmix64(fmix64(y ^ 0x9E3779B97F4A7C15ULL) ^ x);
  k1 += fmix64(fmix64(x ^ 0xC2B2AE3D27D4EB4FULL) + y);
}

// ---- policy -----------------------------------------------------------------------------------------------------
// Agent.argmaxs (agent.py:124-137, pit_agent.py:16-23) with its tie rule: a tie between 0 and 1 goes to 1 or 2, ties with 2 go to 2
__device__ __forceinline__ int argmax3(const float z[3]) {
  if (z[0] > z[1]) return (z[0] > z[2]) ? 0 : 2;
  return (z[1] > z[2]) ? 1 : 2;
}
// AlphaNNet.v's obstacle mask (alpha_nnet.py:63-76) on one plane: a move whose target cell next to the viewer's head holds a
// body value (ch1) of at least 0.04 is valued -1.  numpy1_mask: compared in float64 (NumPy 1.18), otherwise in float32
// (NumPy >= 2).  Only the masked entries of v are written.
__device__ __forceinline__ void obstacle_mask3(const float* plane, int side, int numpy1_mask, float v[3]) {
  const int N = 2 * side - 1, c = side - 1;
  const float b[3] = {plane[((size_t)c * N + (c - 1)) * 3 + 1], plane[((size_t)(c - 1) * N + c) * 3 + 1], plane[((size_t)c * N + (c + 1)) * 3 + 1]};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const bool obs = numpy1_mask ? ((double)b[k] >= 0.04) : (b[k] >= 0.04f);
    if (obs) v[k] = -1.0f;
  }
}
// deterministic stand-in for the value network: three 16-bit fields of a plane-key word mapped to [-1, 1)
__device__ __forceinline__ void stub_value3(uint64_t word, float v[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] = ((float)(uint32_t)((word >> (16 * k)) & 0xFFFFull) - 32767.5f) * (1.0f / 32768.0f);
}

// ---- warp helpers -----------------------------------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return (int)(threadIdx.x & 31u); }
__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum_i32(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_excl_scan_i32(int v, int lane) {
  int s = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, s, o);
    if (lane >= o) s += t;
  }
  return s - v;
}

// ---- L2 residency hints ---------------------------------------------------------------------------------------------
// The game records (21 MB at 65,536 games) are read and rewritten by every launch and fit in L2 many times over; the
// planes (1 GB per launch) stream through it.  Records are accessed with an evict_last policy, planes with evict_first.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint32_t ld_hint_u32(const uint32_t* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ uint64_t ld_hint_u64(const uint64_t* p, uint64_t pol) {
  uint64_t v;
  asm volatile("ld.global.L2::cache_hint.b64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_hint_u32(uint32_t* p, uint32_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.b32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint_u64(uint64_t* p, uint64_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.b64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint_v2u32(uint32_t* p, uint32_t a, uint32_t b, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.b32 [%0], {%1, %2}, %3;" ::"l"(p), "r"(a), "r"(b), "l"(pol) : "memory");
}

// streaming 16-byte store that does not allocate in L1 (planes are written once and read by another kernel)
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

}  // namespace asz
