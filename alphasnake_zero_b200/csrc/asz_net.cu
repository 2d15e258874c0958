// asz_net.cu -- the value network of alpha_nnet.py:19-56 as hand-written sm_100a kernels (inference only).
//
// The only dense contraction of the self-play loop (99.7 % of the FLOPs are the eight 128->128 3x3 convolutions,
// SURVEY.md 8(a) a14) runs as implicit GEMM on the 5th-generation tensor cores:
//
//   activations  bf16, "channel-chunk major": act[kc][pos][8] (kc = channel / 8), pos = flat position of a padded
//                22x22 raster per image (21 real rows/cols + one zero row/col shared by neighbours), so that the
//                input of tap (dy,dx) for output rows [m, m+128) is simply rows [m+s, m+s+128), s = (dy-1)*22+(dx-1);
//   A operand    one halo tile (256 + 2*24 rows, all 16 channel chunks) per CTA and super-tile, fetched with cp.async.bulk
//                and reused by all 9 taps through the shared-memory descriptor's start address (no-swizzle K-major core
//                matrices: 8 rows x 16 B contiguous, SBO = 128 B => rows are linear, any row offset is legal);
//   B operand    weights [tap][kc][cout][8] bf16 in half-tap chunks of 8 KB per CTA of a pair, which holds only half of the
//                output channels: resident for a whole launch where they fit (RESW), else streamed through an mbarrier ring;
//   D            two 128 x 128 fp32 accumulators per CTA and super-tile in TMEM (double buffered: 512 columns), 144
//                tcgen05.mma (M256 N128 K16, cta_group::2 over a CTA pair) issued by one elected thread;
//   epilogue     8 warps read TMEM (tcgen05.ld 32x32b), apply the folded BatchNorm scale/bias, the residual add and
//                the ReLU (alpha_nnet.py:22-47), zero the padding positions and store bf16 in the same layout; the
//                last convolution instead applies the 1x1 head convolution + BN + ReLU (alpha_nnet.py:49-50).
//   dense head   Flatten + Dense(128) + ReLU + Dense(3) + tanh (alpha_nnet.py:52-54): 8 images per CTA, fp32.
//
// fp8 networks (asz_net_create_fp8, opt-in; DESIGN.md 4.3): the same kernel with F8 = true.  Activations are e4m3,
// act[8][pos][16] (16 channels per 16-byte chunk, the same byte geometry), each layer's stored with a power-of-two scale;
// convolutions 1..8 contract e4m3 x e4m3 with tcgen05.mma kind::f8f6f4 (M256 N128 K32), the first keeps bf16 operands and
// only stores e4m3.  The epilogue is y = acc * scale' + bias (+ residual * res_scale), ReLU, mask, e4m3(y / act_scale).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "asz_engine.hpp"

namespace asz {

constexpr int kC = 128;          // channels of the tower
constexpr int kKC = kC / 8;      // 16-byte channel chunks
constexpr int kTileM = 128;      // output rows (positions) per accumulator
constexpr int kHalo = 40;        // >= pitch + 1 = max |tap shift| (39 for the 38-pitch raster of 19x19 boards)
constexpr int kGuard = 48;       // zero rows before and after the activation arrays

__host__ __device__ constexpr int pitch_of(int side) { return 2 * side; }            // 2*side-1 real + 1 pad
__host__ __device__ constexpr int img_rows_of(int side) { return 2 * side; }         // 2*side-1 real + 1 pad
static_assert(pitch_of(19) + 1 <= kHalo, "conv_umma_kernel<kHalo, ..> must cover every tap shift of 19x19 boards");

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- CTA-pair (cta_group::2) wrappers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
// arrive on a barrier of another CTA of the cluster.  Default semantics (release at CTA scope) on purpose: a cluster-scope
// release compiles to MEMBAR.ALL.GPU, and what these arrivals order (bulk-copy bytes seen through complete_tx, TMEM reads
// fenced by tcgen05.fence::before_thread_sync) does not travel through the generic proxy.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// one MMA over the CTA pair: M = 256 (128 rows of A and of D in each CTA), B split along N between the two CTAs
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z)
      : "memory");
}
// the same with e4m3 A and B (kind::f8f6f4): K = 32 per instruction, the same 32 bytes of each row as a bf16 K = 16 step
__device__ __forceinline__ void umma_f8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in both CTAs once every MMA issued so far has completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// instruction descriptor kind::f16: D fp32 (bits 4-5 = 1), A and B bf16 (bits 7-9, 10-12 = 1), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t kIdescPair = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kC >> 3) << 17) | ((uint32_t)((2 * kTileM) >> 4) << 24);
// kind::f8f6f4: the same with A and B e4m3 (format code 0 in bits 7-9 and 10-12)
constexpr uint32_t kIdescPairF8 = (1u << 4) | ((uint32_t)(kC >> 3) << 17) | ((uint32_t)((2 * kTileM) >> 4) << 24);

// ---- convolution kernel -----------------------------------------------------------------------------------------
struct ConvParams {
  const __nv_bfloat16* in;     // [16][P_tot][8], or [1][P_tot][8] for the first layer's raster
  const __nv_bfloat16* wt;     // pair layouts of pair_weight_layout_kernel / first_weight_layout_kernel
  const float* scale;          // [128] folded BN
  const float* bias;           // [128]
  const __nv_bfloat16* res;    // [16][P_tot][8] or null
  __nv_bfloat16* out;          // [16][P_tot][8] or null (head mode)
  const float* head_w;         // [128] or null
  float head_scale, head_bias;
  float* head_out;             // [P_tot] (head mode)
  int pitch;                   // raster pitch (22 at 11x11)
  int img_stride;              // positions per image (pitch * rows)
  int real;                    // real rows / cols per image (21)
  int P_tot;                   // rows of every activation array (guards included)
  int P_real;                  // positions that belong to images of this launch
  float res_scale;             // F8: the residual's stored e4m3 values times this are its values
  float out_inv_scale;         // F8: 1 / act_scale of this layer (the stored e4m3 values are y * out_inv_scale)
};

// ---- persistent convolution kernel over CTA pairs -----------------------------------------------------------------------
// The two CTAs of a cluster (the two SMs of a TPC) issue ONE tcgen05.mma.cta_group::2 of M = 256: every CTA supplies its own
// 128 rows of A (its own halo tile) but only HALF of the weights (64 of the 128 output channels).  One pair per TPC loops over
// pair super-tiles of 512 positions; CTA r owns positions [512 st + 256 r, +256).  Per super-tile the weights stream through
// shared memory once (half a tap per stage; or stay resident, RESW) and feed two M=128 accumulators per CTA; TMEM holds two
// accumulator pairs (4 x 128 columns) so that the epilogue of super-tile i overlaps the MMAs of super-tile i+1.
//   warp 0      producer  : cp.async.bulk of the A halo tile and of the weight chunks, mbarrier complete_tx
//   warp 1      rank 0: MMA issuer, one elected thread, tcgen05.commit releases stages / publishes accumulators;
//               rank 1: relays "my operands have landed" to rank 0's full barriers
//   warps 2..9  epilogue  : tcgen05.ld, BN scale/bias, residual, ReLU, padding mask, bf16 store (or the fused head conv)
// Loop order inside a super-tile: channel half c (8 of the 16 chunks) outermost, then the 9 taps.  The A half c is
// released as soon as its 9 taps are issued, so the next super-tile's half 0 streams in while half 1 is being consumed:
// the halo tile is effectively double buffered at 1x its size, which leaves room for 9+ weight stages.
//   barriers    full barriers of rank 0 count 2 arrivals (own producer + the relay); empty / accumulator-full barriers are
//               signalled in both CTAs by a multicast tcgen05.commit; accumulator-empty lives in rank 0 and counts the 16
//               epilogue warps of the pair.
//   weights     pair layout [tap][half][rank][8 kc][64 cout][8] (pair_weight_layout_kernel): a chunk is one bulk copy and
//               is fetched from L2 once per CTA pair.
//
// The MMA issue loop is written for issue rate: an M128 N128 K16 MMA lasts 64 tensor cycles, and ONE thread has to issue
// them back to back.  (tools/umma_probe.cu: the tensor pipe sustains 64.1 clk per MMA for every operand layout and shape
// tried, with bulk-copy fills running; the first version of this loop spent 196 SASS instructions per 8 MMAs rebuilding
// descriptors and walking divergence waterfalls and reached 46 % of that.)  So: the whole warp runs the loop in uniform
// control flow, one elected lane issues; loops have compile-time trip counts; a descriptor's low word is base + constant.
// IN8: e4m3 operands, 16 channels per 16-byte chunk, so the halo tile and a weight chunk (half a tap) take half the bytes
template <int HALO, bool IN8 = false>
struct UmmaSmem {
  static constexpr int kSuper = 256;                               // positions per CTA and weight pass
  static constexpr int rows = kSuper + 2 * HALO;
  static constexpr int kc = IN8 ? kKC / 2 : kKC;                   // 16-byte channel chunks of a row
  static constexpr size_t a_bytes = (size_t)kc * rows * 16;        // one halo tile, managed as two channel halves
  static constexpr int b_rows = kC / 2;                            // output channels whose weights this CTA holds
  static constexpr size_t b_chunk = (size_t)(kc / 2) * b_rows * 16;   // half a tap: 8 KB per CTA (IN8: 4 KB)
  static constexpr int max_stages = 18;                            // 18 = every weight chunk of a 3x3 layer (9 taps x 2 channel halves)
  static constexpr size_t tail = 3 * kC * sizeof(float) + (8 + 2 * max_stages) * sizeof(uint64_t) + 64;
  static constexpr int raw_stages = (int)((232448 - a_bytes - tail) / b_chunk);
  static constexpr int b_stages = raw_stages > max_stages ? max_stages : raw_stages;   // 18 (HALO 24) / 17 (HALO 40); IN8: 18
  static constexpr size_t total = a_bytes + b_stages * b_chunk + tail;
};

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xFFFFFFFF;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// shared-memory matrix descriptor, K-major, no swizzle: 8x(16 B) core matrices, LBO = byte distance between the two
// 16-byte K chunks of one K=16 step, SBO = byte distance between 8-row groups (cute/arch/mma_sm100_desc.hpp layout:
// start [0,14), LBO [16,30), SBO [32,46), version [46,48) = 1, layout type [61,64) = 0); lo = bits 0-31, hi = bits 32-63
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | (uint64_t)lo; }

// FIRST = the first convolution (alpha_nnet.py:21-22, 3 input channels).  Its input is the same raster as every other layer's,
// with ONE 16-byte channel chunk per position (3 real channels + 5 zeros; planes_to_raster_kernel), and its 9 taps are contracted
// TWO PER MMA: in the K-major no-swizzle layout the second 16-byte K chunk of an operand lies LBO bytes after the first, and the
// descriptor does not care what is there -- so with LBO = the row distance between two taps one K = 16 step multiplies the
// (8 channels of tap 2j | 8 channels of tap 2j+1) of every row with the matching weight rows.  Five MMAs (the fifth pairs tap 8
// with zero weights) instead of an im2col buffer: the layer reads 16 B per position where the im2col rows were 64 B, and the
// separate im2col pass (write 64 B + read 64 B per position) is gone.  Weights: two chunks per tile, K steps 0..3 and K step 4.
// F8 = a layer of an fp8 network: it stores (and adds as residual) e4m3 activations; unless FIRST it also reads e4m3 ones and
// contracts them with e4m3 weights (IN8): a half is 4 chunks of 16 channels, one K = 32 MMA per 2 chunks, so the issue loop,
// its descriptors and the weight ring are those of bf16 with 4 instead of 8 chunks per half.
template <int HALO, bool FIRST, bool F8 = false>
__global__ void __launch_bounds__(320, 1) conv_umma_kernel(const ConvParams p, int n_tiles) {
  constexpr bool IN8 = F8 && !FIRST;
  using SM = UmmaSmem<HALO, IN8>;
  constexpr int NS = SM::b_stages;
  constexpr int KC_HALF = FIRST ? 1 : SM::kc / 2;                  // channel chunks of A per half
  constexpr int HALVES = FIRST ? 1 : 2;
  constexpr int TAPS = FIRST ? 2 : 9;                              // weight chunks per half (FIRST: K steps 0..3, K step 4)
  constexpr int TILE = 2 * SM::kSuper;                             // positions per work unit (pair super-tile)
  constexpr uint32_t chunk_bytes = (uint32_t)SM::b_chunk;          // a full weight chunk: 8 K chunks (IN8: 4)
  constexpr uint32_t last_chunk_bytes = FIRST ? (uint32_t)(2 * SM::b_rows * 16) : chunk_bytes;   // FIRST: K step 4 alone
  // RESW: the CTA's half of the layer's weights (9 taps x 2 halves x 8 KB = 144 KB) fits next to the halo tile (HALO 24: 7x7 and
  // 11x11 boards): it is loaded ONCE per launch and stays resident, instead of streaming through the stage ring once per super-tile
  // (52 times per CTA and layer at 4,096 images).  Stage index = chunk index t * HALVES + c; b_full[0] is the only weight barrier.
  constexpr bool RESW = !FIRST && NS >= TAPS * HALVES;
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* sA = smem;
  unsigned char* sB = smem + SM::a_bytes;
  float* s_scale = reinterpret_cast<float*>(sB + NS * SM::b_chunk);
  float* s_bias = s_scale + kC;
  float* s_head = s_bias + kC;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_head + kC);
  uint64_t* a_full = bars;             // [2] channel halves
  uint64_t* a_empty = bars + 2;        // [2]
  uint64_t* acc_full = bars + 4;       // [2] accumulator pairs
  uint64_t* acc_empty = bars + 6;      // [2] (of rank 0)
  uint64_t* b_full = bars + 8;         // [NS]
  uint64_t* b_empty = bars + 8 + SM::max_stages;   // [NS]
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 8 + 2 * SM::max_stages);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = (int)(threadIdx.x & 31);
  const uint32_t rank = cluster_ctarank();
  const int first_tile = (int)(blockIdx.x >> 1);
  const int tile_step = (int)(gridDim.x >> 1);

  for (int i = (int)threadIdx.x; i < kC; i += (int)blockDim.x) {
    s_scale[i] = p.scale[i]; s_bias[i] = p.bias[i];
    s_head[i] = p.head_w ? p.head_w[i] : 0.0f;
  }
  if (threadIdx.x == 0) {
    const uint32_t full_count = rank == 0 ? 2u : 1u;
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], full_count); mbar_init(&a_empty[i], 1);
      mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 16);
    }
    for (int i = 0; i < NS; ++i) { mbar_init(&b_full[i], full_count); mbar_init(&b_empty[i], 1); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(s_tmem, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0) {
    if (lane == 0) {
      // ---- producer ----
      uint32_t stage = 0, phase = 0, it = 0;
      constexpr size_t chunk_stride = (size_t)2 * (chunk_bytes / 2);                     // bf16 elements between chunks
      if constexpr (RESW) {
        if (first_tile < n_tiles) {
          mbar_expect_tx(&b_full[0], (uint32_t)(TAPS * HALVES) * chunk_bytes);
#pragma unroll 1
          for (int ch = 0; ch < TAPS * HALVES; ++ch)
            bulk_g2s(sB + (size_t)ch * SM::b_chunk, p.wt + (size_t)rank * (chunk_bytes / 2) + (size_t)ch * chunk_stride, chunk_bytes, &b_full[0]);
        }
      }
      for (int st = first_tile; st < n_tiles; st += tile_step, ++it) {
        const size_t row0 = (size_t)kGuard + (size_t)st * TILE + (size_t)rank * SM::kSuper - HALO;
#pragma unroll 1
        for (int c = 0; c < HALVES; ++c) {
          mbar_wait(&a_empty[c], (it & 1u) ^ 1u);
          mbar_expect_tx(&a_full[c], (uint32_t)(KC_HALF * SM::rows * 16));
#pragma unroll
          for (int k = 0; k < KC_HALF; ++k) {
            const int kc = c * KC_HALF + k;
            bulk_g2s(sA + (size_t)kc * SM::rows * 16, p.in + ((size_t)kc * p.P_tot + row0) * 8, SM::rows * 16, &a_full[c]);
          }
          if constexpr (!RESW) {
#pragma unroll 1
          for (int t = 0; t < TAPS; ++t) {
            const uint32_t bytes = (t == TAPS - 1) ? last_chunk_bytes : chunk_bytes;
            mbar_wait(&b_empty[stage], phase ^ 1u);
            mbar_expect_tx(&b_full[stage], bytes);
            // pair layout [tap][half][rank][8][64][8]: chunk (t, c, rank) = ((t * HALVES + c) * 2 + rank) * chunk
            // (FIRST: chunk 1 is short, and its two rank parts follow the two full parts of chunk 0)
            const size_t off = (FIRST && t == 1) ? (size_t)2 * (chunk_bytes / 2) + (size_t)rank * (last_chunk_bytes / 2)
                                                 : (size_t)rank * (chunk_bytes / 2) + (size_t)(t * HALVES + c) * chunk_stride;
            bulk_g2s(sB + (size_t)stage * SM::b_chunk, p.wt + off, bytes, &b_full[stage]);
            if (++stage == NS) { stage = 0; phase ^= 1u; }
          }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---- MMA issuer: the whole warp runs the loop (uniform control flow), one elected lane issues ----
      const bool issuer = elect_one();
      const uint32_t a_lo0 = ((smem_u32(sA) >> 4) & 0x3FFFu) | ((uint32_t)SM::rows << 16);      // LBO = rows * 16 B
      const uint32_t b_lo0 = ((smem_u32(sB) >> 4) & 0x3FFFu) | ((uint32_t)SM::b_rows << 16);    // LBO = b_rows * 16 B
      constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);                                     // SBO = 128 B, version 1
      const int pitch = p.pitch;
      uint32_t stage = 0, phase = 0, it = 0;
      if constexpr (RESW) {
        if (first_tile < n_tiles) { mbar_wait(&b_full[0], 0u); tc_fence_after(); }   // the resident weights of both CTAs have landed
      }
      for (int st = first_tile; st < n_tiles; st += tile_step, ++it) {
        const uint32_t buf = it & 1u;
        mbar_wait(&acc_empty[buf], ((it >> 1) & 1u) ^ 1u);     // the epilogue(s) have drained this accumulator pair
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * 256u;
#pragma unroll 1
        for (int c = 0; c < HALVES; ++c) {
          mbar_wait(&a_full[c], it & 1u);
          tc_fence_after();
          const uint32_t a_c = a_lo0 + (uint32_t)(c * KC_HALF * SM::rows + HALO);
#pragma unroll
          for (int t = 0; t < TAPS; ++t) {
            const int shift = FIRST ? 0 : ((t / 3) - 1) * pitch + ((t % 3) - 1);
            if constexpr (!RESW) {
              mbar_wait(&b_full[stage], phase);
              tc_fence_after();
            }
            if (issuer) {
              const uint32_t b_s = b_lo0 + (RESW ? (uint32_t)(t * HALVES + c) : stage) * (uint32_t)(SM::b_chunk >> 4);
              if (FIRST) {
                // K step j = taps (2j, 2j+1): start address = the rows of tap 2j, LBO = the row distance to tap 2j+1
                const uint32_t a_rows = ((smem_u32(sA) >> 4) & 0x3FFFu) + (uint32_t)HALO;
#pragma unroll
                for (int sub = 0; sub < 2; ++sub) {
#pragma unroll
                  for (int ks = 0; ks < (t == 0 ? 4 : 1); ++ks) {
                    const int j = t * 4 + ks, ta = 2 * j, tb = (2 * j + 1 < 9) ? 2 * j + 1 : 2 * j;
                    const int sa = ((ta / 3) - 1) * pitch + ((ta % 3) - 1), sb = ((tb / 3) - 1) * pitch + ((tb % 3) - 1);
                    const uint32_t lbo = (tb == ta) ? 1u : (uint32_t)(sb - sa);          // rows of 16 B = the LBO field's unit
                    const uint64_t ad = desc64((a_rows + (uint32_t)(sa + sub * kTileM)) | (lbo << 16), desc_hi);
                    const uint64_t bd = desc64(b_s + (uint32_t)(2 * ks * SM::b_rows), desc_hi);
                    const uint32_t acc = (j == 0) ? 0u : 1u;
                    umma_bf16_pair(tmem_d + (uint32_t)(sub * kC), ad, bd, kIdescPair, acc);
                  }
                }
              } else {
                const uint32_t a_t = a_c + (uint32_t)shift;
#pragma unroll
                for (int sub = 0; sub < 2; ++sub) {
#pragma unroll
                  for (int ks = 0; ks < KC_HALF / 2; ++ks) {
                    const uint64_t ad = desc64(a_t + (uint32_t)(sub * kTileM + 2 * ks * SM::rows), desc_hi);
                    const uint64_t bd = desc64(b_s + (uint32_t)(2 * ks * SM::b_rows), desc_hi);
                    const uint32_t acc = (t == 0 && ks == 0) ? (uint32_t)c : 1u;
                    if constexpr (IN8) umma_f8_pair(tmem_d + (uint32_t)(sub * kC), ad, bd, kIdescPairF8, acc);
                    else umma_bf16_pair(tmem_d + (uint32_t)(sub * kC), ad, bd, kIdescPair, acc);
                  }
                }
              }
              if constexpr (!RESW) umma_commit_pair(&b_empty[stage]);
            }
            __syncwarp();
            if constexpr (!RESW) { if (++stage == NS) { stage = 0; phase ^= 1u; } }
          }
          if (issuer) umma_commit_pair(&a_empty[c]);
        }
        if (issuer) umma_commit_pair(&acc_full[buf]);
        __syncwarp();
      }
    } else if (lane == 0) {
      // ---- relay of rank 1: tell rank 0's full barriers that this CTA's operands have landed ----
      uint32_t stage = 0, phase = 0, it = 0;
      if constexpr (RESW) {
        if (first_tile < n_tiles) { mbar_wait(&b_full[0], 0u); mbar_arrive_cluster(mapa_u32(smem_u32(&b_full[0]), 0)); }
      }
      for (int st = first_tile; st < n_tiles; st += tile_step, ++it) {
#pragma unroll 1
        for (int c = 0; c < HALVES; ++c) {
          mbar_wait(&a_full[c], it & 1u);
          mbar_arrive_cluster(mapa_u32(smem_u32(&a_full[c]), 0));
          if constexpr (!RESW) {
#pragma unroll 1
          for (int t = 0; t < TAPS; ++t) {
            mbar_wait(&b_full[stage], phase);
            mbar_arrive_cluster(mapa_u32(smem_u32(&b_full[stage]), 0));
            if (++stage == NS) { stage = 0; phase ^= 1u; }
          }
          }
        }
      }
    }
  } else {
    // 8 epilogue warps: warps 2..5 take rows 0..127 of this CTA's super-tile (sub 0), warps 6..9 rows 128..255 (sub 1);
    // a warp may only touch the TMEM lane quarter warp % 4.  One thread = one output row (position), 128 channels.
    const int q = warp & 3;
    const int sub = (warp - 2) >> 2;
    uint32_t it = 0;
    for (int st = first_tile; st < n_tiles; st += tile_step, ++it) {
      const int buf = (int)(it & 1u);
      const int pos = st * TILE + (int)rank * SM::kSuper + sub * kTileM + q * 32 + lane;
      const int rem = pos % p.img_stride;
      const int y = rem / p.pitch, x = rem - y * p.pitch;
      const bool valid = pos < p.P_real && y < p.real && x < p.real;
      const size_t grow = (size_t)kGuard + (size_t)pos;
      // the residual row does not depend on the accumulator: fetch it while the MMAs of this super-tile run
      constexpr int RKC = F8 ? kKC / 2 : kKC;                      // 16-byte chunks of a stored row
      uint4 rv[RKC];
      if (p.res != nullptr) {
#pragma unroll
        for (int kc = 0; kc < RKC; ++kc) rv[kc] = *reinterpret_cast<const uint4*>(p.res + ((size_t)kc * p.P_tot + grow) * 8);
      }
      mbar_wait(&acc_full[buf], (it >> 1) & 1u);
      tc_fence_after();
      float head_acc = 0.0f;
#pragma unroll
      for (int cb = 0; cb < kC / 32; ++cb) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (uint32_t)(buf * 256 + sub * kC + cb * 32) + ((uint32_t)(q * 32) << 16), v);
        if constexpr (F8) {
#pragma unroll
          for (int j16 = 0; j16 < 2; ++j16) {
            const int kc = cb * 2 + j16;                           // 16-channel chunk
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j16 * 16 + j]) * s_scale[kc * 16 + j] + s_bias[kc * 16 + j];
            if (p.res != nullptr) {
              const __nv_fp8x2_storage_t* rb = reinterpret_cast<const __nv_fp8x2_storage_t*>(&rv[kc]);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const __half2_raw h = __nv_cvt_fp8x2_to_halfraw2(rb[j], __NV_E4M3);   // exact: e4m3 -> f16 -> f32
                const float2 t2 = __half22float2(__half2(h));
                f[2 * j] += t2.x * p.res_scale; f[2 * j + 1] += t2.y * p.res_scale;   // power-of-two scale: exact product
              }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = valid ? fmaxf(f[j], 0.0f) : 0.0f;
            if (p.out != nullptr) {
              uint4 ov;
              __nv_fp8x2_storage_t* ob = reinterpret_cast<__nv_fp8x2_storage_t*>(&ov);
#pragma unroll
              for (int j = 0; j < 8; ++j)       // cvt.rn.satfinite.e4m3x2.f32: nearest even, +-448 past the range
                ob[j] = __nv_cvt_float2_to_fp8x2(make_float2(f[2 * j] * p.out_inv_scale, f[2 * j + 1] * p.out_inv_scale), __NV_SATFINITE,
                                                 __NV_E4M3);
              *reinterpret_cast<uint4*>(p.out + ((size_t)kc * p.P_tot + grow) * 8) = ov;
            }
            if (p.head_out != nullptr) {
#pragma unroll
              for (int j = 0; j < 16; ++j) head_acc = fmaf(__bfloat162float(__float2bfloat16_rn(f[j])), s_head[kc * 16 + j], head_acc);
            }
          }
        } else {
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            const int kc = cb * 4 + j8;
            float f[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(v[j8 * 8 + j]) * s_scale[kc * 8 + j] + s_bias[kc * 8 + j];
            if (p.res != nullptr) {
              const __nv_bfloat162* rb = reinterpret_cast<const __nv_bfloat162*>(&rv[kc]);
#pragma unroll
              for (int j = 0; j < 4; ++j) { const float2 t2 = __bfloat1622float2(rb[j]); f[2 * j] += t2.x; f[2 * j + 1] += t2.y; }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = valid ? fmaxf(f[j], 0.0f) : 0.0f;
            if (p.out != nullptr) {
              uint4 ov;
              __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&ov);
#pragma unroll
              for (int j = 0; j < 4; ++j) ob[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
              *reinterpret_cast<uint4*>(p.out + ((size_t)kc * p.P_tot + grow) * 8) = ov;
            }
            if (p.head_out != nullptr) {
#pragma unroll
              for (int j = 0; j < 8; ++j) head_acc = fmaf(__bfloat162float(__float2bfloat16_rn(f[j])), s_head[kc * 8 + j], head_acc);
            }
          }
        }
      }
      if (p.head_out != nullptr) p.head_out[grow] = valid ? fmaxf(head_acc * p.head_scale + p.head_bias, 0.0f) : 0.0f;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&acc_empty[buf]), 0));
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // nobody leaves (or frees tensor memory) while the peer can still signal or accumulate
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

// [tap][kc][128 cout][8] -> [tap][half][rank][kc % 8][64 cout][8]: each (tap, half, rank) chunk is one contiguous bulk copy
__global__ void pair_weight_layout_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int taps, int kc_in) {
  const int kc_half = kc_in < 8 ? kc_in : 8, halves = kc_in / kc_half;
  const int total = taps * kc_in * kC;                       // 16-byte elements
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= total) return;
  const int cout = i % kC, kc = (i / kC) % kc_in, t = i / (kC * kc_in);
  const int c = kc / kc_half, k = kc % kc_half, r = cout / (kC / 2), co = cout % (kC / 2);
  const size_t o = ((((size_t)t * halves + c) * 2 + r) * kc_half + k) * (kC / 2) + co;
  reinterpret_cast<uint4*>(dst)[o] = reinterpret_cast<const uint4*>(src)[i];
}

// ---- input of the persistent first convolution: fp32 NHWC planes -> the raster with one 16-byte chunk per position (3 channels
// + 5 zeros, bf16), zero at the padding positions -----------------------------------------------------------------------------
__global__ void planes_to_raster_kernel(const float* __restrict__ planes, size_t plane_stride, int n_img, int real, int pitch, int img_stride,
                                        __nv_bfloat16* __restrict__ out /* [P_tot][8] */) {
  const int pos = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (pos >= n_img * img_stride) return;
  const int n = pos / img_stride, rem = pos - n * img_stride;
  const int y = rem / pitch, x = rem - y * pitch;
  uint4 ov = make_uint4(0u, 0u, 0u, 0u);
  if (y < real && x < real) {
    const float* s = planes + (size_t)n * plane_stride + ((size_t)y * real + x) * 3;
    __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&ov);
    ob[0] = __floats2bfloat162_rn(s[0], s[1]);
    ob[1] = __floats2bfloat162_rn(s[2], 0.0f);
  }
  *reinterpret_cast<uint4*>(out + ((size_t)kGuard + (size_t)pos) * 8) = ov;
}

// first-layer weights for the tap-paired contraction: the caller's im2col layout [4 kc][128][8] (k = tap * 3 + channel, 27 of 32
// used) -> K chunk t = the 8 channel slots of tap t (3 real), 10 chunks (tap 9 = zeros), split for CTA pairs:
//   [chunk 0: rank][8][64][8] then [chunk 1: rank][2][64][8]
__global__ void first_weight_layout_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);      // (tap chunk, cout)
  if (i >= 10 * kC) return;
  const int t = i / kC, cout = i - t * kC;
  __align__(16) __nv_bfloat16 v[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int k = t * 3 + c;
    v[c] = (t < 9 && c < 3) ? src[((size_t)(k >> 3) * kC + cout) * 8 + (k & 7)] : __float2bfloat16_rn(0.0f);
  }
  const int r = cout / (kC / 2), co = cout % (kC / 2);
  const size_t o = t < 8 ? ((size_t)r * 8 + t) * (kC / 2) + co : (size_t)2 * 8 * (kC / 2) + ((size_t)r * 2 + (t - 8)) * (kC / 2) + co;
  reinterpret_cast<uint4*>(dst)[o] = *reinterpret_cast<const uint4*>(v);
}

// ---- dense head: Flatten + Dense(128) + ReLU + Dense(3) + tanh (alpha_nnet.py:52-54), 8 images per CTA ------------------
// The dense1 weights are re-laid out once on the padded raster ([img_stride][128], zero rows at padding positions), so the
// head activations of an image are one contiguous run of img_stride floats (the epilogue wrote zeros at the padding).
// 256 threads: thread t owns hidden units 2 (t % 64), +1 for all 8 images over one quarter of the raster (t / 64); one pass
// over the weights serves 8 images; the four quarters are added in a fixed order (batch invariant).
constexpr int kHeadImg = 8;
__global__ void __launch_bounds__(256) dense_head_kernel(const float* __restrict__ head /* [P_tot] */, int n_img, int img_stride,
                                                         const float* __restrict__ w1r /* [img_stride][128] */,
                                                         const float* __restrict__ b1, const float* __restrict__ w2 /* [128][3] */,
                                                         const float* __restrict__ b2, float* __restrict__ out /* [n][3] */) {
  extern __shared__ __align__(16) float sh[];          // [img_stride][8] inputs, [4][8][128] partial sums
  float* s_in = sh;
  float* s_h = sh + kHeadImg * img_stride;
  const int n0 = (int)blockIdx.x * kHeadImg, tid = (int)threadIdx.x;
  const int up = tid & 63, quarter = tid >> 6;          // hidden units 2 up, 2 up + 1 over one quarter of the raster
  const float* src = head + kGuard + (size_t)n0 * img_stride;
  const int n_here = min(kHeadImg, n_img - n0);
  for (int i = tid; i < kHeadImg * img_stride; i += 256) {
    const int j = i / img_stride, r = i - j * img_stride;
    s_in[r * kHeadImg + j] = j < n_here ? src[i] : 0.0f;
  }
  __syncthreads();
  float a0[kHeadImg], a1[kHeadImg];
#pragma unroll
  for (int j = 0; j < kHeadImg; ++j) { a0[j] = 0.0f; a1[j] = 0.0f; }
  const int qlen = (img_stride + 3) / 4;
  const int i_begin = quarter * qlen, i_end = min(img_stride, i_begin + qlen);
#pragma unroll 8
  for (int i = i_begin; i < i_end; ++i) {
    const float2 w = *reinterpret_cast<const float2*>(w1r + (size_t)i * 128 + 2 * up);
    const float4 a = *reinterpret_cast<const float4*>(s_in + i * kHeadImg);
    const float4 b = *reinterpret_cast<const float4*>(s_in + i * kHeadImg + 4);
    const float x[kHeadImg] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < kHeadImg; ++j) { a0[j] = fmaf(x[j], w.x, a0[j]); a1[j] = fmaf(x[j], w.y, a1[j]); }
  }
#pragma unroll
  for (int j = 0; j < kHeadImg; ++j) {
    *reinterpret_cast<float2*>(s_h + (quarter * kHeadImg + j) * 128 + 2 * up) = make_float2(a0[j], a1[j]);
  }
  __syncthreads();
  if (tid < 128) {
#pragma unroll
    for (int j = 0; j < kHeadImg; ++j) {
      float v = b1[tid];
#pragma unroll
      for (int q = 0; q < 4; ++q) v += s_h[(q * kHeadImg + j) * 128 + tid];     // fixed order: batch invariant
      s_h[j * 128 + tid] = fmaxf(v, 0.0f);
    }
  }
  __syncthreads();
  if (tid < kHeadImg * 3) {
    const int j = tid / 3, k = tid - j * 3;
    if (j < n_here) {
      float o = b2[k];
      for (int u = 0; u < 128; ++u) o = fmaf(s_h[j * 128 + u], w2[u * 3 + k], o);
      out[(size_t)(n0 + j) * 3 + k] = tanhf(o);
    }
  }
}

// dense1 weights [real*real][128] -> padded raster [img_stride][128]
__global__ void dense1_raster_kernel(const float* __restrict__ w1, int real, int pitch, int img_stride, float* __restrict__ w1r) {
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= img_stride * 128) return;
  const int pos = i >> 7, u = i & 127;
  const int y = pos / pitch, x = pos - y * pitch;
  w1r[i] = (y < real && x < real) ? w1[((size_t)y * real + x) * 128 + u] : 0.0f;
}




template <int HALO, bool FIRST, bool F8>
constexpr size_t conv_smem_bytes() { return UmmaSmem<HALO, F8 && !FIRST>::total; }
template <int HALO, bool FIRST, bool F8>
static int configure_one() {
  return cuda_ok(cudaFuncSetAttribute(conv_umma_kernel<HALO, FIRST, F8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)conv_smem_bytes<HALO, FIRST, F8>()), "cudaFuncSetAttribute(conv_umma_kernel)") ? ASZ_OK : ASZ_ERR_CUDA;
}
template <bool F8>
static int configure_umma_kernels() {
  int rc = ASZ_OK;
  if ((rc = configure_one<24, false, F8>()) != ASZ_OK) return rc;
  if ((rc = configure_one<24, true, F8>()) != ASZ_OK) return rc;
  if ((rc = configure_one<kHalo, false, F8>()) != ASZ_OK) return rc;
  if ((rc = configure_one<kHalo, true, F8>()) != ASZ_OK) return rc;
  return rc;
}
template <int HALO, bool FIRST, bool F8>
static int launch_one(int grid, const ConvParams& p, int n_tiles, cudaStream_t st) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(320); cfg.dynamicSmemBytes = conv_smem_bytes<HALO, FIRST, F8>(); cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cuda_ok(cudaLaunchKernelEx(&cfg, conv_umma_kernel<HALO, FIRST, F8>, p, n_tiles), "conv_umma_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}
template <bool F8>
static int launch_umma(bool big, bool first, int grid, const ConvParams& p, int n_tiles, cudaStream_t st) {
  if (!big) return first ? launch_one<24, true, F8>(grid, p, n_tiles, st) : launch_one<24, false, F8>(grid, p, n_tiles, st);
  return first ? launch_one<kHalo, true, F8>(grid, p, n_tiles, st) : launch_one<kHalo, false, F8>(grid, p, n_tiles, st);
}

}  // namespace asz

using namespace asz;

struct asz_net {
  asz_net_weights w;
  int side = 0, real = 0, pitch = 0, img_stride = 0;
  int chunk = 0;           // images per pass
  int P_tot = 0;           // rows of the activation arrays (guards + padded positions)
  __nv_bfloat16* act[3] = {nullptr, nullptr, nullptr};
  __nv_bfloat16* col = nullptr;   // input raster of the first layer [P_tot][8] (planes_to_raster_kernel)
  float* head = nullptr;          // [P_tot]
  float* w1r = nullptr;           // dense1 weights on the padded raster [img_stride][128]
  int n_sm = 148;
  int device = 0;                 // the device this network lives on (asz_net_create's current device)
  __nv_bfloat16* w_pair[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  __nv_bfloat16* w_first_pair = nullptr;   // first-layer weights, tap-paired and split for CTA pairs (first_weight_layout_kernel)
  bool fp8 = false;               // asz_net_create_fp8: e4m3 activations and residual-layer weights
  float act_scale[9] = {1, 1, 1, 1, 1, 1, 1, 1, 1};   // fp8: stored e4m3 value of layer i's output = output / act_scale[i]
};

static int net_forward_impl(asz_net* n, const float* d_planes, int32_t count, float* d_values, int stop_layer, float* d_act, cudaStream_t st,
                            size_t plane_stride = 0);

namespace asz {
int net_side(const asz_net* n) { return n->side; }
int net_device(const asz_net* n) { return n->device; }
}  // namespace asz

extern "C" {

// operands derived from the caller's weight arrays: dense1 on the padded raster, convolution weights split for CTA pairs
static int net_derive(asz_net* n, cudaStream_t st) {
  dense1_raster_kernel<<<(n->img_stride * 128 + 255) / 256, 256, 0, st>>>(n->w.dense1_w, n->real, n->pitch, n->img_stride, n->w1r);
  if (!cuda_ok(cudaGetLastError(), "dense1_raster_kernel")) return ASZ_ERR_CUDA;
  first_weight_layout_kernel<<<(10 * kC + 255) / 256, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(n->w.w_conv[0]), n->w_first_pair);
  if (!cuda_ok(cudaGetLastError(), "first_weight_layout_kernel")) return ASZ_ERR_CUDA;
  for (int l = 1; l < 9; ++l) {
    // fp8 [tap][8][128][16 B] read as [tap * 2 + half][4][128][16 B]: the pair layout [tap][half][rank][4][64][16 B] of the
    // 4 KB weight chunks of conv_umma_kernel<.., F8>
    const int taps = n->fp8 ? 18 : 9, kc_in = n->fp8 ? kKC / 4 : kKC, total = taps * kc_in * kC;
    pair_weight_layout_kernel<<<(total + 255) / 256, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(n->w.w_conv[l]), n->w_pair[l], taps, kc_in);
    if (!cuda_ok(cudaGetLastError(), "pair_weight_layout_kernel")) return ASZ_ERR_CUDA;
  }
  return ASZ_OK;
}

// allocations of asz_net_create; on failure the caller destroys the partially built object (cudaFree(nullptr) is a no-op)
static int net_alloc(asz_net* n, const asz_net_weights* w, int32_t chunk_images) {
  n->w = *w;
  n->side = w->side; n->real = 2 * w->side - 1; n->pitch = pitch_of(w->side); n->img_stride = n->pitch * img_rows_of(w->side);
  n->chunk = chunk_images;
  const size_t P = (size_t)chunk_images * n->img_stride;
  const size_t P_pad = (P + 511) / 512 * 512;                 // whole pair super-tiles
  n->P_tot = (int)(kGuard + P_pad + kGuard + kHalo);
  const size_t act_bytes = (size_t)(n->fp8 ? kKC / 2 : kKC) * n->P_tot * 16;
  for (int i = 0; i < 3; ++i) {
    ASZ_CUDA(cudaMalloc(&n->act[i], act_bytes));
    ASZ_CUDA(cudaMemset(n->act[i], 0, act_bytes));
  }
  ASZ_CUDA(cudaMalloc(&n->col, (size_t)n->P_tot * 8 * sizeof(__nv_bfloat16)));
  ASZ_CUDA(cudaMemset(n->col, 0, (size_t)n->P_tot * 8 * sizeof(__nv_bfloat16)));
  ASZ_CUDA(cudaMalloc(&n->head, (size_t)n->P_tot * sizeof(float)));
  ASZ_CUDA(cudaMemset(n->head, 0, (size_t)n->P_tot * sizeof(float)));
  {
    int dev = 0; cudaDeviceProp prop;
    ASZ_CUDA(cudaGetDevice(&dev));
    ASZ_CUDA(cudaGetDeviceProperties(&prop, dev));
    n->n_sm = prop.multiProcessorCount;
    n->device = dev;
  }
  { int rc = n->fp8 ? configure_umma_kernels<true>() : configure_umma_kernels<false>(); if (rc != ASZ_OK) return rc; }
  ASZ_CUDA(cudaFuncSetAttribute(dense_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  ASZ_CUDA(cudaMalloc(&n->w1r, (size_t)n->img_stride * 128 * sizeof(float)));
  for (int l = 1; l < 9; ++l) ASZ_CUDA(cudaMalloc(&n->w_pair[l], (size_t)9 * kKC * kC * 16));
  ASZ_CUDA(cudaMalloc(&n->w_first_pair, (size_t)10 * kC * 16));
  { int rc = net_derive(n, nullptr); if (rc != ASZ_OK) return rc; }
  ASZ_CUDA(cudaDeviceSynchronize());
  return ASZ_OK;
}


static int net_create(asz_net** out, const asz_net_weights* w, const float* act_scale, int32_t chunk_images) {
  if (!out || !w) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (w->side != 7 && w->side != 11 && w->side != 19) { set_error("side must be 7, 11 or 19"); return ASZ_ERR_ARG; }
  if (chunk_images < 1) { set_error("chunk_images must be >= 1"); return ASZ_ERR_ARG; }
  asz_net* n = new asz_net();
  if (act_scale) { n->fp8 = true; std::copy(act_scale, act_scale + 9, n->act_scale); }
  const int rc = net_alloc(n, w, chunk_images);
  if (rc != ASZ_OK) { asz_net_destroy(n); return rc; }
  *out = n;
  return ASZ_OK;
}

int asz_net_create(asz_net** out, const asz_net_weights* w, int32_t chunk_images) { return net_create(out, w, nullptr, chunk_images); }

// an fp8 activation scale: a power of two whose reciprocal is a normal fp32 number too (so both products are exact)
static bool act_scales_ok(const float* s) {
  for (int i = 0; i < 9; ++i) {
    int e = 0;
    if (!(s[i] > 0.0f) || !std::isfinite(s[i]) || std::frexp(s[i], &e) != 0.5f || e < -124 || e > 127) {
      set_error("act_scale must hold positive powers of two in [2^-125, 2^126]");
      return false;
    }
  }
  return true;
}

int asz_net_create_fp8(asz_net** out, const asz_net_weights_fp8* w, int32_t chunk_images) {
  if (!out || !w) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (!act_scales_ok(w->act_scale)) return ASZ_ERR_ARG;
  return net_create(out, &w->w, w->act_scale, chunk_images);
}

// New weights for an existing network (the per-generation weight push, alpha_snake_zero_trainer.py:52-57, 79-83): the
// pointers of *w replace the old ones (same board side; the caller keeps the arrays alive) and the derived operands are
// rebuilt on `stream`, ordered after whatever the caller enqueued there to fill the arrays (e.g. an NCCL broadcast).
int asz_net_update_weights(asz_net* n, const asz_net_weights* w, void* stream) {
  if (!n || !w) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (w->side != n->side) { set_error("asz_net_update_weights: board side differs from the network's"); return ASZ_ERR_ARG; }
  if (n->fp8) { set_error("asz_net_update_weights: an fp8 network takes asz_net_update_weights_fp8"); return ASZ_ERR_ARG; }
  DeviceGuard guard(n->device);
  n->w = *w;
  return net_derive(n, (cudaStream_t)stream);
}

int asz_net_update_weights_fp8(asz_net* n, const asz_net_weights_fp8* w, void* stream) {
  if (!n || !w) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (w->w.side != n->side) { set_error("asz_net_update_weights_fp8: board side differs from the network's"); return ASZ_ERR_ARG; }
  if (!n->fp8) { set_error("asz_net_update_weights_fp8: a bf16 network takes asz_net_update_weights"); return ASZ_ERR_ARG; }
  if (!act_scales_ok(w->act_scale)) return ASZ_ERR_ARG;
  DeviceGuard guard(n->device);
  n->w = w->w;
  std::copy(w->act_scale, w->act_scale + 9, n->act_scale);
  return net_derive(n, (cudaStream_t)stream);
}

int asz_net_destroy(asz_net* n) {
  if (!n) return ASZ_OK;
  DeviceGuard guard(n->device);
  for (int i = 0; i < 3; ++i) cudaFree(n->act[i]);
  cudaFree(n->col); cudaFree(n->head); cudaFree(n->w1r);
  for (int l = 0; l < 9; ++l) cudaFree(n->w_pair[l]);
  cudaFree(n->w_first_pair);
  delete n;
  return ASZ_OK;
}

static int launch_conv(asz_net* n, int layer, const __nv_bfloat16* in, const __nv_bfloat16* res, __nv_bfloat16* outp, bool head,
                       int n_img, cudaStream_t st) {
  ConvParams p;
  memset(&p, 0, sizeof p);
  p.in = in; p.wt = layer == 0 ? n->w_first_pair : n->w_pair[layer];
  p.scale = n->w.scale[layer]; p.bias = n->w.bias[layer];
  p.res = res; p.out = outp;
  if (head) { p.head_w = n->w.head_w; p.head_scale = n->w.head_scale; p.head_bias = n->w.head_bias; p.head_out = n->head; }
  p.pitch = n->pitch; p.img_stride = n->img_stride; p.real = n->real; p.P_tot = n->P_tot;
  p.P_real = n_img * n->img_stride;
  const bool big = n->pitch + 1 > 24;
  const int n_tiles = (p.P_real + 511) / 512;                   // pair super-tiles
  const int grid = 2 * std::min(n_tiles, n->n_sm / 2);
  if (!n->fp8) return launch_umma<false>(big, layer == 0, grid, p, n_tiles, st);
  p.res_scale = res ? n->act_scale[layer - 2] : 1.0f;            // the residual of layer 2b+2 is the output of layer 2b
  p.out_inv_scale = 1.0f / n->act_scale[layer];
  return launch_umma<true>(big, layer == 0, grid, p, n_tiles, st);
}

int asz_net_forward(asz_net* n, const float* d_planes, int32_t count, float* d_values, void* stream) {
  if (!n || !d_planes || !d_values) { set_error("null argument"); return ASZ_ERR_ARG; }
  DeviceGuard guard(n->device);
  NvtxRange nvtx("asz:net forward");
  return net_forward_impl(n, d_planes, count, d_values, -1, nullptr, (cudaStream_t)stream);
}

int asz_net_forward_pitched(asz_net* n, const float* d_planes, int32_t plane_pitch, int32_t count, float* d_values, void* stream) {
  if (!n || !d_planes || !d_values) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (plane_pitch < n->real * n->real * 3) { set_error("plane_pitch is smaller than a plane"); return ASZ_ERR_ARG; }
  DeviceGuard guard(n->device);
  NvtxRange nvtx("asz:net forward");
  return net_forward_impl(n, d_planes, count, d_values, -1, nullptr, (cudaStream_t)stream, (size_t)plane_pitch);
}

int asz_net_debug_layer(asz_net* n, const float* d_planes, int32_t count, int32_t layer, float* d_act, void* stream) {
  if (!n || !d_planes || !d_act) { set_error("null argument"); return ASZ_ERR_ARG; }
  if (count > n->chunk) { set_error("debug export handles one chunk"); return ASZ_ERR_ARG; }
  if (layer < 0 || layer > 8) { set_error("layer must be in 0..8"); return ASZ_ERR_ARG; }
  DeviceGuard guard(n->device);
  return net_forward_impl(n, d_planes, count, nullptr, layer, d_act, (cudaStream_t)stream);
}

}  // extern "C"

namespace asz {
// activation buffer -> fp32 [n][real][real][128] (debug / tests); F8: e4m3 act[8][pos][16] times `scale` (exact)
template <bool F8 = false>
__global__ void export_act_kernel(const __nv_bfloat16* act, const float* head, int n_img, int real, int pitch, int img_stride, int P_tot,
                                  float* out, float scale = 1.0f) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t per = (size_t)real * real * (head ? 1 : kC);
  if (i >= (size_t)n_img * per) return;
  const int n = (int)(i / per);
  size_t r = i - (size_t)n * per;
  int c = 0;
  if (!head) { c = (int)(r % kC); r /= kC; }
  const int y = (int)(r / real), x = (int)(r % real);
  const size_t grow = (size_t)kGuard + (size_t)n * img_stride + (size_t)y * pitch + x;
  if constexpr (F8) {
    const __nv_fp8_storage_t* a8 = reinterpret_cast<const __nv_fp8_storage_t*>(act);
    out[i] = head ? head[grow] : __half2float(__half(__nv_cvt_fp8_to_halfraw(a8[((size_t)(c >> 4) * P_tot + grow) * 16 + (c & 15)], __NV_E4M3))) * scale;
  } else {
    out[i] = head ? head[grow] : __bfloat162float(act[((size_t)(c >> 3) * P_tot + grow) * 8 + (c & 7)]);
  }
}
}  // namespace asz

static int net_forward_impl(asz_net* n, const float* d_planes, int32_t count, float* d_values, int stop_layer, float* d_act, cudaStream_t st,
                            size_t plane_stride) {
  const size_t plane = plane_stride ? plane_stride : (size_t)n->real * n->real * 3;     // floats between consecutive input planes
  auto dump = [&](const __nv_bfloat16* act, const float* head, int m) -> int {
    const size_t tot = (size_t)m * n->real * n->real * (head ? 1 : kC);
    if (n->fp8)
      export_act_kernel<true><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(act, head, m, n->real, n->pitch, n->img_stride, n->P_tot, d_act,
                                                                              n->act_scale[stop_layer]);
    else
      export_act_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(act, head, m, n->real, n->pitch, n->img_stride, n->P_tot, d_act);
    return cuda_ok(cudaGetLastError(), "export_act_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
  };
  // balanced passes: ceil(count / chunk) passes of (almost) equal size, so that no pass is a sliver that leaves SMs idle
  const int n_pass = (count + n->chunk - 1) / n->chunk;
  const int per_pass = n_pass > 0 ? (count + n_pass - 1) / n_pass : 0;
  for (int i0 = 0; i0 < count; i0 += per_pass) {
    const int m = std::min(per_pass, count - i0);
    const int P = m * n->img_stride;
    planes_to_raster_kernel<<<(P + 255) / 256, 256, 0, st>>>(d_planes + (size_t)i0 * plane, plane, m, n->real, n->pitch, n->img_stride, n->col);
    if (!cuda_ok(cudaGetLastError(), "planes_to_raster_kernel")) return ASZ_ERR_CUDA;
    int rc = launch_conv(n, 0, n->col, nullptr, n->act[0], false, m, st);          // alpha_nnet.py:21-22
    if (rc != ASZ_OK) return rc;
    if (stop_layer == 0) return dump(n->act[0], nullptr, m);
    int x = 0;                                                                     // index of the block input
    for (int b = 0; b < 4; ++b) {                                                  // alpha_nnet.py:24-47
      const int t = (x + 1) % 3, y = (x + 2) % 3;
      rc = launch_conv(n, 1 + 2 * b, n->act[x], nullptr, n->act[t], false, m, st);
      if (rc != ASZ_OK) return rc;
      if (stop_layer == 1 + 2 * b) return dump(n->act[t], nullptr, m);
      const bool last = b == 3;
      rc = launch_conv(n, 2 + 2 * b, n->act[t], n->act[x], last ? nullptr : n->act[y], last, m, st);
      if (rc != ASZ_OK) return rc;
      if (stop_layer == 2 + 2 * b) return last ? dump(nullptr, n->head, m) : dump(n->act[y], nullptr, m);
      x = y;
    }
    dense_head_kernel<<<(m + kHeadImg - 1) / kHeadImg, 256, (size_t)kHeadImg * (n->img_stride + 4 * 128) * sizeof(float), st>>>(
        n->head, m, n->img_stride, n->w1r, n->w.dense1_b, n->w.dense2_w, n->w.dense2_b, d_values + (size_t)i0 * 3);
    if (!cuda_ok(cudaGetLastError(), "dense_head_kernel")) return ASZ_ERR_CUDA;
  }
  return ASZ_OK;
}
