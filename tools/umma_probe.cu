// umma_probe.cu -- measurement tool (not product code): cycles per tcgen05.mma for the operand layouts / shapes the
// convolution kernel can choose from.  One CTA (or CTA pair) per SM issues a long chain of MMAs on static shared
// memory and times it with clock64.  Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o umma_probe umma_probe.cu
// Run:   ./umma_probe            (prints one line per configuration)
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nW_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra D_%=;\nbra W_%=;\nD_%=:\n}\n" ::"r"(
          smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  if (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// F8: kind::f8f6f4 with e4m3 A and B, K = 32 per MMA (the same 32 bytes of a row as a bf16 K = 16 step)
template <int CG, bool F8>
__device__ __forceinline__ void umma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  if (F8 && CG == 1) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n}\n" ::"r"(d),
                 "l"(a), "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
  } else if (F8) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n}\n" ::"r"(d),
                 "l"(a), "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
  } else if (CG == 1) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d), "l"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
  } else {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d), "l"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
  }
}
template <int CG>
__device__ __forceinline__ void commit(uint64_t* bar) {
  if (CG == 1) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
  else {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
  }
}
__device__ __forceinline__ uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
         (1ull << 46) | ((uint64_t)layout << 61);
}

// MODE 0: no swizzle, K-major core matrices (8 rows x 16 B), rows linear (SBO 128), LBO = rows*16 (the convolution's layout)
// MODE 1: 128-byte swizzle, K-major (rows of 128 B = 64 bf16, SBO 1024)
// MODE 2: like 0 but the descriptors are rebuilt from integers for every MMA (the product kernel's issue loop)
// FILL > 0: a second thread keeps FILL bytes per MMA of bulk copies (global -> shared) in flight, as the producer does
// F8: the same chain with kind::f8f6f4 (e4m3, K = 32: twice the MACs per MMA of a bf16 K = 16 step)
template <int CG, int N, int MODE, int FILL, bool F8 = false>
__global__ void __launch_bounds__(128, 1) probe_kernel(int iters, const unsigned char* gsrc, long long* out) {
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sA = smem;                 // 80 KB
  unsigned char* sB = smem + 80 * 1024;     // 64 KB
  unsigned char* sF = smem + 144 * 1024;    // 64 KB fill target
  __shared__ uint64_t bar, fbar[4];
  __shared__ uint32_t s_tmem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 208 * 1024 / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&fbar[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 0) tmem_alloc<CG>(&s_tmem, 512);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (CG == 2) cluster_sync_all();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = s_tmem;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0;
  constexpr int M = CG == 2 ? 256 : 128;
  constexpr uint32_t idesc = (1u << 4) | (F8 ? 0u : (1u << 7) | (1u << 10)) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
  constexpr int NB = CG == 2 ? N / 2 : N;    // rows of B in this CTA
  if (warp == 1 && lane == 0 && rank == 0) {
    const uint32_t a_base = smem_u32(sA), b_base = smem_u32(sB);
    long long t0 = clock64();
    uint32_t acc = 0;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        uint64_t ad, bd;
        if (MODE == 1) {
          // 4 K-steps inside one 128-byte swizzled row, two row blocks
          ad = desc(a_base + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024, 2);
          bd = desc(b_base + (k >> 2) * (NB * 128) + (k & 3) * 32, 16, 1024, 2);
        } else if (MODE == 0) {
          ad = desc(a_base + (2 * k) * 304 * 16 + ((i & 3) * 24) * 16, 304 * 16, 128, 0);
          bd = desc(b_base + (2 * k) * NB * 16, NB * 16, 128, 0);
        } else {
          const int kc = 2 * k;
          const int shift = ((i % 3) - 1) * 22 + ((i & 1));
          const uint32_t a_addr = a_base + (uint32_t)((kc * 304 + 24 + shift) * 16);
          const uint32_t b_addr = b_base + (uint32_t)(kc * NB * 16);
          ad = desc(a_addr, 304 * 16, 128, 0);
          bd = desc(b_addr, NB * 16, 128, 0);
        }
        umma<CG, F8>(tmem + (uint32_t)((i & 1) * N), ad, bd, idesc, acc);
        acc = 1;
      }
    }
    commit<CG>(&bar);
    mbar_wait(&bar, 0);
    long long t1 = clock64();
    out[blockIdx.x] = t1 - t0;
  }
  if (FILL > 0 && warp == 2 && lane == 0) {
    // keep 4 bulk copies of FILL*8 bytes (one per 8 MMAs) in flight
    const uint32_t bytes = FILL * 8;
    for (int i = 0; i < iters; ++i) {
      const int s = i & 3;
      if (i >= 4) mbar_wait(&fbar[s], ((i >> 2) - 1) & 1);
      mbar_expect_tx(&fbar[s], bytes);
      bulk_g2s(sF + s * 16384, gsrc + ((size_t)blockIdx.x * 65536 + (size_t)s * 16384), bytes, &fbar[s]);
    }
    for (int i = iters; i < iters + 4; ++i) { if (i >= 4) mbar_wait(&fbar[i & 3], ((i >> 2) - 1) & 1); }
  }
  if (CG == 2 && rank == 1 && warp == 1 && lane == 0) mbar_wait(&bar, 0);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (CG == 2) cluster_sync_all();
  if (warp == 0) { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); tmem_dealloc<CG>(tmem, 512); }
}

template <int CG, int N, int MODE, int FILL, bool F8 = false>
static void run(const char* name, int grid, const unsigned char* gsrc, long long* d_out) {
  const int iters = 512;
  const size_t smem = 208 * 1024;
  cudaFuncSetAttribute(probe_kernel<CG, N, MODE, FILL, F8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaMemset(d_out, 0, 148 * sizeof(long long));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = CG; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  for (int rep = 0; rep < 2; ++rep) {
    cudaError_t e = cudaLaunchKernelEx(&cfg, probe_kernel<CG, N, MODE, FILL, F8>, iters, gsrc, d_out);
    if (e != cudaSuccess) { printf("%s: launch error %s\n", name, cudaGetErrorString(e)); return; }
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: error %s\n", name, cudaGetErrorString(e)); exit(1); }
  }
  long long h[148];
  cudaMemcpy(h, d_out, sizeof h, cudaMemcpyDeviceToHost);
  double sum = 0; int cnt = 0; long long mx = 0;
  for (int i = 0; i < grid; ++i) if (h[i] > 0) { sum += h[i]; ++cnt; if (h[i] > mx) mx = h[i]; }
  const double per = sum / cnt / (iters * 8.0);
  const double macs = (CG == 2 ? 128.0 : 128.0) * N * (F8 ? 32 : 16);     // per SM
  const double peak = F8 ? 8192.0 : 4096.0;                                 // dense MAC/clk/SM: e4m3 twice bf16
  printf("%-44s grid %3d: %7.1f clk/MMA (max %7.1f)  %6.0f MAC/clk/SM  (%.0f%% of %.0f)\n", name, grid, per, mx / (iters * 8.0), macs / per,
         100.0 * macs / per / peak, peak);
}

int main() {
  unsigned char* gsrc; long long* d_out;
  cudaMalloc(&gsrc, (size_t)148 * 65536 + 65536);
  cudaMemset(gsrc, 0, (size_t)148 * 65536 + 65536);
  cudaMalloc(&d_out, 148 * sizeof(long long));
  run<1, 128, 0, 0>("cg1 N128 noswz", 148, gsrc, d_out);
  run<1, 128, 2, 0>("cg1 N128 noswz desc-in-loop", 148, gsrc, d_out);
  run<1, 256, 0, 0>("cg1 N256 noswz", 148, gsrc, d_out);
  run<1, 64, 0, 0>("cg1 N64  noswz", 148, gsrc, d_out);
  run<1, 128, 1, 0>("cg1 N128 sw128", 148, gsrc, d_out);
  run<1, 256, 1, 0>("cg1 N256 sw128", 148, gsrc, d_out);
  run<2, 128, 0, 0>("cg2 M256 N128 noswz", 148, gsrc, d_out);
  run<2, 256, 0, 0>("cg2 M256 N256 noswz", 148, gsrc, d_out);
  run<2, 128, 1, 0>("cg2 M256 N128 sw128", 148, gsrc, d_out);
  run<2, 256, 1, 0>("cg2 M256 N256 sw128", 148, gsrc, d_out);
  run<1, 128, 0, 2048>("cg1 N128 noswz + 2 KB fill per MMA", 148, gsrc, d_out);
  run<1, 128, 1, 2048>("cg1 N128 sw128 + 2 KB fill per MMA", 148, gsrc, d_out);
  run<2, 128, 0, 1024>("cg2 M256 N128 noswz + 1 KB fill per MMA", 148, gsrc, d_out);
  run<1, 128, 0, 0, true>("f8 K32 cg1 N128 noswz", 148, gsrc, d_out);
  run<2, 128, 0, 0, true>("f8 K32 cg2 M256 N128 noswz", 148, gsrc, d_out);
  run<2, 128, 2, 0, true>("f8 K32 cg2 M256 N128 noswz desc-in-loop", 148, gsrc, d_out);
  run<2, 128, 0, 1024, true>("f8 K32 cg2 M256 N128 noswz + 1 KB fill/MMA", 148, gsrc, d_out);
  run<1, 128, 0, 0>("cg1 N128 noswz, 1 CTA", 1, gsrc, d_out);
  return 0;
}
