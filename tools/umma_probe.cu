// tools/umma_probe.cu -- measured tcgen05.mma issue-rate ceilings for the instruction shapes an ON-CHIP fused
// GEMM1 -> GEMM2 kernel would have to use (VERDICT r1 "next" #4: build the experiment instead of arguing it).
//
// Every SM (or SM pair) runs one CTA whose single MMA thread issues a long stream of kind::f16 UMMAs (bf16 in, fp32
// accumulate in TMEM) over operands that already sit in 128B-swizzled shared memory (a ring of 4 k-blocks, contents
// irrelevant), commits to an mbarrier and waits; MACs per SM clock per SM are reported per shape:
//
//   cg2 M256 N256 SS   the 256 x 256 CTA-pair tile of gemm_kernel                                   (reference point)
//   cg2 M256 N128 SS   a pair tile with a 128-wide accumulator (what a TMEM budget of Y + H-chunk forces)
//   cg1 M128 N256 SS   one CTA per 128 rows, d_out split across the pair (the DSMEM-exchange design of SURVEY 7.3)
//   cg1 M128 N128 SS   ... with 128-wide hidden chunks
//   cg1 M128 N256 TS   A operand (GELU'd hidden chunk) read from TMEM instead of shared memory
//   cg2 M256 N256 TS   pair tile with A from TMEM
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/bin/umma_probe tools/umma_probe.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../glom_pytorch_b200/csrc/ptx.cuh"

using namespace glom;

__device__ __forceinline__ void umma_bf16_1sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_1sm_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit_1sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_alloc_1sm(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_1sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

struct Result { unsigned long long cycles; unsigned long long mmas; };

// CG = cta_group (1 or 2); M = UMMA M (128 for CG 1, 256 for CG 2); N = UMMA N; TS = A operand from TMEM
template <int CG, int M, int N, bool TS>
__global__ void __launch_bounds__(128, 1) probe_kernel(Result* out, int kblocks) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // ring of 4 k-blocks: A 128 rows x 64 (16 KB) + this CTA's B rows x 64 (N / CG rows)
  constexpr uint32_t B_BYTES = (N / CG) * 128;
  constexpr uint32_t STAGE = 16384 + B_BYTES;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0;
  for (uint32_t i = threadIdx.x; i < 4 * STAGE / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u + i;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  if (threadIdx.x < 32) { if (CG == 2) tmem_alloc_2sm(&tmem_slot, 512); else tmem_alloc_1sm(&tmem_slot, 512); }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  if (CG == 2) cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_slot;
  if (threadIdx.x == 0 && rank == 0) {
    constexpr uint32_t idesc = umma_idesc_bf16(M, N, 0, 0);
    const long long c0 = clock64();
    unsigned long long issued = 0;
    for (int kb = 0; kb < kblocks; ++kb) {
      const uint32_t a_addr = smem_u32(smem + (size_t)(kb & 3) * STAGE);
      const uint32_t b_addr = a_addr + 16384;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint64_t bd = umma_desc_sw128(b_addr + k * 32, 16, 1024);
        const uint32_t d_tmem = tmem_base + (uint32_t)((kb >> 4) & 1) * (TS ? 0u : 256u);      // two accumulator regions (SS)
        if (TS) {
          const uint32_t a_tmem = tmem_base + 256u + (uint32_t)((kb & 3) * 32 + k * 8);        // bf16 A: 8 columns per K=16
          if (CG == 2) umma_bf16_2sm_ts(d_tmem, a_tmem, bd, idesc, (kb | k) ? 1u : 0u);
          else umma_bf16_1sm_ts(d_tmem, a_tmem, bd, idesc, (kb | k) ? 1u : 0u);
        } else {
          const uint64_t ad = umma_desc_sw128(a_addr + k * 32, 16, 1024);
          if (CG == 2) umma_bf16_2sm(d_tmem, ad, bd, idesc, (kb | k) ? 1u : 0u);
          else umma_bf16_1sm(d_tmem, ad, bd, idesc, (kb | k) ? 1u : 0u);
        }
        ++issued;
      }
    }
    if (CG == 2) umma_commit_2sm(&bar, 1); else umma_commit_1sm(&bar);
    mbar_wait(&bar, 0);
    const long long c1 = clock64();
    out[blockIdx.x / CG].cycles = (unsigned long long)(c1 - c0);
    out[blockIdx.x / CG].mmas = issued;
  }
  tc_fence_before_sync();
  __syncthreads();
  if (CG == 2) cluster_sync_all();
  if (threadIdx.x < 32) { tc_fence_after_sync(); if (CG == 2) tmem_dealloc_2sm(tmem_base, 512); else tmem_dealloc_1sm(tmem_base, 512); }
}

template <int CG, int M, int N, bool TS>
static void run(const char* name, int sms, int kblocks, Result* dres) {
  const size_t smem = 1024 + 4 * (16384 + (N / CG) * 128);
  cudaFuncSetAttribute(probe_kernel<CG, M, N, TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(sms / CG * CG); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 2; ++rep) {
    cudaMemset(dres, 0, sizeof(Result) * sms);
    cudaEventRecord(e0);
    cudaError_t e = cudaLaunchKernelEx(&cfg, probe_kernel<CG, M, N, TS>, dres, kblocks);
    cudaEventRecord(e1);
    e = e == cudaSuccess ? cudaDeviceSynchronize() : e;
    if (e != cudaSuccess) { printf("%-18s FAILED: %s\n", name, cudaGetErrorString(e)); exit(1); }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  Result* h = (Result*)malloc(sizeof(Result) * sms);
  cudaMemcpy(h, dres, sizeof(Result) * sms, cudaMemcpyDeviceToHost);
  const int units = sms / CG;
  double worst = 0, sum = 0;
  for (int i = 0; i < units; ++i) { sum += (double)h[i].cycles; if ((double)h[i].cycles > worst) worst = (double)h[i].cycles; }
  const double macs_per_mma = (double)M * N * 16;
  const double rate = macs_per_mma * (double)h[0].mmas / (sum / units) / CG;       // MAC / clk / SM
  const double smem_rd = ((TS ? 0.0 : 128.0 * 32) + (double)(N / CG) * 32) * (double)h[0].mmas / (sum / units);   // operand bytes / clk / SM
  printf("%-18s %7.0f MAC/clk/SM  (%5.1f %% of 4096)   operand smem reads %5.1f B/clk/SM   %.3f ms, %.0f TFLOP/s chip\n", name, rate,
         100.0 * rate / 4096.0, smem_rd, ms, 2.0 * macs_per_mma * (double)h[0].mmas * units / (ms * 1e-3) / 1e12);
  free(h);
}

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  Result* dres;
  cudaMalloc(&dres, sizeof(Result) * sms);
  const int kb = 20000;       // 80 k UMMAs per issuing thread: tens of ms per shape
  printf("UMMA issue-rate ceilings, %d SMs, all SMs busy, operands resident in shared memory / TMEM (no TMA traffic)\n", sms);
  run<2, 256, 256, false>("cg2 M256 N256 SS", sms, kb, dres);
  run<2, 256, 128, false>("cg2 M256 N128 SS", sms, kb, dres);
  run<1, 128, 256, false>("cg1 M128 N256 SS", sms, kb, dres);
  run<1, 128, 128, false>("cg1 M128 N128 SS", sms, kb, dres);
  run<1, 128, 256, true>("cg1 M128 N256 TS", sms, kb, dres);
  run<2, 256, 256, true>("cg2 M256 N256 TS", sms, kb, dres);
  return 0;
}
