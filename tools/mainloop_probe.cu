// tools/mainloop_probe.cu -- the GEMM main loop WITHOUT an epilogue: how fast can a CTA pair run
// TMA (L2 -> 128B-swizzled smem ring) + tcgen05.mma cta_group::2 256 x 256 x 64 k-blocks back to back?
//
// umma_probe.cu shows the tensor pipe sustains 4096 MAC/clk/SM from resident operands, l2_feed_probe.cu that the L2
// delivers 73 B/clk/SM into all shared memories at once (the main loop needs 64).  This probe runs both together,
// exactly as gemm_kernel does (5-slot ring of 32 KB per CTA, producer lane + MMA lane, mbarrier full / empty
// pairs, tcgen05.commit frees the slot), with NO epilogue: accumulators are simply overwritten.  What is left between
// this number and the real kernels is the epilogue (TMEM read-out, GELU / combine math, transposes through shared
// memory, global stores); what is left between this number and 4096 is contention between TMA writes and UMMA reads
// of shared memory plus pipeline latency.
//   operands: A rows walk a 64 MB region (one 128-row x K slab per tile, like the state rows), B = 256 weight rows
//   re-read for every tile (L2-resident), K = 512 (GEMM1) or 4096 (GEMM2).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/bin/mainloop_probe tools/mainloop_probe.cu -lcuda
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../glom_pytorch_b200/csrc/ptx.cuh"

using namespace glom;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct Result { unsigned long long cycles, kblocks, wait_full, wait_empty; };

constexpr uint32_t STAGE_BYTES = 32768;

template <int STAGES>
__global__ void __launch_bounds__(128, 1)
mainloop_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, Result* out, int tiles,
                int nkb, int a_rows_total) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], done_bar;
  __shared__ uint32_t tmem_slot;
  const uint32_t rank = cluster_ctarank();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&done_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm(&tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_slot;
  const int K = nkb * 64;
  if (warp == 0 && lane == 0) {
    // TMA producer (both CTAs): A rows of this CTA, its half of the 256 B rows
    int stage = 0; uint32_t phase = 0;
    unsigned long long w = 0;
    for (int t = 0; t < tiles; ++t) {
      const int a_row = (int)(((long long)(cluster_id + (long long)t * num_clusters) * 256) % (a_rows_total - 256)) / 256 * 256 + (int)rank * 128;
      for (int kb = 0; kb < nkb; ++kb) {
        const long long t0 = clock64();
        mbar_wait(&empty_bar[stage], phase ^ 1);
        w += (unsigned long long)(clock64() - t0);
        uint8_t* sa = smem + (size_t)stage * STAGE_BYTES;
        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * STAGE_BYTES);
        const uint32_t bar = mapa_shared(smem_u32(&full_bar[stage]), 0);
        tma_load_2d_2sm(sa, &map_a, bar, kb * 64, a_row);
        tma_load_2d_2sm(sa + 16384, &map_b, bar, kb * 64, (int)rank * 128);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    out[blockIdx.x].wait_empty = w;
  } else if (warp == 1 && lane == 0 && rank == 0) {
    constexpr uint32_t idesc = umma_idesc_bf16(256, 256, 0, 0);
    int stage = 0; uint32_t phase = 0;
    unsigned long long w = 0;
    const long long c0 = clock64();
    for (int t = 0; t < tiles; ++t) {
      const uint32_t d_tmem = tmem_base + (uint32_t)(t & 1) * 256u;
      for (int kb = 0; kb < nkb; ++kb) {
        const long long t0 = clock64();
        mbar_wait(&full_bar[stage], phase);
        w += (unsigned long long)(clock64() - t0);
        tc_fence_after_sync();
        const uint32_t a_addr = smem_u32(smem + (size_t)stage * STAGE_BYTES);
        const uint32_t b_addr = a_addr + 16384;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_2sm(d_tmem, umma_desc_sw128(a_addr + k * 32, 16, 1024), umma_desc_sw128(b_addr + k * 32, 16, 1024), idesc,
                        (kb | k) ? 1u : 0u);
        umma_commit_2sm(&empty_bar[stage], 3);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    umma_commit_2sm(&done_bar, 1);
    mbar_wait(&done_bar, 0);
    out[blockIdx.x].cycles = (unsigned long long)(clock64() - c0);
    out[blockIdx.x].kblocks = (unsigned long long)tiles * nkb;
    out[blockIdx.x].wait_full = w;
  }
  (void)K;
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) { tc_fence_after_sync(); tmem_dealloc_2sm(tmem_base, 512); }
}

template <int STAGES>
static void run(const CUtensorMap& ma, const CUtensorMap& mb, int sms, int nkb, int tiles, int a_rows_total, Result* dres) {
  const size_t smem = 1024 + (size_t)STAGES * STAGE_BYTES;
  cudaFuncSetAttribute(mainloop_kernel<STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(sms / 2 * 2); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 2; ++rep) {
    cudaMemset(dres, 0, sizeof(Result) * sms);
    cudaEventRecord(e0);
    cudaError_t e = cudaLaunchKernelEx(&cfg, mainloop_kernel<STAGES>, ma, mb, dres, tiles, nkb, a_rows_total);
    cudaEventRecord(e1);
    e = e == cudaSuccess ? cudaDeviceSynchronize() : e;
    if (e != cudaSuccess) { printf("FAILED: %s\n", cudaGetErrorString(e)); exit(1); }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  Result* h = (Result*)malloc(sizeof(Result) * sms);
  cudaMemcpy(h, dres, sizeof(Result) * sms, cudaMemcpyDeviceToHost);
  double cyc = 0, wf = 0, we = 0;
  const int pairs = sms / 2;
  for (int i = 0; i < pairs; ++i) { cyc += (double)h[2 * i].cycles; wf += (double)h[2 * i].wait_full; we += (double)h[2 * i].wait_empty; }
  cyc /= pairs; wf /= pairs; we /= pairs;
  const double kb = (double)h[0].kblocks;
  const double rate = kb * 256.0 * 256.0 * 64.0 / cyc / 2.0;      // MAC / clk / SM
  printf("K = %4d  %d-slot ring  %6.0f MAC/clk/SM (%5.1f %% of 4096)   %5.1f clk per k-block (512 ideal)   MMA lane waits for operands %4.1f %% of the time, "
         "producer for a free slot %4.1f %%   %.2f ms, %.0f TFLOP/s chip\n",
         nkb * 64, STAGES, rate, 100.0 * rate / 4096.0, cyc / kb, 100.0 * wf / cyc, 100.0 * we / cyc, ms,
         2.0 * kb * pairs * 256.0 * 256.0 * 64.0 / (ms * 1e-3) / 1e12);
  free(h);
}

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const int a_rows_total = 16384;                     // 16384 rows x 4096 bf16 = 128 MB of A
  const int KMAX = 4096;
  void *a, *b;
  cudaMalloc(&a, (size_t)a_rows_total * KMAX * 2);
  cudaMalloc(&b, (size_t)256 * KMAX * 2);
  cudaMemset(a, 0, (size_t)a_rows_total * KMAX * 2);
  cudaMemset(b, 0, (size_t)256 * KMAX * 2);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn) { printf("no cuTensorMapEncodeTiled\n"); return 1; }
  EncodeTiledFn enc = (EncodeTiledFn)fn;
  CUtensorMap ma, mb;
  {
    cuuint64_t gd[2] = {(cuuint64_t)KMAX, (cuuint64_t)a_rows_total};
    cuuint64_t gs[1] = {(cuuint64_t)KMAX * 2};
    cuuint32_t bx[2] = {64, 128};
    cuuint32_t es[2] = {1, 1};
    if (enc(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a, gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return 1;
    cuuint64_t gdb[2] = {(cuuint64_t)KMAX, 256};
    if (enc(&mb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, b, gdb, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return 1;
  }
  Result* dres;
  cudaMalloc(&dres, sizeof(Result) * sms);
  printf("GEMM main loop without epilogue: TMA ring + tcgen05.mma cta_group::2 256x256x64 k-blocks, %d SMs (%d pairs)\n", sms, sms / 2);
  run<5>(ma, mb, sms, 8, 600, a_rows_total, dres);     // GEMM1-like: K = 512
  run<5>(ma, mb, sms, 64, 80, a_rows_total, dres);     // GEMM2-like: K = 4096
  run<6>(ma, mb, sms, 8, 600, a_rows_total, dres);
  run<6>(ma, mb, sms, 64, 80, a_rows_total, dres);
  run<4>(ma, mb, sms, 8, 600, a_rows_total, dres);
  run<3>(ma, mb, sms, 64, 80, a_rows_total, dres);
  return 0;
}
