// tools/l2_feed_probe.cu -- how many operand bytes per clock can the L2 deliver into the shared memories of all SMs?
//
// The GEMM kernels stage 64 KB of operands per 256 x 256 x 64 pair k-block = 64 B / clk / SM at the full MMA rate
// (tools/umma_probe.cu shows the tensor pipe itself sustains that rate for every shape).  This probe runs the TMA
// producer side ALONE: every SM streams 16 KB boxes of an L2-resident bf16 matrix into a 5-slot shared-memory ring
// (cp.async.bulk.tensor.2d, 128B swizzle, mbarrier completion; a consumer lane frees the slots immediately) and
// reports bytes per SM clock per SM, chip-wide.  Variants:
//   unicast       every CTA loads its own 32 KB per stage (what gemm_kernel does: A box + half-B box)
//   multicast x2  clusters of 2: each CTA loads 16 KB and multicasts it to both CTAs (both receive 32 KB per stage, the
//                 L2 serves 16 KB per CTA): the cost of DELIVERED bytes when half of them are shared
//   multicast x4  clusters of 4, each CTA loads 8 KB, multicast to all four
// `same` = all CTAs walk the same 8 MB region in the same order (maximal L2 hit / request merging), `spread` = every
// CTA starts at a different offset of a 64 MB region.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/bin/l2_feed_probe tools/l2_feed_probe.cu -lcuda
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

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                   smem_u32(dst)),
               "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}

struct Result { unsigned long long cycles, bytes; };

constexpr int STAGES = 5;
constexpr uint32_t STAGE_BYTES = 32768;

// CS = cluster size (1: unicast; 2 / 4: every CTA loads 32 KB / CS per stage and multicasts it to the whole cluster)
template <int CS>
__global__ void __launch_bounds__(64, 1) feed_kernel(const __grid_constant__ CUtensorMap map, Result* out, int iters, int rows_total,
                                                     int spread) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES];
  const uint32_t rank = CS > 1 ? cluster_ctarank() : 0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], CS); }
    fence_barrier_init();
  }
  __syncthreads();
  if (CS > 1) cluster_sync_all();
  constexpr int BOX_ROWS = 256 / CS;                // rows of 128 B this CTA loads per stage (256 rows = 32 KB per stage)
  const int row_base = spread ? (int)(((long long)blockIdx.x * 7919 * 256) % (rows_total - 256)) / 256 * 256 : 0;
  if (threadIdx.x == 0) {
    // producer
    int stage = 0; uint32_t phase = 0;
    const long long c0 = clock64();
    for (int it = 0; it < iters; ++it) {
      mbar_wait(&empty_bar[stage], phase ^ 1);
      mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES);
      int row = (row_base + it * 256) % (rows_total - 256);
      row = row / 256 * 256;
      uint8_t* dst = smem + (size_t)stage * STAGE_BYTES + (size_t)rank * BOX_ROWS * 128;
      if (CS == 1) tma_load_2d(dst, &map, &full_bar[stage], 0, row);
      else tma_load_2d_mc(dst, &map, &full_bar[stage], 0, row + (int)rank * BOX_ROWS, (uint16_t)((1u << CS) - 1));
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
    out[blockIdx.x].cycles = (unsigned long long)(clock64() - c0);
    out[blockIdx.x].bytes = (unsigned long long)iters * STAGE_BYTES;
  } else if (threadIdx.x == 32) {
    // consumer: frees a slot in every CTA of the cluster as soon as its bytes have landed here
    int stage = 0; uint32_t phase = 0;
    for (int it = 0; it < iters; ++it) {
      mbar_wait(&full_bar[stage], phase);
      if (CS == 1) mbar_arrive(&empty_bar[stage]);
      else for (int r = 0; r < CS; ++r) mbar_arrive_cluster(mapa_shared(smem_u32(&empty_bar[stage]), r));
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  }
  __syncthreads();
  if (CS > 1) cluster_sync_all();
}

template <int CS>
static void run(const char* name, const CUtensorMap& map, int sms, int iters, int rows_total, int spread, Result* dres) {
  const size_t smem = 1024 + STAGES * STAGE_BYTES;
  cudaFuncSetAttribute(feed_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (CS > 4) cudaFuncSetAttribute(feed_kernel<CS>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg{};
  int grid = sms / CS * CS;
  if (CS > 1) {
    cfg.gridDim = dim3(CS); cfg.blockDim = dim3(64); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute a[1];
    a[0].id = cudaLaunchAttributeClusterDimension; a[0].val.clusterDim.x = CS; a[0].val.clusterDim.y = 1; a[0].val.clusterDim.z = 1;
    cfg.attrs = a; cfg.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, feed_kernel<CS>, &cfg) == cudaSuccess && nc * CS < grid) grid = nc * CS;
  }
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(64); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 2; ++rep) {
    cudaMemset(dres, 0, sizeof(Result) * sms);
    cudaEventRecord(e0);
    cudaError_t e = cudaLaunchKernelEx(&cfg, feed_kernel<CS>, map, dres, iters, rows_total, spread);
    cudaEventRecord(e1);
    e = e == cudaSuccess ? cudaDeviceSynchronize() : e;
    if (e != cudaSuccess) { printf("%-28s FAILED: %s\n", name, cudaGetErrorString(e)); return; }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  Result* h = (Result*)malloc(sizeof(Result) * sms);
  cudaMemcpy(h, dres, sizeof(Result) * sms, cudaMemcpyDeviceToHost);
  double cyc = 0;
  for (int i = 0; i < grid; ++i) cyc += (double)h[i].cycles;
  cyc /= grid;
  const double per_sm = (double)h[0].bytes / cyc;              // bytes DELIVERED into one SM's shared memory per clock
  printf("%-28s %3d CTAs  delivered %6.1f B/clk/SM = %6.0f B/clk chip (%5.2f TB/s wall)   L2 requests %6.1f B/clk/SM   MMA-rate cap at 64 B/clk/SM: %3.0f %%\n",
         name, grid, per_sm, per_sm * grid, (double)h[0].bytes * grid / (ms * 1e-3) / 1e12, per_sm / CS,
         100.0 * (per_sm < 64.0 ? per_sm / 64.0 : 1.0));
  free(h);
}

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const int rows_total = 64 * 1024 * 1024 / 128;      // 64 MB of 128-byte rows (L2-resident after the first pass)
  void* buf;
  cudaMalloc(&buf, (size_t)rows_total * 128);
  cudaMemset(buf, 1, (size_t)rows_total * 128);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn) { printf("no cuTensorMapEncodeTiled\n"); return 1; }
  EncodeTiledFn enc = (EncodeTiledFn)fn;
  Result* dres;
  cudaMalloc(&dres, sizeof(Result) * sms);
  printf("L2 -> shared-memory feed, %d SMs, TMA only (no MMA), 32 KB delivered per stage and CTA, 5-slot ring\n", sms);
  for (int cs = 1; cs <= 4; cs *= 2) {
    CUtensorMap map;
    cuuint64_t gd[2] = {64, (cuuint64_t)rows_total};
    cuuint64_t gs[1] = {128};
    cuuint32_t bx[2] = {64, (cuuint32_t)(256 / cs)};
    cuuint32_t es[2] = {1, 1};
    if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, buf, gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { printf("encode failed\n"); return 1; }
    const int iters = 40000;
    for (int spread = 0; spread <= 1; ++spread) {
      char name[64];
      snprintf(name, sizeof(name), "%s x%d, %s", cs == 1 ? "unicast" : "multicast", cs, spread ? "spread" : "same");
      if (cs == 1) run<1>(name, map, sms, iters, spread ? rows_total : 8 * 1024 * 1024 / 128, spread, dres);
      if (cs == 2) run<2>(name, map, sms, iters, spread ? rows_total : 8 * 1024 * 1024 / 128, spread, dres);
      if (cs == 4) run<4>(name, map, sms, iters, spread ? rows_total : 8 * 1024 * 1024 / 128, spread, dres);
    }
  }
  return 0;
}
