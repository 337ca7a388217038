// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA +
// TMEM).  Bit layouts follow the PTX ISA's shared-memory / instruction descriptor tables.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

namespace glom {

#ifndef GLOM_WAIT_TIMEOUT_CYCLES
#define GLOM_WAIT_TIMEOUT_CYCLES (4000000000LL)   // ~2 s at 1.9 GHz: trap instead of hanging the box
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug traps (the launch fails with an error) instead of hanging.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > GLOM_WAIT_TIMEOUT_CYCLES) {
      printf("glom_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// same with acquire semantics at cluster scope: the arrivals come from the peer CTA (mbar_arrive_cluster after a
// fence.proxy.async; a release.cluster arrive costs a GPU-scope MEMBAR per warp and item and is not needed for
// shared-memory data consumed by the tensor core of the writing CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  auto try_wait = [&]() -> uint32_t {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
  };
  if (try_wait()) return;
  const long long t0 = clock64();
  while (!try_wait()) {
    if (clock64() - t0 > GLOM_WAIT_TIMEOUT_CYCLES) {
      printf("glom_b200: cluster mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// One lane of a converged warp (all 32 lanes must execute this).  Control warps run their loops warp-converged and
// predicate the TMA / MMA instructions on the elected lane: issued from inside a divergent `if (lane == 0)` region every
// uniform-datapath instruction (UTMALDG, UTCHMMA, UTCBAR) is wrapped in an ELECT / BRA.U.ANY loop and its operands
// are re-materialised, ~80 instructions per k-block -- measured (profiles/r2_epilogue_probe2.txt): that issue stream, not
// the L2 feed, held the main loop at 81 % of the tensor peak; warp-converged it reaches 100 %.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred;
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {  // generic-proxy smem writes -> async proxy (TMA/UMMA)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}

// fire-and-forget vector atomic add to global memory (no return value: the reduction happens in L2)
__device__ __forceinline__ void red_add_f32x4(float* dst, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// ---------------------------------------------------------------- TMEM (allocation: see the CTA-pair section)
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets row (lane base + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors (tcgen05.mma, kind::f16)
// Shared-memory matrix descriptor, 128-byte swizzle.  start address / LBO / SBO are encoded >> 4.
//   K-major operand  (rows x 64 bf16, 128 B per row):   SBO = 1024 (8 rows), LBO unused (canonical 1)
//   MN-major operand (64 bf16 of MN contiguous per K row): LBO = bytes between 64-wide MN blocks,
//                                                          SBO = 1024 (8 K rows)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;  // layout type: SWIZZLE_128B
  return d;
}
// Instruction descriptor: D=f32, A=B=bf16, dense, no negate.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// ---------------------------------------------------------------- CTA pairs (cta_group::2, cluster of 2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {   // every thread of both CTAs
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_addr` (a shared::cta address) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// TMA load into THIS CTA's shared memory whose bytes are accounted on an mbarrier given as a
// shared::cluster address (the pair leader's barrier).
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm_sa(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(dst_smem),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm_sa_hint(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                        int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst_smem),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// same with an L2 cache policy (createpolicy value), e.g. evict-first for operands that stream through once
__device__ __forceinline__ void tma_load_2d_2sm_hint(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                     int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_3d_2sm(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm_sa(uint32_t dst_smem, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                   int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(dst_smem),
      "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t ncols) {  // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[256 x N] (+)= A[256 x 16] . B[N x 16]^T over the CTA pair: each CTA supplies 128 rows of A and
// N/2 rows of B from its own shared memory and receives its 128 rows of D in its own TMEM.
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once) on the mbarrier at this shared-memory offset in every CTA of `cta_mask` when all
// previously issued MMAs have completed.
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// Programmatic dependent launch: `pdl_wait` blocks until the preceding kernel in the stream has completed and its
// writes are visible; everything before it (barrier init, TMEM allocation, descriptor prefetch) overlaps that
// kernel's tail.  `pdl_launch_dependents` lets the next kernel's CTAs be scheduled as soon as SMs free up.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }


// ---------------------------------------------------------------- in-kernel clock sample
// One thread of block 0 brackets the kernel's working phase with (clock64, %globaltimer) and adds the two deltas to a
// per-kernel accumulator: cycles / ns = the SM clock the kernel actually ran at (under the power cap this differs from
// what NVML or a probe kernel between launches reports).  Cost: four special-register reads and two atomics per launch.
struct ClockSample { long long c0; unsigned long long t0; };
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ ClockSample clock_sample_begin() {
  ClockSample s; s.c0 = clock64(); s.t0 = globaltimer_ns(); return s;
}
__device__ __forceinline__ void clock_sample_end(const ClockSample& s, unsigned long long* acc /* [2]: cycles, ns */) {
  atomicAdd(&acc[0], (unsigned long long)(clock64() - s.c0));
  atomicAdd(&acc[1], globaltimer_ns() - s.t0);
}

// ---------------------------------------------------------------- small math helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


// Packed-pair version for the GEMM1 epilogue (FFMA2 / FADD2: two fp32 lanes per instruction):
// gelu(acc + bias) for two neighbouring columns, returned as a bf16x2 word.  Uses u = -|x| (one OR per
// lane instead of abs) and a degree-5 fit of log2(0.5*erfc(a/sqrt2)) on [0,6] whose leading coefficient
// is negative, so it needs no clamp (p -> -inf, 2^p -> 0 for large |x|); |gelu error| <= 1.9e-6.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// (r2: a relu-free packed form x/2 + u (e - 1/2) with a degree-4 fit was tried -- 11 instead of 12 instructions per pair,
// FFMA2 takes -|x| as an operand modifier and the coefficients as immediates either way -- and dropped: an even-degree fit
// needs a clamp for |x| > 12 (the peaky golden case overflowed), which costs the instruction it saved; a degree-3 fit is
// off by up to 6 bf16 ulps on small outputs.  profiles/r2_epilogue_probe.txt: the GELU's ALU work is what slows the tensor
// pipe in the GEMM1 tiles, 80.7 % -> 62.7 % of peak.)
__device__ __forceinline__ uint32_t gelu_pair_bf16(float acc0, float acc1, float bias0, float bias1) {
  const uint64_t x = f2_add(f2_pack(acc0, acc1), f2_pack(bias0, bias1));
  float x0, x1;
  f2_unpack(x, x0, x1);
  const float u0 = __uint_as_float(__float_as_uint(x0) | 0x80000000u);   // -|x|
  const float u1 = __uint_as_float(__float_as_uint(x1) | 0x80000000u);
  const uint64_t u = f2_pack(u0, u1);
  // p(a) with a = -u: odd coefficients change sign
  uint64_t q = f2_fma(f2_pack(0.00036467931931838393f, 0.00036467931931838393f), u,
                      f2_pack(0.006363349035382271f, 0.006363349035382271f));
  q = f2_fma(q, u, f2_pack(0.05013200640678406f, 0.05013200640678406f));
  q = f2_fma(q, u, f2_pack(-0.4617065489292145f, -0.4617065489292145f));
  q = f2_fma(q, u, f2_pack(1.150075078010559f, 1.150075078010559f));
  q = f2_fma(q, u, f2_pack(-1.0001276731491089f, -1.0001276731491089f));
  float q0, q1;
  f2_unpack(q, q0, q1);
  const uint64_t e = f2_pack(ex2_approx(q0), ex2_approx(q1));
  const uint64_t g = f2_fma(u, e, f2_pack(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f)));   // relu(x) - |x| Phi(-|x|)
  float g0, g1;
  f2_unpack(g, g0, g1);
  return pack_bf16x2(g0, g1);
}

}  // namespace glom
