// Column-contrastive loss on selected levels (DESIGN §9): the regulariser the reference's README lists as its open Todo
// ("contrastive / consistency regularization of top-ish levels").  Two views za, zb (B, n, L, d); per selected level the
// R = B n unit-normalised rows a_r, b_r; logits s_rc = <a_r, b_c> / tau over the candidate set {r} u {other images}:
//   loss = mean_(level, r) 1/2 [ (lse_c s_rc - s_rr) + (lse_c s_cr - s_rr) ].
//
//   ct_normalise_kernel   (CUDA cores) rows of the selected levels -> bf16 A, B (level, row, d), 1 / |z|, s_rr
//   ct_kernel<false>      (tcgen05)    E_r = sum over other-image columns of 2^((<a_r, b_c> - 1) log2e / tau)
//                                      (run on (A, B) and on (B, A): row and column sums)
//   ct_rows_kernel        per row: the loss term, lse (log2 units), G_rr - 1; a fixed-order block partial of the loss
//   ct_sum_kernel         one block: the partials in a fixed order -> the loss scalar
//   ct_kernel<true>       (tcgen05)    dA_r = g (O_r + (G_rr - 1) b_r) / (tau R_total),  O_r = sum_c G_rc b_c  over
//                                      other-image columns, G recomputed per tile (run again with A, B swapped for dB)
//   ct_normalise_bwd_kernel (CUDA cores) dz = (dA - a <a, dA>) / |z| at the selected levels, zeros elsewhere
//
// Stabiliser: rows are unit vectors, so |s| <= 1 / tau and 1 / tau replaces the running maximum; with tau >= 0.03 every
// exponent (s - 1/tau) log2e lies in [-96, ~0.1] log2 units, inside fp32's normal range (the ATTN_BOUND_MAX argument).
// No buffer grows with R^2: S and G only ever exist as one 128 x 128 tile in TMEM / shared memory.  No atomics: every
// sum has one owner and a fixed order, so the loss and both gradients are bit-reproducible.
#include "engine.h"
#include "ptx.cuh"

#include <stdio.h>

namespace glom {

namespace {

constexpr int CT_BM = 128;                  // rows per tile = UMMA M = TMEM lanes
constexpr int CT_BN = 128;                  // columns per S tile
constexpr int CT_BK = 64;                   // bf16 per 128-byte swizzle row
constexpr uint32_t CT_CHUNK = 16384;        // 128 rows x 64 bf16
constexpr uint32_t CT_SLOT = 32768;         // ring slot: A chunk + B chunk, or 64 keys x 256 d-columns of V
constexpr int CT_EPI_WARPS = 8;             // 4 TMEM lane quadrants x 2 column halves
constexpr int CT_THREADS = 32 * (CT_EPI_WARPS + 2);
constexpr int CT_LSE_STAGES = 3;            // ~100 KB: two lse CTAs per SM
constexpr int CT_GRAD_STAGES = 4;
constexpr int CT_OSLICE = 256;              // d-columns of O per grad CTA (TMEM: 2 x 128 S + 256 O = 512 columns)

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_1sm(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_1sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[128 x N] (+)= A[128 x 16] . B[N x 16]^T, operands in this CTA's shared memory
__device__ __forceinline__ void umma_bf16_1sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_1sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct CtParams {
  int R, Rp, n, d, nlev;          // rows per level, R rounded up to 128, columns per image, dim, selected levels
  int row_tiles, col_tiles;
  int nsplit, tiles_per_split;    // lse: column range split of a row tile (partial sums in esum[split])
  int nslice;                     // grad: 256-wide d-slices of O
  float k;                        // log2(e) / tau
  float* esum;                    // lse: [nsplit][nlev][Rp]
  const float* m_row;             // grad: [nlev][Rp] (lse_r - 1/tau) log2e of the row operand
  const float* m_col;             //       same for the column operand
  const float* dg;                //       [nlev][Rp] G_rr - 1
  const __nv_bfloat16* v;         //       column operand rows (nlev, R, d): the diagonal term
  const float* grad_loss;         //       device scalar dL/dloss
  float inv_tau_rtot;             //       1 / (tau R_total)
  float* dz;                      //       (B, n, L, d) contiguous; this call writes the selected levels' slots
  int L;
  int lev[GLOM_CT_MAX_SEL];
};

// Column tile c0 lies wholly inside the single image of row tile r0: no candidate there, skipped by every role.
__device__ __forceinline__ bool tile_skipped(const CtParams& p, int r0, int c0) {
  const int ib = r0 / p.n;
  return min(r0 + CT_BM - 1, p.R - 1) / p.n == ib && c0 / p.n == ib && min(c0 + CT_BN - 1, p.R - 1) / p.n == ib;
}
// Some (row, column) of the tile pair shares an image, or columns run past R: the epilogue masks per element.
__device__ __forceinline__ bool tile_masked(const CtParams& p, int r0, int c0) {
  if (c0 + CT_BN > p.R) return true;
  const int rlo = r0 / p.n, rhi = min(r0 + CT_BM - 1, p.R - 1) / p.n;
  const int clo = c0 / p.n, chi = (c0 + CT_BN - 1) / p.n;
  return !(chi < rlo || clo > rhi);
}

// grid: one CTA per (level, row tile, column split) [lse] or (level, row tile, d-slice) [grad]; warps 0-7 epilogue,
// warp 8 TMA producer, warp 9 MMA issuer + TMEM allocator.
template <bool GRAD>
__global__ void __launch_bounds__(CT_THREADS, 1)
ct_kernel(const __grid_constant__ CUtensorMap map_a,   // row operand (d, R, nlev) box (64, 128, 1)
          const __grid_constant__ CUtensorMap map_b,   // column operand, same box
          const __grid_constant__ CUtensorMap map_v,   // column operand, box (64, 64, 1): MN-major V of O = G V
          const __grid_constant__ CtParams p) {
  constexpr int STAGES = GRAD ? CT_GRAD_STAGES : CT_LSE_STAGES;
  constexpr uint32_t TMEM_COLS = GRAD ? 512 : 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = smem;
  uint8_t* gsm = ring + STAGES * CT_SLOT;                                    // grad: 2 x [2 chunks of 128 x 64] bf16 G
  float* red = reinterpret_cast<float*>(gsm + (GRAD ? 2 * 2 * CT_CHUNK : 0)); // lse: [2][128] row sums of the two halves
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(red + 2 * CT_BM);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* sfull = empty_bar + STAGES;      // [2] S tile in TMEM buffer
  uint64_t* sempty = sfull + 2;              // [2] buffer read out by the 8 epilogue warps
  uint64_t* gfull = sempty + 2;              // [2] G tile in shared memory
  uint64_t* gempty = gfull + 2;              // [2] G buffer consumed by its O MMAs
  uint64_t* ofull = gempty + 2;              // O slice complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ofull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_TMA = CT_EPI_WARPS, W_MMA = CT_EPI_WARPS + 1;
  int item = blockIdx.x;
  const int sub = item % (GRAD ? p.nslice : p.nsplit);   // d-slice | column split
  item /= GRAD ? p.nslice : p.nsplit;
  const int rt = item % p.row_tiles, ls = item / p.row_tiles;
  const int r0 = rt * CT_BM;
  const int ct_beg = GRAD ? 0 : sub * p.tiles_per_split;
  const int ct_end = GRAD ? p.col_tiles : min(p.col_tiles, ct_beg + p.tiles_per_split);
  const int kchunks = p.d / CT_BK;
  const int ow = min(CT_OSLICE, p.d - sub * CT_OSLICE);   // grad: O slice width (multiple of 64)
  const int nbox = ow / 64;

  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&map_a); tma_prefetch_desc(&map_b);
    if (GRAD) tma_prefetch_desc(&map_v);
  }
  if (warp == W_MMA) {
    if (lane == 0) {
      for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
      for (int i = 0; i < 2; ++i) {
        mbar_init(&sfull[i], 1); mbar_init(&sempty[i], CT_EPI_WARPS);
        mbar_init(&gfull[i], CT_EPI_WARPS); mbar_init(&gempty[i], 1);
      }
      mbar_init(ofull, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc_1sm(tmem_slot, TMEM_COLS);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == W_TMA) {
    // ------------------------------------------------------------------ TMA producer, warp-converged
    // ring order: S_0 operands, [grad: S_1, V_0, S_2, V_1, ...], i.e. V_(j-1) after S_j (the MMA issuer's order)
    const uint32_t elected = elect_one();
    int stage = 0; uint32_t phase = 0;
    const uint32_t ring0 = smem_u32(ring);
    auto load_s = [&](int c0) {
      for (int kc = 0; kc < kchunks; ++kc) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elected) {
          const uint32_t s = ring0 + (uint32_t)stage * CT_SLOT;
          mbar_arrive_expect_tx(&full_bar[stage], 2 * CT_CHUNK);
          tma_load_3d(s, &map_a, &full_bar[stage], kc * CT_BK, r0, ls);
          tma_load_3d(s + CT_CHUNK, &map_b, &full_bar[stage], kc * CT_BK, c0, ls);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    };
    auto load_v = [&](int c0) {
      for (int kc = 0; kc < 2; ++kc) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elected) {
          const uint32_t s = ring0 + (uint32_t)stage * CT_SLOT;
          mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)nbox * 8192u);
          for (int i = 0; i < nbox; ++i)
            tma_load_3d(s + i * 8192, &map_v, &full_bar[stage], sub * CT_OSLICE + i * 64, c0 + kc * 64, ls);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    };
    int prev = -1;
    for (int ct = ct_beg; ct < ct_end; ++ct) {
      const int c0 = ct * CT_BN;
      if (tile_skipped(p, r0, c0)) continue;
      load_s(c0);
      if (GRAD && prev >= 0) load_v(prev);
      prev = c0;
    }
    if (GRAD && prev >= 0) load_v(prev);
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer, warp-converged
    const uint32_t elected = elect_one();
    int stage = 0; uint32_t phase = 0;
    const uint32_t ring_lo = smem_u32(ring) >> 4;
    const uint64_t kdesc0 = umma_desc_sw128(0, 16, 1024);      // K-major: A, B chunks and G
    const uint64_t vdesc0 = umma_desc_sw128(0, 8192, 1024);    // MN-major V: 64-column boxes 8 KB apart
    const uint32_t idesc_s = umma_idesc_bf16(CT_BM, CT_BN, 0, 0);
    const uint32_t idesc_o = umma_idesc_bf16(CT_BM, ow, 0, 1);
    auto mma_s = [&](int j) {
      const uint32_t buf = j & 1;
      mbar_wait(&sempty[buf], ((j >> 1) & 1) ^ 1);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + buf * CT_BN;
      for (int kc = 0; kc < kchunks; ++kc) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elected) {
          const uint32_t s_lo = ring_lo + (uint32_t)stage * (CT_SLOT >> 4);
          const uint64_t ad = kdesc0 + s_lo, bd = kdesc0 + s_lo + (CT_CHUNK >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_1sm(d_tmem, ad + 2 * k, bd + 2 * k, idesc_s, (kc | k) != 0 ? 1u : 0u);
          umma_commit_1sm(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (elected) umma_commit_1sm(&sfull[buf]);
      __syncwarp();
    };
    auto mma_o = [&](int j) {
      const uint32_t gb = j & 1;
      mbar_wait(&gfull[gb], (j >> 1) & 1);
      tc_fence_after_sync();
      const uint32_t g_lo = (smem_u32(gsm) >> 4) + gb * (2 * CT_CHUNK >> 4);
      for (int kc = 0; kc < 2; ++kc) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elected) {
          const uint64_t ad = kdesc0 + g_lo + kc * (CT_CHUNK >> 4);
          const uint64_t bd = vdesc0 + ring_lo + (uint32_t)stage * (CT_SLOT >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_1sm(tmem_base + 2 * CT_BN, ad + 2 * k, bd + (2048 >> 4) * k, idesc_o, (j | kc | k) != 0 ? 1u : 0u);
          umma_commit_1sm(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (elected) umma_commit_1sm(&gempty[gb]);
      __syncwarp();
    };
    int j = 0;
    for (int ct = ct_beg; ct < ct_end; ++ct) {
      if (tile_skipped(p, r0, ct * CT_BN)) continue;
      mma_s(j);
      if (GRAD && j > 0) mma_o(j - 1);
      ++j;
    }
    if (GRAD && j > 0) {
      mma_o(j - 1);
      if (elected) umma_commit_1sm(ofull);
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ epilogue: warp = (quad, half)
    const int quad = warp & 3, half = warp >> 2;
    const int t = quad * 32 + lane;              // row inside the tile == TMEM lane
    const int r = r0 + t;
    const bool row_ok = r < p.R;
    const int own_lo = (r / p.n) * p.n, own_hi = own_lo + p.n;   // this row's image: not a candidate
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const float k = p.k;
    const size_t lrow = (size_t)ls * p.Rp;
    const float m_r = GRAD ? p.m_row[lrow + r] : 0.f;     // Rp-padded: rows >= R read a finite 0
    float acc = 0.f;
    int j = 0;
    for (int ct = ct_beg; ct < ct_end; ++ct) {
      const int c0 = ct * CT_BN;
      if (tile_skipped(p, r0, c0)) continue;
      const bool masked = tile_masked(p, r0, c0);
      const uint32_t buf = j & 1;
      mbar_wait(&sfull[buf], (j >> 1) & 1);
      tc_fence_after_sync();
      if (GRAD) mbar_wait(&gempty[buf], ((j >> 1) & 1) ^ 1);
#pragma unroll 1
      for (int c = 0; c < 64; c += 32) {
        uint32_t v[32];
        tmem_ld32(lane_addr + buf * CT_BN + half * 64 + c, v);
        tmem_ld_wait();
        const int col0 = c0 + half * 64 + c;
        if (!GRAD) {
          float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            float x = ex2_approx(fmaf(__uint_as_float(v[e]), k, -k));
            const int col = col0 + e;
            if (masked && (col >= p.R || (col >= own_lo && col < own_hi))) x = 0.f;
            part[e & 3] += x;
          }
          acc += (part[0] + part[1]) + (part[2] + part[3]);
        } else {
          const float4* mc4 = reinterpret_cast<const float4*>(p.m_col + lrow + col0);
          uint32_t pk[16];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 mc = __ldg(mc4 + q);
            const float mcv[4] = {mc.x, mc.y, mc.z, mc.w};
            float g[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float sk = fmaf(__uint_as_float(v[4 * q + e]), k, -k);
              g[e] = 0.5f * (ex2_approx(sk - m_r) + ex2_approx(sk - mcv[e]));
              const int col = col0 + 4 * q + e;
              if (masked && (col >= p.R || (col >= own_lo && col < own_hi))) g[e] = 0.f;
            }
            pk[2 * q] = pack_bf16x2(g[0], g[1]);
            pk[2 * q + 1] = pack_bf16x2(g[2], g[3]);
          }
          // G row t, keys [half * 64 + c, +32): chunk `half` of buffer `buf`, UMMA K-major SW128 layout
          uint8_t* rowp = gsm + buf * (2 * CT_CHUNK) + half * CT_CHUNK + (size_t)t * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(rowp + ((((c >> 3) + q) ^ (t & 7)) << 4)) =
                make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sempty[buf]);
      if (GRAD) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&gfull[buf]);
      }
      ++j;
    }
    if (!GRAD) {
      red[half * CT_BM + t] = acc;
      named_bar_sync(1, CT_EPI_WARPS * 32);
      if (half == 0 && row_ok) p.esum[((size_t)sub * p.nlev + ls) * p.Rp + r] = red[t] + red[CT_BM + t];
    } else {
      // dA_r = g (O_r + (G_rr - 1) b_r) / (tau R_total), this half of the slice's columns, straight into dz
      if (j > 0) {
        mbar_wait(ofull, 0);
        tc_fence_after_sync();
      }
      const float scale = __ldg(p.grad_loss) * p.inv_tau_rtot;
      const float dg = p.dg[lrow + r];
      const int hw = ow >> 1;
      const __nv_bfloat16* vrow = p.v + ((size_t)ls * p.R + (row_ok ? r : 0)) * p.d + sub * CT_OSLICE;
      float* dst = p.dz + ((size_t)(row_ok ? r : 0) * p.L + p.lev[ls]) * p.d + sub * CT_OSLICE;
#pragma unroll 1
      for (int c = half * hw; c < half * hw + hw; c += 32) {
        uint32_t v[32];
        if (j > 0) {
          tmem_ld32(lane_addr + 2 * CT_BN + c, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = 0u;
        }
        if (!row_ok) continue;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 bw = __ldg(reinterpret_cast<const uint4*>(vrow + c + 8 * q));
          const uint32_t bb[4] = {bw.x, bw.y, bw.z, bw.w};
          float o[8];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            o[2 * e] = fmaf(dg, __uint_as_float(bb[e] << 16), __uint_as_float(v[8 * q + 2 * e])) * scale;
            o[2 * e + 1] = fmaf(dg, __uint_as_float(bb[e] & 0xFFFF0000u), __uint_as_float(v[8 * q + 2 * e + 1])) * scale;
          }
          reinterpret_cast<float4*>(dst + c + 8 * q)[0] = make_float4(o[0], o[1], o[2], o[3]);
          reinterpret_cast<float4*>(dst + c + 8 * q)[1] = make_float4(o[4], o[5], o[6], o[7]);
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == W_MMA) {
    tc_fence_after_sync();
    tmem_dealloc_1sm(tmem_base, TMEM_COLS);
  }
}

struct SelLevels { int lev[GLOM_CT_MAX_SEL]; };

// one warp per (selected level, row): F.normalize in fp32, bf16 operands, 1/|z| and s_rr = <bf16 a_r, bf16 b_r>
__global__ void __launch_bounds__(256)
ct_normalise_kernel(const float* __restrict__ za, const float* __restrict__ zb, ContrastiveStrides sa, ContrastiveStrides sb,
                    int R, int Rp, int n, int d, int nlev, const __grid_constant__ SelLevels sel, __nv_bfloat16* __restrict__ ah,
                    __nv_bfloat16* __restrict__ bh, float* __restrict__ inv_a, float* __restrict__ inv_b,
                    float* __restrict__ srr) {
  const long long wid = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (wid >= (long long)nlev * R) return;
  const int ls = (int)(wid / R), r = (int)(wid % R);
  const int b = r / n, i = r % n, l = sel.lev[ls];
  const float* xa = za + b * sa.b + i * sa.n + l * sa.l;
  const float* xb = zb + b * sb.b + i * sb.n + l * sb.l;
  float qa = 0.f, qb = 0.f;
  for (int c = lane; c < d; c += 32) { const float u = xa[c], w = xb[c]; qa = fmaf(u, u, qa); qb = fmaf(w, w, qb); }
  qa = warp_sum(qa); qb = warp_sum(qb);
  const float ia = 1.f / fmaxf(sqrtf(qa), 1e-12f), ib = 1.f / fmaxf(sqrtf(qb), 1e-12f);
  const size_t o = ((size_t)ls * R + r) * d;
  float s = 0.f;
  for (int c = lane; c < d; c += 32) {
    const __nv_bfloat16 u = __float2bfloat16_rn(xa[c] * ia), w = __float2bfloat16_rn(xb[c] * ib);
    ah[o + c] = u; bh[o + c] = w;
    s = fmaf(__bfloat162float(u), __bfloat162float(w), s);
  }
  s = warp_sum(s);
  if (lane == 0) {
    const size_t q = (size_t)ls * Rp + r;
    inv_a[q] = ia; inv_b[q] = ib; srr[q] = s;
  }
}

// one thread per (selected level, padded row): X = sum_(c != r) exp(s_rc - s_rr) in both directions, the row's loss term
// 1/2 (log1p X_a + log1p X_b), the lse of both directions (log2 units, relative to 1/tau) and G_rr - 1; padding rows
// get finite zeros.  Block partials of the loss in a fixed tree order.
__global__ void __launch_bounds__(256)
ct_rows_kernel(const float* __restrict__ ea, const float* __restrict__ eb, const float* __restrict__ srr, int R, int Rp,
               int nlev, int nsplit, float k, float* __restrict__ m_a, float* __restrict__ m_b, float* __restrict__ dg,
               float* __restrict__ partials) {
  __shared__ float red[256];
  const long long q = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long total = (long long)nlev * Rp;
  float loss = 0.f;
  if (q < total) {
    const int r = (int)(q % Rp);
    float ma = 0.f, mb = 0.f, g = 0.f;
    if (r < R) {
      float sa = 0.f, sb = 0.f;
      for (int s = 0; s < nsplit; ++s) { sa += ea[(size_t)s * total + q]; sb += eb[(size_t)s * total + q]; }
      const float s = srr[q];
      const float f = exp2f((1.f - s) * k);            // exp(1/tau - s_rr) <= 2^96.5
      const float xa = sa * f, xb = sb * f;
      loss = 0.5f * (log1pf(xa) + log1pf(xb));
      const float e_rr = exp2f((s - 1.f) * k);         // >= 2^-96.5: normal
      ma = log2f(sa + e_rr);
      mb = log2f(sb + e_rr);
      g = -0.5f * (xa / (1.f + xa) + xb / (1.f + xb));  // G_rr - 1 without cancellation
    }
    m_a[q] = ma; m_b[q] = mb; dg[q] = g;
  }
  red[threadIdx.x] = loss;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(1024) ct_sum_kernel(const float* __restrict__ partials, int count, float inv_rows, float* out) {
  __shared__ float red[1024];
  float s = 0.f;
  for (int i = threadIdx.x; i < count; i += 1024) s += partials[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 512; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0] * inv_rows;
}

// one warp per (tensor, row, level): selected levels hold dA from ct_kernel<true>; dz = (dA - a <a, dA>) / |z| in place
// (F.normalize's backward; a clamped norm passes dA / eps through).  Other levels are zeroed.
__global__ void __launch_bounds__(256)
ct_normalise_bwd_kernel(const float* __restrict__ za, const float* __restrict__ zb, ContrastiveStrides sa,
                        ContrastiveStrides sb, const float* __restrict__ inv_a, const float* __restrict__ inv_b, int R, int Rp,
                        int n, int L, int d, int nlev, const __grid_constant__ SelLevels sel, float* __restrict__ dza, float* __restrict__ dzb) {
  const long long wid = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (wid >= (long long)R * L) return;
  const bool second = blockIdx.y == 1;
  const float* z = second ? zb : za;
  const ContrastiveStrides st = second ? sb : sa;
  float* dz = (second ? dzb : dza) + wid * d;
  const int r = (int)(wid / L), l = (int)(wid % L);
  int ls = -1;
  for (int s = 0; s < nlev; ++s) ls = sel.lev[s] == l ? s : ls;
  if (ls < 0) {
    for (int c = lane; c < d; c += 32) dz[c] = 0.f;
    return;
  }
  const float inv = (second ? inv_b : inv_a)[(size_t)ls * Rp + r];
  const float* x = z + (r / n) * st.b + (r % n) * st.n + l * st.l;
  float dot = 0.f, sq = 0.f;
  for (int c = lane; c < d; c += 32) { const float u = x[c]; dot = fmaf(u * inv, dz[c], dot); sq = fmaf(u, u, sq); }
  dot = warp_sum(dot);
  sq = warp_sum(sq);
  const bool clamped = !(sqrtf(sq) > 1e-12f);
  for (int c = lane; c < d; c += 32) dz[c] = clamped ? dz[c] * inv : inv * (dz[c] - x[c] * inv * dot);
}

bool ct_map(EncodeTiledFn enc, CUtensorMap* m, const void* base, int R, int d, int nlev, uint32_t box_rows, char* err,
            size_t errlen, const char* what) {
  cuuint64_t gd[3] = {(cuuint64_t)d, (cuuint64_t)R, (cuuint64_t)nlev};
  cuuint64_t gs[2] = {(cuuint64_t)d * 2, (cuuint64_t)R * d * 2};
  cuuint32_t bx[3] = {(cuuint32_t)CT_BK, box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gd, gs, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { snprintf(err, errlen, "cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r); return false; }
  return true;
}

template <bool GRAD>
constexpr size_t ct_smem_bytes() {
  return 1024 + (size_t)(GRAD ? CT_GRAD_STAGES : CT_LSE_STAGES) * CT_SLOT + (GRAD ? 4 * CT_CHUNK : 0) + 2 * CT_BM * 4 + 256;
}

template <bool GRAD>
cudaError_t ct_launch(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mv, const CtParams& p, int items,
                      cudaStream_t st) {
  static SmemOptIn optin;
  if (cudaError_t e = optin.ensure(ct_kernel<GRAD>, ct_smem_bytes<GRAD>())) return e;
  ct_kernel<GRAD><<<items, CT_THREADS, ct_smem_bytes<GRAD>(), st>>>(ma, mb, mv, p);
  return cudaGetLastError();
}

CtParams ct_params(const ContrastiveGeom& g) {
  CtParams p{};
  p.R = g.R; p.Rp = g.Rp; p.n = g.n; p.d = g.d; p.nlev = g.nsel; p.L = g.L;
  p.row_tiles = g.Rp / CT_BM;
  p.col_tiles = g.Rp / CT_BN;
  p.k = 1.4426950408889634f / g.tau;
  for (int i = 0; i < g.nsel; ++i) p.lev[i] = g.sel[i];
  return p;
}

}  // namespace

ContrastiveLayout contrastive_layout(const ContrastiveGeom& g) {
  ContrastiveLayout w{};
  const size_t rows = (size_t)g.nsel * g.Rp;            // per-row fp32 arrays, Rp-padded per level
  size_t off = 0;
  w.a_off = off; off = align_up(off + (size_t)g.nsel * g.R * g.d * 2, 1024);
  w.b_off = off; off = align_up(off + (size_t)g.nsel * g.R * g.d * 2, 1024);
  w.inv_a_off = off; off = align_up(off + rows * 4, 1024);
  w.inv_b_off = off; off = align_up(off + rows * 4, 1024);
  w.m_a_off = off; off = align_up(off + rows * 4, 1024);
  w.m_b_off = off; off = align_up(off + rows * 4, 1024);
  w.dg_off = off; off = align_up(off + rows * 4, 1024);
  w.saved = off;
  off = 0;
  w.ea_off = off; off = align_up(off + (size_t)GLOM_CT_MAX_SPLIT * rows * 4, 1024);
  w.eb_off = off; off = align_up(off + (size_t)GLOM_CT_MAX_SPLIT * rows * 4, 1024);
  w.srr_off = off; off = align_up(off + rows * 4, 1024);
  w.part_off = off; off = align_up(off + (rows + 255) / 256 * 4, 1024);
  w.scratch = off;
  return w;
}

int contrastive_forward(const ContrastiveGeom& g, const float* za, const float* zb, float* loss, void* saved, void* scratch,
                        EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches, char* err, size_t errlen) {
  const ContrastiveLayout w = contrastive_layout(g);
  uint8_t* sv = static_cast<uint8_t*>(saved);
  uint8_t* sc = static_cast<uint8_t*>(scratch);
  auto* ah = reinterpret_cast<__nv_bfloat16*>(sv + w.a_off);
  auto* bh = reinterpret_cast<__nv_bfloat16*>(sv + w.b_off);
  float* inv_a = reinterpret_cast<float*>(sv + w.inv_a_off);
  float* inv_b = reinterpret_cast<float*>(sv + w.inv_b_off);
  float* ea = reinterpret_cast<float*>(sc + w.ea_off);
  float* eb = reinterpret_cast<float*>(sc + w.eb_off);
  float* srr = reinterpret_cast<float*>(sc + w.srr_off);
  float* part = reinterpret_cast<float*>(sc + w.part_off);
  SelLevels sel{};
  for (int i = 0; i < g.nsel; ++i) sel.lev[i] = g.sel[i];
  cudaError_t e;
  {
    const long long warps = (long long)g.nsel * g.R;
    ct_normalise_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(za, zb, g.sa, g.sb, g.R, g.Rp, g.n, g.d, g.nsel, sel, ah,
                                                                     bh, inv_a, inv_b, srr);
    if (launches) ++*launches;
    if ((e = cudaGetLastError()) != cudaSuccess) { snprintf(err, errlen, "contrastive normalise: %s", cudaGetErrorString(e)); return -3; }
  }
  CtParams p = ct_params(g);
  // split each row tile's columns so that the grid covers the SMs about twice (partial sums, summed in ct_rows_kernel)
  const int base_items = g.nsel * p.row_tiles;
  int nsplit = (4 * num_sms + base_items - 1) / base_items;
  nsplit = nsplit < 1 ? 1 : nsplit > GLOM_CT_MAX_SPLIT ? GLOM_CT_MAX_SPLIT : nsplit;
  if (nsplit > p.col_tiles) nsplit = p.col_tiles;
  p.tiles_per_split = (p.col_tiles + nsplit - 1) / nsplit;
  p.nsplit = (p.col_tiles + p.tiles_per_split - 1) / p.tiles_per_split;
  CUtensorMap mapa, mapb;
  if (!ct_map(enc, &mapa, ah, g.R, g.d, g.nsel, CT_BM, err, errlen, "contrastive.a")) return -3;
  if (!ct_map(enc, &mapb, bh, g.R, g.d, g.nsel, CT_BM, err, errlen, "contrastive.b")) return -3;
  for (int dir = 0; dir < 2; ++dir) {
    p.esum = dir ? eb : ea;
    e = dir ? ct_launch<false>(mapb, mapa, mapa, p, base_items * p.nsplit, st)
            : ct_launch<false>(mapa, mapb, mapb, p, base_items * p.nsplit, st);
    if (launches) ++*launches;
    if (e != cudaSuccess) { snprintf(err, errlen, "contrastive lse kernel: %s", cudaGetErrorString(e)); return -3; }
  }
  const long long rows = (long long)g.nsel * g.Rp;
  const int blocks = (int)((rows + 255) / 256);
  ct_rows_kernel<<<blocks, 256, 0, st>>>(ea, eb, srr, g.R, g.Rp, g.nsel, p.nsplit, p.k,
                                         reinterpret_cast<float*>(sv + w.m_a_off), reinterpret_cast<float*>(sv + w.m_b_off),
                                         reinterpret_cast<float*>(sv + w.dg_off), part);
  if (launches) ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) { snprintf(err, errlen, "contrastive rows: %s", cudaGetErrorString(e)); return -3; }
  ct_sum_kernel<<<1, 1024, 0, st>>>(part, blocks, 1.0f / (float)((double)g.nsel * g.R), loss);
  if (launches) ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) { snprintf(err, errlen, "contrastive sum: %s", cudaGetErrorString(e)); return -3; }
  return 0;
}

int contrastive_backward(const ContrastiveGeom& g, const float* za, const float* zb, const float* grad_loss, const void* saved,
                         float* dza, float* dzb, EncodeTiledFn enc, cudaStream_t st, int* launches, char* err, size_t errlen) {
  const ContrastiveLayout w = contrastive_layout(g);
  const uint8_t* sv = static_cast<const uint8_t*>(saved);
  auto* ah = reinterpret_cast<const __nv_bfloat16*>(sv + w.a_off);
  auto* bh = reinterpret_cast<const __nv_bfloat16*>(sv + w.b_off);
  const float* m_a = reinterpret_cast<const float*>(sv + w.m_a_off);
  const float* m_b = reinterpret_cast<const float*>(sv + w.m_b_off);
  CtParams p = ct_params(g);
  p.nslice = (g.d + CT_OSLICE - 1) / CT_OSLICE;
  p.dg = reinterpret_cast<const float*>(sv + w.dg_off);
  p.grad_loss = grad_loss;
  p.inv_tau_rtot = (float)(1.0 / ((double)g.tau * g.nsel * g.R));
  CUtensorMap mapa, mapb, mapva, mapvb;
  if (!ct_map(enc, &mapa, ah, g.R, g.d, g.nsel, CT_BM, err, errlen, "contrastive.a")) return -3;
  if (!ct_map(enc, &mapb, bh, g.R, g.d, g.nsel, CT_BM, err, errlen, "contrastive.b")) return -3;
  if (!ct_map(enc, &mapva, ah, g.R, g.d, g.nsel, 64, err, errlen, "contrastive.va")) return -3;
  if (!ct_map(enc, &mapvb, bh, g.R, g.d, g.nsel, 64, err, errlen, "contrastive.vb")) return -3;
  const int items = g.nsel * p.row_tiles * p.nslice;
  cudaError_t e;
  for (int dir = 0; dir < 2; ++dir) {      // dA: rows A, columns B;  dB: the same with the operands and lse vectors swapped
    p.m_row = dir ? m_b : m_a;
    p.m_col = dir ? m_a : m_b;
    p.v = dir ? ah : bh;
    p.dz = dir ? dzb : dza;
    e = dir ? ct_launch<true>(mapb, mapa, mapva, p, items, st) : ct_launch<true>(mapa, mapb, mapvb, p, items, st);
    if (launches) ++*launches;
    if (e != cudaSuccess) { snprintf(err, errlen, "contrastive grad kernel: %s", cudaGetErrorString(e)); return -3; }
  }
  SelLevels sel{};
  for (int i = 0; i < g.nsel; ++i) sel.lev[i] = g.sel[i];
  const long long warps = (long long)g.R * g.L;
  ct_normalise_bwd_kernel<<<dim3((unsigned)((warps + 7) / 8), 2), 256, 0, st>>>(
      za, zb, g.sa, g.sb, reinterpret_cast<const float*>(sv + w.inv_a_off), reinterpret_cast<const float*>(sv + w.inv_b_off),
      g.R, g.Rp, g.n, g.L, g.d, g.nsel, sel, dza, dzb);
  if (launches) ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) { snprintf(err, errlen, "contrastive normalise backward: %s", cudaGetErrorString(e)); return -3; }
  return 0;
}

}  // namespace glom
