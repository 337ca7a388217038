// Tensor-core (tcgen05 / TMEM / TMA) kernels of the GLOM column update for sm_100a.
//
//   gemm_kernel<0>  K1: H = gelu_erf(A_g . W1_g^T + b1_g)         all 2L-1 MLP groups, one launch
//                       (GroupedFeedForward first Conv1d + GELU, glom_pytorch.py:29-30, calls :134/:136)
//   gemm_kernel<1>  K2: S' = (S + C + [H_bu,l | H_td,l] . [W2bu_l | W2td_l]^T + b2) / c_l
//                       (second Conv1d :31 of both nets, F.pad zero top level :137, combine :141-142)
//   attn_kernel     K3: C = softmax_j(<S_i, S_j/|S_j|> d^-1/2, diag := -5e-4, radius mask) . S
//                       (ConsensusAttention.forward :56-73)
//
// All three are warp-specialised: warp 0 = TMA producer (one lane), warp 1 = MMA issuer (one
// lane), warp 2 = TMEM allocator, remaining warps = TMEM->register epilogue / softmax.  The GEMMs
// run on CTA pairs (cluster of 2, tcgen05 cta_group::2, UMMA 256 x BN x 16).
// Operands are staged by TMA into 128B-swizzled shared memory; accumulators live in TMEM.
#include "engine.h"
#include "ptx.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace glom {

constexpr int BM = 128;            // UMMA M (rows of the state per tile)
constexpr int BK = 64;             // bf16 elements per 128-byte swizzle row
constexpr uint32_t A_STAGE_BYTES = BM * BK * 2;   // 16 KB

// =====================================================================================
// K1 / K2: persistent grouped GEMM on CTA pairs (cta_group::2), fused epilogues
//   cluster of 2 CTAs = one 256 x BN output tile; CTA r owns rows [128 r, 128 r + 128) of it,
//   loads its 128 rows of A and its half (BN/2 rows) of B; the leader CTA issues UMMA 256xBNx16.
//   Epilogue warps read their 32-row TMEM quadrant row-per-thread, then transpose each 32x32 chunk
//   through a private shared-memory patch so that every global load/store instruction covers whole
//   cache lines (the reference's 4-way combine / residual write, glom_pytorch.py:141-142).
// =====================================================================================
constexpr int GEMM_CTRL_WARPS = 4;

// in-kernel clock samples (see clock_sample_begin): [kind][cycles, ns], kinds = ProfKind
// + wait-cycle counters of block 0's control / epilogue warps: [2] MMA lane waiting for operands, [3] for a free accumulator
// stage, [4] TMA lane waiting for a free ring slot, [5] epilogue warp 0 waiting for an accumulator, [6] its busy cycles
__device__ unsigned long long g_kernel_clk[PROF_KINDS][8];


struct GemmParams {
  int rows, d, L, n, G;
  int num_m, num_n, num_tiles;       // num_m counts 256-row pair tiles
  int m128;                          // 128-row blocks of the (padded) hidden buffer H
  int z0;                            // first MLP group (K1) / level (K2) of this launch, see level batching below
  int n_half;                        // K2: number of half-cost (top-level) tiles in this launch
  const float* bias;
  // K1
  __nv_bfloat16* h_out;
  // K2
  const float* s32_in;
  int s_bcast;                       // s32_in = init_levels broadcast (see K2Chunk)
  const __nv_bfloat16* c_in;
  const float* pos;
  float* s32_out;
  __nv_bfloat16* sb_out;
  __nv_bfloat16* sp_out;
  float* nsq_out;
  int nparts;
  // tokeniser (MODE 2)
  float* tok_out;
  int tok_kb;      // K blocks of 64 of the zero-padded patch dimension
};

template <int MODE, int BN>
struct GemmCfg {
  // column parts of a tile = epilogue warp groups: K1 (GELU-heavy) uses 4 parts when the tile allows
  static constexpr int PARTS = (BN == 256) ? 4 : 2;
  static constexpr int PART_COLS = BN / PARTS;                      // 64 / 64 / 32
  static constexpr int EPI_WARPS = 4 * PARTS;
  static constexpr int THREADS = 32 * (GEMM_CTRL_WARPS + EPI_WARPS);
  static constexpr uint32_t B_STAGE_BYTES = (BN / 2) * BK * 2;      // this CTA's half of the B tile
  static constexpr uint32_t STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = (BN == 256) ? 5 : 8;   // 32 KB stages + patches must fit 227 KB; for K1 five measured
                                                        // better than four or six (the sixth would fit)
  static constexpr uint32_t TMEM_COLS = 2 * BN;                     // two accumulator stages
  static constexpr uint32_t PATCH_BYTES = (MODE == 0) ? 2048 : 4096; // per-warp 32x32 transpose patch (bf16 | f32)
  static_assert(MODE >= 0 && MODE <= 2, "0 = GEMM1+GELU, 1 = GEMM2+combine, 2 = tokeniser");
  // K1: one private bias slice (PART_COLS floats) per epilogue warp; K2 / tokeniser keep their 8 bias values per lane in registers
  static constexpr uint32_t BIAS_BYTES = (MODE == 0) ? EPI_WARPS * PART_COLS * 4 : 0;
  static constexpr size_t SMEM_BYTES = 1024 /*align slack*/ + (size_t)STAGES * STAGE_BYTES +
                                       (size_t)EPI_WARPS * PATCH_BYTES + BIAS_BYTES + 256;
};

struct TileInfo {
  int z;        // K1: group g ; K2: level l
  int m_blk, n_blk;
  int num_kb;   // K blocks of 64
};

template <int MODE>
__device__ __forceinline__ TileInfo decode_tile(const GemmParams& p, int tile) {
  TileInfo t;
  t.n_blk = tile % p.num_n;
  const int r = tile / p.num_n;
  t.m_blk = r % p.num_m;
  t.z = p.z0 + r / p.num_m;
  if (MODE == 0) t.num_kb = p.d / BK;
  else if (MODE == 1) t.num_kb = ((t.z == p.L - 1) ? 4 * p.d : 8 * p.d) / BK;   // top level: no top-down half (:137)
  else t.num_kb = p.tok_kb;
  return t;
}

// Round-robin tile walk of the uniform-cost kernels (K1, tokeniser) for the epilogue warps: the same sequence as
// sched_tile / decode_tile, advanced by mixed-radix addition instead of two integer divisions per tile and thread.
struct RRIter {
  int tile, n_blk, m_blk, z, dn, dm, dz, C;
  __device__ __forceinline__ void init(const GemmParams& p, int c, int C_) {
    C = C_; tile = c;
    n_blk = c % p.num_n; int r = c / p.num_n; m_blk = r % p.num_m; z = r / p.num_m;      // z: position in the group walk
    dn = C_ % p.num_n; r = C_ / p.num_n; dm = r % p.num_m; dz = r / p.num_m;
  }
  __device__ __forceinline__ void next(const GemmParams& p) {
    tile += C;
    n_blk += dn; int carry = n_blk >= p.num_n ? 1 : 0; n_blk -= carry ? p.num_n : 0;
    m_blk += dm + carry; carry = m_blk >= p.num_m ? 1 : 0; m_blk -= carry ? p.num_m : 0;
    z += dz + carry;
  }
};

// Static tile schedule of cluster `c` (of `C`): the it-th tile it processes, or -1 when done.
//   K1 / tokeniser: uniform tiles, plain round-robin.
//   K2: the top level's tiles cost half (K = 4d instead of 8d, :137).  Full-cost tiles are dealt round-robin
//   first; the half-cost ones then go to the clusters that received one full tile fewer (up to two each, which
//   levels them with the others) and only after that round-robin over everybody.  Closed form, so every warp
//   role of both CTAs walks the same list without communication.
template <int MODE>
__device__ __forceinline__ int sched_tile(const GemmParams& p, int c, int C, int it) {
  if (MODE != 1) { const int t = c + it * C; return t < p.num_tiles ? t : -1; }
  const int S = p.n_half;                     // half-cost tiles (top level, last in the launch), ids [B, B + S)
  const int B = p.num_tiles - S;              // full-cost tiles, ids [0, B)
  const int heavy = B % C;                    // clusters [0, heavy) hold one more full tile than the rest
  const int nb = (B - c + C - 1) / C;         // full tiles of this cluster (B - c may be <= 0)
  const int nbig = nb > 0 ? nb : 0;
  if (it < nbig) return c + it * C;
  int k = it - nbig;                          // k-th half-cost tile of this cluster
  const int light = C - heavy;
  const int first = (2 * light < S) ? 2 * light : S;     // half tiles dealt to the light clusters first
  if (c >= heavy) {
    if (k < 2) { const int j = k * light + (c - heavy); if (j < first) return B + j; }
    k -= 2;
    if (k < 0) return -1;
  }
  const int j = first + k * C + c;            // the rest: round-robin over all clusters
  return j < S ? B + j : -1;
}

// Sum of squares of a 32-column chunk row, in the canonical order shared with prep_state_kernel:
// 8 lanes hold 4 consecutive columns each (sequential fmaf), then an xor tree over the 8 lanes.
__device__ __forceinline__ float row_chunk_sumsq(float a, float b, float c, float d) {
  float q = a * a;
  q = fmaf(b, b, q);
  q = fmaf(c, c, q);
  q = fmaf(d, d, q);
  q += __shfl_xor_sync(0xffffffffu, q, 1);
  q += __shfl_xor_sync(0xffffffffu, q, 2);
  q += __shfl_xor_sync(0xffffffffu, q, 4);
  return q;
}

// ---- K1 epilogue chunk: 32 rows x 32 columns.  Row-per-thread bias + exact-erf GELU + bf16 pack, transpose
// through the warp's 2 KB patch (16-byte chunk c of row r stored at chunk c ^ ((r >> 1) & 3)), then 64-byte
// row segments out (8 rows x 64 B per store instruction).
template <bool FULL>
__device__ __forceinline__ void k1_chunk(const uint32_t (&v)[32], const float* bias, uint8_t* patch,
                                         __nv_bfloat16* hdst /* &H[row0][col] */, size_t pitch, int lane, int rows_left) {
  uint32_t pk[16];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    // bias slice read per use (broadcast LDS.128): 32 fewer live registers, so the polynomial's constant pairs stay in
    // registers instead of being re-materialised for every pair
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * i);
    pk[2 * i] = gelu_pair_bf16(__uint_as_float(v[4 * i + 0]), __uint_as_float(v[4 * i + 1]), b.x, b.y);
    pk[2 * i + 1] = gelu_pair_bf16(__uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]), b.z, b.w);
  }
#pragma unroll
  for (int c = 0; c < 4; ++c)
    *reinterpret_cast<uint4*>(patch + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) =
        make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
  __syncwarp();
  const int c = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i * 8 + (lane >> 2);
    const uint4 val = *reinterpret_cast<const uint4*>(patch + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
    // streaming (evict-first) stores: H (369 MB per step) never fits L2, and letting it through the normal policy
    // evicts the state shadows and weights the GEMMs and the consensus kernel re-read (measured: K1 -4 %)
    if (FULL || r < rows_left) __stcs(reinterpret_cast<uint4*>(hdst + (size_t)r * pitch + c * 8), val);
  }
  __syncwarp();
}

// ---- K2 epilogue chunk: the 4-way combine (glom_pytorch.py:141-142) on a 32 x 32 accumulator chunk.
// The accumulators go through the warp's 4 KB patch (f32, 128-byte rows, chunk c of row r at c ^ (r & 7)) so
// that each lane then owns 4 consecutive columns of 8 rows and every global access covers whole 128-byte lines.
struct K2Chunk {
  int l, L, d, n, row0;
  int prow0;            // row0 % n: patch index of the band's first row (position table row), computed once per tile
  int s_bcast;          // 1: s32_in is init_levels (L, d), the same for every row (first step of a call without carried state)
  const float* s32_in; const __nv_bfloat16* c_in; const float* pos;
  float* s32_out; __nv_bfloat16* sb_out; __nv_bfloat16* sp_out;
};
template <bool FULL>
__device__ __forceinline__ void k2_chunk(const uint32_t (&v)[32], const float4 b4, uint8_t* patch, const K2Chunk& k,
                                         int col, int lane, int rows_left, float (&rowsq)[8]) {
#pragma unroll
  for (int c = 0; c < 8; ++c)
    *reinterpret_cast<uint4*>(patch + lane * 128 + ((c ^ (lane & 7)) << 4)) =
        make_uint4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
  __syncwarp();
  const int c = lane & 7, rsub = lane >> 3;
  const bool top = (k.l == k.L - 1);                  // 3 contributions on the top level, 4 elsewhere (:128-129)
  const bool has_td = (k.l >= 1);
  const size_t ld = (size_t)k.L * k.d;
  const size_t base = ((size_t)k.row0 * k.L + k.l) * k.d + col + c * 4;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    // global loads of four rows first (independent, all in flight), then combine + store
    float4 sv[4], pp[4];
    uint2 cw[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = (h * 4 + j) * 4 + rsub;
      sv[j] = make_float4(0.f, 0.f, 0.f, 0.f); pp[j] = sv[j]; cw[j] = make_uint2(0u, 0u);
      if (FULL || r < rows_left) {
        sv[j] = k.s_bcast ? __ldg(reinterpret_cast<const float4*>(k.s32_in + (size_t)k.l * k.d + col + c * 4))
                          : __ldcs(reinterpret_cast<const float4*>(k.s32_in + base + (size_t)r * ld));
        cw[j] = __ldcs(reinterpret_cast<const uint2*>(k.c_in + base + (size_t)r * ld));
        if (has_td) {
          int pr = k.prow0 + r;                       // (row0 + r) % n without a division per row (r < 32)
          if (k.n >= 32) { if (pr >= k.n) pr -= k.n; } else pr %= k.n;
          pp[j] = __ldg(reinterpret_cast<const float4*>(k.pos + (size_t)pr * k.d + col + c * 4));
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int i = h * 4 + j;
      const int r = i * 4 + rsub;
      const float4 acc = *reinterpret_cast<const float4*>(patch + r * 128 + ((c ^ (r & 7)) << 4));
      float o0 = (sv[j].x + (acc.x + b4.x)) + __uint_as_float(cw[j].x << 16);               // (:141)
      float o1 = (sv[j].y + (acc.y + b4.y)) + __uint_as_float(cw[j].x & 0xFFFF0000u);
      float o2 = (sv[j].z + (acc.z + b4.z)) + __uint_as_float(cw[j].y << 16);
      float o3 = (sv[j].w + (acc.w + b4.w)) + __uint_as_float(cw[j].y & 0xFFFF0000u);
      if (top) { o0 = o0 / 3.0f; o1 = o1 / 3.0f; o2 = o2 / 3.0f; o3 = o3 / 3.0f; }          // (:142) IEEE division
      else { o0 *= 0.25f; o1 *= 0.25f; o2 *= 0.25f; o3 *= 0.25f; }                          // x/4 == x*0.25 exactly
      if (FULL || r < rows_left) {
        const size_t o = base + (size_t)r * ld;
        __stcs(reinterpret_cast<float4*>(k.s32_out + o), make_float4(o0, o1, o2, o3));
        *reinterpret_cast<uint2*>(k.sb_out + o) = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
        if (has_td)
          *reinterpret_cast<uint2*>(k.sp_out + ((size_t)(k.row0 + r) * (k.L - 1) + (k.l - 1)) * k.d + col + c * 4) =
              make_uint2(pack_bf16x2(o0 + pp[j].x, o1 + pp[j].y), pack_bf16x2(o2 + pp[j].z, o3 + pp[j].w));
      } else {
        o0 = o1 = o2 = o3 = 0.f;
      }
      rowsq[i] += row_chunk_sumsq(o0, o1, o2, o3);
    }
  }
  __syncwarp();
}

// ---- tokeniser epilogue chunk (image_to_tokens Linear bias, glom_pytorch.py:96): f32 out, whole 128-byte lines.
__device__ __forceinline__ void tok_chunk(const uint32_t (&v)[32], const float4 b4, uint8_t* patch, float* dst,
                                          size_t pitch, int lane, int rows_left) {
#pragma unroll
  for (int c = 0; c < 8; ++c)
    *reinterpret_cast<uint4*>(patch + lane * 128 + ((c ^ (lane & 7)) << 4)) =
        make_uint4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
  __syncwarp();
  const int c = lane & 7, rsub = lane >> 3;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + rsub;
    const float4 a = *reinterpret_cast<const float4*>(patch + r * 128 + ((c ^ (r & 7)) << 4));
    if (r < rows_left)
      *reinterpret_cast<float4*>(dst + (size_t)r * pitch + c * 4) = make_float4(a.x + b4.x, a.y + b4.y, a.z + b4.z, a.w + b4.w);
  }
  __syncwarp();
}

template <int MODE, int BN, bool CNT>
__global__ void __launch_bounds__(GemmCfg<MODE, BN>::THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap map_a0,   // K1: tokens Xb (rows, d)        K2: H (rows, G*4d)
            const __grid_constant__ CUtensorMap map_a1,   // K1: state shadow Sb (rows, L*d)
            const __grid_constant__ CUtensorMap map_a2,   // K1: Sb[:,1:]+pos shadow Sp (rows, (L-1)*d)
            const __grid_constant__ CUtensorMap map_b,    // K1: W1p (G*4d, d)              K2: W2p (L*d, 8d)
            const GemmParams p) {
  using Cfg = GemmCfg<MODE, BN>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int EPI_THREADS = Cfg::EPI_WARPS * 32;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic on the __shared__ array (keeps the shared address space
  // visible to the compiler: LDS/STS instead of generic LD/ST for every patch / bias / P access)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* patches = smem + (size_t)STAGES * Cfg::STAGE_BYTES;
  float* bias_s = reinterpret_cast<float*>(patches + (size_t)Cfg::EPI_WARPS * Cfg::PATCH_BYTES);    // K1: [EPI_WARPS][PART_COLS]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(bias_s) + Cfg::BIAS_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  // Warp roles: epilogue warps come FIRST (ids 0 .. EPI_WARPS-1), the single-lane control warps last: the SM's
  // warp arbiter favours higher warp ids, and the TMA / MMA issuers must never wait behind epilogue math.
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int W_TMA = Cfg::EPI_WARPS, W_MMA = Cfg::EPI_WARPS + 1, W_ALLOC = Cfg::EPI_WARPS + 2;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;

  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_b);
    if (MODE == 0) { tma_prefetch_desc(&map_a1); tma_prefetch_desc(&map_a2); }
  }
  if (warp == W_MMA && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * Cfg::EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == W_ALLOC) tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();          // peer barriers initialised + both TMEM allocations done before any cross-CTA traffic
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();     // the next kernel may start its own set-up on SMs we vacate
  pdl_wait();                  // ... and we touch global memory only after the previous kernel has finished
  const bool clk_thread = blockIdx.x == 0 && warp == W_ALLOC && lane == 0;
  ClockSample clk_s{};
  if (clk_thread) clk_s = clock_sample_begin();
  const bool cnt_cta = CNT && blockIdx.x == 0;          // wait-cycle counters (diagnostic instantiation): block 0 only
  unsigned long long* const cnt = g_kernel_clk[MODE == 0 ? PROF_GEMM1 : MODE == 1 ? PROF_GEMM2 : PROF_TOKENIZE];
  unsigned long long w0 = 0, w1 = 0;
#define GLOM_CNT_WAIT(acc, stmt) do { if (cnt_cta) { const long long t_ = clock64(); stmt; acc += (unsigned long long)(clock64() - t_); } else { stmt; } } while (0)

  if (warp == W_TMA) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    // warp-converged: all lanes walk the schedule and poll the barriers, the elected lane issues (see elect_one)
    const uint32_t elected = elect_one();
    int stage = 0; uint32_t phase = 0;
    const uint32_t smem0 = smem_u32(smem);
    const uint32_t bar0 = mapa_shared(smem_u32(&full_bar[0]), 0);
    const uint64_t pol_first = l2_policy_evict_first();
    const int kbg_n = 4 * p.d / BK;
    const int blk_skip = (p.m128 - 1) * kbg_n;
    for (int it = 0, tile; (tile = sched_tile<MODE>(p, cluster_id, num_clusters, it)) >= 0; ++it) {
      const TileInfo t = decode_tile<MODE>(p, tile);
      const CUtensorMap* amap;
      int a_col, b_row;
      if (MODE == 0) {
        const int l = t.z >> 1;
        if (t.z == 0) { amap = &map_a0; a_col = 0; }                        // bottom-up level 0 reads the tokens (:132)
        else if (t.z & 1) { amap = &map_a2; a_col = l * p.d; }              // top-down l reads S[l+1]+pos (:136)
        else { amap = &map_a1; a_col = (l - 1) * p.d; }                     // bottom-up l reads S[l-1]   (:134)
        b_row = t.z * 4 * p.d + t.n_blk * BN;
      } else if (MODE == 1) {
        amap = &map_a0; a_col = 0;             // H is stored as contiguous 16 KB (128 x 64) blocks, see below
        b_row = t.z * p.d + t.n_blk * BN;
      } else {
        amap = &map_a0; a_col = 0;               // patches (rows, Kp) x Wtok (d, Kp)
        b_row = t.n_blk * BN;
      }
      const int a_row = t.m_blk * 256 + (int)cta_rank * BM;
      b_row += (int)cta_rank * (BN / 2);
      // K2: block (group g, 128-row block, 64-wide k block); [H_bu,l | H_td,l] are groups 2l and 2l+1, so k block kb
      // of the concatenation is block blk0 + kb of group 2l and, from kb = kbg_n on, of the group behind it
      const int blk0 = (2 * t.z * p.m128 + (a_row >> 7)) * kbg_n;
      for (int kb = 0; kb < t.num_kb; ++kb) {
        GLOM_CNT_WAIT(w0, mbar_wait(&empty_bar[stage], phase ^ 1));
        if (elected) {
          const uint32_t sa = smem0 + (uint32_t)stage * Cfg::STAGE_BYTES;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);   // both CTAs' bytes land here
          const uint32_t bar = bar0 + 8u * (uint32_t)stage;
          if (MODE == 1) {
            const int blk = blk0 + kb + (kb >= kbg_n ? blk_skip : 0);
            // H streams through once per pair of column tiles: evict-first keeps it from displacing weights / state
            // (measured best on every load).  An L2 prefetch cursor running ahead of these loads measured slower
            // (profiles/r2_k2_prefetch_ab.txt).
            tma_load_2d_2sm_sa_hint(sa, amap, bar, 0, blk * BM, pol_first);
          } else {
            tma_load_2d_2sm_sa(sa, amap, bar, a_col + kb * BK, a_row);
          }
          tma_load_2d_2sm_sa(sa + A_STAGE_BYTES, &map_b, bar, kb * BK, b_row);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    if (cnt_cta && elected) atomicAdd(&cnt[4], w0);
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN, 0, 0);
      const uint32_t elected = elect_one();
      // descriptors of stage 0; stage s / 16-element k step k: + s * (STAGE_BYTES >> 4) + 2 k (start address field, >> 4)
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(smem), 16, 1024);
      const uint64_t b_desc0 = umma_desc_sw128(smem_u32(smem) + A_STAGE_BYTES, 16, 1024);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      for (int it = 0, tile; (tile = sched_tile<MODE>(p, cluster_id, num_clusters, it)) >= 0; ++it) {
        const TileInfo t = decode_tile<MODE>(p, tile);
        GLOM_CNT_WAIT(w1, mbar_wait(&tempty_bar[as], aphase ^ 1));      // both CTAs' epilogues drained this accumulator stage
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < t.num_kb; ++kb) {
          GLOM_CNT_WAIT(w0, mbar_wait(&full_bar[stage], phase));
          tc_fence_after_sync();
          if (elected) {
            const uint64_t ad = a_desc0 + (uint64_t)(stage * (int)(Cfg::STAGE_BYTES >> 4));
            const uint64_t bd = b_desc0 + (uint64_t)(stage * (int)(Cfg::STAGE_BYTES >> 4));
            umma_bf16_2sm(d_tmem, ad, bd, idesc, kb != 0 ? 1u : 0u);
#pragma unroll
            for (int k = 1; k < BK / 16; ++k) umma_bf16_2sm(d_tmem, ad + 2 * k, bd + 2 * k, idesc, 1u);
            umma_commit_2sm(&empty_bar[stage], 3);     // frees the slot in both CTAs
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (elected) umma_commit_2sm(&tfull_bar[as], 3);          // accumulator complete -> both epilogues
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
      if (cnt_cta && elected) { atomicAdd(&cnt[2], w0); atomicAdd(&cnt[3], w1); }
    }
  } else if (warp < Cfg::EPI_WARPS) {
    // ------------------------------------------------------------------ epilogue (4 * PARTS warps)
    const int ew = warp;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int part = ew >> 2;                  // column part of the tile
    constexpr int PART_COLS = Cfg::PART_COLS;
    uint8_t* patch = patches + (size_t)ew * Cfg::PATCH_BYTES;
    int as = 0; uint32_t aphase = 0;
    // Bias.  K1: every warp owns a slice of PART_COLS floats in shared memory (read as broadcast LDS.128 by the GELU); the
    // next tile's slice is fetched into registers one tile ahead (its L2 latency overlaps this tile's epilogue) and
    // swapped in behind a warp barrier -- no CTA-wide barrier, the 16 warps are free to drift apart.  K2 / tokeniser: the
    // 2 x 4 values a lane needs are loaded into registers before the accumulator wait.
    float* bias_w = bias_s + ew * PART_COLS;
    RRIter rr{};
    if (MODE != 1) rr.init(p, cluster_id, num_clusters);
    if (MODE == 0 && rr.tile < p.num_tiles) {
      static_assert(MODE != 0 || PART_COLS == 64, "K1: one float2 of bias per lane");
      *reinterpret_cast<float2*>(bias_w + 2 * lane) =
          __ldg(reinterpret_cast<const float2*>(p.bias + (size_t)(p.z0 + rr.z) * 4 * p.d + rr.n_blk * BN + part * PART_COLS) + lane);
      __syncwarp();
    }
    for (int it = 0;; ++it) {
      TileInfo t;
      bool has_next = false;
      float2 next_bias = make_float2(0.f, 0.f);
      if (MODE == 1) {
        const int tile = sched_tile<MODE>(p, cluster_id, num_clusters, it);
        if (tile < 0) break;
        t = decode_tile<MODE>(p, tile);
      } else {
        if (rr.tile >= p.num_tiles) break;
        t.z = p.z0 + rr.z; t.m_blk = rr.m_blk; t.n_blk = rr.n_blk; t.num_kb = 0;
        rr.next(p);                                  // rr now describes the NEXT tile
        has_next = rr.tile < p.num_tiles;
        if (MODE == 0 && has_next)
          next_bias = __ldg(reinterpret_cast<const float2*>(p.bias + (size_t)(p.z0 + rr.z) * 4 * p.d + rr.n_blk * BN + part * PART_COLS) + lane);
      }
      float4 b4r[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
      if (MODE != 0) {
        const float* bsrc = p.bias + (MODE == 1 ? (size_t)t.z * p.d : (size_t)0) + t.n_blk * BN + part * PART_COLS + (lane & 7) * 4;
        b4r[0] = __ldg(reinterpret_cast<const float4*>(bsrc));
        if (PART_COLS > 32) b4r[1] = __ldg(reinterpret_cast<const float4*>(bsrc + 32));
      }
      const int row0 = t.m_blk * 256 + (int)cta_rank * BM + quad * 32;   // first row of this warp's 32-row band
      const int rows_left = p.rows - row0;                                // >= 32: whole band valid (warp-uniform)
      if (MODE == 1 && lane < rows_left) {
        // The combine reads this warp's 32 x 64 patch of the fp32 state (streamed to HBM by the previous step) and of C:
        // pull those lines into L2 now, a whole main loop (~25 us) before the accumulator is complete, so the epilogue's
        // dependent global loads hit L2 instead of paying the HBM latency four times per tile
        const size_t o = ((size_t)(row0 + lane) * p.L + t.z) * p.d + t.n_blk * BN + part * PART_COLS;
        if (!p.s_bcast) {
          prefetch_l2(p.s32_in + o);
          if (PART_COLS > 32) prefetch_l2(p.s32_in + o + 32);
        }
        prefetch_l2(p.c_in + o);
      }
      GLOM_CNT_WAIT(w0, mbar_wait(&tfull_bar[as], aphase));
      tc_fence_after_sync();
      const long long busy_t0 = cnt_cta ? clock64() : 0;
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN + part * PART_COLS);
      const float* bias = bias_w;
      if (MODE == 0) {
        // H block (group, 128-row block, k block = this warp's 64-column part): 16 KB contiguous, row pitch 64
        const int hblk = (t.z * p.m128 + (t.m_blk * 2 + (int)cta_rank)) * (4 * p.d / BK) + t.n_blk * (BN / BK) + part;
        __nv_bfloat16* hrow = p.h_out + ((size_t)hblk * BM + quad * 32) * BK;
#pragma unroll 1
        for (int c0 = 0; c0 < PART_COLS; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_addr + c0, v);
          tmem_ld_wait();
          if (rows_left >= 32) k1_chunk<true>(v, bias + c0, patch, hrow + c0, (size_t)BK, lane, 32);
          else k1_chunk<false>(v, bias + c0, patch, hrow + c0, (size_t)BK, lane, rows_left);
        }
      } else if (MODE == 2) {
        float* trow = p.tok_out + (size_t)row0 * p.d + t.n_blk * BN + part * PART_COLS;
#pragma unroll 1
        for (int c0 = 0; c0 < PART_COLS; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_addr + c0, v);
          tmem_ld_wait();
          tok_chunk(v, c0 ? b4r[1] : b4r[0], patch, trow + c0, (size_t)p.d, lane, rows_left);
        }
      } else {
        K2Chunk kc;
        kc.l = t.z; kc.L = p.L; kc.d = p.d; kc.n = p.n; kc.row0 = row0; kc.prow0 = row0 % p.n; kc.s_bcast = p.s_bcast;
        kc.s32_in = p.s32_in; kc.c_in = p.c_in; kc.pos = p.pos;
        kc.s32_out = p.s32_out; kc.sb_out = p.sb_out; kc.sp_out = p.sp_out;
        float rowsq[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) rowsq[i] = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < PART_COLS; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_addr + c0, v);
          tmem_ld_wait();
          const int col = t.n_blk * BN + part * PART_COLS + c0;
          const float4 b4 = c0 ? b4r[1] : b4r[0];
          if (rows_left >= 32) k2_chunk<true>(v, b4, patch, kc, col, lane, 32, rowsq);
          else k2_chunk<false>(v, b4, patch, kc, col, lane, rows_left, rowsq);
        }
        if ((lane & 7) == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = i * 4 + (lane >> 3);
            if (r < rows_left)
              p.nsq_out[((size_t)(row0 + r) * p.L + t.z) * p.nparts + t.n_blk * Cfg::PARTS + part] = rowsq[i];
          }
        }
      }
      // release this accumulator stage to the leader's MMA issuer: one arrival per epilogue warp of either CTA
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty_bar[as]), 0));
      if (++as == 2) { as = 0; aphase ^= 1; }
      if (cnt_cta) w1 += (unsigned long long)(clock64() - busy_t0);
      if (MODE == 0 && has_next) {          // (the __syncwarp above: every lane is done with this tile's slice)
        *reinterpret_cast<float2*>(bias_w + 2 * lane) = next_bias;
        __syncwarp();
      }
    }
    if (cnt_cta && warp == 0 && lane == 0) { atomicAdd(&cnt[5], w0); atomicAdd(&cnt[6], w1); }
  }
#undef GLOM_CNT_WAIT

  tc_fence_before_sync();
  __syncthreads();
  if (clk_thread) clock_sample_end(clk_s, g_kernel_clk[MODE == 0 ? PROF_GEMM1 : MODE == 1 ? PROF_GEMM2 : PROF_TOKENIZE]);
  cluster_sync_all();          // no CTA exits (or frees TMEM) while its pair can still touch it
  if (warp == W_ALLOC) {
    tc_fence_after_sync();
    tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
  }
}

// =====================================================================================
// K3: consensus attention on CTA pairs.  Persistent clusters of two CTAs (one per SM); a work item is
// (pair of 128-query tiles, level l, image b), CTA r of the pair owning query tile 2u + r.
//   phase 1: S = Q K^T per key block (<= 256 keys) over d as one 256 x w cta_group::2 MMA: each CTA feeds its
//            own 128 query rows and HALF of the key block and receives its rows of S (fp32) in a 256-column TMEM
//            buffer.  The softmax warps turn them into unnormalised bf16 probabilities P in shared memory
//            (UMMA A-operand layout).
//   phase 2: O = P V in 256-wide slices of d (V read MN-major straight from the state shadow, each CTA
//            feeding half of the slice's columns); each slice is scaled by 1/rowsum and written as bf16 C while
//            the next one is being multiplied.
// Every byte of the state shadow is therefore fetched once per pair and phase instead of once per query tile,
// which halves the L2 -> shared-memory traffic.  The TMA / MMA threads keep their ring and buffer counters
// running across items: the two TMEM buffers alternate S, O0, O1, S', O0', ... so Q K^T of item i+1 is issued
// as soon as slice 0 of item i has been read out and overlaps the rest of its output phase.
// Softmax stabiliser: every key is unit-normalised, so |logit_ij| <= |S_i| d^-1/2 (Cauchy-Schwarz); that bound
// replaces the row maximum (softmax is shift-invariant) and S is read from TMEM once instead of twice.  The
// diagonal is never masked (its logit is -5e-4 or, with attend_self, ~ the bound itself), so the row sum cannot
// underflow while the bound stays below 2^BOUND_MAX; rows beyond that take the exact-maximum pass.
// With n in (240, 256] a CTA's query tile IS its half of the single key block and is not loaded separately.
// Measured (profiles/README.md): the softmax / output warps are bound by TMEM read-out (64 B/clk/SM), the XU pipe
// (ex2 + fp32->bf16 packing) and the burst of C stores, the Q K^T phase by the first touch of the shadow in HBM.
// =====================================================================================
constexpr int ATTN_SM_WARPS = 16;                 // softmax / output warps: 4 TMEM quadrants x 4 column parts
constexpr int ATTN_THREADS = 640;                 // 16 softmax warps + TMA + MMA + TMEM-alloc + 1 idle
constexpr int ATTN_RED_FLOATS = 1536;             // block maxima [2][4][128] + row sums [4][128]
constexpr int ATTN_SM_THREADS = ATTN_SM_WARPS * 32;
constexpr int ATTN_MAX_KB = 4;
constexpr uint32_t ATTN_SLOT_BYTES = 32768;       // ring slot: Q + K-half chunk(s), or 2 key chunks x 2 column boxes of V
constexpr uint32_t ATTN_PATCH_BYTES = ATTN_SM_WARPS * 2048;
constexpr float ATTN_BOUND_MAX = 96.f;            // log2 units
constexpr int ATTN_SINGLE_PASS_MAX = 576;         // columns whose probabilities (128 queries x all keys) fit in shared memory
constexpr int ATTN_PASS_KEYS = 512;               // keys per pass beyond that (two key blocks of 256)

struct AttnParams {
  int n, L, d;
  int attend_self, mask_side, mask_d2_max;
  int n_pad16, n_pad64, nkb, nchunk;   // key padding, key blocks (<=256), 64-key chunks
  int khalf_rows;                      // rows fetched per K box: half of the (widest) key block
  int num_stages;
  int q_in_k;                          // 1: the CTA's query tile is its half of the single key block
  int lean;                            // 1: no transpose patches (P of many columns leaves no room): row-per-thread stores
  int npairs, num_items;               // query-tile pairs per (l, b); npairs * L * B
  int nparts;
  const float* nsq;                    // (rows, L, nparts) squared-norm partials of the state
  __nv_bfloat16* c_out;                // (rows, L, d)
  float scale;                         // d^-1/2 (:60)
  // Key passes (n > 576 columns: the probabilities of a 128-query tile against ALL keys no longer fit in shared memory).
  // One launch handles the keys [key0, key0 + nk) (the n_pad* / nkb / nchunk fields above describe THIS range); the
  // unnormalised output and the per-row (stabiliser, row sum) are carried in fp32 scratch from pass to pass and the last
  // pass normalises and writes C.  A single pass (key0 = 0, nk = n, first = last = 1) is the plain kernel.
  int key0, nk, pass_first, pass_last;
  float* o_acc;                        // (rows, L, d) fp32
  float* ml_acc;                       // (rows, L, 2) fp32: stabiliser (log2 units), row sum
};

template <bool CNT>
__global__ void __launch_bounds__(ATTN_THREADS, 1)
attn_kernel(const __grid_constant__ CUtensorMap map_q,    // (L*d, n, B) box (64, 128, 1)
            const __grid_constant__ CUtensorMap map_k,    // box (64, khalf_rows, 1)
            const __grid_constant__ CUtensorMap map_v,    // box (64, 64, 1)
            const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic on the __shared__ array (keeps the shared address space
  // visible to the compiler: LDS/STS instead of generic LD/ST for every patch / bias / P access)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* p_smem = smem;                                                  // nchunk x [128 x 64] bf16, SW128
  uint8_t* stages = p_smem + (size_t)p.nchunk * A_STAGE_BYTES;
  uint8_t* patches = stages + (size_t)p.num_stages * ATTN_SLOT_BYTES;      // 16 x 2 KB transpose patches
  float* rs = reinterpret_cast<float*>(patches + (p.lean ? 0u : ATTN_PATCH_BYTES));   // [2][n_pad16] per-key scales, by item parity
  float* bnd = rs + 2 * p.n_pad16;                                         // [2][n_pad16] per-row logit bounds
  uint32_t* key_hw = reinterpret_cast<uint32_t*>(bnd + 2 * p.n_pad16);     // [n_pad16] (grid row << 16) | grid column
  float* red = reinterpret_cast<float*>(key_hw + p.n_pad16);               // block maxima (2 parities), row sums
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(red + ATTN_RED_FLOATS); // leader's: both CTAs' TMA bytes
  uint64_t* empty_bar = full_bar + p.num_stages;                           // own: slot consumed by the pair MMA
  uint64_t* afull_bar = empty_bar + p.num_stages;      // own [2]: S block / O slice complete in TMEM buffer
  uint64_t* aempty_bar = afull_bar + 2;                // leader's [2]: buffer drained by the softmax warps of both CTAs
  uint64_t* pready_bar = aempty_bar + 2;               // leader's: P of the item complete in both CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pready_bar + 1);

  // softmax / output warps are warps 0-15, control warps 16-18 (higher ids win the warp arbiter)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int W_TMA = ATTN_SM_WARPS, W_MMA = ATTN_SM_WARPS + 1, W_ALLOC = ATTN_SM_WARPS + 2;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int nsub = (p.d + 255) / 256;                  // O slices per item
  const int nvslot = (p.nchunk + 1) / 2;               // ring slots per O slice (two 64-key chunks each)
  const int cps = p.q_in_k ? 2 : 1;                    // d-chunks of Q K^T per ring slot
  const uint32_t kv_off = p.q_in_k ? 0u : A_STAGE_BYTES;
  const int pairs_per_img = p.npairs * p.L;

  if (warp == W_TMA && lane == 0) { tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_k); tma_prefetch_desc(&map_v); }
  if (warp == W_MMA && lane == 0) {
    for (int i = 0; i < p.num_stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 2 * ATTN_SM_WARPS); }
    mbar_init(pready_bar, 2 * ATTN_SM_WARPS);
    fence_barrier_init();
  }
  if (warp == W_ALLOC) tmem_alloc_2sm(tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();          // peer barriers initialised + both TMEM allocations done before any cross-CTA traffic
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();
  const bool clk_thread = blockIdx.x == 0 && warp == W_ALLOC && lane == 0;
  ClockSample clk_s{};
  if (clk_thread) clk_s = clock_sample_begin();
  // diagnostic instantiation (GLOM_B200_WAIT_COUNTERS=1): block 0's wait / busy cycles per role, in g_kernel_clk[PROF_ATTN]:
  // [2] MMA lane waiting for operands, [3] for a free TMEM buffer or for P, [4] TMA lane waiting for a free slot,
  // [5] softmax warp 0 waiting for S / O in TMEM, [6] its softmax work, [7] its output work
  const bool cnt_cta = CNT && blockIdx.x == 0;
  unsigned long long* const cnt = g_kernel_clk[PROF_ATTN];
  unsigned long long w0 = 0, w1 = 0, w2 = 0;
#define GLOM_CNT_WAIT(acc, stmt) do { if (cnt_cta) { const long long t_ = clock64(); stmt; acc += (unsigned long long)(clock64() - t_); } else { stmt; } } while (0)

  if (warp == W_TMA) {
    // ------------------------------------------------------------------ TMA producer (both CTAs), warp-converged
    // (all lanes walk the item list and poll the ring, the elected lane issues: see elect_one)
    const uint32_t elected = elect_one();
    int stage = 0; uint32_t phase = 0;
    const uint32_t stages0 = smem_u32(stages);
    const uint32_t bar0 = mapa_shared(smem_u32(&full_bar[0]), 0);
    const uint32_t qk_tx = kv_off + (uint32_t)p.khalf_rows * 128u;
    for (int it = cluster_id; it < p.num_items; it += num_clusters) {
      const int b = it / pairs_per_img, l = (it % pairs_per_img) / p.npairs;
      const int q0 = (2 * (it % p.npairs) + (int)cta_rank) * BM;
      for (int kb = 0; kb < p.nkb; ++kb) {
        const int w = min(256, p.n_pad16 - kb * 256);
        const int key0 = p.key0 + kb * 256 + (int)cta_rank * (w >> 1);        // this CTA's half of the key block
        for (int dc = 0; dc < p.d / BK; dc += cps) {
          const int nc = min(cps, p.d / BK - dc);
          GLOM_CNT_WAIT(w0, mbar_wait(&empty_bar[stage], phase ^ 1));
          if (elected) {
            const uint32_t s = stages0 + (uint32_t)stage * ATTN_SLOT_BYTES;
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2u * (uint32_t)nc * qk_tx);
            const uint32_t bar = bar0 + 8u * (uint32_t)stage;
            for (int c = 0; c < nc; ++c) {
              if (!p.q_in_k) tma_load_3d_2sm_sa(s, &map_q, bar, l * p.d + (dc + c) * BK, q0, b);
              tma_load_3d_2sm_sa(s + kv_off + c * 16384, &map_k, bar, l * p.d + (dc + c) * BK, key0, b);
            }
          }
          __syncwarp();
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
      }
      for (int sp = 0; sp < nsub; ++sp) {
        const int wdp = (min(256, p.d - sp * 256) + 127) & ~127;     // slice width as issued (128 or 256)
        const int nbox = wdp >> 7;                                   // 64-column boxes in this CTA's half
        for (int vs = 0; vs < nvslot; ++vs) {
          const int nkc = min(2, p.nchunk - 2 * vs);               // 64-key chunks in this slot
          GLOM_CNT_WAIT(w0, mbar_wait(&empty_bar[stage], phase ^ 1));
          if (elected) {
            const uint32_t s = stages0 + (uint32_t)stage * ATTN_SLOT_BYTES;
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2u * (uint32_t)(nkc * nbox) * 8192u);
            const uint32_t bar = bar0 + 8u * (uint32_t)stage;
            for (int kc = 0; kc < nkc; ++kc)
              for (int i = 0; i < nbox; ++i) {
                const int dcol = sp * 256 + (int)cta_rank * (wdp >> 1) + i * 64;   // this CTA's half of the slice
                tma_load_3d_2sm_sa(s + kc * 16384 + i * 8192, &map_v, bar, dcol < p.d ? l * p.d + dcol : p.L * p.d,
                                   p.key0 + (2 * vs + kc) * 64, b);                // past d: out of bounds -> zeros
              }
          }
          __syncwarp();
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
    if (cnt_cta && elected) atomicAdd(&cnt[4], w0);
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only), warp-converged
    if (leader) {
      const uint32_t elected = elect_one();
      const uint32_t stages0 = smem_u32(stages);
      // K-major operand descriptors (Q, K halves, P) and the MN-major one of V, all relative to shared-memory offset 0:
      // the start-address field (>> 4) of a concrete operand is added per use
      const uint64_t kdesc0 = umma_desc_sw128(0, 16, 1024);
      const uint64_t vdesc0 = umma_desc_sw128(0, 8192, 1024);
      const uint32_t p_lo = smem_u32(p_smem) >> 4;
      int stage = 0; uint32_t phase = 0;
      uint32_t job = 0, item_par = 0;
      for (int it = cluster_id; it < p.num_items; it += num_clusters, item_par ^= 1) {
        // phase 1: S_kb = Q K_kb^T
        for (int kb = 0; kb < p.nkb; ++kb, ++job) {
          const int w = min(256, p.n_pad16 - kb * 256);
          const uint32_t idesc = umma_idesc_bf16(256, w, 0, 0);
          const uint32_t buf = job & 1;
          GLOM_CNT_WAIT(w1, mbar_wait(&aempty_bar[buf], ((job >> 1) & 1) ^ 1));
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + buf * 256u;
          for (int dc = 0; dc < p.d / BK; dc += cps) {
            const int nc = min(cps, p.d / BK - dc);
            GLOM_CNT_WAIT(w0, mbar_wait(&full_bar[stage], phase));
            tc_fence_after_sync();
            if (elected) {
              const uint32_t s_lo = (stages0 + (uint32_t)stage * ATTN_SLOT_BYTES) >> 4;
              for (int c = 0; c < nc; ++c) {
                const uint64_t bd = kdesc0 + (uint64_t)(s_lo + ((kv_off + (uint32_t)c * 16384u) >> 4));
                const uint64_t ad = p.q_in_k ? bd : kdesc0 + (uint64_t)s_lo;
                umma_bf16_2sm(d_tmem, ad, bd, idesc, (dc | c) != 0 ? 1u : 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16_2sm(d_tmem, ad + 2 * k, bd + 2 * k, idesc, 1u);
              }
              umma_commit_2sm(&empty_bar[stage], 3);
            }
            __syncwarp();
            if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
          }
          if (elected) umma_commit_2sm(&afull_bar[buf], 3);
          __syncwarp();
        }
        // phase 2: O = P V   (A = P from smem, K-major; B = V slice, MN-major, 64 columns from each CTA)
        GLOM_CNT_WAIT(w1, mbar_wait_cluster(pready_bar, item_par));
        tc_fence_after_sync();
        for (int sp = 0; sp < nsub; ++sp, ++job) {
          const int wdp = (min(256, p.d - sp * 256) + 127) & ~127;
          const uint32_t idesc = umma_idesc_bf16(256, wdp, 0, 1);
          const uint32_t buf = job & 1;
          GLOM_CNT_WAIT(w1, mbar_wait(&aempty_bar[buf], ((job >> 1) & 1) ^ 1));
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + buf * 256u;
          for (int vs = 0; vs < nvslot; ++vs) {
            const int nkc = min(2, p.nchunk - 2 * vs);
            GLOM_CNT_WAIT(w0, mbar_wait(&full_bar[stage], phase));
            tc_fence_after_sync();
            if (elected) {
              const uint32_t s_lo = (stages0 + (uint32_t)stage * ATTN_SLOT_BYTES) >> 4;
              for (int kc = 0; kc < nkc; ++kc) {
                const uint64_t ad = kdesc0 + (uint64_t)(p_lo + (uint32_t)(2 * vs + kc) * (A_STAGE_BYTES >> 4));
                const uint64_t bd = vdesc0 + (uint64_t)(s_lo + (uint32_t)kc * (16384u >> 4));
                umma_bf16_2sm(d_tmem, ad, bd, idesc, (vs | kc) != 0 ? 1u : 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16_2sm(d_tmem, ad + 2 * k, bd + (2048 >> 4) * k, idesc, 1u);
              }
              umma_commit_2sm(&empty_bar[stage], 3);
            }
            __syncwarp();
            if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
          }
          if (elected) umma_commit_2sm(&afull_bar[buf], 3);
          __syncwarp();
        }
      }
      if (cnt_cta && elected) { atomicAdd(&cnt[2], w0); atomicAdd(&cnt[3], w1); }
    }
  } else if (warp < ATTN_SM_WARPS) {
    // ------------------------------------------------------------------ softmax + output warps (16 per CTA)
    // warp = (quad, part): TMEM lane quadrant `quad` (32 query rows, one per thread) x column quarter `part`
    // of every key block / output slice; row sums (and exact maxima) are combined across the four parts in smem.
    // These loops are chains of dependent latencies (TMEM load -> math -> shared-memory transpose -> store), so
    // four warps per scheduler are what hides them.
    const int quad = warp & 3, part = warp >> 2;
    const int t = quad * 32 + lane;          // query row inside the tile == TMEM lane
    const int tid = threadIdx.x;
    constexpr float LOG2E = 1.4426950408889634f;
    const float NEG_INF = __int_as_float(0xff800000);
    const bool use_mask = p.mask_side > 0;
    uint8_t* patch = patches + (size_t)warp * 2048;
    // releases towards the leader's MMA issuer: one arrival per warp of either CTA
    const uint32_t pready_remote = mapa_shared(smem_u32(pready_bar), 0);
    const uint32_t aempty_remote = mapa_shared(smem_u32(&aempty_bar[0]), 0);     // [buf]: + 8 * buf

    // per-key scale  log2(e) d^-1/2 / max(|S_j|, 1e-12)  (F.normalize eps, :58; logits are kept in log2 units)
    // and per-row bound  log2(e) d^-1/2 |S_j|  on the magnitude of row j's logits
    auto key_scales = [&](int item, int par) {
      const int b_ = item / pairs_per_img, l_ = (item % pairs_per_img) / p.npairs;
      for (int j = tid; j < p.n_pad16; j += ATTN_SM_THREADS) {
        float v = 0.f, bd = 0.f;
        if (j < p.nk) {
          const float* ns = p.nsq + (((size_t)b_ * p.n + p.key0 + j) * p.L + l_) * p.nparts;
          float ss = 0.f;
          if ((p.nparts & 3) == 0 && p.nparts <= 16) {      // one round trip: all partials in flight, then summed in order
            float4 q[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              q[i] = 4 * i < p.nparts ? __ldg(reinterpret_cast<const float4*>(ns) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) ss = (((ss + q[i].x) + q[i].y) + q[i].z) + q[i].w;
          } else {
            for (int i = 0; i < p.nparts; ++i) ss += ns[i];
          }
          const float nrm = sqrtf(ss);
          v = p.scale * LOG2E / fmaxf(nrm, 1e-12f);
          bd = p.scale * LOG2E * nrm;
        }
        rs[par * p.n_pad16 + j] = v;
        bnd[par * p.n_pad16 + j] = bd;
      }
    };
    if (cluster_id < p.num_items) key_scales(cluster_id, 0);
    // key coordinates for the careful path: padding keys sit 20000 rows away, so one distance test masks them as well
    // (:67-69; without a radius every real key is at (0, 0), the query at (0, 0) and the threshold 1)
    for (int j = tid; j < p.n_pad16; j += ATTN_SM_THREADS)
      key_hw[j] = j >= p.nk ? (20000u << 16)
                            : use_mask ? ((uint32_t)((p.key0 + j) / p.mask_side) << 16) | (uint32_t)((p.key0 + j) % p.mask_side) : 0u;
    const int d2_max = use_mask ? p.mask_d2_max : 1;
    if (part == 3) {                          // K-padding keys of the last 64-key chunk: P = 0, never written again
      for (int key = p.n_pad16; key < p.n_pad64; key += 8) {
        uint4* ptr = reinterpret_cast<uint4*>(p_smem + (size_t)(key >> 6) * A_STAGE_BYTES + (size_t)t * 128 +
                                              ((((key & 63) >> 3) ^ (t & 7)) << 4));
        *ptr = make_uint4(0, 0, 0, 0);
      }
    }

    uint32_t job = 0;
    int item_par = 0;
    for (int it = cluster_id; it < p.num_items; it += num_clusters, item_par ^= 1) {
      const int b = it / pairs_per_img, l = (it % pairs_per_img) / p.npairs;
      const int q0 = (2 * (it % p.npairs) + (int)cta_rank) * BM;
      const int qi = q0 + t;
      const size_t img_row0 = (size_t)b * p.n;
      const float* rsc = rs + item_par * p.n_pad16;
      named_bar_sync(1, ATTN_SM_THREADS);      // this item's key scales are visible
      const long long cnt_t0 = cnt_cta ? clock64() : 0;
      const unsigned long long cnt_w0 = w0;

      const int qh = use_mask ? qi / p.mask_side : 0, qw = use_mask ? qi % p.mask_side : 0;
      const int diag = p.attend_self ? -1 : qi;
      const int diag_blk = p.attend_self ? -1 : (q0 + quad * 32) >> 5;      // the 32 keys holding this warp's diagonals
      // logits (log2 units) of 16 keys starting at j0 (multiple of 16).  Plain blocks - no diagonal, padding or
      // radius mask, a warp-uniform property - take one multiply per key; the others a branch-free select chain.
      auto plain = [&](int j0) -> bool { return !use_mask && j0 + 16 <= p.nk && ((p.key0 + j0) >> 5) != diag_blk; };
      auto logits16 = [&](const uint32_t (&v)[16], int j0, float (&lg)[16]) {
        const float4* r4 = reinterpret_cast<const float4*>(rsc + j0);
        if (plain(j0)) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 r = r4[q];
            lg[4 * q] = __uint_as_float(v[4 * q]) * r.x;         lg[4 * q + 1] = __uint_as_float(v[4 * q + 1]) * r.y;
            lg[4 * q + 2] = __uint_as_float(v[4 * q + 2]) * r.z; lg[4 * q + 3] = __uint_as_float(v[4 * q + 3]) * r.w;
          }
        } else {
          const uint4* h4 = reinterpret_cast<const uint4*>(key_hw + j0);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 r = r4[q];
            const uint4 h = h4[q];
            const float rr[4] = {r.x, r.y, r.z, r.w};
            const uint32_t hh[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = p.key0 + j0 + 4 * q + e;                                  // global key index
              float sv = __uint_as_float(v[4 * q + e]) * rr[e];                       // (:60)
              sv = (j == diag) ? -5e-4f * LOG2E : sv;                                 // (:62-65)
              const int dh = qh - (int)(hh[e] >> 16), dw = qw - (int)(hh[e] & 0xFFFFu);
              lg[4 * q + e] = (dh * dh + dw * dw > d2_max) ? NEG_INF : sv;            // (:67-69) and key padding
            }
          }
        }
      };

      // stabiliser: the row's logit bound, or (beyond 2^BOUND_MAX, decided per warp) the exact running maximum
      const bool multi = !(p.pass_first && p.pass_last);
      float row_bound = 0.f;
      if (qi < p.n) {
        if (!multi) row_bound = bnd[item_par * p.n_pad16 + qi];
        else {                                   // the pass's scale arrays cover its keys only: this row's norm from the partials
          const float* ns = p.nsq + ((img_row0 + qi) * p.L + l) * p.nparts;
          float ss = 0.f;
          if ((p.nparts & 3) == 0 && p.nparts <= 16) {
            float4 q4[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              q4[i] = 4 * i < p.nparts ? __ldg(reinterpret_cast<const float4*>(ns) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) ss = (((ss + q4[i].x) + q4[i].y) + q4[i].z) + q4[i].w;
          } else {
            for (int i = 0; i < p.nparts; ++i) ss += ns[i];
          }
          row_bound = p.scale * LOG2E * sqrtf(ss);
        }
      }
      const bool exact_max = __any_sync(0xffffffffu, !(row_bound <= ATTN_BOUND_MAX));
      float m_run = exact_max ? NEG_INF : row_bound, l_run = 0.f;      // l_run: this warp's column part only
      float m_used[ATTN_MAX_KB];
      for (int kb = 0; kb < p.nkb; ++kb, ++job) {
        const int w = min(256, p.n_pad16 - kb * 256);
        const int cbeg = (((w >> 4) * part) >> 2) << 4, cend = (((w >> 4) * (part + 1)) >> 2) << 4;   // 16-key blocks
        const uint32_t buf = job & 1;
        GLOM_CNT_WAIT(w0, mbar_wait(&afull_bar[buf], (job >> 1) & 1));
        tc_fence_after_sync();
        const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * 256u;
        // S is read from TMEM 16 columns at a time; the loops stay rolled (one copy of the block body each)
        uint32_t cur[16];
        float lg[16];
        float m_safe = m_run;
        if (exact_max) {
          float bm = NEG_INF;
#pragma unroll 1
          for (int c0 = cbeg; c0 < cend; c0 += 16) {
            tmem_ld16(t_addr + c0, cur);
            tmem_ld_wait();
            logits16(cur, kb * 256 + c0, lg);
#pragma unroll
            for (int i = 0; i < 16; i += 4) bm = fmaxf(bm, fmaxf(fmaxf(lg[i], lg[i + 1]), fmaxf(lg[i + 2], lg[i + 3])));
          }
          red[(kb & 1) * 512 + part * 128 + t] = bm;                     // exchange the block max with the other parts
          named_bar_sync(2 + quad, 128);
#pragma unroll
          for (int q = 0; q < 4; ++q) bm = fmaxf(bm, red[(kb & 1) * 512 + q * 128 + t]);
          const float m_new = fmaxf(m_run, bm);
          m_safe = (m_new == NEG_INF) ? 0.f : m_new;
          l_run *= (m_run == NEG_INF) ? 0.f : ex2_approx(m_run - m_safe);
          m_run = m_new;
        }
        // unnormalised probabilities 2^(logit - m) -> bf16 P (UMMA A-operand layout) and their running sum
        uint32_t nxt[16];
        if (cbeg < cend) tmem_ld16(t_addr + cbeg, nxt);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cend; c0 += 16) {
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) cur[i] = nxt[i];
          if (c0 + 16 < cend) tmem_ld16(t_addr + c0 + 16, nxt);      // in flight while this block is processed
          const int j0 = kb * 256 + c0;
          logits16(cur, j0, lg);
          uint32_t pk[8];
          float acc = 0.f;
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float e0 = ex2_approx(lg[i] - m_safe), e1 = ex2_approx(lg[i + 1] - m_safe);
            const float e2 = ex2_approx(lg[i + 2] - m_safe), e3 = ex2_approx(lg[i + 3] - m_safe);
            acc += (e0 + e1) + (e2 + e3);
            pk[i / 2] = pack_bf16x2(e0, e1);
            pk[i / 2 + 1] = pack_bf16x2(e2, e3);
          }
          l_run += acc;
          uint8_t* rowp = p_smem + (size_t)(j0 >> 6) * A_STAGE_BYTES + (size_t)t * 128;
          const int ch = (j0 & 63) >> 3;                     // 16-byte chunk index inside the 128-byte row (even)
          *reinterpret_cast<uint4*>(rowp + (((ch) ^ (t & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          *reinterpret_cast<uint4*>(rowp + (((ch + 1) ^ (t & 7)) << 4)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        }
        m_used[kb] = m_safe;
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(aempty_remote + 8u * buf);
      }
      if (exact_max) {
        const float m_fin = (m_run == NEG_INF) ? 0.f : m_run;
        // bring every block's probabilities onto the final stabiliser
        for (int kb = 0; kb < p.nkb; ++kb) {
          if (m_used[kb] == m_fin) continue;
          const float f = ex2_approx(m_used[kb] - m_fin);
          const int w = min(256, p.n_pad16 - kb * 256);
          const int cbeg = (((w >> 4) * part) >> 2) << 4, cend = (((w >> 4) * (part + 1)) >> 2) << 4;
          for (int c0 = cbeg; c0 < cend; c0 += 8) {
            const int key = kb * 256 + c0;
            uint4* ptr = reinterpret_cast<uint4*>(p_smem + (size_t)(key >> 6) * A_STAGE_BYTES + (size_t)t * 128 +
                                                  ((((key & 63) >> 3) ^ (t & 7)) << 4));
            uint4 u = *ptr;
            uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float lo = __uint_as_float(wv[i] << 16) * f, hi = __uint_as_float(wv[i] & 0xFFFF0000u) * f;
              wv[i] = pack_bf16x2(lo, hi);
            }
            *ptr = make_uint4(wv[0], wv[1], wv[2], wv[3]);
          }
        }
      }
      red[1024 + part * 128 + t] = l_run;                                // row sum = sum of the four parts
      fence_proxy_async_smem();                // this thread's P rows -> visible to the tensor core's reads
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(pready_remote);
      const long long cnt_t1 = cnt_cta ? clock64() : 0;
      const unsigned long long cnt_w1 = w0;
      if (cnt_cta) w1 += (unsigned long long)(cnt_t1 - cnt_t0) - (cnt_w1 - cnt_w0);       // softmax work (waits excluded)
      // while P V runs: key scales of this cluster's next item (other parity; last read in the previous item)
      if (it + num_clusters < p.num_items) key_scales(it + num_clusters, item_par ^ 1);
      // key passes: this row's carried (stabiliser, row sum), read before the barrier below (part 0 rewrites it after it)
      const size_t acc_row = (img_row0 + (size_t)qi) * p.L + l;
      float m_acc = NEG_INF, l_acc = 0.f;
      if (multi && !p.pass_first && qi < p.n) {
        const float2 ml = *reinterpret_cast<const float2*>(p.ml_acc + acc_row * 2);
        m_acc = ml.x; l_acc = ml.y;
      }
      named_bar_sync(2 + quad, 128);
      const float l_pass = (red[1024 + t] + red[1152 + t]) + (red[1280 + t] + red[1408 + t]);
      float inv_l = 1.0f / l_pass, f_old = 0.f, f_new = 1.f;
      if (multi) {
        // partial results of different key ranges are on different stabilisers only for rows on the exact-maximum path
        float m_pass = exact_max ? m_run : row_bound;
        if (l_pass == 0.f) m_pass = NEG_INF;                       // no unmasked key in this range
        const float m_new = fmaxf(m_acc, m_pass);
        f_old = (m_acc == NEG_INF) ? 0.f : ex2_approx(m_acc - m_new);
        f_new = (m_pass == NEG_INF) ? 0.f : ex2_approx(m_pass - m_new);
        const float l_new = l_acc * f_old + l_pass * f_new;
        inv_l = p.pass_last ? 1.0f / l_new : 1.0f;
        if (!p.pass_last && part == 0 && qi < p.n) *reinterpret_cast<float2*>(p.ml_acc + acc_row * 2) = make_float2(m_new, l_new);
      }

      // output: O slice (128 x <=256) from TMEM, scaled by 1/rowsum, bf16, transposed through a 2 KB patch
      // so that stores cover 64-byte row segments
      const int rows_left = p.n - (q0 + quad * 32);
      for (int sp = 0; sp < nsub; ++sp, ++job) {
        const int wdp = (min(256, p.d - sp * 256) + 127) & ~127;
        const int cbeg = part * (wdp >> 2), cend = min(cbeg + (wdp >> 2), p.d - sp * 256);   // columns past d hold zeros
        const uint32_t buf = job & 1;
        GLOM_CNT_WAIT(w0, mbar_wait(&afull_bar[buf], (job >> 1) & 1));
        tc_fence_after_sync();
        const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * 256u;
        __nv_bfloat16* cdst = p.c_out + ((img_row0 + q0 + quad * 32) * p.L + l) * p.d + sp * 256;
        // 32 columns of this thread's row are scaled by 1/rowsum, rounded to bf16 and transposed through the warp's
        // 2 KB patch so that stores cover 64-byte row segments
        auto emit32 = [&](const uint32_t (&v)[32], int c0) {
          if (p.lean) {        // this thread's own row: 32 columns = 64 contiguous bytes (slower stores, no shared memory)
            uint4* dst = reinterpret_cast<uint4*>(cdst + (size_t)lane * p.L * p.d + c0);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint4 val = make_uint4(
                  pack_bf16x2(__uint_as_float(v[8 * c + 0]) * inv_l, __uint_as_float(v[8 * c + 1]) * inv_l),
                  pack_bf16x2(__uint_as_float(v[8 * c + 2]) * inv_l, __uint_as_float(v[8 * c + 3]) * inv_l),
                  pack_bf16x2(__uint_as_float(v[8 * c + 4]) * inv_l, __uint_as_float(v[8 * c + 5]) * inv_l),
                  pack_bf16x2(__uint_as_float(v[8 * c + 6]) * inv_l, __uint_as_float(v[8 * c + 7]) * inv_l));
              if (lane < rows_left) dst[c] = val;
            }
            return;
          }
#pragma unroll
          for (int c = 0; c < 4; ++c)
            *reinterpret_cast<uint4*>(patch + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) = make_uint4(
                pack_bf16x2(__uint_as_float(v[8 * c + 0]) * inv_l, __uint_as_float(v[8 * c + 1]) * inv_l),
                pack_bf16x2(__uint_as_float(v[8 * c + 2]) * inv_l, __uint_as_float(v[8 * c + 3]) * inv_l),
                pack_bf16x2(__uint_as_float(v[8 * c + 4]) * inv_l, __uint_as_float(v[8 * c + 5]) * inv_l),
                pack_bf16x2(__uint_as_float(v[8 * c + 6]) * inv_l, __uint_as_float(v[8 * c + 7]) * inv_l));
          __syncwarp();
          const int c = lane & 3;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = i * 8 + (lane >> 2);
            const uint4 val = *reinterpret_cast<const uint4*>(patch + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
            if (r < rows_left) *reinterpret_cast<uint4*>(cdst + (size_t)r * p.L * p.d + c0 + c * 8) = val;
          }
          __syncwarp();
        };
        uint32_t cur[32];
#pragma unroll 1
        for (int c0 = cbeg; c0 < cend; c0 += 32) {
          tmem_ld32(t_addr + c0, cur);
          tmem_ld_wait();
          if (multi) {
            // this thread's row, 32 consecutive fp32 columns (128 bytes) of the carried output
            float4* acc = reinterpret_cast<float4*>(p.o_acc + acc_row * p.d + sp * 256 + c0);
            const bool row_ok = qi < p.n;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
              if (!p.pass_first && row_ok) o = acc[q];
              const float4 v = make_float4(__uint_as_float(cur[4 * q]) * f_new + o.x * f_old, __uint_as_float(cur[4 * q + 1]) * f_new + o.y * f_old,
                                           __uint_as_float(cur[4 * q + 2]) * f_new + o.z * f_old, __uint_as_float(cur[4 * q + 3]) * f_new + o.w * f_old);
              if (!p.pass_last) { if (row_ok) acc[q] = v; }
              else { cur[4 * q] = __float_as_uint(v.x); cur[4 * q + 1] = __float_as_uint(v.y); cur[4 * q + 2] = __float_as_uint(v.z); cur[4 * q + 3] = __float_as_uint(v.w); }
            }
            if (!p.pass_last) continue;
          }
          emit32(cur, c0);
        }
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(aempty_remote + 8u * buf);
      }
      if (cnt_cta) w2 += (unsigned long long)(clock64() - cnt_t1) - (w0 - cnt_w1);          // key scales + output work
    }
    if (cnt_cta && warp == 0 && lane == 0) { atomicAdd(&cnt[5], w0); atomicAdd(&cnt[6], w1); atomicAdd(&cnt[7], w2); }
  }
#undef GLOM_CNT_WAIT

  tc_fence_before_sync();
  __syncthreads();
  if (clk_thread) clock_sample_end(clk_s, g_kernel_clk[PROF_ATTN]);
  cluster_sync_all();          // no CTA exits (or frees TMEM) while its pair can still touch it
  if (warp == W_ALLOC) {
    tc_fence_after_sync();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// cycles / ns accumulated by the kernels of this translation unit since the last call (and reset)
cudaError_t tc_kernel_clocks(unsigned long long* out /* [PROF_KINDS][8] */, bool reset) {
  cudaError_t e = cudaMemcpyFromSymbol(out, g_kernel_clk, sizeof(unsigned long long) * PROF_KINDS * 8);
  if (e == cudaSuccess && reset) {
    static const unsigned long long zeros[PROF_KINDS * 8] = {};
    e = cudaMemcpyToSymbol(g_kernel_clk, zeros, sizeof(zeros));
  }
  return e;
}

// =====================================================================================
// Host side: tensor maps + launches for one Jacobi step
// =====================================================================================
static inline bool encode_map(EncodeTiledFn enc, CUtensorMap* m, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, char* err, size_t errlen,
                       const char* what) {
  cuuint64_t gd[3]; cuuint64_t gs[2]; cuuint32_t bx[3]; cuuint32_t es[3] = {1, 1, 1};
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(err, errlen, "cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r);
    return false;
  }
  return true;
}

static inline bool map2d(EncodeTiledFn enc, CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                  char* err, size_t errlen, const char* what) {
  const uint64_t dims[2] = {cols, rows};
  const uint64_t strides[1] = {cols * 2};
  const uint32_t box[2] = {(uint32_t)BK, box_rows};
  return encode_map(enc, m, base, 2, dims, strides, box, err, errlen, what);
}

template <int MODE, int BN, bool CNT>
static cudaError_t launch_gemm_impl(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& bm,
                                    const GemmParams& p, int num_sms, cudaStream_t st);

template <int MODE, int BN>
static cudaError_t launch_gemm(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& bm,
                               const GemmParams& p, int num_sms, cudaStream_t st) {
  // GLOM_B200_WAIT_COUNTERS=1 (diagnostics): the instantiation whose block 0 accumulates its roles' wait cycles
  static int count_waits = -1;
  if (count_waits < 0) { const char* ev = getenv("GLOM_B200_WAIT_COUNTERS"); count_waits = (ev && ev[0] == '1') ? 1 : 0; }
  if (count_waits) return launch_gemm_impl<MODE, BN, true>(a0, a1, a2, bm, p, num_sms, st);
  return launch_gemm_impl<MODE, BN, false>(a0, a1, a2, bm, p, num_sms, st);
}

template <int MODE, int BN, bool CNT>
static cudaError_t launch_gemm_impl(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& bm,
                                    const GemmParams& p, int num_sms, cudaStream_t st) {
  using Cfg = GemmCfg<MODE, BN>;
  static SmemOptIn optin;
  if (cudaError_t e = optin.ensure(gemm_kernel<MODE, BN, CNT>, Cfg::SMEM_BYTES)) return e;
  const int max_clusters = num_sms / 2;
  const int clusters = p.num_tiles < max_clusters ? p.num_tiles : max_clusters;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // PDL: see pdl_wait() in the kernel
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, gemm_kernel<MODE, BN, CNT>, a0, a1, a2, bm, p);
}

// K3: consensus attention -> C
static int launch_attention(const Geometry& g, const Bf16Buffers& b, EncodeTiledFn enc, int num_sms, cudaStream_t st,
                            int* launches, char* err, size_t errlen, Profiler* prof) {
  const int d = g.d, L = g.L, n = g.n;
  // Up to 576 columns the probabilities of a 128-query tile against all keys fit in shared memory: one launch.  Beyond,
  // the keys are processed in passes of ATTN_PASS_KEYS (one launch each, see AttnParams): no shape falls to CUDA cores.
  const int npass = (n <= ATTN_SINGLE_PASS_MAX) ? 1 : (n + ATTN_PASS_KEYS - 1) / ATTN_PASS_KEYS;
  if (npass > 1 && !b.attn_acc) {
    snprintf(err, errlen, "consensus for n = %d columns needs the key-pass scratch buffer (workspace too old?)", n);
    return -3;
  }
  CUtensorMap mq, mk, mv;
  const uint64_t dims[3] = {(uint64_t)L * d, (uint64_t)n, (uint64_t)g.B};
  const uint64_t strides[2] = {(uint64_t)L * d * 2, (uint64_t)n * L * d * 2};
  const uint32_t boxq[3] = {(uint32_t)BK, (uint32_t)BM, 1}, boxv[3] = {(uint32_t)BK, 64, 1};
  if (!encode_map(enc, &mq, b.sb_in, 3, dims, strides, boxq, err, errlen, "attn.q")) return -3;
  if (!encode_map(enc, &mv, b.sb_in, 3, dims, strides, boxv, err, errlen, "attn.v")) return -3;
  for (int pass = 0; pass < npass; ++pass) {
    AttnParams ap{};
    ap.n = n; ap.L = L; ap.d = d;
    ap.attend_self = g.attend_self; ap.mask_side = g.mask_side; ap.mask_d2_max = g.mask_d2_max;
    ap.key0 = npass == 1 ? 0 : pass * ATTN_PASS_KEYS;
    ap.nk = npass == 1 ? n : (n - ap.key0 < ATTN_PASS_KEYS ? n - ap.key0 : ATTN_PASS_KEYS);
    ap.pass_first = pass == 0; ap.pass_last = pass == npass - 1;
    ap.o_acc = b.attn_acc;
    ap.ml_acc = b.attn_acc ? b.attn_acc + (size_t)g.rows * L * d : nullptr;
    ap.n_pad16 = (ap.nk + 15) / 16 * 16;
    ap.n_pad64 = (ap.nk + 63) / 64 * 64;
    ap.nkb = (ap.n_pad16 + 255) / 256;
    ap.nchunk = ap.n_pad64 / 64;
    ap.khalf_rows = (ap.n_pad16 < 256 ? ap.n_pad16 : 256) / 2;
    ap.nparts = g.nparts;
    ap.nsq = b.nsq_in;
    ap.c_out = b.c;
    ap.scale = 1.0f / sqrtf((float)d);
    const int ntiles = (n + BM - 1) / BM;
    ap.npairs = (ntiles + 1) / 2;
    ap.q_in_k = npass == 1 && ap.n_pad16 == 256;    // one key block of 256: CTA r's queries are keys [128 r, 128 r + 128)
    ap.num_items = ap.npairs * L * g.B;
    size_t fixed = 1024 + (size_t)ap.nchunk * A_STAGE_BYTES + ATTN_PATCH_BYTES + (size_t)ap.n_pad16 * 20 +
                   ATTN_RED_FLOATS * 4 + 256;
    const size_t max_smem = 227 * 1024;
    int stages = 4;
    while (stages > 0 && fixed + (size_t)stages * ATTN_SLOT_BYTES > max_smem) --stages;
    if (stages < 2 && fixed - ATTN_PATCH_BYTES + ATTN_SLOT_BYTES <= max_smem) {
      // P of this many columns leaves at most one ring slot: give up the transpose patches (row-per-thread stores) so
      // that loads and MMAs can overlap at all
      ap.lean = 1;
      fixed -= ATTN_PATCH_BYTES;
      stages = 4;
      while (stages > 0 && fixed + (size_t)stages * ATTN_SLOT_BYTES > max_smem) --stages;
    }
    if (stages < 1 || ap.nkb > ATTN_MAX_KB) {
      snprintf(err, errlen, "consensus pass of %d keys does not fit shared memory", ap.nk);
      return -3;
    }
    ap.num_stages = stages;
    const size_t smem = fixed + (size_t)stages * ATTN_SLOT_BYTES;
    static SmemOptIn optin;
    static int count_waits = -1;
    if (count_waits < 0) { const char* ev = getenv("GLOM_B200_WAIT_COUNTERS"); count_waits = (ev && ev[0] == '1') ? 1 : 0; }
    static SmemOptIn optin_cnt;
    if (cudaError_t e = count_waits ? optin_cnt.ensure(attn_kernel<true>, smem) : optin.ensure(attn_kernel<false>, smem)) {
      snprintf(err, errlen, "cudaFuncSetAttribute(attn): %s", cudaGetErrorString(e));
      return -3;
    }
    const uint32_t boxk[3] = {(uint32_t)BK, (uint32_t)ap.khalf_rows, 1};
    if (!encode_map(enc, &mk, b.sb_in, 3, dims, strides, boxk, err, errlen, "attn.k")) return -3;
    const int max_clusters = num_sms / 2;
    const int clusters = ap.num_items < max_clusters ? ap.num_items : max_clusters;
    ProfScope scope(prof, PROF_ATTN, st);
    cudaLaunchConfig_t acfg{};
    acfg.gridDim = dim3(2 * clusters); acfg.blockDim = dim3(ATTN_THREADS); acfg.dynamicSmemBytes = smem; acfg.stream = st;
    cudaLaunchAttribute aattr[2];
    aattr[0].id = cudaLaunchAttributeClusterDimension;
    aattr[0].val.clusterDim.x = 2; aattr[0].val.clusterDim.y = 1; aattr[0].val.clusterDim.z = 1;
    aattr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // PDL: see pdl_wait() in the kernel
    aattr[1].val.programmaticStreamSerializationAllowed = 1;
    acfg.attrs = aattr; acfg.numAttrs = 2;
    const cudaError_t e = count_waits ? cudaLaunchKernelEx(&acfg, attn_kernel<true>, mq, mk, mv, ap)
                                      : cudaLaunchKernelEx(&acfg, attn_kernel<false>, mq, mk, mv, ap);
    if (launches) ++*launches;
    if (e != cudaSuccess) { snprintf(err, errlen, "attn_kernel launch: %s", cudaGetErrorString(e)); return -3; }
  }
  return 0;
}

int step_bf16(const Geometry& g, const Bf16Buffers& b, int step_index, EncodeTiledFn enc, int num_sms, cudaStream_t st,
              int* launches, char* err, size_t errlen, Profiler* prof) {
  const int d = g.d, L = g.L, n = g.n, rows = g.rows;
  // One launch each of K1 (all groups), K3, K2 (all levels).  Splitting K1/K2 into per-level batches so that H stays
  // L2-resident was measured slower (5.3 / 5.6 / 6.5 ms per step for 3 / 2 / 1 levels per batch vs 5.06 ms): the extra
  // kernel boundaries and partial waves cost more than the saved HBM traffic (profiles/README.md).
  CUtensorMap mh;
  const int m128 = (rows + BM - 1) / BM;
  if (!map2d(enc, &mh, b.h, (uint64_t)g.G * m128 * (4 * d / BK) * BM, BK, BM, err, errlen, "H")) return -3;
  CUtensorMap mx, msb, msp, mw1, mw2;
  if (!map2d(enc, &mx, b.xb, rows, d, BM, err, errlen, "Xb")) return -3;
  if (!map2d(enc, &msb, b.sb_in, rows, (uint64_t)L * d, BM, err, errlen, "Sb")) return -3;
  if (!map2d(enc, &msp, b.sp_in, rows, (uint64_t)(L - 1) * d, BM, err, errlen, "Sp")) return -3;
  if (!map2d(enc, &mw1, b.w1, (uint64_t)g.G * 4 * d, d, 128, err, errlen, "W1p")) return -3;
  if (!map2d(enc, &mw2, b.w2, (uint64_t)L * d, (uint64_t)8 * d, (uint32_t)g.bn2 / 2, err, errlen, "W2p")) return -3;
  // ---------------- K1: grouped GEMM1 + bias + GELU -> H   (all 2L-1 groups)
  {
    GemmParams p{};
    p.rows = rows; p.d = d; p.L = L; p.n = n; p.G = g.G;
    // group 0 (bottom-up net of level 0) reads the tokens, which are the same in every step of a call (:132-134): its block
    // of H is written by the call's first step and stays valid; the later steps run the other 2L - 2 groups only.
    // Groups are walked bottom-up and every H block is a streaming store: a reverse walk and normal-policy stores for
    // the groups GEMM2 reads first measured no effect (profiles/r2_k1_order_ab.txt).
    p.z0 = (step_index > 0 && g.G > 1) ? 1 : 0;
    p.num_m = (rows + 255) / 256; p.num_n = 4 * d / 256; p.num_tiles = (g.G - p.z0) * p.num_m * p.num_n;
    p.bias = b.b1; p.h_out = b.h; p.m128 = m128;
    ProfScope scope(prof, PROF_GEMM1, st);
    cudaError_t e = launch_gemm<0, 256>(mx, msb, msp, mw1, p, num_sms, st);
    if (launches) ++*launches;
    if (e != cudaSuccess) { snprintf(err, errlen, "gemm1 launch: %s", cudaGetErrorString(e)); return -3; }
  }
  // ---------------- K3 between K1 and K2 (C is then still L2-resident when K2's epilogue reads it; launching it
  // first instead measured the same within 0.2 %)
  if (int rc = launch_attention(g, b, enc, num_sms, st, launches, err, errlen, prof)) return rc;
  // ---------------- K2: grouped GEMM2 + combine -> state t+1 (+ shadows, norms)   (all levels)
  {
    GemmParams p{};
    p.rows = rows; p.d = d; p.L = L; p.n = n; p.G = g.G;
    p.num_m = (rows + 255) / 256; p.num_n = d / g.bn2; p.z0 = 0; p.num_tiles = L * p.num_m * p.num_n;
    p.n_half = p.num_m * p.num_n;
    p.m128 = m128;
    p.bias = b.b2; p.s32_in = b.s32_in; p.s_bcast = b.s32_in_bcast; p.c_in = b.c; p.pos = b.pos;
    p.s32_out = b.s32_out; p.sb_out = b.sb_out; p.sp_out = b.sp_out; p.nsq_out = b.nsq_out; p.nparts = g.nparts;
    cudaError_t e;
    ProfScope scope(prof, PROF_GEMM2, st);
    if (g.bn2 == 256) e = launch_gemm<1, 256>(mh, mh, mh, mw2, p, num_sms, st);
    else if (g.bn2 == 128) e = launch_gemm<1, 128>(mh, mh, mh, mw2, p, num_sms, st);
    else e = launch_gemm<1, 64>(mh, mh, mh, mw2, p, num_sms, st);
    if (launches) ++*launches;
    if (e != cudaSuccess) { snprintf(err, errlen, "gemm2 launch: %s", cudaGetErrorString(e)); return -3; }
  }
  return 0;
}


// ---------------- tensor-core tokeniser: tokens = patches(bf16) . Wtok(bf16)^T + bias   (glom_pytorch.py:94-97)
int tokenize_tc(const __nv_bfloat16* patches, const __nv_bfloat16* wtok, const float* bias, float* tokens, int rows,
                int d, int kp, EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches, char* err, size_t errlen) {
  const int bn = (d % 256 == 0) ? 256 : (d % 128 == 0) ? 128 : 64;
  CUtensorMap ma, mb;
  if (!map2d(enc, &ma, patches, rows, kp, BM, err, errlen, "patches")) return -3;
  if (!map2d(enc, &mb, wtok, d, kp, (uint32_t)bn / 2, err, errlen, "Wtok")) return -3;
  GemmParams p{};
  p.rows = rows; p.d = d; p.L = 1; p.n = 1; p.G = 1;
  p.num_m = (rows + 255) / 256; p.num_n = d / bn; p.num_tiles = p.num_m * p.num_n;
  p.bias = bias; p.tok_out = tokens; p.tok_kb = kp / BK;
  cudaError_t e;
  if (bn == 256) e = launch_gemm<2, 256>(ma, ma, ma, mb, p, num_sms, st);
  else if (bn == 128) e = launch_gemm<2, 128>(ma, ma, ma, mb, p, num_sms, st);
  else e = launch_gemm<2, 64>(ma, ma, ma, mb, p, num_sms, st);
  if (launches) ++*launches;
  if (e != cudaSuccess) { snprintf(err, errlen, "tokeniser gemm launch: %s", cudaGetErrorString(e)); return -3; }
  return 0;
}

}  // namespace glom
