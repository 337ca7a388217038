// Internal engine declarations shared by the C-ABI translation unit and the kernel files.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stddef.h>
#include <stdint.h>
#include <mutex>
#include <vector>

namespace glom {

// Optional per-kernel CUDA-event timing (bench.py's roofline numbers).  Events are recorded on the
// launch stream around each kernel; nothing is synchronised until the caller reads them.
enum ProfKind { PROF_ATTN = 0, PROF_GEMM1 = 1, PROF_GEMM2 = 2, PROF_PREP = 3, PROF_TOKENIZE = 4, PROF_KINDS = 5 };
struct Profiler {
  bool enabled = false;
  std::vector<cudaEvent_t> ev;
  size_t used = 0;
  struct Span { int kind; size_t a, b; };
  std::vector<Span> spans;
  size_t mark(cudaStream_t st) {
    if (used == ev.size()) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); }
    cudaEventRecord(ev[used], st);
    return used++;
  }
};
struct ProfScope {   // RAII: events around one launch when profiling is on
  Profiler* p; int kind; cudaStream_t st; size_t a;
  ProfScope(Profiler* p_, int kind_, cudaStream_t st_) : p(p_ && p_->enabled ? p_ : nullptr), kind(kind_), st(st_), a(0) {
    if (p) a = p->mark(st);
  }
  ~ProfScope() { if (p) { const size_t b = p->mark(st); p->spans.push_back({kind, a, b}); } }
};

struct Geometry {
  int d, L, n, B;
  int rows;        // B * n   (columns of the batch = GEMM M)
  int G;           // 2L - 1  MLP groups, ordered bu_0, td_0, bu_1, td_1, ..., bu_{L-1}
  int hidden;      // 4d
  int attend_self, mask_side, mask_d2_max;
  int bn2;         // N tile of the second GEMM: 256 / 128 / 64 (largest dividing d)
  int part_w;      // columns covered by one squared-norm partial (one epilogue warp group)
  int nparts;      // squared-norm partials per (row, level) = d / part_w
};

// ---- packed weights -------------------------------------------------------------------------
// bf16 engine:  W1p [(G*4d) x d] bf16 | W2p [(L*d) x 8d] bf16 | b1p [G*4d] f32 | b2p [L*d] f32
// fp32 engine:  same shapes, all f32.
struct PackedLayout {
  size_t w1_off, w2_off, b1_off, b2_off, total;
};
PackedLayout packed_layout(int d, int L, int precision);

// ---- workspace ------------------------------------------------------------------------------
struct WorkspaceLayout {
  size_t s32_off;      // one fp32 state slab (ping-pong partner of state_out); 0 bytes if return_all
  size_t s32_bytes;
  size_t sb_off[2];    // bf16 shadow of the state           (rows, L, d)
  size_t sp_off[2];    // bf16 shadow of state[:, :, 1:] + pos (rows, L-1, d)
  size_t xb_off;       // bf16 tokens                        (rows, d)
  size_t h_off;        // hidden activations: bf16 engine = 16 KB blocks [G][rows/128][4d/64][128][64]; f32 = (rows, G*4d)
  size_t h_bytes;
  size_t c_off;        // consensus output                   (rows, L, d)   bf16 | f32
  size_t c_bytes;
  size_t nsq_off[2];   // squared-norm partials              (rows, L, nparts) f32
  size_t nsq_bytes;
  size_t attn_acc_off; // bf16 engine, n > 576 columns: fp32 output / (stabiliser, row sum) carried between the consensus kernel's key passes
  size_t attn_acc_bytes;
  size_t total;
};
WorkspaceLayout workspace_layout(const Geometry& g, int precision, int iters, int return_all);

// ---- launchers (return cudaError_t of the launch; all asynchronous on `st`) -----------------
struct Bf16Buffers {
  const float* s32_in;  float* s32_out;              // fp32 master state of step t / t+1
  int s32_in_bcast;                                   // 1: s32_in is init_levels (L, d) broadcast over the rows (step 0, no carried state)
  const __nv_bfloat16* sb_in;  __nv_bfloat16* sb_out;
  const __nv_bfloat16* sp_in;  __nv_bfloat16* sp_out;
  const __nv_bfloat16* xb;
  __nv_bfloat16* h;  __nv_bfloat16* c;
  float* attn_acc;                                    // n > 576 columns only: (rows, L, d) + (rows, L, 2) fp32 carried between key passes
  const float* nsq_in;  float* nsq_out;
  const float* pos;                                   // (n, d) fp32
  const __nv_bfloat16* w1;  const __nv_bfloat16* w2;  const float* b1;  const float* b2;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// state prologue: S_0 -> fp32 master copy (dst may equal src => skipped), bf16 shadows, norms, bf16 tokens
cudaError_t launch_prep(const Geometry& g, const float* state_in, const float* init_levels, const float* pos,
                        const float* tokens, float* s32_dst, __nv_bfloat16* sb, __nv_bfloat16* sp,
                        __nv_bfloat16* xb, float* nsq, cudaStream_t st, int* launches, Profiler* prof);

// one Jacobi step on tensor cores, three launches: GEMM1+GELU -> H ; consensus -> C ; GEMM2+combine -> state t+1.
// step_index: position of the step inside the forward call.  The bottom-up net of level 0 reads the tokens, which do not
// change during a call (glom_pytorch.py:132-134), so its hidden activations (MLP group 0 of H) are computed by step 0 only
// and re-read by GEMM2 of the later steps.
int step_bf16(const Geometry& g, const Bf16Buffers& b, int step_index, EncodeTiledFn enc, int num_sms, cudaStream_t st,
              int* launches, char* err, size_t errlen, Profiler* prof);

struct F32Buffers {
  const float* s_in;  float* s_out;
  const float* x;  const float* pos;
  float* h;  float* c;
  const float* w1;  const float* w2;  const float* b1;  const float* b2;
};
cudaError_t step_f32(const Geometry& g, const F32Buffers& b, cudaStream_t st, int* launches, Profiler* prof);
cudaError_t launch_broadcast_init(const Geometry& g, const float* state_in, const float* init_levels, float* dst,
                                  cudaStream_t st, int* launches, Profiler* prof);

cudaError_t launch_pack(int d, int L, int precision, const float* bu_w1, const float* bu_b1, const float* bu_w2,
                        const float* bu_b2, const float* td_w1, const float* td_b1, const float* td_w2,
                        const float* td_b2, void* packed, cudaStream_t st, int* launches);

cudaError_t launch_tokenize(const float* img, const float* w, const float* bias, float* tokens, int B, int H, int W,
                            int p, int d, cudaStream_t st, int* launches, Profiler* prof);

// island analytics on state slabs (islands.cu)
cudaError_t launch_islands(const float* states, int slabs, int side_h, int side_w, int L, int d, float threshold,
                           float* cos_right, float* cos_down, float* agreement, int* labels, int* num_islands,
                           cudaStream_t st, int* launches);

cudaError_t launch_clock_probe(unsigned long long* out, unsigned long long spin_ns, cudaStream_t st);
// (cycles, ns) sampled INSIDE the tensor-core kernels since the last reset, by ProfKind (tc_kernels.cu)
cudaError_t tc_kernel_clocks(unsigned long long* out /* [PROF_KINDS][8] */, bool reset);

// bf16 tokeniser: patchify + cast (CUDA cores), then the tcgen05 GEMM
cudaError_t launch_patchify_bf16(const float* img, const float* w, __nv_bfloat16* patches, __nv_bfloat16* wtok, int B,
                                 int H, int W, int p, int d, int kp, cudaStream_t st, int* launches);
int tokenize_tc(const __nv_bfloat16* patches, const __nv_bfloat16* wtok, const float* bias, float* tokens, int rows,
                int d, int kp, EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches, char* err, size_t errlen);

// ---- backward (fp32, CUDA cores; bwd_kernels.cu) ---------------------------------------------------------
struct BackwardArgs {
  const float* tokens;   // (R, d)
  const float* pos;      // (n, d)
  const float* states;   // (T+1, R, L, d): S_0 .. S_T of the forward
  const float* grad_out; // (T+1, R, L, d) if grad_all else (R, L, d): dL/d(returned tensor)
  const float *bu_w1, *bu_b1, *bu_w2, *td_w1, *td_b1, *td_w2;   // reference layout, fp32 (second biases are not needed)
  // outputs, ACCUMULATED into (caller zero-initialises); d_state0 / d_init: exactly one is non-NULL
  float *d_tokens, *d_pos, *d_state0, *d_init;
  float *d_bu_w1, *d_bu_b1, *d_bu_w2, *d_bu_b2, *d_td_w1, *d_td_b1, *d_td_w2, *d_td_b2;
};
struct BackwardLayout {
  size_t g_off, gs_off, ds_off, khat_off, dkhat_off, rnorm_off, pre_off, h_off, dh_off, xp_off, dx_off, attn_off,
      dattn_off;
  // bf16 (tensor-core) MLP backward only
  size_t xb_off, sb_off, sp_off, gsb_off, w1p_off, w2t_off, w1t_off, b1p_off, bpre_off, bh_off, bdpre_off;
  size_t khatb_off, ab_off, dsimb_off;     // bf16 khat (state-like), probabilities and scaled dsim (Z, n, n)
  size_t blocked_bytes;
  size_t total;
};
// tensor-core MLP backward (tc_bwd_kernels.cu)
struct MlpBwdTc {
  const __nv_bfloat16 *xb, *sb, *sp, *gsb;      // bf16 shadows: tokens, S_t, S_t[:,1:]+pos, dL/dS_{t+1}/c
  const __nv_bfloat16 *w1p, *w2t, *w1t;        // (G*4d, d), (G*4d, d) = W2^T, (G*d, 4d) = W1^T, groups interleaved bu/td
  const float* b1p;                            // (G*4d)
  __nv_bfloat16 *pre, *h, *dpre;               // blocked (G, R_pad/128, 4d/64, 128, 64)
  float *ds, *d_tokens, *d_pos;                // input gradients of the groups are reduced straight into these:
                                               // dL/dS_t (R, L, d), dL/dtokens (R, d), dL/dpos (n, d)
  float *d_bu_w1, *d_bu_w2, *d_td_w1, *d_td_w2;
  float *d_bu_b1, *d_td_b1;                    // first-layer bias gradients, reduced in the DH epilogue
};
int mlp_backward_tc(const Geometry& g, const MlpBwdTc& a, EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches,
                    char* err, size_t errlen);

// (optional trailing arguments: a second product accumulated into the same output tile, see tc_bwd_kernels.cu)
int attn_bwd_gemm_tc(const Geometry& g, const void* a_src, int a_state, int a_mn, const void* b_src, int b_state, int b_mn,
                     int N, int K, int out_kind, float* out, EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches,
                     char* err, size_t errlen, const void* a2_src = nullptr, int a2_state = 0, int a2_mn = 0,
                     const void* b2_src = nullptr, int b2_state = 0, int b2_mn = 0);

BackwardLayout backward_layout(const Geometry& g, int precision);
// tokeniser backward (fp32, CUDA cores; bwd_kernels.cu): any of d_weight / d_bias / d_img may be NULL; all ACCUMULATED into
size_t tokenize_backward_workspace_bytes(int B, int H, int W, int p, int need_dimg);
cudaError_t tokenize_backward(const float* img, const float* weight, const float* d_tokens, float* d_weight, float* d_bias,
                              float* d_img, int B, int H, int W, int p, int d, void* workspace, cudaStream_t st, int* launches);
int backward_run(const Geometry& g, const BackwardArgs& a, int precision, int iters, int grad_all, void* workspace,
                 EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches, char* err, size_t errlen);

// ---- column-contrastive loss (contrastive.cu) ------------------------------------------------------------
#define GLOM_CT_MAX_SEL 32      // selected levels per call
#define GLOM_CT_MAX_SPLIT 8     // column splits of the lse kernel (partial sums in the scratch buffer)
struct ContrastiveStrides { long long b, n, l; };   // element strides of a (B, n, L, d) input whose d is contiguous
struct ContrastiveGeom {
  int R, Rp, n, d, L, nsel;     // R = B n rows per level, Rp = R rounded up to 128
  int sel[GLOM_CT_MAX_SEL];
  float tau;
  ContrastiveStrides sa, sb;
};
struct ContrastiveLayout {
  // saved for the backward: bf16 unit rows A, B (nsel, R, d); fp32 per row (nsel, Rp): 1/|z_a|, 1/|z_b|, the lse of both
  // directions (log2 units, relative to 1/tau) and G_rr - 1
  size_t a_off, b_off, inv_a_off, inv_b_off, m_a_off, m_b_off, dg_off, saved;
  // forward scratch: lse partial sums [GLOM_CT_MAX_SPLIT][nsel][Rp] per direction, s_rr, loss block partials
  size_t ea_off, eb_off, srr_off, part_off, scratch;
};
ContrastiveLayout contrastive_layout(const ContrastiveGeom& g);
int contrastive_forward(const ContrastiveGeom& g, const float* za, const float* zb, float* loss, void* saved, void* scratch,
                        EncodeTiledFn enc, int num_sms, cudaStream_t st, int* launches, char* err, size_t errlen);
int contrastive_backward(const ContrastiveGeom& g, const float* za, const float* zb, const float* grad_loss, const void* saved,
                         float* dza, float* dzb, EncodeTiledFn enc, cudaStream_t st, int* launches, char* err, size_t errlen);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device and per function: remember, per device, the
// largest size already configured for one kernel (one instance of this per kernel template instantiation).
struct SmemOptIn {
  size_t configured[64] = {};
  std::mutex mu;
  template <typename K>
  cudaError_t ensure(K kernel, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lk(mu);
    if (bytes <= configured[dev]) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) configured[dev] = bytes;
    return e;
  }
};

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace glom
