/*
 * glom_b200.h -- C ABI of the B200-native GLOM column-update engine (libglom_b200.so).
 *
 * The reference (lucidrains/glom-pytorch) has no FFI: its hot path is the Python loop
 * glom_pytorch/glom_pytorch.py:131-145 calling GroupedFeedForward (:23-36) and
 * ConsensusAttention (:38-73).  This header is the boundary a maintainer would bind
 * instead of that loop (ctypes stub in INTEGRATION.md).  Conventions:
 *
 *   - plain C symbols, POD structs with a leading struct_size, no torch types;
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch's allocator);
 *     the library never allocates device memory, never synchronises the stream and
 *     never throws: 0 on success, a negative glom_b200_status otherwise, text via
 *     glom_b200_last_error() (thread-local);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*) of the CURRENT
 *     device (caller does cudaSetDevice / torch.cuda.device);
 *   - state layout is the reference's: (B, n, L, d) contiguous, d fastest, fp32
 *     (the reference carries the state in fp32 even under autocast, SURVEY 5.1).
 */
#ifndef GLOM_B200_H_
#define GLOM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLOM_B200_ABI_VERSION 1

#if defined(__GNUC__)
#define GLOM_B200_API __attribute__((visibility("default")))
#else
#define GLOM_B200_API
#endif

typedef enum glom_b200_status {
  GLOM_B200_OK = 0,
  GLOM_B200_ERR_INVALID = -1,     /* bad argument / unsupported shape              */
  GLOM_B200_ERR_WORKSPACE = -2,   /* workspace or packed buffer too small          */
  GLOM_B200_ERR_CUDA = -3,        /* a CUDA runtime/driver call failed             */
  GLOM_B200_ERR_DEVICE = -4       /* device is not sm_100 (no CPU / other-arch fallback) */
} glom_b200_status;

typedef enum glom_b200_precision {
  GLOM_B200_FP32 = 0,  /* CUDA-core fp32 path: matches the reference's fp32 forward     */
  GLOM_B200_BF16 = 1   /* tcgen05 path: bf16 operands, fp32 accumulate, fp32 state --
                          the arithmetic of the reference under torch.autocast(bf16)     */
} glom_b200_precision;

/* Static description of one Glom module + one call geometry.
 * Mirrors Glom.__init__ kwargs (glom_pytorch.py:78-87) and ConsensusAttention (:39-54). */
typedef struct glom_b200_cfg {
  uint32_t struct_size;   /* = sizeof(glom_b200_cfg)                                     */
  int32_t dim;            /* d                                                           */
  int32_t levels;         /* L  (>= 2: the reference cannot build top_down for L == 1)    */
  int32_t n;              /* columns (patches) of THIS call, n <= num_patches (:115)     */
  int32_t attend_self;    /* consensus_self (:85); 0 => diagonal logit := -5e-4 (:11)    */
  int32_t mask_side;      /* patches per grid row for the radius mask; 0 => no mask      */
  int32_t mask_d2_max;    /* logits with (dh^2+dw^2) > mask_d2_max are masked (:44-54,
                             :67-69).  The host derives it from non_local_mask.          */
  int32_t precision;      /* glom_b200_precision                                         */
} glom_b200_cfg;

/* Device pointers to the reference's parameters in state_dict layout (fp32, contiguous):
 *   bottom_up.net.1.weight (L*4d, d, 1)   .bias (L*4d)      glom_pytorch.py:29
 *   bottom_up.net.3.weight (L*d, 4d, 1)   .bias (L*d)       glom_pytorch.py:31
 *   top_down.*  same with L-1 groups                         glom_pytorch.py:105   */
typedef struct glom_b200_weights_ref {
  uint32_t struct_size;
  const float* bu_w1; const float* bu_b1; const float* bu_w2; const float* bu_b2;
  const float* td_w1; const float* td_b1; const float* td_w2; const float* td_b2;
} glom_b200_weights_ref;

GLOM_B200_API int glom_b200_abi_version(void);

/* Thread-local text of the last error returned on this thread ("" if none). */
GLOM_B200_API const char* glom_b200_last_error(void);

/* Bytes of the packed-weight buffer for cfg (depends on dim, levels, precision). */
GLOM_B200_API int glom_b200_packed_weight_bytes(const glom_b200_cfg* cfg, size_t* out_bytes);

/* Repack the reference-layout MLP weights into the engine layout (per level: W1 rows of
 * bottom-up and top-down interleaved, W2 K-concatenated [bu | td], biases summed where the
 * combine adds them).  Replaces nothing in the reference: it is the one-time cost of
 * swapping GroupedFeedForward's Conv1d weights (:29, :31) for GEMM operands. */
GLOM_B200_API int glom_b200_pack_weights(const glom_b200_cfg* cfg, const glom_b200_weights_ref* w,
                           void* packed, size_t packed_bytes, void* stream);

/* Workspace bytes glom_b200_forward needs for (cfg, batch, iters, return_all). */
GLOM_B200_API int glom_b200_workspace_bytes(const glom_b200_cfg* cfg, int batch, int iters,
                              int return_all, size_t* out_bytes);

/* The hot path: `iters` Jacobi column updates.  Replaces glom_pytorch.py:123-148
 * (state init/carry, the loop :131-145, hiddens/return_all :147-148).
 *
 *   tokens      (B, n, d) fp32   image_to_tokens(img)                     (:114)
 *   pos         (n, d)    fp32   pos_emb.weight[:n]                       (:117)
 *   state_in    (B, n, L, d) fp32 contiguous, or NULL                     (:123)
 *   init_levels (L, d)    fp32   used (broadcast) when state_in == NULL   (:124)
 *   state_out   return_all ? (iters+1, B, n, L, d) : (B, n, L, d), fp32; slab 0 of the
 *               return_all form is S_0 (:126).  Must not alias state_in.
 */
GLOM_B200_API int glom_b200_forward(const glom_b200_cfg* cfg, const void* packed_weights,
                      const float* tokens, const float* pos, const float* state_in,
                      const float* init_levels, float* state_out, int batch, int iters,
                      int return_all, void* workspace, size_t workspace_bytes, void* stream);

/* Cross-call persistence (SURVEY 8 row f3, README.md:94-112: levels carried from frame to frame).  Same as
 * glom_b200_forward with a carried-in state, for the case that `state_in` is bit for bit the FINAL state the previous
 * glom_b200_forward / _forward_resume call on this workspace wrote (same cfg, batch, and `pos`): the workspace then still
 * holds that state's bf16 shadows and norm partials in shadow buffer `shadow_parity` (0 after a plain forward with an even
 * number of steps, 1 after an odd one; in general what the previous _resume call returned), so the state prologue is
 * skipped and step 0 reads the fp32 master straight from `state_in`.  bf16 engine, iters >= 1.  *out_shadow_parity = the
 * buffer holding the new final state's shadows.  Passing a state that does not match the workspace gives wrong results;
 * the host side (glom.py) checks tensor identity and version before taking this path. */
GLOM_B200_API int glom_b200_forward_resume(const glom_b200_cfg* cfg, const void* packed_weights, const float* tokens,
                                           const float* pos, const float* state_in, float* state_out, int batch, int iters,
                                           int return_all, void* workspace, size_t workspace_bytes, void* stream,
                                           int shadow_parity, int* out_shadow_parity);

/* Tokeniser, the step before the loop (SURVEY 8f-1): replaces image_to_tokens
 * (glom_pytorch.py:94-97, call :114): patchify 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)'
 * fused with the Linear(3*p*p -> d).
 *   img (B, 3, H, W) fp32;  weight (d, 3*p*p) fp32;  bias (d) fp32;  tokens (B, n, d) fp32
 * precision GLOM_B200_FP32: one CUDA-core fp32 kernel, no workspace.
 * precision GLOM_B200_BF16: gather + cast to a zero-padded bf16 operand, then a tcgen05 GEMM with
 *   fp32 accumulation (what autocast does to this Linear); needs the workspace below, 1024-aligned. */
GLOM_B200_API int glom_b200_tokenize_workspace_bytes(int batch, int height, int width, int patch,
                                                     int dim, int precision, size_t* out_bytes);
GLOM_B200_API int glom_b200_tokenize(const float* img, const float* weight, const float* bias,
                       float* tokens, int batch, int height, int width, int patch,
                       int dim, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* Number of kernels the last glom_b200_forward / glom_b200_tokenize call on this thread
 * enqueued (bench.py reports it as gpu_launches). */
GLOM_B200_API int glom_b200_last_launch_count(void);

/* Diagnostics: byte offsets of intermediate buffers inside the workspace for the same
 * (cfg, batch, iters, return_all); tests use them to check single stages.
 * which: 0 = hidden activations H -- bf16 engine: 16 KB blocks [2L-1][ceil(rows/128)][4d/64][128][64]
 *            (group, 128-row block, 64-column block, row, column), fp32 engine: (rows, (2L-1)*4d);
 *        1 = consensus C (rows, L, d),
 *        2 = squared-norm partials. Returns GLOM_B200_ERR_INVALID for unknown ids. */
GLOM_B200_API int glom_b200_workspace_offset(const glom_b200_cfg* cfg, int batch, int iters, int return_all,
                               int which, size_t* out_offset, size_t* out_bytes);

/* Backward of the column update (SURVEY 8 row f2): gradients of glom_b200_forward's loop
 * (glom_pytorch.py:123-148) with respect to tokens, pos, the initial state (or init_levels) and the
 * eight MLP tensors, given dL/d(output).  Per-step intermediates are recomputed from the saved states.  precision
 * GLOM_B200_BF16 with dim % 256 == 0: the MLP and consensus GEMMs of the reverse pass run on tcgen05 tensor cores (bf16
 * operands, fp32 accumulation), softmax / normalisation / bias reductions in fp32 on CUDA cores; otherwise everything
 * is fp32 on CUDA cores.  All d_* buffers are ACCUMULATED into (zero them first); weights and their
 * gradients use the reference's state_dict layout.
 *   states    (iters+1, B, n, L, d) fp32: S_0..S_T as returned by forward(return_all=1)
 *   grad_out  (iters+1, B, n, L, d) if grad_all else (B, n, L, d)
 *   d_state0  (B, n, L, d) or NULL;  d_init (L, d) or NULL  (the one matching how the forward was started) */
typedef struct glom_b200_grads {
  uint32_t struct_size;
  float* d_tokens; float* d_pos; float* d_state0; float* d_init;
  float* d_bu_w1; float* d_bu_b1; float* d_bu_w2; float* d_bu_b2;
  float* d_td_w1; float* d_td_b1; float* d_td_w2; float* d_td_b2;
} glom_b200_grads;
GLOM_B200_API int glom_b200_backward_workspace_bytes(const glom_b200_cfg* cfg, int batch, size_t* out_bytes);
GLOM_B200_API int glom_b200_backward(const glom_b200_cfg* cfg, const glom_b200_weights_ref* weights,
                       const float* tokens, const float* pos, const float* states, const float* grad_out,
                       const glom_b200_grads* grads, int batch, int iters, int grad_all,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Backward of glom_b200_tokenize (image_to_tokens, glom_pytorch.py:94-97; SURVEY 8 rows f1 + f2), fp32 on CUDA cores:
 *   d_weight (dim, 3 patch^2) += d_tokens^T . patches,   d_bias (dim) += column sums of d_tokens,
 *   d_img (B, 3, H, W) += fold(d_tokens . weight).
 * Any of the three outputs may be NULL (skipped); they are ACCUMULATED into.  workspace: see _workspace_bytes
 * (need_d_img = whether d_img is requested). */
GLOM_B200_API int glom_b200_tokenize_backward_workspace_bytes(int batch, int height, int width, int patch, int need_d_img,
                                                              size_t* out_bytes);
GLOM_B200_API int glom_b200_tokenize_backward(const float* img, const float* weight, const float* d_tokens, float* d_weight,
                                              float* d_bias, float* d_img, int batch, int height, int width, int patch, int dim,
                                              void* workspace, size_t workspace_bytes, void* stream);

/* Per-kernel device timing for the roofline report (bench.py).  Between _begin and _end every
 * kernel the forward/tokenize calls of THIS thread enqueue is bracketed by CUDA events on the
 * launch stream (no synchronisation is added to the calls).  _end waits for those events and
 * returns summed milliseconds and launch counts per kernel kind:
 *   0 consensus attention, 1 GEMM1+GELU, 2 GEMM2+combine, 3 state prologue, 4 tokeniser.
 * `kinds` is the capacity of both arrays (>= 5; kinds beyond the capacity are dropped). */
#define GLOM_B200_PROFILE_KINDS 5
GLOM_B200_API int glom_b200_profile_begin(void);
GLOM_B200_API int glom_b200_profile_end(double* ms_by_kind, int* launches_by_kind, int kinds);

/* Island analytics on column states (SURVEY 8 row f4; the consumer of return_all the reference's README.md:34-36
 * describes: "all the level data across iterations for clustering, from which one can inspect for the theorized
 * islands").  states: `slabs` contiguous (side_h * side_w, levels, dim) fp32 state slabs, e.g. the (iters+1) * B slabs of
 * glom_b200_forward(return_all = 1).  Per (slab, level), on the patch grid (patch i = h * side_w + w):
 *   cos_right / cos_down (slabs, levels, n)  cosine similarity with the right / lower neighbour (0 where there is none)
 *   agreement            (slabs, levels, n)  mean cosine similarity with the existing 4-neighbours
 *   labels               (slabs, levels, n)  island id = smallest patch index of the 4-connected component in the graph
 *                                            of neighbour pairs with cosine similarity >= threshold
 *   num_islands          (slabs, levels)     number of such components
 * HBM-bound CUDA-core kernels (3 dot products per patch, no Gram matrix); all outputs device memory of the caller. */
GLOM_B200_API int glom_b200_islands(const float* states, int slabs, int side_h, int side_w, int levels, int dim, float threshold,
                                    float* cos_right, float* cos_down, float* agreement, int32_t* labels,
                                    int32_t* num_islands, void* stream);

/* Column-contrastive loss on selected levels of two views (the regulariser the reference's README lists as its open Todo,
 * "contrastive / consistency regularization of top-ish levels"; DESIGN section 9).  za, zb: (B, n, L, d) fp32 with d
 * contiguous and element strides given in the cfg.  Per selected level, rows r = (b, i), R = B n of them:
 *   a_r = za[b,i,l] / max(|za[b,i,l]|, 1e-12), b_r likewise;  s_rc = <a_r, b_c> / tau;
 *   candidates of r: {r} and every column of another image;
 *   l_r = 1/2 [ (lse_(c in cand r) s_rc - s_rr) + (lse_(c in cand r) s_cr - s_rr) ];  loss = mean over levels and rows.
 * tcgen05 kernels: bf16 unit vectors as GEMM operands, fp32 accumulation, fp32 softmax sums and gradients; no buffer of
 * R x R (or R x R / 128) elements exists.  Requires dim % 64 == 0, temperature >= 0.03 (then 1/tau is a valid fixed
 * stabiliser: 2 log2(e) / tau <= 96), 1 <= num_selected <= 32 distinct levels.  No atomics: results are bit-reproducible. */
#define GLOM_B200_CONTRASTIVE_MAX_LEVELS 32
typedef struct glom_b200_contrastive_cfg {
  uint32_t struct_size;   /* = sizeof(glom_b200_contrastive_cfg)                                  */
  int32_t batch, n, levels, dim;
  int32_t num_selected;   /* entries of `selected` in use                                          */
  int32_t selected[GLOM_B200_CONTRASTIVE_MAX_LEVELS];   /* level indices in [0, levels), distinct  */
  float temperature;      /* tau >= 0.03                                                           */
  int64_t stride_a[3];    /* element strides of za over (B, n, L); d has stride 1                  */
  int64_t stride_b[3];
} glom_b200_contrastive_cfg;

/* Bytes of the two caller-owned buffers (no device needed; both grow linearly in B n):
 *   saved:   what the backward reads (bf16 unit rows of both views, per-row fp32 norms / lse / diagonal terms); it must
 *            stay untouched from _forward until _backward of the same loss.  1024-byte aligned.
 *   scratch: forward-only (lse partial sums, loss partials); may be reused as soon as _forward's work has run.
 * GLOM_B200_ERR_INVALID for an unsupported cfg (dim % 64 != 0, tau < 0.03, bad level list, ...). */
GLOM_B200_API int glom_b200_contrastive_workspace_bytes(const glom_b200_contrastive_cfg* cfg, size_t* saved_bytes,
                                                        size_t* scratch_bytes);
/* loss: one fp32 device word, overwritten (not accumulated).  za / zb may alias each other. */
GLOM_B200_API int glom_b200_contrastive_forward(const glom_b200_contrastive_cfg* cfg, const float* za, const float* zb,
                                                float* loss, void* saved, size_t saved_bytes, void* scratch,
                                                size_t scratch_bytes, void* stream);
/* grad_loss: one fp32 device word (dL/dloss; read on the device, no host synchronisation).  dza, dzb: (B, n, L, d)
 * contiguous fp32, OVERWRITTEN with the full gradients (exact zeros at unselected levels); must not alias za, zb or each
 * other.  `saved` as filled by the matching _forward. */
GLOM_B200_API int glom_b200_contrastive_backward(const glom_b200_contrastive_cfg* cfg, const float* za, const float* zb,
                                                 const float* grad_loss, const void* saved, size_t saved_bytes, float* dza,
                                                 float* dzb, void* stream);

/* Measurement aid (bench.py): one device thread spins for `spin_us` microseconds of %globaltimer and writes
 * {SM cycles elapsed, nanoseconds elapsed} to out_cycles_ns[0..1] (device memory, 16 bytes): cycles / ns is the SM
 * clock in GHz the device actually ran at when the probe executed.  Enqueued on `stream`; the caller synchronises. */
GLOM_B200_API int glom_b200_clock_probe(uint64_t* out_cycles_ns, int spin_us, void* stream);

/* Measurement aid (bench.py): the SM clock the tensor-core kernels ACTUALLY ran at.  One thread of block 0 of every
 * tcgen05 kernel brackets the kernel's working phase with (clock64, %globaltimer); the deltas accumulate per kernel kind
 * (indices as in glom_b200_profile_end: 0 consensus, 1 GEMM1+GELU, 2 GEMM2+combine, 4 tokeniser GEMM).
 * Writes MHz (cycles per microsecond of in-kernel time) and the in-kernel milliseconds per kind since the last reset;
 * kinds without samples report 0.  wait_frac (may be NULL, else 6 doubles per kind): fractions of block 0's in-kernel
 * cycles that {the MMA lane waited for operands, the MMA lane waited for a free accumulator stage (consensus: TMEM buffer
 * or P), the TMA lane waited for a free ring slot, epilogue / softmax warp 0 waited for an accumulator, that warp was
 * busy (consensus: softmax work), consensus only: its output work}; filled by the diagnostic instantiations only
 * (environment variable GLOM_B200_WAIT_COUNTERS=1).
 * Synchronises the device; `reset` != 0 clears the accumulators. */
GLOM_B200_API int glom_b200_kernel_clocks(double* mhz_by_kind, double* ms_by_kind, double* wait_frac, int kinds, int reset);

#ifdef __cplusplus
}
#endif
#endif /* GLOM_B200_H_ */
