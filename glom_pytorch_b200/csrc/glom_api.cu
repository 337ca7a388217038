// C ABI of libglom_b200.so (see include/glom_b200.h).  Host logic only: argument checking,
// buffer layout, the per-step launch sequence.  No device allocation, no stream sync.
#include "../../include/glom_b200.h"
#include "engine.h"

#include <mutex>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace glom {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;
static thread_local Profiler g_prof;

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

PackedLayout packed_layout(int d, int L, int precision) {
  const size_t es = precision == GLOM_B200_BF16 ? 2 : 4;
  const size_t G = 2 * (size_t)L - 1;
  PackedLayout p;
  size_t off = 0;
  p.w1_off = off; off = align_up(off + G * 4 * d * d * es, 1024);
  p.w2_off = off; off = align_up(off + (size_t)L * d * 8 * d * es, 1024);
  p.b1_off = off; off = align_up(off + G * 4 * d * 4, 1024);
  p.b2_off = off; off = align_up(off + (size_t)L * d * 4, 1024);
  p.total = off;
  return p;
}

WorkspaceLayout workspace_layout(const Geometry& g, int precision, int iters, int return_all) {
  WorkspaceLayout w{};
  const size_t state_elems = (size_t)g.rows * g.L * g.d;
  size_t off = 0;
  w.s32_off = off;
  w.s32_bytes = (return_all || iters == 0) ? 0 : state_elems * 4;
  off = align_up(off + w.s32_bytes, 1024);
  if (precision == GLOM_B200_BF16) {
    for (int i = 0; i < 2; ++i) { w.sb_off[i] = off; off = align_up(off + state_elems * 2, 1024); }
    for (int i = 0; i < 2; ++i) { w.sp_off[i] = off; off = align_up(off + (size_t)g.rows * (g.L - 1) * g.d * 2, 1024); }
    w.xb_off = off; off = align_up(off + (size_t)g.rows * g.d * 2, 1024);
    w.h_bytes = (size_t)((g.rows + 127) / 128 * 128) * g.G * 4 * g.d * 2;   // 128-row blocks, padded
    w.c_bytes = state_elems * 2;
    w.nsq_bytes = (size_t)g.rows * g.L * g.nparts * 4;
  } else {
    w.h_bytes = (size_t)g.rows * g.G * 4 * g.d * 4;
    w.c_bytes = state_elems * 4;
    w.nsq_bytes = 0;
  }
  w.h_off = off; off = align_up(off + w.h_bytes, 1024);
  w.c_off = off; off = align_up(off + w.c_bytes, 1024);
  for (int i = 0; i < 2; ++i) { w.nsq_off[i] = off; off = align_up(off + w.nsq_bytes, 1024); }
  w.attn_acc_off = off;
  w.attn_acc_bytes = (precision == GLOM_B200_BF16 && g.n > 576) ? (state_elems + (size_t)g.rows * g.L * 2) * 4 : 0;
  off = align_up(off + w.attn_acc_bytes, 1024);
  w.total = off > 0 ? off : 1024;
  return w;
}

static int check_cfg(const glom_b200_cfg* cfg) {
  if (!cfg) return fail(GLOM_B200_ERR_INVALID, "cfg is NULL");
  if (cfg->struct_size != sizeof(glom_b200_cfg))
    return fail(GLOM_B200_ERR_INVALID, "cfg.struct_size %u != %zu (ABI mismatch)", cfg->struct_size, sizeof(glom_b200_cfg));
  if (cfg->levels < 2) return fail(GLOM_B200_ERR_INVALID, "levels must be >= 2 (got %d)", cfg->levels);
  if (cfg->dim < 4 || cfg->dim % 4) return fail(GLOM_B200_ERR_INVALID, "dim must be a positive multiple of 4 (got %d)", cfg->dim);
  if (cfg->n < 1) return fail(GLOM_B200_ERR_INVALID, "n must be >= 1 (got %d)", cfg->n);
  if (cfg->precision != GLOM_B200_FP32 && cfg->precision != GLOM_B200_BF16)
    return fail(GLOM_B200_ERR_INVALID, "unknown precision %d", cfg->precision);
  if (cfg->precision == GLOM_B200_BF16 && cfg->dim % 64)
    return fail(GLOM_B200_ERR_INVALID, "bf16 (tcgen05) precision needs dim %% 64 == 0 (got %d); use fp32 precision", cfg->dim);
  if (cfg->mask_side < 0 || (cfg->mask_side > 0 && cfg->n % cfg->mask_side))
    return fail(GLOM_B200_ERR_INVALID, "mask_side %d does not tile n = %d", cfg->mask_side, cfg->n);
  return 0;
}

static Geometry make_geometry(const glom_b200_cfg* cfg, int batch) {
  Geometry g{};
  g.d = cfg->dim; g.L = cfg->levels; g.n = cfg->n; g.B = batch;
  g.rows = batch * cfg->n;
  g.G = 2 * g.L - 1;
  g.hidden = 4 * g.d;
  g.attend_self = cfg->attend_self; g.mask_side = cfg->mask_side; g.mask_d2_max = cfg->mask_d2_max;
  g.bn2 = (g.d % 256 == 0) ? 256 : (g.d % 128 == 0) ? 128 : 64;
  g.part_w = (g.bn2 == 256) ? 64 : g.bn2 / 2;   // columns per GEMM2 epilogue warp group (GemmCfg<1, BN>::PART_COLS)
  g.nparts = g.d / g.part_w;
  return g;
}

struct DeviceInfo { bool ok; int sms; };
static std::mutex g_mu;
static DeviceInfo g_dev[64];
static bool g_dev_known[64];
static EncodeTiledFn g_encode = nullptr;

static int device_info(DeviceInfo* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  if (dev < 0 || dev >= 64) return fail(GLOM_B200_ERR_CUDA, "device ordinal %d out of range", dev);
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_dev_known[dev]) {
    int major = 0, sms = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
    g_dev[dev].ok = (major == 10);
    g_dev[dev].sms = sms;
    g_dev_known[dev] = true;
  }
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr);
    if (e != cudaSuccess || qr != cudaDriverEntryPointSuccess || !fn)
      return fail(GLOM_B200_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable (%s)", cudaGetErrorString(e));
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *out = g_dev[dev];
  if (!out->ok) return fail(GLOM_B200_ERR_DEVICE, "device %d is not compute capability 10.x (sm_100a kernels only)", dev);
  return 0;
}

}  // namespace glom

using namespace glom;

extern "C" {

GLOM_B200_API int glom_b200_abi_version(void) { return GLOM_B200_ABI_VERSION; }

GLOM_B200_API const char* glom_b200_last_error(void) { return g_err; }

GLOM_B200_API int glom_b200_last_launch_count(void) { return g_launches; }

GLOM_B200_API int glom_b200_packed_weight_bytes(const glom_b200_cfg* cfg, size_t* out_bytes) {
  if (int r = check_cfg(cfg)) return r;
  if (!out_bytes) return fail(GLOM_B200_ERR_INVALID, "out_bytes is NULL");
  *out_bytes = packed_layout(cfg->dim, cfg->levels, cfg->precision).total;
  return 0;
}

GLOM_B200_API int glom_b200_pack_weights(const glom_b200_cfg* cfg, const glom_b200_weights_ref* w, void* packed, size_t packed_bytes,
                           void* stream) {
  if (int r = check_cfg(cfg)) return r;
  if (!w || w->struct_size != sizeof(glom_b200_weights_ref)) return fail(GLOM_B200_ERR_INVALID, "weights struct missing or wrong size");
  if (!w->bu_w1 || !w->bu_b1 || !w->bu_w2 || !w->bu_b2 || !w->td_w1 || !w->td_b1 || !w->td_w2 || !w->td_b2)
    return fail(GLOM_B200_ERR_INVALID, "a weight pointer is NULL");
  const PackedLayout pl = packed_layout(cfg->dim, cfg->levels, cfg->precision);
  if (!packed || packed_bytes < pl.total) return fail(GLOM_B200_ERR_WORKSPACE, "packed buffer: need %zu bytes, got %zu", pl.total, packed_bytes);
  if (reinterpret_cast<uintptr_t>(packed) % 1024) return fail(GLOM_B200_ERR_INVALID, "packed buffer must be 1024-byte aligned");
  g_launches = 0;
  cudaError_t e = launch_pack(cfg->dim, cfg->levels, cfg->precision, w->bu_w1, w->bu_b1, w->bu_w2, w->bu_b2, w->td_w1,
                              w->td_b1, w->td_w2, w->td_b2, packed, static_cast<cudaStream_t>(stream), &g_launches);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "pack_weights launch: %s", cudaGetErrorString(e));
  return 0;
}

GLOM_B200_API int glom_b200_workspace_bytes(const glom_b200_cfg* cfg, int batch, int iters, int return_all, size_t* out_bytes) {
  if (int r = check_cfg(cfg)) return r;
  if (batch < 1 || iters < 0 || !out_bytes) return fail(GLOM_B200_ERR_INVALID, "bad batch/iters/out_bytes");
  *out_bytes = workspace_layout(make_geometry(cfg, batch), cfg->precision, iters, return_all).total;
  return 0;
}

GLOM_B200_API int glom_b200_workspace_offset(const glom_b200_cfg* cfg, int batch, int iters, int return_all, int which,
                               size_t* out_offset, size_t* out_bytes) {
  if (int r = check_cfg(cfg)) return r;
  if (batch < 1 || iters < 0 || !out_offset || !out_bytes) return fail(GLOM_B200_ERR_INVALID, "bad arguments");
  const WorkspaceLayout w = workspace_layout(make_geometry(cfg, batch), cfg->precision, iters, return_all);
  switch (which) {
    case 0: *out_offset = w.h_off; *out_bytes = w.h_bytes; return 0;
    case 1: *out_offset = w.c_off; *out_bytes = w.c_bytes; return 0;
    case 2: *out_offset = w.nsq_off[0]; *out_bytes = w.nsq_bytes; return 0;
    default: return fail(GLOM_B200_ERR_INVALID, "unknown workspace buffer id %d", which);
  }
}

static int forward_impl(const glom_b200_cfg* cfg, const void* packed_weights, const float* tokens, const float* pos,
                        const float* state_in, const float* init_levels, float* state_out, int batch, int iters,
                        int return_all, void* workspace, size_t workspace_bytes, void* stream, int resume_parity);

GLOM_B200_API int glom_b200_forward(const glom_b200_cfg* cfg, const void* packed_weights, const float* tokens, const float* pos,
                      const float* state_in, const float* init_levels, float* state_out, int batch, int iters,
                      int return_all, void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(cfg, packed_weights, tokens, pos, state_in, init_levels, state_out, batch, iters, return_all, workspace,
                      workspace_bytes, stream, -1);
}

GLOM_B200_API int glom_b200_forward_resume(const glom_b200_cfg* cfg, const void* packed_weights, const float* tokens,
                                           const float* pos, const float* state_in, float* state_out, int batch, int iters,
                                           int return_all, void* workspace, size_t workspace_bytes, void* stream,
                                           int shadow_parity, int* out_shadow_parity) {
  if (!cfg || cfg->precision != GLOM_B200_BF16) return fail(GLOM_B200_ERR_INVALID, "forward_resume: bf16 engine only");
  if (!state_in || (shadow_parity != 0 && shadow_parity != 1) || iters < 1)
    return fail(GLOM_B200_ERR_INVALID, "forward_resume: need state_in, shadow_parity in {0, 1} and iters >= 1");
  const int r = forward_impl(cfg, packed_weights, tokens, pos, state_in, nullptr, state_out, batch, iters, return_all, workspace,
                             workspace_bytes, stream, shadow_parity);
  if (r == 0 && out_shadow_parity) *out_shadow_parity = (shadow_parity + iters) & 1;
  return r;
}

static int forward_impl(const glom_b200_cfg* cfg, const void* packed_weights, const float* tokens, const float* pos,
                        const float* state_in, const float* init_levels, float* state_out, int batch, int iters,
                        int return_all, void* workspace, size_t workspace_bytes, void* stream, int resume_parity) {
  if (int r = check_cfg(cfg)) return r;
  if (batch < 1 || iters < 0) return fail(GLOM_B200_ERR_INVALID, "batch must be >= 1 and iters >= 0");
  if (!packed_weights || !tokens || !pos || !state_out) return fail(GLOM_B200_ERR_INVALID, "a required pointer is NULL");
  if (!state_in && !init_levels) return fail(GLOM_B200_ERR_INVALID, "need state_in or init_levels");
  if (state_in == state_out) return fail(GLOM_B200_ERR_INVALID, "state_out must not alias state_in");
  if (reinterpret_cast<uintptr_t>(packed_weights) % 1024 || reinterpret_cast<uintptr_t>(workspace) % 1024)
    return fail(GLOM_B200_ERR_INVALID, "packed weights and workspace must be 1024-byte aligned");
  if (reinterpret_cast<uintptr_t>(tokens) % 16 || reinterpret_cast<uintptr_t>(pos) % 16 ||
      reinterpret_cast<uintptr_t>(state_out) % 16 || reinterpret_cast<uintptr_t>(state_in) % 16 ||
      reinterpret_cast<uintptr_t>(init_levels) % 16)
    return fail(GLOM_B200_ERR_INVALID, "tensor pointers must be 16-byte aligned");
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  const Geometry g = make_geometry(cfg, batch);
  const WorkspaceLayout wl = workspace_layout(g, cfg->precision, iters, return_all);
  if (!workspace || workspace_bytes < wl.total)
    return fail(GLOM_B200_ERR_WORKSPACE, "workspace: need %zu bytes, got %zu", wl.total, workspace_bytes);
  const PackedLayout pl = packed_layout(g.d, g.L, cfg->precision);
  const char* pw = static_cast<const char*>(packed_weights);
  char* ws = static_cast<char*>(workspace);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t slab = (size_t)g.rows * g.L * g.d;
  g_launches = 0;

  // where the fp32 master of step t lives
  float* wslab = reinterpret_cast<float*>(ws + wl.s32_off);
  auto loc = [&](int t) -> float* {
    if (return_all) return state_out + (size_t)t * slab;
    return ((iters - t) % 2 == 0) ? state_out : wslab;
  };

  if (cfg->precision == GLOM_B200_BF16) {
    __nv_bfloat16* sb[2] = {reinterpret_cast<__nv_bfloat16*>(ws + wl.sb_off[0]), reinterpret_cast<__nv_bfloat16*>(ws + wl.sb_off[1])};
    __nv_bfloat16* sp[2] = {reinterpret_cast<__nv_bfloat16*>(ws + wl.sp_off[0]), reinterpret_cast<__nv_bfloat16*>(ws + wl.sp_off[1])};
    float* nsq[2] = {reinterpret_cast<float*>(ws + wl.nsq_off[0]), reinterpret_cast<float*>(ws + wl.nsq_off[1])};
    __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(ws + wl.xb_off);
    // resumed call (glom_b200_forward_resume): the shadows / norm partials of state_in are the ones the previous call left
    // in buffer `p0`; the state prologue is skipped and step 0 reads the fp32 master straight from state_in
    const bool resume = resume_parity >= 0;
    const int p0 = resume ? resume_parity : 0;
    const bool s0_direct = resume || (!return_all && iters >= 1);
    cudaError_t e;
    if (resume) {
      e = launch_prep(g, nullptr, nullptr, pos, tokens, nullptr, nullptr, nullptr, xb, nullptr, st, &g_launches, &g_prof);
      if (e == cudaSuccess && return_all) {       // slab 0 of the return_all form is S_0 (:126)
        e = cudaMemcpyAsync(state_out, state_in, slab * sizeof(float), cudaMemcpyDeviceToDevice, st);
        ++g_launches;
      }
    } else {
      // S_0 as an fp32 slab is only materialised when it is part of the result (return_all slab 0, iters == 0): otherwise
      // step 0 reads the carried state from the caller's tensor, or init_levels broadcast over the rows
      e = launch_prep(g, state_in, init_levels, pos, tokens, s0_direct ? nullptr : loc(0), sb[0], sp[0], xb, nsq[0], st,
                      &g_launches, &g_prof);
    }
    if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "prep launch: %s", cudaGetErrorString(e));
    for (int t = 0; t < iters; ++t) {
      Bf16Buffers b{};
      b.s32_in = (s0_direct && t == 0) ? (state_in ? state_in : init_levels) : loc(t); b.s32_out = loc(t + 1);
      b.s32_in_bcast = (s0_direct && t == 0 && !state_in) ? 1 : 0;
      b.sb_in = sb[(t + p0) & 1]; b.sb_out = sb[(t + p0 + 1) & 1];
      b.sp_in = sp[(t + p0) & 1]; b.sp_out = sp[(t + p0 + 1) & 1];
      b.xb = xb;
      b.h = reinterpret_cast<__nv_bfloat16*>(ws + wl.h_off);
      b.attn_acc = wl.attn_acc_bytes ? reinterpret_cast<float*>(ws + wl.attn_acc_off) : nullptr;
      b.c = reinterpret_cast<__nv_bfloat16*>(ws + wl.c_off);
      b.nsq_in = nsq[(t + p0) & 1]; b.nsq_out = nsq[(t + p0 + 1) & 1];
      b.pos = pos;
      b.w1 = reinterpret_cast<const __nv_bfloat16*>(pw + pl.w1_off);
      b.w2 = reinterpret_cast<const __nv_bfloat16*>(pw + pl.w2_off);
      b.b1 = reinterpret_cast<const float*>(pw + pl.b1_off);
      b.b2 = reinterpret_cast<const float*>(pw + pl.b2_off);
      char msg[400] = "";
      const int r = step_bf16(g, b, t, g_encode, di.sms, st, &g_launches, msg, sizeof(msg), &g_prof);
      if (r) return fail(r == -1 ? GLOM_B200_ERR_INVALID : GLOM_B200_ERR_CUDA, "step %d: %s", t, msg);
    }
  } else {
    cudaError_t e = launch_broadcast_init(g, state_in, init_levels, loc(0), st, &g_launches, &g_prof);
    if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "init launch: %s", cudaGetErrorString(e));
    for (int t = 0; t < iters; ++t) {
      F32Buffers b{};
      b.s_in = loc(t); b.s_out = loc(t + 1);
      b.x = tokens; b.pos = pos;
      b.h = reinterpret_cast<float*>(ws + wl.h_off);
      b.c = reinterpret_cast<float*>(ws + wl.c_off);
      b.w1 = reinterpret_cast<const float*>(pw + pl.w1_off);
      b.w2 = reinterpret_cast<const float*>(pw + pl.w2_off);
      b.b1 = reinterpret_cast<const float*>(pw + pl.b1_off);
      b.b2 = reinterpret_cast<const float*>(pw + pl.b2_off);
      e = step_f32(g, b, st, &g_launches, &g_prof);
      if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "fp32 step %d launch: %s", t, cudaGetErrorString(e));
    }
  }
  g_err[0] = 0;
  return 0;
}

static int tok_kp(int patch) { return (3 * patch * patch + 63) / 64 * 64; }

GLOM_B200_API int glom_b200_tokenize_workspace_bytes(int batch, int height, int width, int patch, int dim, int precision,
                                                     size_t* out_bytes) {
  if (!out_bytes || batch < 1 || patch < 1 || dim < 1 || height < patch || width < patch || height % patch || width % patch)
    return fail(GLOM_B200_ERR_INVALID, "bad tokeniser geometry");
  if (precision == GLOM_B200_BF16) {
    const size_t rows = (size_t)batch * (height / patch) * (width / patch);
    *out_bytes = align_up(rows * tok_kp(patch) * 2, 1024) + align_up((size_t)dim * tok_kp(patch) * 2, 1024);
  } else {
    *out_bytes = 0;
  }
  return 0;
}

GLOM_B200_API int glom_b200_tokenize(const float* img, const float* weight, const float* bias, float* tokens, int batch, int height,
                       int width, int patch, int dim, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!img || !weight || !bias || !tokens) return fail(GLOM_B200_ERR_INVALID, "a required pointer is NULL");
  if (batch < 1 || patch < 1 || dim < 1 || height < patch || width < patch || height % patch || width % patch)
    return fail(GLOM_B200_ERR_INVALID, "image %dx%d is not a positive multiple of patch %d", height, width, patch);
  if (precision != GLOM_B200_FP32 && precision != GLOM_B200_BF16) return fail(GLOM_B200_ERR_INVALID, "unknown precision %d", precision);
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  g_launches = 0;
  if (precision == GLOM_B200_FP32) {
    cudaError_t e = launch_tokenize(img, weight, bias, tokens, batch, height, width, patch, dim, st, &g_launches, &g_prof);
    if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "tokenize launch: %s", cudaGetErrorString(e));
    return 0;
  }
  if (dim % 64) return fail(GLOM_B200_ERR_INVALID, "bf16 tokeniser needs dim %% 64 == 0 (got %d)", dim);
  size_t need = 0;
  glom_b200_tokenize_workspace_bytes(batch, height, width, patch, dim, precision, &need);
  if (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 1024)
    return fail(GLOM_B200_ERR_WORKSPACE, "tokeniser workspace: need %zu bytes 1024-aligned, got %zu", need, workspace_bytes);
  const int kp = tok_kp(patch);
  const int rows = batch * (height / patch) * (width / patch);
  __nv_bfloat16* patches = static_cast<__nv_bfloat16*>(workspace);
  __nv_bfloat16* wtok = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(workspace) + align_up((size_t)rows * kp * 2, 1024));
  ProfScope scope(&g_prof, PROF_TOKENIZE, st);
  cudaError_t e = launch_patchify_bf16(img, weight, patches, wtok, batch, height, width, patch, dim, kp, st, &g_launches);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "patchify launch: %s", cudaGetErrorString(e));
  char msg[300] = "";
  if (int r = tokenize_tc(patches, wtok, bias, tokens, rows, dim, kp, g_encode, di.sms, st, &g_launches, msg, sizeof(msg)))
    return fail(GLOM_B200_ERR_CUDA, "%s", msg);
  return 0;
}

GLOM_B200_API int glom_b200_tokenize_backward_workspace_bytes(int batch, int height, int width, int patch, int need_d_img,
                                                              size_t* out_bytes) {
  if (!out_bytes || batch < 1 || patch < 1 || height < patch || width < patch || height % patch || width % patch)
    return fail(GLOM_B200_ERR_INVALID, "tokeniser backward: bad arguments");
  *out_bytes = tokenize_backward_workspace_bytes(batch, height, width, patch, need_d_img);
  return 0;
}

GLOM_B200_API int glom_b200_tokenize_backward(const float* img, const float* weight, const float* d_tokens, float* d_weight,
                                              float* d_bias, float* d_img, int batch, int height, int width, int patch, int dim,
                                              void* workspace, size_t workspace_bytes, void* stream) {
  if (!img || !weight || !d_tokens) return fail(GLOM_B200_ERR_INVALID, "a required pointer is NULL");
  if (batch < 1 || patch < 1 || dim < 1 || height < patch || width < patch || height % patch || width % patch)
    return fail(GLOM_B200_ERR_INVALID, "image %dx%d is not a positive multiple of patch %d", height, width, patch);
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  const size_t need = tokenize_backward_workspace_bytes(batch, height, width, patch, d_img != nullptr);
  if ((d_weight || d_img) && (!workspace || workspace_bytes < need))
    return fail(GLOM_B200_ERR_WORKSPACE, "tokeniser backward workspace: need %zu bytes, got %zu", need, workspace_bytes);
  g_launches = 0;
  const cudaError_t e = tokenize_backward(img, weight, d_tokens, d_weight, d_bias, d_img, batch, height, width, patch, dim,
                                          workspace, static_cast<cudaStream_t>(stream), &g_launches);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "tokeniser backward: %s", cudaGetErrorString(e));
  return 0;
}

GLOM_B200_API int glom_b200_backward_workspace_bytes(const glom_b200_cfg* cfg, int batch, size_t* out_bytes) {
  if (int r = check_cfg(cfg)) return r;
  if (batch < 1 || !out_bytes) return fail(GLOM_B200_ERR_INVALID, "bad batch/out_bytes");
  *out_bytes = backward_layout(make_geometry(cfg, batch), cfg->precision).total;
  return 0;
}

GLOM_B200_API int glom_b200_backward(const glom_b200_cfg* cfg, const glom_b200_weights_ref* w, const float* tokens,
                                     const float* pos, const float* states, const float* grad_out,
                                     const glom_b200_grads* gr, int batch, int iters, int grad_all, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  if (int r = check_cfg(cfg)) return r;
  if (batch < 1 || iters < 0) return fail(GLOM_B200_ERR_INVALID, "batch must be >= 1 and iters >= 0");
  if (!w || w->struct_size != sizeof(glom_b200_weights_ref) || !gr || gr->struct_size != sizeof(glom_b200_grads))
    return fail(GLOM_B200_ERR_INVALID, "weights / grads struct missing or wrong size");
  if (!tokens || !pos || !states || !grad_out) return fail(GLOM_B200_ERR_INVALID, "a required pointer is NULL");
  if (!w->bu_w1 || !w->bu_b1 || !w->bu_w2 || !w->td_w1 || !w->td_b1 || !w->td_w2)
    return fail(GLOM_B200_ERR_INVALID, "a weight pointer is NULL");
  if (!gr->d_tokens || !gr->d_pos || !gr->d_bu_w1 || !gr->d_bu_b1 || !gr->d_bu_w2 || !gr->d_bu_b2 || !gr->d_td_w1 ||
      !gr->d_td_b1 || !gr->d_td_w2 || !gr->d_td_b2 || (!gr->d_state0 == !gr->d_init))
    return fail(GLOM_B200_ERR_INVALID, "gradient pointers: all MLP/token/pos outputs and exactly one of d_state0 / d_init");
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  const Geometry g = make_geometry(cfg, batch);
  const BackwardLayout wl = backward_layout(g, cfg->precision);
  if (!workspace || workspace_bytes < wl.total || reinterpret_cast<uintptr_t>(workspace) % 1024)
    return fail(GLOM_B200_ERR_WORKSPACE, "backward workspace: need %zu bytes 1024-aligned, got %zu", wl.total, workspace_bytes);
  BackwardArgs a{};
  a.tokens = tokens; a.pos = pos; a.states = states; a.grad_out = grad_out;
  a.bu_w1 = w->bu_w1; a.bu_b1 = w->bu_b1; a.bu_w2 = w->bu_w2; a.td_w1 = w->td_w1; a.td_b1 = w->td_b1; a.td_w2 = w->td_w2;
  a.d_tokens = gr->d_tokens; a.d_pos = gr->d_pos; a.d_state0 = gr->d_state0; a.d_init = gr->d_init;
  a.d_bu_w1 = gr->d_bu_w1; a.d_bu_b1 = gr->d_bu_b1; a.d_bu_w2 = gr->d_bu_w2; a.d_bu_b2 = gr->d_bu_b2;
  a.d_td_w1 = gr->d_td_w1; a.d_td_b1 = gr->d_td_b1; a.d_td_w2 = gr->d_td_w2; a.d_td_b2 = gr->d_td_b2;
  g_launches = 0;
  char msg[400] = "";
  if (int r = backward_run(g, a, cfg->precision, iters, grad_all, workspace, g_encode, di.sms,
                           static_cast<cudaStream_t>(stream), &g_launches, msg, sizeof(msg)))
    return fail(r == -1 ? GLOM_B200_ERR_INVALID : GLOM_B200_ERR_CUDA, "%s", msg);
  g_err[0] = 0;
  return 0;
}

GLOM_B200_API int glom_b200_islands(const float* states, int slabs, int side_h, int side_w, int levels, int dim, float threshold,
                                    float* cos_right, float* cos_down, float* agreement, int32_t* labels, int32_t* num_islands,
                                    void* stream) {
  if (!states || !cos_right || !cos_down || !agreement || !labels || !num_islands)
    return fail(GLOM_B200_ERR_INVALID, "a required pointer is NULL");
  if (slabs < 1 || slabs > 65535 || side_h < 1 || side_w < 1 || (long long)side_h * side_w > 8192 || levels < 1 ||
      levels > 65535 || dim < 4 || dim % 4)
    return fail(GLOM_B200_ERR_INVALID, "islands: need 1 <= slabs, levels <= 65535, side_h * side_w <= 8192, dim %% 4 == 0");
  if (reinterpret_cast<uintptr_t>(states) % 16) return fail(GLOM_B200_ERR_INVALID, "states must be 16-byte aligned");
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  g_launches = 0;
  cudaError_t e = launch_islands(states, slabs, side_h, side_w, levels, dim, threshold, cos_right, cos_down, agreement, labels,
                                 num_islands, static_cast<cudaStream_t>(stream), &g_launches);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "islands launch: %s", cudaGetErrorString(e));
  return 0;
}

static_assert(GLOM_B200_CONTRASTIVE_MAX_LEVELS == GLOM_CT_MAX_SEL, "selected-level capacity of the ABI and the kernels");

// The tensor-map encoder is a driver call and needs a current context.  A thread whose first CUDA work is this call (the
// autograd engine's worker thread running the backward) has none yet: cudaSetDevice makes the primary context current.
static int bind_current_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaSetDevice(dev);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  return 0;
}

static int contrastive_geometry(const glom_b200_contrastive_cfg* cfg, ContrastiveGeom* g) {
  if (!cfg) return fail(GLOM_B200_ERR_INVALID, "contrastive cfg is NULL");
  if (cfg->struct_size != sizeof(glom_b200_contrastive_cfg))
    return fail(GLOM_B200_ERR_INVALID, "contrastive cfg.struct_size %u != %zu (ABI mismatch)", cfg->struct_size,
                sizeof(glom_b200_contrastive_cfg));
  if (cfg->batch < 1 || cfg->n < 1 || cfg->levels < 1)
    return fail(GLOM_B200_ERR_INVALID, "contrastive: batch, n, levels must be >= 1");
  if (cfg->dim < 64 || cfg->dim % 64)
    return fail(GLOM_B200_ERR_INVALID, "contrastive: dim must be a positive multiple of 64 (tcgen05 operands), got %d", cfg->dim);
  const long long rows = (long long)cfg->batch * cfg->n;
  if (rows > (1LL << 30)) return fail(GLOM_B200_ERR_INVALID, "contrastive: batch * n = %lld rows is too many", rows);
  if (!(cfg->temperature >= 0.03f))
    return fail(GLOM_B200_ERR_INVALID, "contrastive: temperature must be >= 0.03 (got %g)", (double)cfg->temperature);
  if (cfg->num_selected < 1 || cfg->num_selected > GLOM_B200_CONTRASTIVE_MAX_LEVELS)
    return fail(GLOM_B200_ERR_INVALID, "contrastive: 1 <= num_selected <= %d", GLOM_B200_CONTRASTIVE_MAX_LEVELS);
  g->R = (int)rows;
  g->Rp = (int)((rows + 127) / 128 * 128);
  g->n = cfg->n; g->d = cfg->dim; g->L = cfg->levels; g->nsel = cfg->num_selected; g->tau = cfg->temperature;
  for (int i = 0; i < g->nsel; ++i) {
    const int l = cfg->selected[i];
    if (l < 0 || l >= cfg->levels) return fail(GLOM_B200_ERR_INVALID, "contrastive: level %d out of range [0, %d)", l, cfg->levels);
    for (int j = 0; j < i; ++j)
      if (cfg->selected[j] == l) return fail(GLOM_B200_ERR_INVALID, "contrastive: level %d selected twice", l);
    g->sel[i] = l;
  }
  g->sa = {cfg->stride_a[0], cfg->stride_a[1], cfg->stride_a[2]};
  g->sb = {cfg->stride_b[0], cfg->stride_b[1], cfg->stride_b[2]};
  return 0;
}

GLOM_B200_API int glom_b200_contrastive_workspace_bytes(const glom_b200_contrastive_cfg* cfg, size_t* saved_bytes,
                                                        size_t* scratch_bytes) {
  ContrastiveGeom g{};
  if (int r = contrastive_geometry(cfg, &g)) return r;
  if (!saved_bytes || !scratch_bytes) return fail(GLOM_B200_ERR_INVALID, "contrastive: output pointer is NULL");
  const ContrastiveLayout w = contrastive_layout(g);
  *saved_bytes = w.saved;
  *scratch_bytes = w.scratch;
  return 0;
}

GLOM_B200_API int glom_b200_contrastive_forward(const glom_b200_contrastive_cfg* cfg, const float* za, const float* zb,
                                                float* loss, void* saved, size_t saved_bytes, void* scratch,
                                                size_t scratch_bytes, void* stream) {
  ContrastiveGeom g{};
  if (int r = contrastive_geometry(cfg, &g)) return r;
  if (!za || !zb || !loss || !saved || !scratch) return fail(GLOM_B200_ERR_INVALID, "contrastive forward: a pointer is NULL");
  const ContrastiveLayout w = contrastive_layout(g);
  if (saved_bytes < w.saved || scratch_bytes < w.scratch)
    return fail(GLOM_B200_ERR_WORKSPACE, "contrastive forward: need %zu saved / %zu scratch bytes, got %zu / %zu", w.saved,
                w.scratch, saved_bytes, scratch_bytes);
  if (reinterpret_cast<uintptr_t>(saved) % 1024 || reinterpret_cast<uintptr_t>(scratch) % 1024)
    return fail(GLOM_B200_ERR_INVALID, "contrastive forward: saved and scratch must be 1024-byte aligned");
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  if (int r = bind_current_device()) return r;
  g_launches = 0;
  if (contrastive_forward(g, za, zb, loss, saved, scratch, g_encode, di.sms, static_cast<cudaStream_t>(stream), &g_launches,
                          g_err, sizeof(g_err)))
    return GLOM_B200_ERR_CUDA;
  return 0;
}

GLOM_B200_API int glom_b200_contrastive_backward(const glom_b200_contrastive_cfg* cfg, const float* za, const float* zb,
                                                 const float* grad_loss, const void* saved, size_t saved_bytes, float* dza,
                                                 float* dzb, void* stream) {
  ContrastiveGeom g{};
  if (int r = contrastive_geometry(cfg, &g)) return r;
  if (!za || !zb || !grad_loss || !saved || !dza || !dzb)
    return fail(GLOM_B200_ERR_INVALID, "contrastive backward: a pointer is NULL");
  if (dza == dzb || (const float*)dza == za || (const float*)dza == zb || (const float*)dzb == za || (const float*)dzb == zb)
    return fail(GLOM_B200_ERR_INVALID, "contrastive backward: dza / dzb must not alias the inputs or each other");
  const ContrastiveLayout w = contrastive_layout(g);
  if (saved_bytes < w.saved) return fail(GLOM_B200_ERR_WORKSPACE, "contrastive backward: need %zu saved bytes, got %zu", w.saved, saved_bytes);
  if (reinterpret_cast<uintptr_t>(saved) % 1024 || reinterpret_cast<uintptr_t>(dza) % 16 || reinterpret_cast<uintptr_t>(dzb) % 16)
    return fail(GLOM_B200_ERR_INVALID, "contrastive backward: saved must be 1024-byte, dza / dzb 16-byte aligned");
  DeviceInfo di{};
  if (int r = device_info(&di)) return r;
  if (int r = bind_current_device()) return r;
  g_launches = 0;
  if (contrastive_backward(g, za, zb, grad_loss, saved, dza, dzb, g_encode, static_cast<cudaStream_t>(stream), &g_launches,
                           g_err, sizeof(g_err)))
    return GLOM_B200_ERR_CUDA;
  return 0;
}

GLOM_B200_API int glom_b200_clock_probe(uint64_t* out_cycles_ns, int spin_us, void* stream) {
  if (!out_cycles_ns || spin_us < 1 || spin_us > 100000) return fail(GLOM_B200_ERR_INVALID, "clock probe: bad arguments");
  cudaError_t e = launch_clock_probe(reinterpret_cast<unsigned long long*>(out_cycles_ns), (unsigned long long)spin_us * 1000ull,
                                     static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "clock probe launch: %s", cudaGetErrorString(e));
  return 0;
}

GLOM_B200_API int glom_b200_kernel_clocks(double* mhz_by_kind, double* ms_by_kind, double* wait_frac, int kinds, int reset) {
  if (!mhz_by_kind || !ms_by_kind || kinds < 1) return fail(GLOM_B200_ERR_INVALID, "kernel clocks: bad arguments");
  unsigned long long acc[PROF_KINDS][8];
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = tc_kernel_clocks(&acc[0][0], reset != 0);
  if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "kernel clocks: %s", cudaGetErrorString(e));
  for (int i = 0; i < kinds; ++i) {
    const bool have = i < PROF_KINDS && acc[i][1] > 0;
    mhz_by_kind[i] = have ? 1e3 * (double)acc[i][0] / (double)acc[i][1] : 0.0;     // cycles per ns -> MHz
    ms_by_kind[i] = have ? 1e-6 * (double)acc[i][1] : 0.0;
    if (wait_frac)
      for (int j = 0; j < 6; ++j) wait_frac[6 * i + j] = have && acc[i][0] ? (double)acc[i][2 + j] / (double)acc[i][0] : 0.0;
  }
  return 0;
}

GLOM_B200_API int glom_b200_profile_begin(void) {
  g_prof.enabled = true;
  g_prof.used = 0;
  g_prof.spans.clear();
  return 0;
}

GLOM_B200_API int glom_b200_profile_end(double* ms_by_kind, int* launches_by_kind, int kinds) {
  if (!ms_by_kind || !launches_by_kind || kinds < 5) return fail(GLOM_B200_ERR_INVALID, "need room for at least 5 kinds");
  for (int i = 0; i < kinds; ++i) { ms_by_kind[i] = 0.0; launches_by_kind[i] = 0; }
  g_prof.enabled = false;
  for (const Profiler::Span& s : g_prof.spans) {
    cudaError_t e = cudaEventSynchronize(g_prof.ev[s.b]);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, g_prof.ev[s.a], g_prof.ev[s.b]);
    if (e != cudaSuccess) return fail(GLOM_B200_ERR_CUDA, "profile events: %s", cudaGetErrorString(e));
    if (s.kind >= kinds) continue;              // a caller built against an older header
    ms_by_kind[s.kind] += ms;
    launches_by_kind[s.kind] += 1;
  }
  g_prof.spans.clear();
  g_prof.used = 0;
  return 0;
}

}  // extern "C"
