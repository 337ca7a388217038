"""ctypes binding of libglom_b200.so (include/glom_b200.h).  No torch types cross the ABI:
only raw device pointers, sizes and the stream handle.  There is no fallback: if the library
is missing or fails to load, importing the engine raises."""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GLOM_B200_LIB") or os.path.join(_PKG, "libglom_b200.so")   # override: A/B timing of builds

ABI_VERSION = 1
PRECISION = {"fp32": 0, "bf16": 1}

EXPORTS = (
    "glom_b200_abi_version", "glom_b200_last_error", "glom_b200_packed_weight_bytes",
    "glom_b200_pack_weights", "glom_b200_workspace_bytes", "glom_b200_forward", "glom_b200_forward_resume",
    "glom_b200_tokenize", "glom_b200_tokenize_workspace_bytes", "glom_b200_last_launch_count", "glom_b200_workspace_offset",
    "glom_b200_profile_begin", "glom_b200_profile_end",
    "glom_b200_backward", "glom_b200_backward_workspace_bytes",
    "glom_b200_tokenize_backward", "glom_b200_tokenize_backward_workspace_bytes",
    "glom_b200_clock_probe", "glom_b200_islands", "glom_b200_kernel_clocks",
    "glom_b200_contrastive_workspace_bytes", "glom_b200_contrastive_forward", "glom_b200_contrastive_backward",
)
PROFILE_KINDS = ("attention", "gemm1_gelu", "gemm2_combine", "prologue", "tokenize")


class Cfg(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32), ("dim", ctypes.c_int32), ("levels", ctypes.c_int32),
                ("n", ctypes.c_int32), ("attend_self", ctypes.c_int32), ("mask_side", ctypes.c_int32),
                ("mask_d2_max", ctypes.c_int32), ("precision", ctypes.c_int32)]


class WeightsRef(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32)] + [
        (k, ctypes.c_void_p) for k in ("bu_w1", "bu_b1", "bu_w2", "bu_b2", "td_w1", "td_b1", "td_w2", "td_b2")]


class Grads(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32)] + [
        (k, ctypes.c_void_p) for k in ("d_tokens", "d_pos", "d_state0", "d_init", "d_bu_w1", "d_bu_b1", "d_bu_w2",
                                       "d_bu_b2", "d_td_w1", "d_td_b1", "d_td_w2", "d_td_b2")]


CONTRASTIVE_MAX_LEVELS = 32


class ContrastiveCfg(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32), ("batch", ctypes.c_int32), ("n", ctypes.c_int32),
                ("levels", ctypes.c_int32), ("dim", ctypes.c_int32), ("num_selected", ctypes.c_int32),
                ("selected", ctypes.c_int32 * CONTRASTIVE_MAX_LEVELS), ("temperature", ctypes.c_float),
                ("stride_a", ctypes.c_int64 * 3), ("stride_b", ctypes.c_int64 * 3)]


class GlomB200Error(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library once; raise (never fall back) if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GlomB200Error(
            f"{LIB_PATH} not found: build it with `python -m glom_pytorch_b200.build` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the GLOM column update.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.glom_b200_abi_version.restype = i32
    lib.glom_b200_last_error.restype = ctypes.c_char_p
    lib.glom_b200_last_launch_count.restype = i32
    lib.glom_b200_packed_weight_bytes.argtypes = [ctypes.POINTER(Cfg), ctypes.POINTER(sz)]
    lib.glom_b200_pack_weights.argtypes = [ctypes.POINTER(Cfg), ctypes.POINTER(WeightsRef), vp, sz, vp]
    lib.glom_b200_workspace_bytes.argtypes = [ctypes.POINTER(Cfg), i32, i32, i32, ctypes.POINTER(sz)]
    lib.glom_b200_workspace_offset.argtypes = [ctypes.POINTER(Cfg), i32, i32, i32, i32,
                                               ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.glom_b200_forward.argtypes = [ctypes.POINTER(Cfg), vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
    lib.glom_b200_tokenize.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, sz, vp]
    lib.glom_b200_tokenize_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, ctypes.POINTER(sz)]
    lib.glom_b200_tokenize_workspace_bytes.restype = i32
    lib.glom_b200_profile_begin.restype = i32
    lib.glom_b200_profile_end.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i32), i32]
    lib.glom_b200_profile_end.restype = i32
    lib.glom_b200_backward_workspace_bytes.argtypes = [ctypes.POINTER(Cfg), i32, ctypes.POINTER(sz)]
    lib.glom_b200_backward_workspace_bytes.restype = i32
    lib.glom_b200_backward.argtypes = [ctypes.POINTER(Cfg), ctypes.POINTER(WeightsRef), vp, vp, vp, vp,
                                       ctypes.POINTER(Grads), i32, i32, i32, vp, sz, vp]
    lib.glom_b200_backward.restype = i32
    lib.glom_b200_islands.argtypes = [vp, i32, i32, i32, i32, i32, ctypes.c_float, vp, vp, vp, vp, vp, vp]
    lib.glom_b200_islands.restype = i32
    lib.glom_b200_tokenize_backward_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, ctypes.POINTER(sz)]
    lib.glom_b200_tokenize_backward_workspace_bytes.restype = i32
    lib.glom_b200_tokenize_backward.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, sz, vp]
    lib.glom_b200_tokenize_backward.restype = i32
    lib.glom_b200_forward_resume.argtypes = [ctypes.POINTER(Cfg), vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp, i32,
                                             ctypes.POINTER(i32)]
    lib.glom_b200_forward_resume.restype = i32
    lib.glom_b200_clock_probe.argtypes = [vp, i32, vp]
    lib.glom_b200_clock_probe.restype = i32
    lib.glom_b200_kernel_clocks.argtypes = [vp, vp, vp, i32, i32]
    lib.glom_b200_kernel_clocks.restype = i32
    cc = ctypes.POINTER(ContrastiveCfg)
    lib.glom_b200_contrastive_workspace_bytes.argtypes = [cc, ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.glom_b200_contrastive_workspace_bytes.restype = i32
    lib.glom_b200_contrastive_forward.argtypes = [cc, vp, vp, vp, vp, sz, vp, sz, vp]
    lib.glom_b200_contrastive_forward.restype = i32
    lib.glom_b200_contrastive_backward.argtypes = [cc, vp, vp, vp, vp, sz, vp, vp, vp]
    lib.glom_b200_contrastive_backward.restype = i32
    for f in ("glom_b200_packed_weight_bytes", "glom_b200_pack_weights", "glom_b200_workspace_bytes",
              "glom_b200_workspace_offset", "glom_b200_forward", "glom_b200_tokenize"):
        getattr(lib, f).restype = i32
    if lib.glom_b200_abi_version() != ABI_VERSION:
        raise GlomB200Error(f"libglom_b200 ABI {lib.glom_b200_abi_version()} != expected {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise GlomB200Error(f"glom_b200 error {rc}: {load().glom_b200_last_error().decode()}")


def make_cfg(dim, levels, n, attend_self, mask_side, mask_d2_max, precision):
    return Cfg(ctypes.sizeof(Cfg), dim, levels, n, int(bool(attend_self)), mask_side, mask_d2_max,
               PRECISION[precision])


def packed_weight_bytes(cfg):
    out = ctypes.c_size_t()
    check(load().glom_b200_packed_weight_bytes(ctypes.byref(cfg), ctypes.byref(out)))
    return out.value


def workspace_bytes(cfg, batch, iters, return_all):
    out = ctypes.c_size_t()
    check(load().glom_b200_workspace_bytes(ctypes.byref(cfg), batch, iters, int(return_all), ctypes.byref(out)))
    return out.value


def workspace_offset(cfg, batch, iters, return_all, which):
    off, nb = ctypes.c_size_t(), ctypes.c_size_t()
    check(load().glom_b200_workspace_offset(ctypes.byref(cfg), batch, iters, int(return_all), which,
                                            ctypes.byref(off), ctypes.byref(nb)))
    return off.value, nb.value


def pack_weights(cfg, ptrs, packed_ptr, packed_bytes, stream):
    w = WeightsRef(ctypes.sizeof(WeightsRef), *ptrs)
    check(load().glom_b200_pack_weights(ctypes.byref(cfg), ctypes.byref(w), packed_ptr, packed_bytes, stream))


def forward(cfg, packed_ptr, tokens_ptr, pos_ptr, state_in_ptr, init_ptr, out_ptr, batch, iters,
            return_all, ws_ptr, ws_bytes, stream):
    check(load().glom_b200_forward(ctypes.byref(cfg), packed_ptr, tokens_ptr, pos_ptr, state_in_ptr, init_ptr,
                                   out_ptr, batch, iters, int(return_all), ws_ptr, ws_bytes, stream))


def tokenize_workspace_bytes(batch, height, width, patch, dim, precision):
    out = ctypes.c_size_t()
    check(load().glom_b200_tokenize_workspace_bytes(batch, height, width, patch, dim, PRECISION[precision],
                                                    ctypes.byref(out)))
    return out.value


def tokenize(img_ptr, w_ptr, b_ptr, out_ptr, batch, height, width, patch, dim, precision, ws_ptr, ws_bytes, stream):
    check(load().glom_b200_tokenize(img_ptr, w_ptr, b_ptr, out_ptr, batch, height, width, patch, dim,
                                    PRECISION[precision], ws_ptr, ws_bytes, stream))


def last_launch_count():
    return load().glom_b200_last_launch_count()


def profile_begin():
    check(load().glom_b200_profile_begin())


def profile_end():
    """-> {kind: (milliseconds, launches)} for the kernels enqueued since profile_begin()."""
    k = len(PROFILE_KINDS)
    ms = (ctypes.c_double * k)()
    cnt = (ctypes.c_int * k)()
    check(load().glom_b200_profile_end(ms, cnt, k))
    return {name: (ms[i], cnt[i]) for i, name in enumerate(PROFILE_KINDS)}


def forward_resume(cfg, packed_ptr, tokens_ptr, pos_ptr, state_in_ptr, out_ptr, batch, iters, return_all, ws_ptr, ws_bytes,
                   stream, shadow_parity):
    """glom_b200_forward_resume: returns the shadow buffer index holding the new final state's shadows."""
    out_par = ctypes.c_int(0)
    check(load().glom_b200_forward_resume(ctypes.byref(cfg), packed_ptr, tokens_ptr, pos_ptr, state_in_ptr, out_ptr, batch, iters,
                                          int(bool(return_all)), ws_ptr, ws_bytes, stream, shadow_parity, ctypes.byref(out_par)))
    return out_par.value


def backward_workspace_bytes(cfg, batch):
    out = ctypes.c_size_t()
    check(load().glom_b200_backward_workspace_bytes(ctypes.byref(cfg), batch, ctypes.byref(out)))
    return out.value


def backward(cfg, weight_ptrs, tokens_ptr, pos_ptr, states_ptr, grad_out_ptr, grad_ptrs, batch, iters, grad_all,
             ws_ptr, ws_bytes, stream):
    """weight_ptrs: the 8 reference-layout tensors; grad_ptrs: dict of the Grads fields (None allowed for
    d_state0 / d_init)."""
    w = WeightsRef(ctypes.sizeof(WeightsRef), *weight_ptrs)
    g = Grads(ctypes.sizeof(Grads), *[grad_ptrs.get(k) for k, _ in Grads._fields_[1:]])
    check(load().glom_b200_backward(ctypes.byref(cfg), ctypes.byref(w), tokens_ptr, pos_ptr, states_ptr,
                                    grad_out_ptr, ctypes.byref(g), batch, iters, int(grad_all), ws_ptr, ws_bytes,
                                    stream))


def tokenize_backward_workspace_bytes(batch, h, w, patch, need_d_img):
    n = ctypes.c_size_t(0)
    check(load().glom_b200_tokenize_backward_workspace_bytes(batch, h, w, patch, int(bool(need_d_img)), ctypes.byref(n)))
    return n.value


def tokenize_backward(img_ptr, weight_ptr, d_tokens_ptr, d_weight_ptr, d_bias_ptr, d_img_ptr, batch, h, w, patch, dim,
                      ws_ptr, ws_bytes, stream):
    """Tokeniser backward; d_* pointers may be None (skipped); outputs are accumulated into."""
    check(load().glom_b200_tokenize_backward(img_ptr, weight_ptr, d_tokens_ptr, d_weight_ptr, d_bias_ptr, d_img_ptr, batch, h, w,
                                             patch, dim, ws_ptr, ws_bytes, stream))


def clock_probe(out_ptr, spin_us, stream):
    """Enqueue the SM clock probe: out_ptr -> 2 x uint64 device words {cycles, ns} (read after a synchronize)."""
    check(load().glom_b200_clock_probe(out_ptr, spin_us, stream))


def kernel_clocks(reset=True):
    """{kind: (SM MHz inside the kernels, in-kernel ms, [wait fractions of block 0: MMA lane on operands, MMA lane on a free
    accumulator, TMA lane on a free slot, epilogue warp 0 on an accumulator, epilogue warp 0 busy])} since the last reset."""
    k = len(PROFILE_KINDS)
    mhz, ms, wf = (ctypes.c_double * k)(), (ctypes.c_double * k)(), (ctypes.c_double * (6 * k))()
    check(load().glom_b200_kernel_clocks(mhz, ms, wf, k, int(bool(reset))))
    return {PROFILE_KINDS[i]: (mhz[i], ms[i], [round(wf[6 * i + j], 4) for j in range(6)]) for i in range(k) if ms[i] > 0}


def islands(states_ptr, slabs, side_h, side_w, levels, dim, threshold, cos_right_ptr, cos_down_ptr, agreement_ptr,
            labels_ptr, num_islands_ptr, stream):
    check(load().glom_b200_islands(states_ptr, slabs, side_h, side_w, levels, dim, threshold, cos_right_ptr, cos_down_ptr,
                                   agreement_ptr, labels_ptr, num_islands_ptr, stream))


def make_contrastive_cfg(batch, n, levels, dim, selected, temperature, stride_a, stride_b):
    """stride_a / stride_b: element strides of the two (B, n, L, d) inputs over (B, n, L)."""
    if len(selected) > CONTRASTIVE_MAX_LEVELS:
        raise ValueError(f"at most {CONTRASTIVE_MAX_LEVELS} levels can be selected")
    sel = (ctypes.c_int32 * CONTRASTIVE_MAX_LEVELS)(*selected)
    return ContrastiveCfg(ctypes.sizeof(ContrastiveCfg), batch, n, levels, dim, len(selected), sel, float(temperature),
                          (ctypes.c_int64 * 3)(*stride_a), (ctypes.c_int64 * 3)(*stride_b))


def contrastive_workspace_bytes(cfg):
    """-> (saved bytes, scratch bytes) of glom_b200_contrastive_forward."""
    saved, scratch = ctypes.c_size_t(), ctypes.c_size_t()
    check(load().glom_b200_contrastive_workspace_bytes(ctypes.byref(cfg), ctypes.byref(saved), ctypes.byref(scratch)))
    return saved.value, scratch.value


def contrastive_forward(cfg, za_ptr, zb_ptr, loss_ptr, saved_ptr, saved_bytes, scratch_ptr, scratch_bytes, stream):
    check(load().glom_b200_contrastive_forward(ctypes.byref(cfg), za_ptr, zb_ptr, loss_ptr, saved_ptr, saved_bytes,
                                               scratch_ptr, scratch_bytes, stream))


def contrastive_backward(cfg, za_ptr, zb_ptr, grad_loss_ptr, saved_ptr, saved_bytes, dza_ptr, dzb_ptr, stream):
    check(load().glom_b200_contrastive_backward(ctypes.byref(cfg), za_ptr, zb_ptr, grad_loss_ptr, saved_ptr, saved_bytes,
                                                dza_ptr, dzb_ptr, stream))
