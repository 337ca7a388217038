"""Column-contrastive loss on the top levels of two views (the reference README's open Todo: "contrastive / consistency
regularization of top-ish levels"; DESIGN section 9).

The top-level embeddings of two views of the same images should agree column by column, with the columns of the other
images as negatives.  Per selected level, rows ``r = (b, i)``, ``R = B n`` of them::

    a_r = F.normalize(za[b, i, l]),  b_r = F.normalize(zb[b, i, l]),  s_rc = <a_r, b_c> / temperature
    cand(r) = {r} u {c : image(c) != image(r)}          (other columns of the same image are not pushed apart)
    l_r = 1/2 [ (logsumexp_{c in cand(r)} s_rc - s_rr) + (logsumexp_{c in cand(r)} s_cr - s_rr) ]

and the loss is the mean of ``l_r`` over the selected levels and rows.  The hot path is fused tcgen05 kernels
(``glom_b200_contrastive_*`` in include/glom_b200.h, csrc/contrastive.cu): bf16 unit vectors as GEMM operands with fp32
accumulation, fp32 softmax sums and gradients -- what torch autocast does to this loss -- and no R x R logit matrix.
"""
import torch

from . import _native

_scratch = {}          # (device index, stream) -> forward-only scratch buffer, grown on demand

MIN_TEMPERATURE = 0.03   # 2 log2(e) / tau <= 96: 1 / tau is a valid fixed softmax stabiliser in fp32


def _aligned(nbytes, device):
    """A 1024-byte aligned byte range of a fresh allocation: (owning tensor, pointer)."""
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    return buf, (buf.data_ptr() + 1023) // 1024 * 1024


def _scratch_ptr(nbytes, device):
    stream = torch.cuda.current_stream(device).cuda_stream
    key = (device.index, stream)
    hit = _scratch.get(key)
    if hit is None or hit[0].numel() < nbytes + 1024:
        hit = _aligned(nbytes, device)
        _scratch[key] = hit
    return hit[1]


def _strides(z):
    return (z.stride(0), z.stride(1), z.stride(2))


class _ColumnContrastive(torch.autograd.Function):
    @staticmethod
    def forward(ctx, za, zb, levels, temperature):
        B, n, L, d = za.shape
        cfg = _native.make_contrastive_cfg(B, n, L, d, levels, temperature, _strides(za), _strides(zb))
        saved_bytes, scratch_bytes = _native.contrastive_workspace_bytes(cfg)
        dev = za.device
        # per call, from the torch allocator: two losses alive in one graph keep their own saved state
        saved, saved_ptr = _aligned(saved_bytes, dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _native.contrastive_forward(cfg, za.data_ptr(), zb.data_ptr(), loss.data_ptr(), saved_ptr, saved_bytes,
                                        _scratch_ptr(scratch_bytes, dev), scratch_bytes,
                                        torch.cuda.current_stream(dev).cuda_stream)
        ctx.save_for_backward(za, zb)
        ctx.cfg, ctx.saved, ctx.saved_ptr, ctx.saved_bytes = cfg, saved, saved_ptr, saved_bytes
        return loss

    @staticmethod
    def backward(ctx, grad):
        za, zb = ctx.saved_tensors
        dev = za.device
        g = grad.detach().to(device=dev, dtype=torch.float32).contiguous()
        dza = torch.empty(za.shape, dtype=torch.float32, device=dev)
        dzb = torch.empty(zb.shape, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _native.contrastive_backward(ctx.cfg, za.data_ptr(), zb.data_ptr(), g.data_ptr(), ctx.saved_ptr, ctx.saved_bytes,
                                         dza.data_ptr(), dzb.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        return dza, dzb, None, None


def column_contrastive_loss(za, zb, *, levels=(-1,), temperature=0.1):
    """Column-contrastive (symmetric InfoNCE) loss between two views' column embeddings.

    za, zb: fp32 CUDA tensors of the same shape (B, n, L, d), e.g. ``all_levels[t]`` of two noised views of the same
    images (``model(img, return_all=True)``), so column i of image b corresponds in both; strided views such as
    ``all_a[7]`` are read in place.  levels: the levels to regularise (negative indices count from the top; no
    duplicates).  temperature: tau >= 0.03.  d must be a multiple of 64 (tcgen05 operands).

    Returns a 0-dim fp32 tensor, differentiable with respect to both inputs; unselected levels receive exactly zero
    gradient and B = 1 (no negatives) gives exactly zero.  Loss and gradients are bit-reproducible from call to call and
    capture in CUDA graphs (no host synchronisation).  Under ``dp.py`` each rank contrasts its own shard's columns: the
    negatives are not gathered across ranks.
    """
    for name, z in (("za", za), ("zb", zb)):
        if not isinstance(z, torch.Tensor) or not z.is_cuda:
            raise RuntimeError("glom_pytorch_b200.column_contrastive_loss runs on CUDA sm_100 only (no CPU fallback)")
        if z.dtype != torch.float32:
            raise ValueError(f"{name} must be float32 (got {z.dtype})")
        if z.dim() != 4:
            raise ValueError(f"{name} must be (B, n, L, d) (got shape {tuple(z.shape)})")
    if za.shape != zb.shape:
        raise ValueError(f"za and zb must have the same shape (got {tuple(za.shape)} and {tuple(zb.shape)})")
    if za.device != zb.device:
        raise ValueError(f"za and zb must be on the same device (got {za.device} and {zb.device})")
    B, n, L, d = za.shape
    if min(B, n, L, d) < 1:
        raise ValueError(f"empty input shape {tuple(za.shape)}")
    if d % 64:
        raise ValueError(f"d = {d} is not a multiple of 64 (tcgen05 operands); there is no CUDA-core path")
    if not float(temperature) >= MIN_TEMPERATURE:
        raise ValueError(f"temperature must be >= {MIN_TEMPERATURE} (got {temperature})")
    if isinstance(levels, int):
        levels = (levels,)
    sel = []
    for l in levels:
        li = int(l)
        if li != l or not -L <= li < L:
            raise ValueError(f"level {l} out of range for L = {L}")
        li %= L
        if li in sel:
            raise ValueError(f"level {l} selected twice")
        sel.append(li)
    if not sel:
        raise ValueError("no level selected")
    if len(sel) > _native.CONTRASTIVE_MAX_LEVELS:
        raise ValueError(f"at most {_native.CONTRASTIVE_MAX_LEVELS} levels can be selected")
    if za.stride(3) != 1:
        za = za.contiguous()
    if zb.stride(3) != 1:
        zb = zb.contiguous()
    return _ColumnContrastive.apply(za, zb, tuple(sel), float(temperature))
