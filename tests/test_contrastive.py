"""Column-contrastive loss (glom_pytorch_b200.column_contrastive_loss): the fp64 oracle against the definition and closed
forms (CPU), the C ABI's workspace sizing and the kernels' compiled form (CPU, nvcc), and the tcgen05 kernels against the
oracle (GPU).

GPU comparisons use ``check`` of tests/test_backward_reference.py on the (B, n, L, d) gradients: per tensor and per
slice (128-row block x level, level x 64 columns).  Thresholds are about twice the worst value measured on a B200
(1000 W power limit; profiles/r4_contrastive.txt), under the caps of 2e-3 (loss, relative) and 1e-2 (gradients):

  quantity                                   worst measured              threshold
  loss relative error                        1.8e-4 (R = 32), <= 1.3e-5 (R >= 588)   4e-4
  input gradients, per tensor / per slice    2.9e-3 / 2.9e-3 (R = 32, tau 0.03)  6e-3 / 6e-3
  aligned views, per slice / |O| scale       1.7e-3 (tau 1.0)            3.5e-3
  Glom end to end, per tensor / per slice    4.7e-3 (image) / 1.4e-3     9.5e-3 / 6e-3

The input-gradient error is the bf16 rounding of the unit vectors and of G in the two GEMMs: 1.66e-3 at every shape with
tau >= 0.1 and R >= 588, more at tau = 0.03 where the logits (and so their rounding) are three times larger, and
most at R = 32, where few rows average it.  The loss error
is the same rounding averaged over the rows, hence larger at tiny R.  The end-to-end image gradient sums the
contrastive gradient of every column through four backward steps and the tokeniser's fold; it is the one number near
a cap, and it is a whole-tensor figure of the image (no slice of any parameter exceeds 1.4e-3).
"""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle.contrastive_oracle import contrastive_naive, contrastive_reference

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL_LOSS = 4e-4
TOL_GRAD = dict(tol_tensor=6e-3, tol_slice=6e-3)
TOL_E2E = dict(tol_tensor=9.5e-3, tol_slice=6e-3)
TOL_ALIGNED = 3.5e-3


# ----------------------------------------------------------------------------- oracle (CPU)
@pytest.mark.parametrize("B,n,L,d,levels,tau,chunk", [(2, 3, 2, 5, (-1,), 0.1, 4), (3, 7, 3, 8, (0, 2), 0.03, 5),
                                                      (4, 5, 1, 6, (0,), 1.0, 64), (1, 6, 2, 4, (1,), 0.2, 4)])
def test_oracle_formulas_match_autograd_of_the_definition(B, n, L, d, levels, tau, chunk):
    g = torch.Generator().manual_seed(B * 100 + n)
    za = torch.randn(B, n, L, d, generator=g, dtype=torch.float64, requires_grad=True)
    zb = torch.randn(B, n, L, d, generator=g, dtype=torch.float64, requires_grad=True)
    ref = contrastive_reference(za, zb, levels, tau, grad_out=0.7, chunk=chunk)
    naive = contrastive_naive(za, zb, [l % L for l in levels], tau)
    dza, dzb = torch.autograd.grad(0.7 * naive, (za, zb))
    assert abs(ref["loss"].item() - naive.item()) <= 1e-12 * max(1.0, abs(naive.item()))
    for got, want in ((ref["dza"], dza), (ref["dzb"], dzb)):
        assert torch.allclose(got, want, rtol=0, atol=1e-12 * max(1.0, want.abs().max().item()))
    unsel = [l for l in range(L) if l not in [x % L for x in levels]]
    assert not ref["dza"][:, :, unsel].any() and not ref["dzb"][:, :, unsel].any()


def test_oracle_closed_forms():
    B, n, d, tau = 3, 4, 16, 0.1
    q, _ = torch.linalg.qr(torch.randn(d, d, dtype=torch.float64, generator=torch.Generator().manual_seed(1)))
    rows = q[: B * n] * (torch.rand(B * n, 1, dtype=torch.float64) * 3 + 0.5)       # orthogonal rows, any norms
    z = rows.reshape(B, n, 1, d)
    want = np.log(np.exp(1 / tau) + B * n - n) - 1 / tau
    assert abs(contrastive_reference(z, z, (0,), tau)["loss"].item() - want) < 1e-12
    za, zb = torch.randn(1, 9, 2, 8, dtype=torch.float64), torch.randn(1, 9, 2, 8, dtype=torch.float64)
    one = contrastive_reference(za, zb, (0, 1), 0.05)
    assert one["loss"].item() == 0.0 and not one["dza"].any() and not one["dzb"].any()
    za, zb = torch.randn(3, 5, 2, 8, dtype=torch.float64), torch.randn(3, 5, 2, 8, dtype=torch.float64)
    ab, ba = contrastive_reference(za, zb, (-1,), 0.1), contrastive_reference(zb, za, (-1,), 0.1)
    assert abs(ab["loss"].item() - ba["loss"].item()) < 1e-13
    assert torch.allclose(ab["dza"], ba["dzb"], rtol=0, atol=1e-15)


# ----------------------------------------------------------------------------- C ABI and compiled form (CPU)
def _ws(batch, n, dim, levels=(0, 1), L=2, tau=0.1):
    from glom_pytorch_b200 import _native
    cfg = _native.make_contrastive_cfg(batch, n, L, dim, levels, tau, (n * L * dim, L * dim, dim), (n * L * dim, L * dim, dim))
    return _native.contrastive_workspace_bytes(cfg)


def test_workspace_bytes_grow_linearly_in_rows():
    from glom_pytorch_b200 import _native
    for dim in (64, 512, 1024):
        for batch, n in ((2, 16), (32, 256), (128, 256), (3, 196)):
            s1, c1 = _ws(batch, n, dim)
            s2, c2 = _ws(2 * batch, n, dim)
            assert s1 > 0 and c1 > 0
            assert s2 <= 2 * s1 + 4096 and c2 <= 2 * c1 + 4096
            rows, rows_p = batch * n, -(-batch * n // 128) * 128
            assert s1 + c1 <= 2 * 2 * rows * dim * 2 + 2 * 100 * rows_p + 16384   # O(R d) bf16 + O(R) fp32, no R^2
    with pytest.raises(_native.GlomB200Error, match="multiple of 64"):
        _ws(2, 16, 96)
    lib = _native.load()
    cfg = _native.make_contrastive_cfg(2, 16, 2, 96, (0,), 0.1, (0, 0, 0), (0, 0, 0))
    import ctypes
    a, b = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.glom_b200_contrastive_workspace_bytes(ctypes.byref(cfg), ctypes.byref(a), ctypes.byref(b)) == -1
    for bad in (dict(tau=0.02), dict(levels=(0, 0)), dict(levels=(2,))):
        with pytest.raises(_native.GlomB200Error):
            _ws(2, 16, 64, **bad)


@pytest.mark.skipif(not shutil.which("nvcc") and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_kernels_compile_for_sm100a_without_spills_on_tensor_cores():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(ROOT, "glom_pytorch_b200", "csrc", "contrastive.cu")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "contrastive.o")
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                            src, "-o", obj], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        spills = [ln for ln in r.stderr.splitlines() if "spill" in ln]
        assert len(spills) >= 6 and all(" 0 bytes spill stores, 0 bytes spill loads" in ln for ln in spills), spills
        sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", obj], capture_output=True,
                              text=True).stdout
    funcs = {}
    for block in sass.split("Function : ")[1:]:
        funcs[block.split()[0]] = block.count("UTCHMMA")
    tc = {k: v for k, v in funcs.items() if "ct_kernel" in k}
    assert len(tc) == 2 and all(v > 0 for v in tc.values()), funcs


def test_non_cuda_input_raises():
    import glom_pytorch_b200 as G
    z = torch.randn(2, 4, 2, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        G.column_contrastive_loss(z, z)


# ----------------------------------------------------------------------------- GPU
def _inputs(B, n, L, d, seed, aligned=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    za = torch.randn(B, n, L, d, generator=g) * (1 + torch.rand(B, n, L, 1, generator=g))
    zb = za + 1e-2 * torch.randn(B, n, L, d, generator=g) if aligned else torch.randn(B, n, L, d, generator=g)
    return za.to(DEV), zb.to(DEV)


def _run(za, zb, levels, tau):
    import glom_pytorch_b200 as G
    a = za.clone().requires_grad_(True)
    b = zb.clone().requires_grad_(True)
    loss = G.column_contrastive_loss(a, b, levels=levels, temperature=tau)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), a.grad, b.grad


def _check(tag, got, ref, L, d, levels):
    from test_backward_reference import check, report
    failures, worst = check(got, ref, L, d, **TOL_GRAD)
    report(tag, worst)
    assert not failures, f"{tag}: {len(failures)} failures:\n" + "\n".join(failures[:20])
    sel = [l % L for l in levels]
    for k, g in got.items():
        unsel = [l for l in range(L) if l not in sel]
        assert not g[:, :, unsel].any(), f"{tag} {k}: unselected level gradient not exactly zero"


CASES = [  # B, n, L, d, levels, tau
    (2, 16, 2, 64, (-1,), 0.1),
    (2, 16, 2, 64, (0, 1), 0.03),
    (2, 16, 2, 64, (-1,), 1.0),
    (32, 256, 6, 512, (-2, -1), 0.1),
    (3, 196, 3, 192, (0, 2), 0.1),
    (3, 196, 3, 192, (0, 2), 0.03),
    (4, 576, 8, 1024, (-1,), 0.1),
    (4, 576, 8, 1024, (-1,), 1.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[f"B{c[0]}_n{c[1]}_L{c[2]}_d{c[3]}_lv{'_'.join(map(str, c[4]))}_t{c[5]}" for c in CASES])
def test_loss_and_grads_match_fp64_oracle(case):
    B, n, L, d, levels, tau = case
    za, zb = _inputs(B, n, L, d, seed=B * 1000 + d)
    loss, ga, gb = _run(za, zb, levels, tau)
    ref = contrastive_reference(za, zb, levels, tau)
    rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    print(f"contrastive {case}: loss {loss.item():.6f} rel err {rel:.2e}", flush=True)
    assert rel <= TOL_LOSS
    _check(f"contrastive {case}", {"levels": ga}, {"levels": ref["dza"]}, L, d, levels)
    _check(f"contrastive {case} zb", {"levels": gb}, {"levels": ref["dzb"]}, L, d, levels)


@pytest.mark.gpu
@pytest.mark.parametrize("tau", [0.03, 0.1, 1.0])
def test_aligned_views_relative_to_norm_of_o(tau):
    """zb = za + 1e-2 noise: p_rr -> 1 and the gradient is O_r - b_r of nearly equal terms; the error is measured against
    the scale of O / (tau R_total) / |z|, per 128-row block and level."""
    B, n, L, d, levels = 8, 100, 2, 256, (0, 1)
    za, zb = _inputs(B, n, L, d, seed=5, aligned=True)
    loss, ga, gb = _run(za, zb, levels, tau)
    ref = contrastive_reference(za, zb, levels, tau)
    assert abs(loss.item() - ref["loss"].item()) <= TOL_LOSS * abs(ref["loss"].item()) + 1e-6
    R = B * n
    worst = 0.0
    for z, g, r in ((za, ga, ref["dza"]), (zb, gb, ref["dzb"])):
        inv = 1.0 / torch.linalg.vector_norm(z.double(), dim=3)                # (B, n, L)
        x, xr, iv = g.double().reshape(R, L, d), r.reshape(R, L, d), inv.reshape(R, L)
        for r0 in range(0, R, 128):
            for lv in levels:
                o = torch.linalg.vector_norm(iv[r0:r0 + 128, lv]).item() / (tau * len(levels) * R)
                worst = max(worst, torch.linalg.norm(x[r0:r0 + 128, lv] - xr[r0:r0 + 128, lv]).item() / o)
    print(f"aligned tau={tau}: worst slice error / |O| scale {worst:.2e}", flush=True)
    assert worst <= TOL_ALIGNED


@pytest.mark.gpu
def test_large_batch_loss_and_sampled_row_blocks():
    B, n, L, d = 256, 256, 1, 512
    za, zb = _inputs(B, n, L, d, seed=11)
    loss, ga, gb = _run(za, zb, (0,), 0.1)
    blocks = [0, 1, 255, 256, 511]                                 # 128-row blocks, first / middle / last
    rows = torch.cat([torch.arange(k * 128, k * 128 + 128) for k in blocks]).to(DEV)
    ref = contrastive_reference(za, zb, (0,), 0.1, grad_rows=rows)
    rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    print(f"B=256: loss {loss.item():.6f} rel err {rel:.2e}", flush=True)
    assert rel <= TOL_LOSS
    pick = lambda t: t.reshape(B * n, L, d)[rows]                  # noqa: E731
    _check("B=256 sampled blocks", {"levels": pick(ga)}, {"levels": pick(ref["dza"])}, L, d, (0,))
    _check("B=256 sampled blocks zb", {"levels": pick(gb)}, {"levels": pick(ref["dzb"])}, L, d, (0,))


@pytest.mark.gpu
def test_single_image_gives_exact_zeros_and_input_checks():
    import glom_pytorch_b200 as G
    za, zb = _inputs(1, 200, 3, 128, seed=3)
    loss, ga, gb = _run(za, zb, (0, 2), 0.05)
    assert loss.item() == 0.0 and not ga.any() and not gb.any()
    za, zb = _inputs(2, 8, 2, 64, seed=4)
    with pytest.raises(ValueError, match="temperature"):
        G.column_contrastive_loss(za, zb, temperature=0.029)
    with pytest.raises(ValueError, match="twice"):
        G.column_contrastive_loss(za, zb, levels=(1, -1))
    with pytest.raises(ValueError, match="out of range"):
        G.column_contrastive_loss(za, zb, levels=(2,))
    with pytest.raises(ValueError, match="multiple of 64"):
        G.column_contrastive_loss(za[..., :32], zb[..., :32])
    with pytest.raises(ValueError, match="float32"):
        G.column_contrastive_loss(za.double(), zb.double())
    with pytest.raises(ValueError, match="same shape"):
        G.column_contrastive_loss(za, zb[:1])


@pytest.mark.gpu
def test_deterministic_and_cuda_graph_replay_bit_identical():
    import glom_pytorch_b200 as G
    za, zb = _inputs(6, 100, 3, 192, seed=8)
    first = _run(za, zb, (1, 2), 0.1)
    second = _run(za, zb, (1, 2), 0.1)
    for x, y in zip(first, second):
        assert torch.equal(x, y)
    a = za.clone().requires_grad_(True)
    b = zb.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                      # warm-up on the capture stream
        for _ in range(2):
            loss = G.column_contrastive_loss(a, b, levels=(1, 2), temperature=0.1)
            torch.autograd.grad(loss, (a, b))
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = G.column_contrastive_loss(a, b, levels=(1, 2), temperature=0.1)
        ga, gb = torch.autograd.grad(loss, (a, b))
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip((loss, ga, gb), first):
        assert torch.equal(x, y)
    with torch.no_grad():                                              # new inputs in place: the replay follows them
        a.copy_(zb); b.copy_(za)
    graph.replay()
    torch.cuda.synchronize()
    swapped = _run(zb, za, (1, 2), 0.1)
    for x, y in zip((loss, ga, gb), swapped):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_two_losses_at_different_steps_in_one_graph():
    import glom_pytorch_b200 as G
    T1, B, n, L, d = 13, 3, 64, 3, 128
    g = torch.Generator().manual_seed(21)
    xa = torch.randn(T1, B, n, L, d, generator=g).to(DEV).requires_grad_(True)
    xb = torch.randn(T1, B, n, L, d, generator=g).to(DEV).requires_grad_(True)
    loss = G.column_contrastive_loss(xa[6], xb[6], levels=(-1,)) + G.column_contrastive_loss(xa[12], xb[12], levels=(-2, -1))
    loss.backward()
    r6 = contrastive_reference(xa[6], xb[6], (-1,), 0.1)
    r12 = contrastive_reference(xa[12], xb[12], (-2, -1), 0.1)
    assert abs(loss.item() - (r6["loss"] + r12["loss"]).item()) <= TOL_LOSS * loss.item()
    for t, r, lv in ((6, r6, (-1,)), (12, r12, (-2, -1))):
        _check(f"two losses t={t}", {"levels": xa.grad[t]}, {"levels": r["dza"]}, L, d, lv)
        _check(f"two losses t={t} zb", {"levels": xb.grad[t]}, {"levels": r["dzb"]}, L, d, lv)
    others = [t for t in range(T1) if t not in (6, 12)]
    assert not xa.grad[others].any() and not xb.grad[others].any()


@pytest.mark.gpu
def test_end_to_end_glom_two_views_matches_fp64_chain():
    import glom_pytorch_b200 as G
    from oracle import glom_oracle_torch as OT
    from oracle.glom_oracle import synth_params
    from test_backward_reference import check, report
    d, L, isz, p, B, T, t = 64, 3, 32, 4, 3, 4, 3
    params = synth_params(d, L, isz, p, seed=2)
    m = G.Glom(dim=d, levels=L, image_size=isz, patch_size=p, precision="bf16")
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    m = m.to(DEV)
    rng = np.random.default_rng(9)
    img = rng.standard_normal((B, 3, isz, isz)).astype(np.float32)
    views = [img + 0.1 * rng.standard_normal(img.shape).astype(np.float32) for _ in range(2)]
    imgs = [torch.from_numpy(v).to(DEV).requires_grad_(True) for v in views]
    outs = [m(x, iters=T, return_all=True) for x in imgs]
    saved = [[s.detach().cpu() for s in o.grad_fn.saved_tensors[:3]] for o in outs]
    loss = G.column_contrastive_loss(outs[0][t], outs[1][t], levels=(-2, -1), temperature=0.1)
    loss.backward()
    torch.cuda.synchronize()
    got = {"img_a": imgs[0].grad, "img_b": imgs[1].grad, **{k: q.grad for k, q in m.named_parameters()}}
    ref_loss = contrastive_reference(outs[0][t], outs[1][t], (-2, -1), 0.1)
    assert abs(loss.item() - ref_loss["loss"].item()) <= TOL_LOSS * abs(ref_loss["loss"].item())
    P = {k: torch.from_numpy(v).double() for k, v in params.items()}
    ref = {}
    for i, (key, (tokens, pos, states)) in enumerate(zip(("dza", "dzb"), saved)):
        cot = torch.zeros((T + 1,) + tuple(outs[i].shape[1:]), dtype=torch.float64)
        cot[t] = ref_loss[key].cpu()
        r = OT.reference_grads(P, views[i], p, states.double(), tokens.double(), pos.double(), cot, return_all=True)
        for k, v in r.items():
            k2 = ("img_a", "img_b")[i] if k == "img" else k
            ref[k2] = ref[k2] + v if k2 in ref else v
    failures, worst = check(got, ref, L, d, **TOL_E2E)
    report("glom two views", worst)
    assert not failures, failures[:20]
