"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the C ABI
(glom_pytorch_b200._native -> libglom_b200.so).  /root/reference does not exist on the box: the
checkers are the committed golden vectors (outputs of the live reference) and the CPU oracle.

Tolerances
  fp32 engine vs reference fp32 golden : max-abs <= 1e-4 * max(1, |ref|max)   (summation order only)
  bf16 engine vs reference fp32 golden : per time step rel-Frobenius <= 1e-2 and
                                         max-abs <= 3e-2 * max(1, |ref|max)
      (SURVEY 8c: anchored on the reference's own autocast-bf16-vs-fp32 gap of 1.7e-3..3.8e-3 rel-Fro,
       6.3e-3 max-abs, with 2-3x head-room as hard caps)
  bf16 engine vs bf16-emulating oracle : rel-Frobenius <= 2e-3 (same roundings, different sum order)
"""
import os

import numpy as np
import pytest
import torch

import glom_pytorch_b200 as G
from glom_pytorch_b200 import _native
from golden_util import CASES, GOLDEN_DIR, inputs, load, model_kwargs
from oracle import glom_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def make_model(case, params, precision):
    m = G.Glom(**model_kwargs(case), precision=precision)
    sd = {k: torch.from_numpy(v) for k, v in params.items()}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k == "attention.non_local_mask" for k in missing)
    return m.to(DEV).eval()


def run_case(name, precision):
    case, params, outs = load(name)
    m = make_model(case, params, precision)
    got = {}
    with torch.no_grad():
        if case.get("frames"):
            levels = None
            for f in range(case["frames"]):
                img, _ = inputs(case, f)
                levels = m(torch.from_numpy(img).to(DEV), iters=case["iters"][f], levels=levels)
                got[f"out{f}"] = levels.cpu().numpy()
        else:
            img, lv = inputs(case)
            out = m(torch.from_numpy(img).to(DEV), iters=case["iters"],
                    levels=None if lv is None else torch.from_numpy(lv).to(DEV),
                    return_all=case.get("return_all", False))
            got["out0"] = out.cpu().numpy()
    torch.cuda.synchronize()
    return case, got, outs


def check_bf16(got, ref, what):
    assert got.shape == ref.shape, what
    assert np.isfinite(got).all(), what
    g, r = (got, ref) if got.ndim == 5 else (got[None], ref[None])
    for t in range(g.shape[0]):
        scale = max(1.0, float(np.abs(r[t]).max()))
        rel = np.linalg.norm(g[t] - r[t]) / max(np.linalg.norm(r[t]), 1e-30)
        mx = float(np.abs(g[t] - r[t]).max())
        assert rel <= 1e-2, (what, t, rel)
        assert mx <= 3e-2 * scale, (what, t, mx, scale)


@pytest.mark.parametrize("name", sorted(CASES))
def test_fp32_engine_matches_reference_golden(name):
    case, got, outs = run_case(name, "fp32")
    for k, ref in outs.items():
        g = outs.pick(k, got[k])
        assert g.shape == ref.shape
        scale = max(1.0, float(np.abs(ref).max()))
        assert np.abs(g - ref).max() <= 1e-4 * scale, (name, k)


@pytest.mark.parametrize("name", sorted(CASES))
def test_bf16_engine_matches_reference_golden(name):
    case, got, outs = run_case(name, "bf16")
    for k, ref in outs.items():
        check_bf16(outs.pick(k, got[k]), ref, (name, k))


def test_bf16_engine_matches_bf16_emulating_oracle():
    case, got, _ = run_case("mid_return_all", "bf16")
    _, params, _ = load("mid_return_all")
    img, _ = inputs(case)
    emu = O.glom_forward(params, img, patch_size=case["patch_size"], iters=case["iters"], return_all=True,
                         dtype=np.float32, emulate="bf16")
    for t in range(1, emu.shape[0]):
        rel = np.linalg.norm(got["out0"][t] - emu[t]) / np.linalg.norm(emu[t])
        assert rel <= 2e-3, (t, rel)


def test_zero_iters_returns_initial_state_and_fresh_tensor():
    case, params, _ = load("c1_return_all")
    m = make_model(case, params, "bf16")
    img, _ = inputs(case)
    x = torch.from_numpy(img).to(DEV)
    with torch.no_grad():
        s0 = m(x, iters=0)
        assert torch.equal(s0[0, 0], m.init_levels.data)
        lv = torch.randn(1, 16, 3, 64, device=DEV)
        out = m(x, iters=0, levels=lv)
        assert torch.equal(out, lv) and out.data_ptr() != lv.data_ptr()


def test_stage_buffers_hidden_and_consensus():
    """Single-stage checks through the workspace: after one bf16 step the hidden activations H and
    the consensus C left in the workspace match the oracle's (localises GEMM1 / attention faults)."""
    case, params, _ = load("mid_return_all")
    m = make_model(case, params, "bf16")
    img, _ = inputs(case)
    x = torch.from_numpy(img).to(DEV)
    with torch.no_grad():
        m(x, iters=1)
    torch.cuda.synchronize()
    B, n, L, d = case["batch"], 64, case["levels"], case["dim"]
    cfg = m.engine_cfg(n)
    ws = m._workspace
    off, nb = _native.workspace_offset(cfg, B, 1, False, 0)
    m128 = (B * n + 127) // 128
    H = ws[off:off + nb].view(torch.bfloat16).float().reshape(2 * L - 1, m128, 4 * d // 64, 128, 64)
    H = H.permute(1, 3, 0, 2, 4).reshape(m128 * 128, 2 * L - 1, 4 * d)[:B * n].cpu().numpy()   # (row, group, 4d)
    off, nb = _native.workspace_offset(cfg, B, 1, False, 1)
    C = ws[off:off + nb].view(torch.bfloat16).float().reshape(B, n, L, d).cpu().numpy()
    P = {k: v.astype(np.float32) for k, v in params.items()}
    tok = O.tokenize(img, P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"], case["patch_size"], emulate="bf16")
    S0 = np.broadcast_to(P["init_levels"], (B, n, L, d)).astype(np.float32)
    pos = P["pos_emb.weight"][:n][None, :, None, :]
    lwi = np.concatenate([tok[:, :, None, :], S0], 2)
    w1bu = P["bottom_up.net.1.weight"].reshape(L, 4 * d, d)
    b1bu = P["bottom_up.net.1.bias"].reshape(L, 4 * d)
    w1td = P["top_down.net.1.weight"].reshape(L - 1, 4 * d, d)
    b1td = P["top_down.net.1.bias"].reshape(L - 1, 4 * d)
    for l in range(L):
        a = O.bf16_round(lwi[:, :, l, :].reshape(B * n, d))
        want = O.gelu_erf(a @ O.bf16_round(w1bu[l]).T + b1bu[l])
        err = np.abs(H[:, 2 * l] - want).max()
        assert err <= 2e-2 * max(1.0, np.abs(want).max()), ("H bu", l, err)
    for l in range(L - 1):
        a = O.bf16_round((lwi[:, :, l + 2, :] + pos[:, :, 0, :]).reshape(B * n, d))
        want = O.gelu_erf(a @ O.bf16_round(w1td[l]).T + b1td[l])
        err = np.abs(H[:, 2 * l + 1] - want).max()
        assert err <= 2e-2 * max(1.0, np.abs(want).max()), ("H td", l, err)
    wantC = O.consensus(S0, False, None)
    assert np.abs(C - wantC).max() <= 2e-2 * max(1.0, np.abs(wantC).max())


def test_native_tokenizer_matches_oracle():
    case, params, _ = load("mid_nonsquare")
    m = make_model(case, params, "fp32")
    img, _ = inputs(case)
    with torch.no_grad():
        tok = m.tokens(torch.from_numpy(img).to(DEV)).cpu().numpy()
    want = O.tokenize(img.astype(np.float64), params["image_to_tokens.1.weight"].astype(np.float64),
                      params["image_to_tokens.1.bias"].astype(np.float64), case["patch_size"])
    assert tok.shape == want.shape and np.abs(tok - want).max() <= 1e-4


def test_tensor_core_tokenizer_matches_oracle():
    """bf16 precision: patchify + cast + tcgen05 GEMM vs the bf16-operand oracle (and the exact one)."""
    for name in ("mid_nonsquare", "c1_return_all"):
        case, params, _ = load(name)
        m = make_model(case, params, "bf16")
        img, _ = inputs(case)
        with torch.no_grad():
            tok = m.tokens(torch.from_numpy(img).to(DEV)).cpu().numpy()
        w, b = params["image_to_tokens.1.weight"], params["image_to_tokens.1.bias"]
        emu = O.tokenize(img, w, b, case["patch_size"], emulate="bf16")
        exact = O.tokenize(img.astype(np.float64), w.astype(np.float64), b.astype(np.float64), case["patch_size"])
        assert tok.shape == emu.shape
        assert np.abs(tok - emu).max() <= 1e-4
        assert np.abs(tok - exact).max() <= 2e-2 * max(1.0, np.abs(exact).max())


EDGE = [
    # dim, L, image_size, patch, img_hw, batch, iters, kwargs
    (192, 3, 24, 4, (24, 24), 2, 2, {}),                       # d % 128 != 0  -> 64-wide GEMM2 tiles, n = 36
    (320, 2, 16, 4, (16, 16), 3, 2, {}),                       # d = 5 x 64: attention output slices 256 + 64
    (64, 3, 224, 14, (140, 140), 3, 2, {}),                    # n = 100 of 256: ragged key padding, rows % 128 != 0
    (128, 3, 96, 4, (96, 96), 1, 2, {}),                       # n = 576: three key blocks, online max across blocks
    (128, 4, 64, 4, (64, 64), 1, 2, dict(local_consensus_radius=3)),   # radius mask on a 16 x 16 grid (n = 256)
    (64, 2, 8, 4, (8, 8), 1, 3, dict(consensus_self=True)),    # n = 4: a single 16-key block mostly padding
    (128, 2, 96, 4, (96, 96), 2, 1, dict(local_consensus_radius=2.5, consensus_self=True)),   # n = 576, mask + self, 5 query tiles (odd)
    (64, 2, 64, 2, (64, 64), 1, 2, {}),                        # n = 1024 > 576: tensor-core consensus in two key passes of 512
    (128, 2, 64, 2, (40, 64), 2, 1, dict(local_consensus_radius=0)),   # n = 640 of 1024: passes of 512 + 128 keys, two images
    (320, 2, 56, 2, (56, 56), 1, 2, dict(local_consensus_radius=6.5, consensus_self=True)),   # n = 784: passes 512 + 272, mask + self, d slices 256 + 64
    (64, 2, 80, 2, (80, 80), 1, 1, {}),                        # n = 1600: four key passes (512 x 3 + 64), 13 query tiles
]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("spec", EDGE, ids=[f"d{e[0]}_L{e[1]}_hw{e[4][0]}x{e[4][1]}_p{e[3]}" for e in EDGE])
def test_shape_edge_cases_against_oracle(spec, precision):
    """Ragged / extreme shapes the reference accepts (SURVEY 8b): checked against the fp64 CPU oracle."""
    dim, L, isz, p, hw, B, T, kw = spec
    params = O.synth_params(dim, L, isz, p, seed=3)
    m = G.Glom(dim=dim, levels=L, image_size=isz, patch_size=p, precision=precision, **kw)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    m = m.to(DEV).eval()
    rng = np.random.default_rng(5)
    img = rng.standard_normal((B, 3) + hw).astype(np.float32)
    n = (hw[0] // p) * (hw[1] // p)
    lv = (rng.standard_normal((B, n, L, dim)) * 2).astype(np.float32)
    with torch.no_grad():
        out = m(torch.from_numpy(img).to(DEV), iters=T, levels=torch.from_numpy(lv).to(DEV),
                return_all=True).cpu().numpy()
    ref = O.glom_forward(params, img, patch_size=p, iters=T, levels=lv, return_all=True, image_size=isz,
                         dtype=np.float64, **kw)
    if precision == "fp32":
        assert np.abs(out - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())
    else:
        check_bf16(out, ref, spec)


def test_key_passes_combine_exact_maximum_rows():
    """n = 784 > 576 columns with levels of rms ~300: the consensus runs in two key passes AND every row is on the
    exact-maximum path, so the passes' partial outputs sit on different stabilisers and are rescaled when combined
    (consensus_self: the diagonal dominates, the result is well conditioned -> standard bf16 tolerance)."""
    dim, L, isz, p = 128, 2, 56, 2                       # n = 784 columns
    params = O.synth_params(dim, L, isz, p, seed=13)
    rng = np.random.default_rng(14)
    img = rng.standard_normal((1, 3, isz, isz)).astype(np.float32)
    lv = (rng.standard_normal((1, 784, L, dim)) * 300).astype(np.float32)
    ref = O.glom_forward(params, img, patch_size=p, iters=2, levels=lv, return_all=True, image_size=isz,
                         dtype=np.float64, consensus_self=True)
    m = G.Glom(dim=dim, levels=L, image_size=isz, patch_size=p, consensus_self=True)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    m = m.to(DEV).eval()
    with torch.no_grad():
        out = m(torch.from_numpy(img).to(DEV), iters=2, levels=torch.from_numpy(lv).to(DEV), return_all=True).cpu().numpy()
    assert np.isfinite(out).all()
    check_bf16(out, ref, "key passes, exact-maximum rows")


@pytest.mark.parametrize("consensus_self", [True, False])
def test_large_magnitude_state_takes_the_exact_maximum_softmax(consensus_self):
    """The bf16 consensus kernel stabilises softmax with the bound |S_i| d^-1/2 on the logits instead of the row
    maximum; rows whose bound is out of range fall back to the exact-maximum pass.  Levels of rms ~300 (bound ~430 in
    log2 units) force that path.  With consensus_self the diagonal logit dominates by hundreds of units, softmax is
    one-hot and the result is well conditioned: standard bf16 tolerance against the oracle.  Without it the attention
    weights depend on logit differences far below bf16 resolution of the dot products (any bf16 implementation is
    ill-conditioned there), so only the fp32 engine is held to the oracle and the bf16 one to finiteness + scale."""
    dim, L, isz, p = 128, 3, 16, 2                       # n = 64 columns
    params = O.synth_params(dim, L, isz, p, seed=11)
    rng = np.random.default_rng(12)
    img = rng.standard_normal((2, 3, isz, isz)).astype(np.float32)
    lv = (rng.standard_normal((2, 64, L, dim)) * 300).astype(np.float32)
    ref = O.glom_forward(params, img, patch_size=p, iters=2, levels=lv, return_all=True, image_size=isz,
                         dtype=np.float64, consensus_self=consensus_self)
    outs = {}
    for precision in ("fp32", "bf16"):
        m = G.Glom(dim=dim, levels=L, image_size=isz, patch_size=p, precision=precision, consensus_self=consensus_self)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
        m = m.to(DEV).eval()
        with torch.no_grad():
            outs[precision] = m(torch.from_numpy(img).to(DEV), iters=2, levels=torch.from_numpy(lv).to(DEV),
                                return_all=True).cpu().numpy()
    assert np.abs(outs["fp32"] - ref).max() <= 1e-4 * np.abs(ref).max()
    assert np.isfinite(outs["bf16"]).all()
    if consensus_self:
        check_bf16(outs["bf16"], ref, "large-magnitude, consensus_self")
    else:
        rel = np.linalg.norm(outs["bf16"] - ref) / np.linalg.norm(ref)
        assert rel <= 0.25, rel


def test_cached_workspaces_side_streams_and_cuda_graph_replay_are_bit_stable():
    """Cross-call persistence (SURVEY 8 f3): packed weights and workspaces are cached per module; interleaving two
    models, changing the batch size, running on a side stream and replaying a captured CUDA graph of `forward`
    (the library never allocates or synchronises) must all reproduce the first results bit for bit."""
    torch.manual_seed(0)
    a = G.Glom(dim=256, levels=4, image_size=64, patch_size=8).to(DEV).eval()
    b = G.Glom(dim=128, levels=3, image_size=32, patch_size=4).to(DEV).eval()
    with torch.no_grad():
        xa = [torch.randn(B, 3, 64, 64, device=DEV) for B in (1, 3, 5)]
        xb = [torch.randn(B, 3, 32, 32, device=DEV) for B in (2, 4)]
        ra = [a(x, iters=3) for x in xa]
        rb = [b(x, iters=2) for x in xb]
        for i in (2, 0, 1):
            assert torch.equal(a(xa[i], iters=3), ra[i])
            if i < 2:
                assert torch.equal(b(xb[i], iters=2), rb[i])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            y = a(xa[1], iters=3)
        torch.cuda.current_stream().wait_stream(side)
        assert torch.equal(y, ra[1])
        static_x = xa[2].clone()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            a(static_x, iters=3)                        # warm-up on a capture-capable stream
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_y = a(static_x, iters=3)
        static_x.copy_(xa[0].expand_as(static_x))       # new input, replay
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y[0], ra[0][0])


# ----------------------------------------------------------------------------- BASELINE sizes
FULL = dict(dim=512, levels=6, image_size=224, patch_size=14)


def full_model(precision, seed=0, **kw):
    torch.manual_seed(seed)
    return G.Glom(**FULL, precision=precision, **kw).to(DEV).eval()


def test_config2_dims_against_cpu_oracle():
    """BASELINE configs[1] dims (d=512 L=6 N=256), B=2, 3 iterations: engine vs the fp32 CPU oracle."""
    m = full_model("bf16")
    g = torch.Generator().manual_seed(1)
    img = torch.randn(2, 3, 224, 224, generator=g)
    with torch.no_grad():
        out = m(img.to(DEV), iters=3, return_all=True).cpu().numpy()
        m32 = full_model("fp32")
        out32 = m32(img.to(DEV), iters=3, return_all=True).cpu().numpy()
    params = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    ref = O.glom_forward(params, img.numpy(), patch_size=14, iters=3, return_all=True, dtype=np.float32)
    assert np.abs(out32 - ref).max() <= 2e-4 * max(1.0, np.abs(ref).max())
    check_bf16(out, ref, "config2-dims")


def _oracle_params(m):
    return {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}


def test_config2_dims_all_12_iterations_against_cpu_oracle():
    """BASELINE configs[1] dims and iteration count (d=512 L=6 N=256, iters=12), B=2, return_all: every one of the 12
    time steps of the bf16 engine against the fp32 CPU oracle (existing bf16 tolerance per step)."""
    m = full_model("bf16")
    img = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(11))
    with torch.no_grad():
        out = m(img.to(DEV), iters=12, return_all=True).cpu().numpy()
    ref = O.glom_forward(_oracle_params(m), img.numpy(), patch_size=14, iters=12, return_all=True, dtype=np.float32)
    assert out.shape == ref.shape == (13, 2, 256, 6, 512)
    check_bf16(out, ref, "config2-dims x 12 iterations")


def test_config5_chain_12_10_6_against_cpu_oracle():
    """BASELINE configs[4] (README.md:105-111): three frames, iters 12 -> 10 -> 6 with the state carried, d=512 L=6
    N=256, B=2: 28 chained iterations.  The engine carries ITS OWN state between the calls, the oracle its own; every
    time step of every call is compared (drift over the whole chain stays inside the per-step bf16 tolerance)."""
    m = full_model("bf16")
    P = _oracle_params(m)
    g = torch.Generator().manual_seed(12)
    lv_e, lv_o = None, None
    for f, T in enumerate((12, 10, 6)):
        img = torch.randn(2, 3, 224, 224, generator=g)
        with torch.no_grad():
            all_e = m(img.to(DEV), iters=T, levels=lv_e, return_all=True)
        all_o = O.glom_forward(P, img.numpy(), patch_size=14, iters=T, levels=lv_o, return_all=True, dtype=np.float32)
        check_bf16(all_e.cpu().numpy(), all_o, f"chain frame {f} ({T} iterations)")
        lv_e, lv_o = all_e[-1].clone(), all_o[-1]


def test_config4_dims_against_cpu_oracle():
    """BASELINE configs[3] dims (d=1024 L=8 384/16 -> N=576, the lean consensus variant), B=1, 3 iterations, against the
    fp32 CPU oracle (not the engine's own fp32 path)."""
    torch.manual_seed(0)
    kw = dict(dim=1024, levels=8, image_size=384, patch_size=16)
    m = G.Glom(**kw, precision="bf16").to(DEV).eval()
    img = torch.randn(1, 3, 384, 384, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        out = m(img.to(DEV), iters=3, return_all=True).cpu().numpy()
    ref = O.glom_forward(_oracle_params(m), img.numpy(), patch_size=16, iters=3, return_all=True, dtype=np.float32)
    check_bf16(out, ref, "config4-dims vs oracle")


def test_radius_mask_and_consensus_self_at_config2_dims():
    """local_consensus_radius = 2.5 together with consensus_self=True at N=256 / d=512 (16 x 16 patch grid), B=1, 3
    iterations, bf16 and fp32 engines against the CPU oracle."""
    torch.manual_seed(3)
    m = G.Glom(**FULL, precision="bf16", consensus_self=True, local_consensus_radius=2.5).to(DEV).eval()
    m32 = G.Glom(**FULL, precision="fp32", consensus_self=True, local_consensus_radius=2.5).to(DEV).eval()
    m32.load_state_dict(m.state_dict())
    img = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(13))
    with torch.no_grad():
        out = m(img.to(DEV), iters=3, return_all=True).cpu().numpy()
        out32 = m32(img.to(DEV), iters=3, return_all=True).cpu().numpy()
    ref = O.glom_forward(_oracle_params(m), img.numpy(), patch_size=14, iters=3, return_all=True, dtype=np.float32,
                         consensus_self=True, local_consensus_radius=2.5)
    assert np.abs(out32 - ref).max() <= 2e-4 * max(1.0, np.abs(ref).max())
    check_bf16(out, ref, "radius 2.5 + consensus_self at N=256")
    # and the default (masked-diagonal) attention with a radius
    m2 = G.Glom(**FULL, precision="bf16", local_consensus_radius=1.5).to(DEV).eval()
    with torch.no_grad():
        out2 = m2(img.to(DEV), iters=2, return_all=True).cpu().numpy()
    ref2 = O.glom_forward(_oracle_params(m2), img.numpy(), patch_size=14, iters=2, return_all=True, dtype=np.float32,
                          local_consensus_radius=1.5)
    check_bf16(out2, ref2, "radius 1.5 at N=256")


def test_packed_weight_cache_follows_the_parameters():
    """ADVICE r1: in-place edits through .data do not bump _version.  train(): repacked every call; eval(): cached,
    dropped by load_state_dict / invalidate_packed()."""
    torch.manual_seed(5)
    m = G.Glom(dim=128, levels=3, image_size=32, patch_size=4).to(DEV)
    x = torch.randn(2, 3, 32, 32, device=DEV)
    with torch.no_grad():
        m.eval()
        a = m(x, iters=2)
        m.bottom_up.net[1].weight.data.mul_(0.5)
        assert torch.equal(m(x, iters=2), a)                # documented: stale until invalidated
        m.invalidate_packed()
        b = m(x, iters=2)
        assert not torch.equal(a, b)
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        sd["bottom_up.net.1.weight"].mul_(2.0)
        m.load_state_dict(sd)                               # back to the original weights
        assert torch.allclose(m(x, iters=2), a, rtol=0, atol=1e-6)
        m.train()
        c = m(x, iters=2)
        m.top_down.net[3].weight.data.mul_(0.25)
        assert not torch.equal(m(x, iters=2), c)            # training mode sees .data edits immediately


def test_hidden_of_mlp_group_0_is_reused_across_the_steps_of_a_call():
    """The bottom-up net of level 0 reads the tokens, which do not change during a call: its hidden activations are
    computed by the call's first step and re-read by the later ones.  Must be bit-identical to one-step calls chained on
    cloned states (every call's first step recomputes them; a clone is not resumed), also for a second call with a
    different image on the same module, which must not reuse the previous call's activations."""
    torch.manual_seed(31)
    m = G.Glom(dim=256, levels=3, image_size=32, patch_size=4).to(DEV).eval()
    a = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(32)).to(DEV)
    b = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(33)).to(DEV)
    with torch.no_grad():
        for img, iters in ((a, 4), (b, 3)):
            out = m(img, iters=iters, return_all=True)
            prev = None
            for t in range(1, iters + 1):
                prev = m(img, iters=1, levels=None if prev is None else prev.clone())
                assert torch.equal(out[t], prev), (iters, t)


def test_resumed_chain_and_staged_tokens_are_bit_identical_to_the_plain_calls():
    """SURVEY 8 row f3 (README.md:94-112, three frames, levels carried).  Passing the very tensor the previous call
    returned lets the engine resume from the bf16 shadows / norm partials it still holds (no state prologue), and
    `stage_tokens` computes the next frame's tokens on a side stream; both must give bit-identical states to plain calls
    on cloned inputs (which take the ordinary prologue), for even and odd step counts, and a modified carried tensor must
    fall back to the ordinary path."""
    torch.manual_seed(41)
    m = G.Glom(dim=256, levels=3, image_size=32, patch_size=4).to(DEV).eval()
    frames = [torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(50 + i)).to(DEV) for i in range(4)]
    with torch.no_grad():
        ref = None                                            # ordinary path: every carried state is a fresh clone
        refs = []
        for f, it in zip(frames, (5, 4, 3, 2)):
            ref = m(f.clone(), iters=it, levels=None if ref is None else ref.clone())
            refs.append(ref)
        launches_plain = m.last_launches
        lv = m(frames[0], iters=5)
        outs = [lv]
        for k, it in ((1, 4), (2, 3), (3, 2)):
            m.stage_tokens(frames[k])
            lv = m(frames[k], iters=it, levels=lv)            # resumed (odd -> even -> odd shadow parity) + staged tokens
            outs.append(lv)
        assert m.last_launches < launches_plain               # no state prologue kernel in the resumed call
        for a, b in zip(outs, refs):
            assert torch.equal(a, b)
        touched = outs[-1]
        touched.mul_(1.0)                                     # version bump: must not resume
        again = m(frames[0], iters=2, levels=touched)
        assert torch.equal(again, m(frames[0].clone(), iters=2, levels=touched.clone()))


def test_in_kernel_clock_samples():
    """Every tensor-core kernel samples (clock64, %globaltimer) around its working phase: after a forward the API
    reports a plausible SM clock and a positive in-kernel time for the three kernels of the step."""
    torch.manual_seed(3)
    m = G.Glom(dim=256, levels=3, image_size=32, patch_size=4).to(DEV).eval()
    img = torch.randn(2, 3, 32, 32, device=DEV)
    _native.kernel_clocks(reset=True)
    with torch.no_grad():
        m(img, iters=3)
    clk = _native.kernel_clocks(reset=True)
    for kind in ("attention", "gemm1_gelu", "gemm2_combine"):
        assert kind in clk, clk
        mhz, ms, _ = clk[kind]
        assert 300.0 < mhz < 3000.0 and ms > 0.0, (kind, mhz, ms)
    assert not _native.kernel_clocks(reset=False)          # reset: no samples left


def test_tokenizer_backward_matches_torch_autograd():
    """glom_b200_tokenize_backward (fp32 CUDA-core GEMMs + fold) against torch's autograd through Rearrange + Linear."""
    torch.manual_seed(5)
    for precision, tol in (("fp32", 2e-4), ("bf16", 2e-2)):
        m = G.Glom(dim=128, levels=2, image_size=32, patch_size=4, precision=precision).to(DEV).train()
        img = torch.randn(3, 3, 32, 32, device=DEV, requires_grad=True)
        lin = m.image_to_tokens[1]
        from glom_pytorch_b200.glom import _Tokenize
        tok = _Tokenize.apply(m, img, lin.weight, lin.bias)
        g = torch.randn_like(tok)
        gi, gw, gb = torch.autograd.grad(tok, (img, lin.weight, lin.bias), g)
        ref = lin(m.image_to_tokens[0](img))
        ri, rw, rb = torch.autograd.grad(ref, (img, lin.weight, lin.bias), g)
        assert (tok - ref).abs().max() <= tol * ref.abs().max()
        for a, b in ((gi, ri), (gw, rw), (gb, rb)):
            assert (a - b).abs().max() <= 2e-4 * b.abs().max().clamp_min(1.0), precision


def test_clock_probe_reports_a_plausible_sm_clock():
    buf = torch.zeros(2, dtype=torch.int64, device=DEV)
    _native.clock_probe(buf.data_ptr(), 200, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    cyc, ns = buf.tolist()
    assert ns >= 200_000 and 500 <= 1e3 * cyc / ns <= 2200, (cyc, ns)


def test_config2_full_size_properties():
    """Size-independent properties at BASELINE configs[1] (B=32, iters=12):
    (1) continuation additivity 12 == 6 + 6 bit-exactly (README.md:105-111);
    (2) batch independence: images 3..5 run alone give bit-identical columns;
    (3) bf16 tensor-core path vs fp32 CUDA-core path of the same engine: rel-Fro <= 1e-2;
    (4) the state contracts (random init): |S_12|max < |S_0|max."""
    m = full_model("bf16")
    g = torch.Generator().manual_seed(1)
    img = torch.randn(32, 3, 224, 224, generator=g).to(DEV)
    with torch.no_grad():
        a = m(img, iters=12)
        b = m(img, iters=6)
        b = m(img, iters=6, levels=b)
        assert torch.equal(a, b)
        sub = m(img[3:6], iters=12)
        assert torch.equal(sub, a[3:6])
        m32 = full_model("fp32")
        c = m32(img[:4], iters=12)
    assert torch.isfinite(a).all()
    rel = (torch.linalg.norm(a[:4] - c) / torch.linalg.norm(c)).item()
    assert rel <= 1e-2, rel
    assert a.abs().max().item() < m.init_levels.abs().max().item()


def test_config4_dims_small_batch():
    """BASELINE configs[3] dims (d=1024 L=8 384/16 -> N=576): bf16 engine vs its own fp32 path, B=1."""
    torch.manual_seed(0)
    kw = dict(dim=1024, levels=8, image_size=384, patch_size=16)
    m = G.Glom(**kw, precision="bf16").to(DEV).eval()
    m32 = G.Glom(**kw, precision="fp32").to(DEV).eval()
    m32.load_state_dict(m.state_dict())
    img = torch.randn(1, 3, 384, 384, generator=torch.Generator().manual_seed(2)).to(DEV)
    with torch.no_grad():
        a = m(img, iters=3, return_all=True).cpu().numpy()
        c = m32(img, iters=3, return_all=True).cpu().numpy()
    check_bf16(a, c, "config4-dims")


def test_permutation_equivariance_over_columns():
    """radius = 0: permuting patches (and pos_emb rows with them) permutes the output columns."""
    case, params, _ = load("mid_return_all")
    m = make_model(case, params, "bf16")
    img, _ = inputs(case)
    x = torch.from_numpy(img).to(DEV)
    perm = torch.randperm(64, generator=torch.Generator().manual_seed(3)).to(DEV)
    with torch.no_grad():
        tok = m.tokens(x)
        base = m(x, iters=3)
        # permuted problem through the C ABI directly: tokens and pos permuted together
        cfg = m.engine_cfg(64)
        stream = torch.cuda.current_stream().cuda_stream
        packed = m._packed_weights(cfg, x.device, stream)
        out = torch.empty_like(base)
        from glom_pytorch_b200.glom import _aligned_bytes
        ws = _aligned_bytes(_native.workspace_bytes(cfg, 2, 3, False), x.device)
        tp = tok[:, perm].contiguous()
        pp = m.pos_emb.weight.data[perm].contiguous()
        init = m.init_levels.data.contiguous()
        _native.forward(cfg, packed.data_ptr(), tp.data_ptr(), pp.data_ptr(), None, init.data_ptr(),
                        out.data_ptr(), 2, 3, False, ws.data_ptr(), ws.numel(), stream)
    torch.cuda.synchronize()
    assert torch.allclose(out, base[:, perm], rtol=0, atol=2e-3 * float(base.abs().max()))


def test_errors_are_reported_not_swallowed():
    case, params, _ = load("c1_return_all")
    m = make_model(case, params, "bf16")
    x = torch.randn(1, 3, 28, 28, device=DEV)
    with torch.no_grad(), pytest.raises(RuntimeError, match="levels must have shape"):
        m(x, levels=torch.zeros(2, 16, 3, 64, device=DEV))
    out = m(x, iters=1)                     # under autograd the loop is a differentiable op (f2)
    assert out.requires_grad and out.grad_fn is not None
    with torch.no_grad(), pytest.raises(IndexError):
        m(torch.randn(1, 3, 56, 56, device=DEV))


# ----------------------------------------------------------------------------- backward (SURVEY 8 f2)
from cases import GRAD_CASES, grad_inputs  # noqa: E402


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", sorted(GRAD_CASES))
def test_gradients_match_reference_autograd(name, precision):
    """loss = sum(out * cot): gradients of every parameter, of the image and of a carried-in state against the
    reference's autograd (golden fixtures from tests/golden/make_golden_grads.py).
    fp32 engine: max-abs <= 2e-4 * max(1, |ref|max) per tensor.  bf16 engine (bf16 forward, fp32 backward evaluated at
    the bf16 forward's states): rel-Frobenius <= 3e-2 per tensor."""
    import os
    case = GRAD_CASES[name]
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        ref = {k: z[k] for k in z.files}
    params = O.synth_params(case["dim"], case["levels"], case["image_size"], case["patch_size"], seed=case["param_seed"])
    m = G.Glom(dim=case["dim"], levels=case["levels"], image_size=case["image_size"], patch_size=case["patch_size"],
               consensus_self=case.get("consensus_self", False),
               local_consensus_radius=case.get("local_consensus_radius", 0), precision=precision)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    m = m.to(DEV)
    img, lv, cot = grad_inputs(case)
    img_t = torch.from_numpy(img).to(DEV).requires_grad_(True)
    lv_t = None if lv is None else torch.from_numpy(lv).to(DEV).requires_grad_(True)
    out = m(img_t, iters=case["iters"], levels=lv_t, return_all=case["return_all"])
    (out * torch.from_numpy(cot).to(DEV)).sum().backward()
    got = {"d_img": img_t.grad}
    if lv_t is not None:
        got["d_levels"] = lv_t.grad
    for k, p in m.named_parameters():
        got["d_" + k] = p.grad
    for k, r in ref.items():
        if k == "out":
            continue
        if got[k] is None:                      # unused parameter (e.g. init_levels when `levels` is given):
            assert not r.any(), k               # the reference leaves .grad None there too (stored as zeros)
            continue
        gk = got[k].detach().cpu().numpy()
        assert gk.shape == r.shape, (k, gk.shape, r.shape)
        if precision == "fp32":
            assert np.abs(gk - r).max() <= 2e-4 * max(1.0, np.abs(r).max()), (k, np.abs(gk - r).max())
        else:
            rel = np.linalg.norm(gk - r) / max(np.linalg.norm(r), 1e-30)
            assert rel <= 3e-2, (k, rel)


def test_readme_denoising_training_step_runs():
    """README.md:58-90: loss on all_levels[7, :, :, -1], backward reaches every parameter."""
    torch.manual_seed(0)
    m = G.Glom(dim=64, levels=3, image_size=28, patch_size=7).to(DEV)
    head = torch.nn.Linear(64, 7 * 7 * 3).to(DEV)
    img = torch.randn(2, 3, 28, 28, device=DEV)
    all_levels = m(img + torch.randn_like(img), return_all=True)
    assert all_levels.shape == (7, 2, 16, 3, 64)
    recon = head(all_levels[5, :, :, -1])
    loss = torch.nn.functional.mse_loss(recon, torch.zeros_like(recon))
    loss.backward()
    for k, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
        if k != "top_down.net.3.bias":
            assert p.grad.abs().max() > 0, k


@pytest.mark.parametrize("spec", [(256, 3, 32, 4, 3, 3), (512, 6, 224, 14, 2, 3)],
                         ids=["d256_L3_n64_rows192", "config2_dims_B2"])
def test_tensor_core_backward_matches_fp32_backward(spec):
    """bf16 engine (dim % 256 == 0): the MLP GEMMs of the backward run on tcgen05.  Checked against the engine's own fp32
    CUDA-core backward (itself pinned on the reference's autograd above): rel-Frobenius <= 3e-2 per gradient tensor."""
    dim, L, isz, p, B, T = spec
    torch.manual_seed(4)
    ms = {}
    for prec in ("fp32", "bf16"):
        torch.manual_seed(4)
        ms[prec] = G.Glom(dim=dim, levels=L, image_size=isz, patch_size=p, precision=prec).to(DEV)
    ms["bf16"].load_state_dict(ms["fp32"].state_dict())
    g = torch.Generator().manual_seed(9)
    img = torch.randn(B, 3, isz, isz, generator=g).to(DEV)
    n = (isz // p) ** 2
    cot = torch.randn(T + 1, B, n, L, dim, generator=g).to(DEV)
    grads = {}
    for prec, m in ms.items():
        x = img.clone().requires_grad_(True)
        out = m(x, iters=T, return_all=True)
        (out * cot).sum().backward()
        grads[prec] = {"img": x.grad, **{k: q.grad for k, q in m.named_parameters()}}
    for k, ref in grads["fp32"].items():
        got = grads["bf16"][k]
        assert got is not None and torch.isfinite(got).all(), k
        rel = (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()
        assert rel <= 3e-2, (k, rel)
