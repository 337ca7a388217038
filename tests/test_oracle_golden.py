"""Pin the CPU oracle against every golden vector produced by the live reference
(tests/golden/make_golden.py).  fp64 oracle vs fp32 reference: <= 2e-5 max-abs relative
to the state scale (the reference itself is only fp32-accurate)."""
import os

import numpy as np
import pytest

from cases import GRAD_CASES, grad_inputs
from golden_util import CASES, GOLDEN_DIR, inputs, load
from oracle import glom_oracle as O

TOL = 2e-5


def _run(case, params, frame=0, levels=None, iters=None, dtype=np.float64, emulate=None):
    img, lv = inputs(case, frame)
    if levels is None:
        levels = lv
    return O.glom_forward(params, img, patch_size=case["patch_size"],
                          iters=case["iters"] if iters is None else iters, levels=levels,
                          return_all=case.get("return_all", False),
                          consensus_self=case.get("consensus_self", False),
                          local_consensus_radius=case.get("local_consensus_radius", 0),
                          image_size=case["image_size"], dtype=dtype, emulate=emulate)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_golden(name):
    case, params, outs = load(name)
    if case.get("frames"):
        levels = None
        for f in range(case["frames"]):
            got = _run(case, params, frame=f, levels=levels, iters=case["iters"][f])
            ref = outs[f"out{f}"]
            assert got.shape == ref.shape
            scale = max(1.0, float(np.abs(ref).max()))
            assert np.abs(got - ref).max() <= TOL * scale
            levels = got
    else:
        got = outs.pick("out0", _run(case, params))
        ref = outs["out0"]
        assert got.shape == ref.shape
        scale = max(1.0, float(np.abs(ref).max()))
        assert np.abs(got - ref).max() <= TOL * scale


def test_oracle_fp32_close_to_fp64():
    case, params, outs = load("mid_return_all")
    a = outs.pick("out0", _run(case, params, dtype=np.float32))
    assert np.abs(a - outs["out0"]).max() <= 1e-4


def test_bf16_emulation_within_autocast_gap():
    """The bf16-operand emulation (what the tensor-core engine computes) must stay inside the
    tolerance the GPU parity tests use: rel-Fro <= 1e-2, max-abs <= 3e-2 per time step."""
    case, params, outs = load("mid_return_all")
    a = outs.pick("out0", _run(case, params, dtype=np.float32, emulate="bf16"))
    ref = outs["out0"]
    for t in range(1, ref.shape[0]):
        rel = np.linalg.norm(a[t] - ref[t]) / np.linalg.norm(ref[t])
        assert rel <= 1e-2, (t, rel)
        assert np.abs(a[t] - ref[t]).max() <= 3e-2


def test_bf16_round_is_rne():
    x = np.array([1.0, 1.00390625, 1.005859375, -2.5, 3.0e38, 1e-40], dtype=np.float32)
    import torch
    want = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(O.bf16_round(x), want)
    r = np.random.default_rng(0).standard_normal(10000).astype(np.float32)
    assert np.array_equal(O.bf16_round(r),
                          torch.from_numpy(r).to(torch.bfloat16).to(torch.float32).numpy())


def test_continuation_additivity():
    """2+2 iterations with the state carried == 4 iterations (SURVEY section 0 [measured])."""
    case, params, _ = load("mid_return_all")
    img, _ = inputs(case)
    kw = dict(patch_size=case["patch_size"], image_size=case["image_size"])
    a = O.glom_forward(params, img, iters=4, **kw)
    b = O.glom_forward(params, img, iters=2, **kw)
    b = O.glom_forward(params, img, iters=2, levels=b, **kw)
    assert np.array_equal(a, b)


def test_radius_mask_matches_reference_semantics():
    m = O.radius_mask(4, 1.5)
    assert m.shape == (16, 16) and not m.diagonal().any()
    # (0,0) -> (1,1) is sqrt2 <= 1.5 (kept); (0,0) -> (0,2) is 2 > 1.5 (masked)
    assert not m[0, 5] and m[0, 2]


@pytest.mark.parametrize("name", sorted(CASES))
def test_torch_cpu_restatement_matches_reference_golden(name):
    """oracle/glom_oracle_torch.py (bench.py's multi-threaded CPU arm when the reference package is not importable)
    against the same golden outputs of the live reference; fp32 arithmetic: <= 1e-4 * scale."""
    import torch
    from oracle import glom_oracle_torch as OT
    case, params, outs = load(name)
    kw = dict(patch_size=case["patch_size"], consensus_self=case.get("consensus_self", False),
              local_consensus_radius=case.get("local_consensus_radius", 0))
    if case.get("frames"):
        levels = None
        for f in range(case["frames"]):
            img, _ = inputs(case, f)
            levels = OT.glom_forward(params, img, iters=case["iters"][f], levels=levels, **kw)
            ref = outs[f"out{f}"]
            assert np.abs(levels.numpy() - ref).max() <= 1e-4 * max(1.0, float(np.abs(ref).max()))
    else:
        img, lv = inputs(case)
        got = OT.glom_forward(params, img, iters=case["iters"], levels=lv, return_all=case.get("return_all", False),
                              **kw).numpy()
        got = outs.pick("out0", got)
        ref = outs["out0"]
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() <= 1e-4 * max(1.0, float(np.abs(ref).max()))


@pytest.mark.parametrize("name", sorted(GRAD_CASES))
def test_fp64_backward_reference_matches_reference_autograd(name):
    """oracle/glom_oracle_torch.py's gradient reference (fp64 autograd through one column_step per time step, walked
    backwards along its own fp64 forward, then the tokenizer's VJP) against the reference's autograd
    (tests/golden/make_golden_grads.py, same seeds): every stored gradient within 1e-6 * max(1, |ref|max)."""
    import torch
    from oracle import glom_oracle_torch as OT
    case = GRAD_CASES[name]
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        ref = {k: z[k] for k in z.files}
    params = O.synth_params(case["dim"], case["levels"], case["image_size"], case["patch_size"], seed=case["param_seed"])
    P = {k: torch.from_numpy(v).double() for k, v in params.items()}
    img, lv, cot = grad_inputs(case)
    cs, radius = case.get("consensus_self", False), case.get("local_consensus_radius", 0)
    states = OT.glom_forward(params, img, patch_size=case["patch_size"], iters=case["iters"], levels=lv,
                             return_all=True, consensus_self=cs, local_consensus_radius=radius, dtype=torch.float64)
    tokens = OT.tokenize(torch.from_numpy(img).double(), P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"],
                         case["patch_size"])
    mask = OT.radius_mask(case["image_size"] // case["patch_size"], radius) if radius > 0 else None
    got = OT.reference_grads(P, img, case["patch_size"], states, tokens, P["pos_emb.weight"][:tokens.shape[1]],
                             torch.from_numpy(cot), return_all=case["return_all"], consensus_self=cs, mask=mask,
                             carried_levels=lv is not None)
    checked = 0
    for k, r in ref.items():
        if k == "out":
            continue
        g = got.get(k[2:])
        if g is None:                           # init_levels when `levels` is carried in: no gradient reaches it
            assert k == "d_init_levels" and lv is not None and not r.any(), k
            continue
        g = g.numpy()
        assert g.shape == r.shape, (k, g.shape, r.shape)
        assert np.abs(g - r).max() <= 1e-6 * max(1.0, float(np.abs(r).max())), (k, np.abs(g - r).max())
        checked += 1
    assert checked == len(got)
