"""Pin the CPU oracle against every golden vector produced by the live reference
(tests/golden/make_golden.py).  fp64 oracle vs fp32 reference: <= 2e-5 max-abs relative
to the state scale (the reference itself is only fp32-accurate)."""
import numpy as np
import pytest

from golden_util import CASES, inputs, load
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
