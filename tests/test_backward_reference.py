"""The engine's backward against an fp64 reference evaluated on the exact states the backward consumes.

Each case runs ``out = m(img, iters=T, levels=..., return_all=...)`` and ``(out * cot).sum().backward()``.  The forward's
autograd node saves ``(tokens, pos, states, *mlp_weights)``; ``oracle.glom_oracle_torch.reference_grads`` walks the loop
backwards in fp64 along those very states (torch autograd through one ``column_step`` per time step), then through
the tokenizer.  Forward drift is therefore not part of the comparison.  What is left is the backward's own arithmetic:
fp32 rounding on the CUDA-core path, bf16 operand rounding where the GEMMs run on tcgen05.

The routing in ``backward_run`` (bwd_kernels.cu) decides which kernels run: ``tc = bf16 && d % 256 == 0`` puts the MLP
GEMMs on tcgen05, and ``attn_tc = tc && n % 8 == 0`` puts the consensus-attention GEMMs there too.  The matrix below
holds at least one case of each of the four paths (``test_matrix_covers_every_backward_path``).

``check`` compares each gradient tensor as a whole and slice by slice, so that a fault in one tile, row block or level
is not averaged away over the tensor:
  * all values finite;
  * per tensor: ``||got - ref||_F / ||ref||_F <= tol_tensor``;
  * per slice s: ``||got_s - ref_s|| <= tol_slice * max(||ref_s||, ||ref|| * sqrt(|s| / |ref|))``;
  * CUDA-core path only: ``max|got - ref| <= maxabs * max|ref|`` per tensor.
Slices: state-like gradients as (B*n, L, d) by (128-row block, level) and by (level, 64-column block); each MLP
group's (4d, d) or (d, 4d) weight matrix by 256 x 256 tiles (the BW_DW tiles); MLP biases per group; ``pos_emb`` by
128-row blocks; the image gradient per image; ``init_levels`` per level.

Thresholds are about twice the worst value measured on a B200 (1000 W power limit) over this matrix and ten random
shapes of tools/fuzz_grads.py (profiles/r3_backward_reference.txt):

  path                                          worst measured: tensor / slice / max-abs   tol_tensor  tol_slice  maxabs
  CUDA cores (fp32 engine; bf16 with d%256!=0)  7.9e-7 / 6.8e-7 / 1.14e-6                  1.5e-6      1.5e-6     2.5e-6
  MLP on tcgen05 (attention on either)          4.2e-3 / 4.5e-3 / -                        8e-3        9e-3       -

Along the saved states the CUDA-core backward is plain fp32 arithmetic, for the bf16 engine too.  The tensor-core
error comes from the bf16 rounding of the GEMM operands; its worst slice measured 3.5e-3 to 4.5e-3 in every case.
"""
import numpy as np
import pytest
import torch

from oracle import glom_oracle_torch as OT
from oracle.glom_oracle import synth_params

DEV = "cuda:0"

TOL_CC = dict(tol_tensor=1.5e-6, tol_slice=1.5e-6, maxabs=2.5e-6)
TOL_TC = dict(tol_tensor=8e-3, tol_slice=9e-3, maxabs=None)

MLP_ROWS = {"net.1.weight": 4, "net.3.weight": 1, "net.1.bias": 4, "net.3.bias": 1}   # rows per group, in units of d


# ----------------------------------------------------------------------------- the checker
def _slices(name, t, L, d):
    """(label, view) pairs of one gradient tensor; see the module docstring."""
    out = []
    if name == "levels":
        x = t.reshape(-1, L, d)
        for r0 in range(0, x.shape[0], 128):
            for lv in range(L):
                out.append((f"rows {r0}:{min(r0 + 128, x.shape[0])} level {lv}", x[r0:r0 + 128, lv]))
        for lv in range(L):
            for c0 in range(0, d, 64):
                out.append((f"level {lv} cols {c0}:{c0 + 64}", x[:, lv, c0:c0 + 64]))
    elif name == "init_levels":
        out = [(f"level {lv}", t[lv]) for lv in range(L)]
    elif name == "pos_emb.weight":
        out = [(f"rows {r0}:{min(r0 + 128, t.shape[0])}", t[r0:r0 + 128]) for r0 in range(0, t.shape[0], 128)]
    elif name == "img":
        out = [(f"image {i}", t[i]) for i in range(t.shape[0])]
    elif name.startswith(("bottom_up.", "top_down.")):
        rows = MLP_ROWS[name.split(".", 1)[1]] * d
        x = t.reshape(-1, rows, t.shape[1] if t.dim() > 1 else 1)
        for g in range(x.shape[0]):
            if t.dim() == 1:
                out.append((f"group {g}", x[g]))
                continue
            for r0 in range(0, rows, 256):
                for c0 in range(0, x.shape[2], 256):
                    out.append((f"group {g} tile {r0}:{r0 + 256},{c0}:{c0 + 256}", x[g, r0:r0 + 256, c0:c0 + 256]))
    return out


def check(got, ref, L, d, *, tol_tensor, tol_slice, maxabs=None):
    """Compare every gradient in ``ref`` (fp64) with ``got``; returns (failures, worst) where ``worst`` holds the largest
    per-tensor rel-Frobenius error, the largest slice error relative to max(||ref_s||, ||ref|| sqrt(|s|/|ref|)) and,
    with ``maxabs``, the largest max-abs error over max|ref|, each with the tensor and slice it came from."""
    failures = []
    worst = {"tensor": (0.0, ""), "slice": (0.0, ""), "maxabs": (0.0, "")}

    def note(kind, value, where):
        if value > worst[kind][0] or not np.isfinite(value):
            worst[kind] = (value, where)

    for name, r in ref.items():
        g = got.get(name)
        if g is None:
            failures.append(f"{name}: no gradient")
            continue
        g, r = g.detach().cpu().double(), r.detach().cpu().double()
        if g.shape != r.shape:
            failures.append(f"{name}: shape {tuple(g.shape)} != {tuple(r.shape)}")
            continue
        if not torch.isfinite(g).all():
            failures.append(f"{name}: non-finite values")
            note("tensor", float("inf"), name)
            continue
        err, rn = torch.linalg.norm(g - r).item(), torch.linalg.norm(r).item()
        rel = err / rn if rn > 0 else (0.0 if err == 0 else float("inf"))
        note("tensor", rel, name)
        if rel > tol_tensor:
            failures.append(f"{name}: rel-Frobenius {rel:.3e} > {tol_tensor:.1e}")
        if maxabs is not None:
            ma = (g - r).abs().max().item() / max(r.abs().max().item(), 1e-300)
            note("maxabs", ma, name)
            if ma > maxabs:
                failures.append(f"{name}: max-abs {ma:.3e} of max|ref| > {maxabs:.1e}")
        for (label, gs), (_, rs) in zip(_slices(name, g, L, d), _slices(name, r, L, d)):
            allow = max(torch.linalg.norm(rs).item(), rn * (rs.numel() / r.numel()) ** 0.5)
            e = torch.linalg.norm(gs - rs).item()
            srel = e / allow if allow > 0 else (0.0 if e == 0 else float("inf"))
            note("slice", srel, f"{name} {label}")
            if srel > tol_slice:
                failures.append(f"{name} {label}: slice error {srel:.3e} > {tol_slice:.1e}")
    return failures, worst


def report(tag, worst):
    line = (f"{tag}: worst tensor rel {worst['tensor'][0]:.2e} ({worst['tensor'][1]}); "
            f"worst slice rel {worst['slice'][0]:.2e} ({worst['slice'][1]})")
    if worst["maxabs"][1]:
        line += f"; worst max-abs/max|ref| {worst['maxabs'][0]:.2e} ({worst['maxabs'][1]})"
    print(line, flush=True)


# ----------------------------------------------------------------------------- the matrix
def C(name, prec, d, L, image_size, patch, B, T, *, img_hw=None, return_all=False, levels=False, consensus_self=False,
      radius=0.0):
    """One case: a Glom(dim=d, levels=L, image_size, patch_size=patch) run on B images of ``img_hw`` (default square)
    for T steps; ``levels`` carries a state in (else it starts from init_levels); n patches used of N = pos_emb rows."""
    side = image_size // patch
    h, w = img_hw or (image_size, image_size)
    return dict(id=name, prec=prec, d=d, L=L, image_size=image_size, patch=patch, img_hw=(h, w),
                n=(h // patch) * (w // patch), N=side * side, B=B, T=T, return_all=return_all, levels=levels,
                consensus_self=consensus_self, radius=radius)


MATRIX = [
    C("fp32_d192_n36", "fp32", 192, 3, 12, 2, 3, 2, return_all=True),
    C("fp32_d320_n784", "fp32", 320, 2, 56, 2, 1, 2, radius=6.5, consensus_self=True, levels=True),
    C("bf16_d192_n100", "bf16", 192, 3, 20, 2, 3, 3, levels=True),
    C("bf16_d256_n100", "bf16", 256, 2, 20, 2, 3, 2, return_all=True),
    C("bf16_d256_n144", "bf16", 256, 4, 24, 2, 2, 2, consensus_self=True, return_all=True, levels=True),
    C("bf16_d256_n784", "bf16", 256, 3, 56, 2, 2, 2, radius=2.5, levels=True),
    C("bf16_d512_n256", "bf16", 512, 6, 224, 14, 2, 3),
    C("bf16_d768_n400", "bf16", 768, 2, 40, 2, 1, 1, return_all=True),
    C("bf16_d1024_n576", "bf16", 1024, 8, 384, 16, 1, 1),
    C("bf16_d256_n32_ns", "bf16", 256, 3, 16, 2, 2, 2, img_hw=(8, 16), return_all=True),
    C("bf16_d256_n16", "bf16", 256, 2, 8, 2, 1, 1, radius=1.5, levels=True),
    C("bf16_d512_n8_ns", "bf16", 512, 3, 8, 2, 2, 2, img_hw=(4, 8)),
    C("bf16_d256_n1600", "bf16", 256, 2, 80, 2, 1, 1, return_all=True),
]


def path(case):
    """The backward path ``backward_run`` routes the case to."""
    if case["prec"] == "fp32":
        return "fp32 CUDA cores"
    if case["d"] % 256:
        return "bf16 CUDA cores"
    return "MLP tcgen05, attention CUDA cores" if case["n"] % 8 else "MLP and attention tcgen05"


def tolerances(case):
    return TOL_TC if "tcgen05" in path(case) else TOL_CC


def make_inputs(case, seed):
    rng = np.random.default_rng(seed)
    B, n, L, d = case["B"], case["n"], case["L"], case["d"]
    img = rng.standard_normal((B, 3) + case["img_hw"]).astype(np.float32)
    lv = rng.standard_normal((B, n, L, d)).astype(np.float32) if case["levels"] else None
    cot = rng.standard_normal(((case["T"] + 1,) if case["return_all"] else ()) + (B, n, L, d)).astype(np.float32)
    return img, lv, cot


def make_model(case, seed):
    import glom_pytorch_b200 as G
    params = synth_params(case["d"], case["L"], case["image_size"], case["patch"], seed=seed)
    m = G.Glom(dim=case["d"], levels=case["L"], image_size=case["image_size"], patch_size=case["patch"],
               consensus_self=case["consensus_self"], local_consensus_radius=case["radius"], precision=case["prec"])
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    return m.to(DEV), params


def engine_and_reference(m, params, case, img, lv, cot):
    """Run the engine's forward + backward once; return (engine grads, fp64 reference grads along the saved states)."""
    m.zero_grad(set_to_none=True)
    B, n, L, d, T = case["B"], case["n"], case["L"], case["d"], case["T"]
    img_t = torch.from_numpy(img).to(DEV).requires_grad_(True)
    lv_t = None if lv is None else torch.from_numpy(lv).to(DEV).requires_grad_(True)
    cot_t = torch.from_numpy(cot).to(DEV)
    out = m(img_t, iters=T, levels=lv_t, return_all=case["return_all"])
    tokens, pos, states = (s.detach().cpu() for s in out.grad_fn.saved_tensors[:3])
    assert tokens.shape == (B, n, d) and pos.shape == (n, d) and states.shape == (T + 1, B, n, L, d)
    (out * cot_t).sum().backward()
    torch.cuda.synchronize()
    got = {"img": img_t.grad, **{k: p.grad for k, p in m.named_parameters()}}
    if lv_t is not None:
        got["levels"] = lv_t.grad
        assert m.init_levels.grad is None           # a carried-in state replaces init_levels: no gradient reaches it
    P = {k: torch.from_numpy(v).double() for k, v in params.items()}
    mask = OT.radius_mask(case["image_size"] // case["patch"], case["radius"]) if case["radius"] > 0 else None
    ref = OT.reference_grads(P, img, case["patch"], states.double(), tokens.double(), pos.double(),
                             torch.from_numpy(cot), return_all=case["return_all"],
                             consensus_self=case["consensus_self"], mask=mask, carried_levels=lv is not None)
    return got, ref


def assert_close(tag, got, ref, case):
    failures, worst = check(got, ref, case["L"], case["d"], **tolerances(case))
    report(f"{tag} [{path(case)}]", worst)
    assert not failures, f"{tag}: {len(failures)} failures:\n" + "\n".join(failures[:20])


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=[c["id"] for c in MATRIX])
def test_backward_matches_fp64_reference_along_saved_states(case):
    seed = 100 + MATRIX.index(case)
    m, params = make_model(case, seed)
    img, lv, cot = make_inputs(case, seed)
    got, ref = engine_and_reference(m, params, case, img, lv, cot)
    if case["n"] < case["N"]:                       # rows of pos_emb no patch used: exactly zero
        assert not got["pos_emb.weight"][case["n"]:].any()
    assert_close(case["id"], got, ref, case)


def test_matrix_covers_every_backward_path():
    paths = {path(c) for c in MATRIX}
    assert paths == {"fp32 CUDA cores", "bf16 CUDA cores", "MLP tcgen05, attention CUDA cores",
                     "MLP and attention tcgen05"}, paths


@pytest.mark.gpu
@pytest.mark.parametrize("with_levels", [True, False], ids=["levels", "init"])
def test_zero_iterations_under_autograd(with_levels):
    """iters = 0 returns S_0: d_levels is the cotangent bit for bit (or d_init_levels its fp64 sum over images and
    patches), and nothing reaches the MLP, the tokenizer or pos_emb."""
    case = C("bf16_d256_n16_t0", "bf16", 256, 2, 8, 2, 2, 0, return_all=not with_levels, levels=with_levels)
    m, _ = make_model(case, 7)
    img, lv, cot = make_inputs(case, 7)
    img_t = torch.from_numpy(img).to(DEV).requires_grad_(True)
    lv_t = torch.from_numpy(lv).to(DEV).requires_grad_(True) if with_levels else None
    out = m(img_t, iters=0, levels=lv_t, return_all=case["return_all"])
    (out * torch.from_numpy(cot).to(DEV)).sum().backward()
    if with_levels:
        assert torch.equal(lv_t.grad.cpu(), torch.from_numpy(cot))
    else:
        ref = torch.from_numpy(cot).double()[0].sum((0, 1))
        got = m.init_levels.grad.cpu().double()
        assert (got - ref).abs().max() <= 1e-6 * ref.abs().max()
    zero = [img_t.grad] + [p.grad for k, p in m.named_parameters() if k != "init_levels"]
    assert all(g is not None and not g.any() for g in zero)


@pytest.mark.gpu
def test_cached_backward_workspace_across_batch_sizes():
    """One module, backward at B = 3, 1, 3: the cached backward workspace is reused across geometries."""
    base = next(c for c in MATRIX if c["id"] == "bf16_d256_n144")
    m, params = make_model(base, 21)
    for i, B in enumerate((3, 1, 3)):
        case = dict(base, B=B)
        img, lv, cot = make_inputs(case, 30 + i)
        got, ref = engine_and_reference(m, params, case, img, lv, cot)
        assert_close(f"{base['id']} B={B} (call {i})", got, ref, case)


# ----------------------------------------------------------------------------- the checker sees indexing faults
def test_checker_rejects_planted_indexing_faults():
    """On the CPU, fp64 reference gradients of a small case (d = 64, L = 3, 12 x 12 patches, B = 2, T = 2): at the
    tensor-core thresholds, 0.3 % element noise passes and each planted fault, modelled on a real indexing bug, fails."""
    case = C("cpu_d64_n144", "bf16", 64, 3, 24, 2, 2, 2, levels=True)
    L, d = case["L"], case["d"]
    params = synth_params(d, L, case["image_size"], case["patch"], seed=5)
    img, lv, cot = make_inputs(case, 5)
    P = {k: torch.from_numpy(v).double() for k, v in params.items()}
    states = OT.glom_forward(params, img, patch_size=case["patch"], iters=case["T"], levels=lv, return_all=True,
                             dtype=torch.float64)
    tokens = OT.tokenize(torch.from_numpy(img).double(), P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"],
                         case["patch"])
    ref = OT.reference_grads(P, img, case["patch"], states, tokens, P["pos_emb.weight"][:case["n"]],
                             torch.from_numpy(cot), return_all=False, carried_levels=True)
    gen = torch.Generator().manual_seed(0)
    noisy = {k: v * (1 + 3e-3 * torch.randn(v.shape, generator=gen, dtype=torch.float64)) for k, v in ref.items()}
    failures, worst = check(noisy, ref, L, d, **TOL_TC)
    report("0.3 % noise", worst)
    assert not failures, failures

    def planted(name, edit):
        g = {k: v.clone() for k, v in noisy.items()}
        edit(g[name])
        failures, _ = check(g, ref, L, d, **TOL_TC)
        assert failures and all(f.startswith(name) for f in failures), (name, failures)

    def swap_db1(t):
        x = t.view(L, 4 * d)
        x[[0, 1]] = x[[1, 0]].clone()

    planted("levels", lambda t: t.view(-1, L, d)[200, 1].zero_())                 # one row at one level
    planted("bottom_up.net.3.weight", lambda t: t.view(L, d, 4 * d)[1, 10].zero_())   # one output row of group 1's dW2
    planted("bottom_up.net.1.bias", swap_db1)                                      # groups 0 and 1 of db1 swapped
    planted("pos_emb.weight", lambda t: t[128:].zero_())                           # the last, ragged 128-row block
    planted("levels", lambda t: t.view(-1, L, d)[:, L - 1].mul_(0.75))             # top level's 1/3 taken as 1/4
