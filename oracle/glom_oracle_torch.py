"""Multi-threaded torch-CPU restatement of the GLOM column update  --  TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE.

Same algorithm and citations as ``oracle/glom_oracle.py`` (the numpy oracle, pinned on the reference's golden
outputs), written with batched torch CPU ops (``torch.bmm`` over the MLP groups, ``F.gelu``, ``torch.softmax``) so
that it uses every host core the way the reference's own torch/oneDNN path does.  ``bench.py`` times it as the CPU
arm (``kind: "port"``) ONLY when the unmodified reference package is not importable on the box
(``$GLOM_REF_PATH`` -> ``oracle/_ref``); ``tests/test_oracle_golden.py`` checks it against
the same golden fixtures as the numpy oracle.

``backward_along`` and ``tokenize_vjp`` are the gradient reference: fp64 torch autograd through one ``column_step`` per
time step, evaluated along the states a forward saved.  ``tests/test_oracle_golden.py`` pins them on the reference's
own autograd (the ``grad_*.npz`` fixtures); ``tests/test_backward_reference.py`` and ``tools/fuzz_grads.py`` compare
the engine's backward with them.  Only ``tests/``, ``tools/`` and ``bench.py``'s CPU legs may import this module.

Restates (``glom_pytorch/glom_pytorch.py``): GroupedFeedForward :23-36, ConsensusAttention.forward :56-73
(F.normalize eps 1e-12 :58, d**-0.5 :60, diagonal -5e-4 :11/:62-65 before the radius mask :67-69), image_to_tokens
:94-97, Glom.forward :110-150 (contributions 4..4,3 :128-129, Jacobi loop :131-145, return_all :147-148).
"""
import math

import torch
import torch.nn.functional as F

TOKEN_ATTEND_SELF_VALUE = -5e-4  # glom_pytorch.py:11


def _grouped_ff(x, w1, b1, w2, b2):
    """x (B, n, G, d) -> (B, n, G, d): per-group d -> 4d -> d MLP with exact-erf GELU (:27-33)."""
    B, n, G, d = x.shape
    a = x.permute(2, 0, 1, 3).reshape(G, B * n, d)                       # group-major rows
    h = F.gelu(torch.baddbmm(b1.reshape(G, 1, 4 * d), a, w1.reshape(G, 4 * d, d).transpose(1, 2)))
    y = torch.baddbmm(b2.reshape(G, 1, d), h, w2.reshape(G, d, 4 * d).transpose(1, 2))
    return y.reshape(G, B, n, d).permute(1, 2, 0, 3)


def _consensus(levels, attend_self, mask):
    """ConsensusAttention.forward (:56-73); levels (B, n, L, d)."""
    B, n, L, d = levels.shape
    q = levels.permute(0, 2, 1, 3)                                       # b l i d
    k = F.normalize(levels, dim=-1).permute(0, 2, 1, 3)                  # (:58)
    sim = torch.matmul(q, k.transpose(-1, -2)) * (d ** -0.5)             # (:60)
    if not attend_self:                                                  # (:62-65)
        eye = torch.eye(n, dtype=torch.bool)
        sim = sim.masked_fill(eye[None, None], TOKEN_ATTEND_SELF_VALUE)
    if mask is not None:                                                 # (:67-69)
        sim = sim.masked_fill(mask[None, None], -torch.finfo(sim.dtype).max)
    attn = sim.softmax(dim=-1)                                           # (:71)
    return torch.matmul(attn, q).permute(0, 2, 1, 3)                     # (:72)


def radius_mask(side, radius):
    """non_local_mask (:44-54): 'ij' meshgrid, '(h w) c' coordinates, cdist > radius."""
    ar = torch.arange(side)
    hh, ww = torch.meshgrid(ar, ar, indexing="ij")
    co = torch.stack((hh.reshape(-1), ww.reshape(-1)), -1).float()
    return torch.cdist(co, co) > radius


def column_step(levels, tokens, pos, P, consensus_self, mask):
    """One iteration of the Jacobi loop (:131-145): S_t (B, n, L, d) -> S_{t+1}.  tokens (B, n, d), pos (n, d), ``P`` the
    parameters keyed like the reference's state_dict.  Differentiable: ``backward_along`` runs autograd through it."""
    L = levels.shape[2]
    bottom = tokens[:, :, None, :]                                                        # (:121)
    contrib = torch.full((L,), 4.0, dtype=levels.dtype)                                   # (:128)
    contrib[-1] = 3.0                                                                     # (:129)
    lwi = torch.cat((bottom, levels), dim=-2)                                             # (:132)
    bu = _grouped_ff(lwi[..., :-1, :], P["bottom_up.net.1.weight"], P["bottom_up.net.1.bias"],
                     P["bottom_up.net.3.weight"], P["bottom_up.net.3.bias"])              # (:134)
    td = _grouped_ff(lwi[..., 2:, :] + pos[None, :, None, :], P["top_down.net.1.weight"], P["top_down.net.1.bias"],
                     P["top_down.net.3.weight"], P["top_down.net.3.bias"])                # (:136)
    td = F.pad(td, (0, 0, 0, 1))                                                          # (:137)
    cons = _consensus(levels, consensus_self, mask)                                       # (:139)
    return (levels + bu + td + cons) / contrib[None, None, :, None]                       # (:141-142)


@torch.no_grad()
def glom_forward(params, img, *, patch_size, iters=None, levels=None, return_all=False, consensus_self=False,
                 local_consensus_radius=0, dtype=torch.float32):
    """Glom.forward (:110-150).  ``params``: reference state_dict keys -> tensors / arrays; img (B, 3, H, W)."""
    P = {k: torch.as_tensor(v).to(dtype) for k, v in params.items() if k != "attention.non_local_mask"}
    L, d = P["init_levels"].shape
    img = torch.as_tensor(img).to(dtype)
    B = img.shape[0]
    tokens = tokenize(img, P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"], patch_size)   # (:114)
    n = tokens.shape[1]
    iters = 2 * L if iters is None else iters                                             # (:112)
    pos = P["pos_emb.weight"][:n]                                                         # (:117-118)
    if levels is None:
        levels = P["init_levels"][None, None].expand(B, n, L, d)                          # (:123-124)
    else:
        levels = torch.as_tensor(levels).to(dtype)
    mask = None
    if local_consensus_radius > 0:
        mask = radius_mask(int(round(math.sqrt(P["pos_emb.weight"].shape[0]))), local_consensus_radius)
    hiddens = [levels]
    for _ in range(iters):                                                                # (:131)
        levels = column_step(levels, tokens, pos, P, consensus_self, mask)
        hiddens.append(levels)                                                            # (:145)
    if return_all:
        return torch.stack(hiddens)                                                       # (:147-148)
    return levels                                                                         # (:150)


def tokenize(img, weight, bias, patch_size):
    """image_to_tokens (:94-97, :114): img (B, 3, H, W) -> (B, n, d); 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)'."""
    B, C, H, W = img.shape
    p = patch_size
    x = img.reshape(B, C, H // p, p, W // p, p).permute(0, 2, 4, 3, 5, 1).reshape(B, (H // p) * (W // p), p * p * C)
    return F.linear(x, weight, bias)


# ----------------------------------------------------------------------------- fp64 gradient reference
MLP_KEYS = ("bottom_up.net.1.weight", "bottom_up.net.1.bias", "bottom_up.net.3.weight", "bottom_up.net.3.bias",
            "top_down.net.1.weight", "top_down.net.1.bias", "top_down.net.3.weight", "top_down.net.3.bias")


def backward_along(states, tokens, pos, P, cot, return_all, consensus_self=False, mask=None):
    """Reverse pass of the loop along a GIVEN trajectory, in fp64: the exact vector-Jacobian product of the column
    update evaluated at ``states`` (S_0..S_T, (T+1, B, n, L, d)), whatever forward produced them.

    For t = T-1 .. 0, ``torch.autograd.grad`` of ``column_step(S_t)`` against the pending cotangent of S_{t+1}; with
    ``return_all`` the cotangent of S_t's own output, ``cot[t]``, is added on the way.  ``cot`` is (T+1, B, n, L, d)
    with ``return_all`` and (B, n, L, d) without.  tokens (B, n, d), pos (n, d), ``P`` holds the eight MLP tensors.
    Returns (d_S0, d_tokens, d_pos, {MLP key: grad}) in fp64."""
    f64 = torch.float64
    T = states.shape[0] - 1
    tokens = tokens.detach().to(f64).requires_grad_(True)
    pos = pos.detach().to(f64).requires_grad_(True)
    W = {k: P[k].detach().to(f64).requires_grad_(True) for k in MLP_KEYS}
    cot = cot.detach().to(f64)
    g = cot[T] if return_all else cot
    d_tokens, d_pos = torch.zeros_like(tokens), torch.zeros_like(pos)
    d_W = {k: torch.zeros_like(w) for k, w in W.items()}
    for t in range(T - 1, -1, -1):
        s = states[t].detach().to(f64).requires_grad_(True)
        with torch.enable_grad():
            out = column_step(s, tokens, pos, W, consensus_self, mask)
            ds, dt, dp, *dw = torch.autograd.grad(out, (s, tokens, pos, *W.values()), g)
        d_tokens += dt
        d_pos += dp
        for k, v in zip(MLP_KEYS, dw):
            d_W[k] += v
        g = ds + cot[t] if return_all else ds
    return g, d_tokens, d_pos, d_W


def tokenize_vjp(img, weight, bias, patch_size, d_tokens):
    """Vector-Jacobian product of image_to_tokens in fp64: d_tokens (B, n, d) -> (d_img, d_weight, d_bias)."""
    f64 = torch.float64
    img = torch.as_tensor(img).detach().to(f64).requires_grad_(True)
    weight = torch.as_tensor(weight).detach().to(f64).requires_grad_(True)
    bias = torch.as_tensor(bias).detach().to(f64).requires_grad_(True)
    with torch.enable_grad():
        tokens = tokenize(img, weight, bias, patch_size)
        return torch.autograd.grad(tokens, (img, weight, bias), d_tokens.to(f64))


def reference_grads(P, img, patch_size, states, tokens, pos, cot, *, return_all, consensus_self=False, mask=None,
                    carried_levels=False):
    """Every gradient of loss = sum(out * cot) in fp64, keyed like ``Glom.named_parameters()`` plus ``"img"`` and, with
    ``carried_levels``, ``"levels"`` (the carried-in state; ``"init_levels"`` otherwise).  ``states``, ``tokens`` and
    ``pos`` are the trajectory the forward saved; ``P`` holds the parameters (reference state_dict keys)."""
    n = tokens.shape[1]
    d_s0, d_tok, d_pos, d_w = backward_along(states, tokens, pos, P, cot, return_all, consensus_self, mask)
    d_img, d_wt, d_bt = tokenize_vjp(img, P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"], patch_size, d_tok)
    d_pos_emb = torch.zeros(tuple(P["pos_emb.weight"].shape), dtype=torch.float64)
    d_pos_emb[:n] = d_pos
    g = {"img": d_img, "image_to_tokens.1.weight": d_wt, "image_to_tokens.1.bias": d_bt, "pos_emb.weight": d_pos_emb,
         **d_w}
    if carried_levels:
        g["levels"] = d_s0
    else:
        g["init_levels"] = d_s0.sum((0, 1))
    return g
