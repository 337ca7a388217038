"""Multi-threaded torch-CPU restatement of the GLOM column update  --  TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE.

Same algorithm and citations as ``oracle/glom_oracle.py`` (the numpy oracle, pinned on the reference's golden
outputs), written with batched torch CPU ops (``torch.bmm`` over the MLP groups, ``F.gelu``, ``torch.softmax``) so
that it uses every host core the way the reference's own torch/oneDNN path does.  ``bench.py`` times it as the CPU
arm (``kind: "port"``) ONLY when the unmodified reference package is not importable on the box
(``$GLOM_REF_PATH`` -> ``oracle/_ref``); ``tests/test_oracle_golden.py`` checks it against
the same golden fixtures as the numpy oracle.  Only ``tests/`` and ``bench.py``'s CPU legs may import this module.

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


@torch.no_grad()
def glom_forward(params, img, *, patch_size, iters=None, levels=None, return_all=False, consensus_self=False,
                 local_consensus_radius=0, dtype=torch.float32):
    """Glom.forward (:110-150).  ``params``: reference state_dict keys -> tensors / arrays; img (B, 3, H, W)."""
    P = {k: torch.as_tensor(v).to(dtype) for k, v in params.items() if k != "attention.non_local_mask"}
    L, d = P["init_levels"].shape
    img = torch.as_tensor(img).to(dtype)
    B, C, H, W = img.shape
    p = patch_size
    x = img.reshape(B, C, H // p, p, W // p, p).permute(0, 2, 4, 3, 5, 1).reshape(B, (H // p) * (W // p), p * p * C)
    tokens = F.linear(x, P["image_to_tokens.1.weight"], P["image_to_tokens.1.bias"])      # (:114)
    n = tokens.shape[1]
    iters = 2 * L if iters is None else iters                                             # (:112)
    pos = P["pos_emb.weight"][:n][None, :, None, :]                                       # (:117-118)
    bottom = tokens[:, :, None, :]                                                        # (:121)
    if levels is None:
        levels = P["init_levels"][None, None].expand(B, n, L, d)                          # (:123-124)
    else:
        levels = torch.as_tensor(levels).to(dtype)
    mask = None
    if local_consensus_radius > 0:
        mask = radius_mask(int(round(math.sqrt(P["pos_emb.weight"].shape[0]))), local_consensus_radius)
    contrib = torch.full((L,), 4.0, dtype=dtype)                                          # (:128)
    contrib[-1] = 3.0                                                                     # (:129)
    hiddens = [levels]
    for _ in range(iters):                                                                # (:131)
        lwi = torch.cat((bottom, levels), dim=-2)                                         # (:132)
        bu = _grouped_ff(lwi[..., :-1, :], P["bottom_up.net.1.weight"], P["bottom_up.net.1.bias"],
                         P["bottom_up.net.3.weight"], P["bottom_up.net.3.bias"])          # (:134)
        td = _grouped_ff(lwi[..., 2:, :] + pos, P["top_down.net.1.weight"], P["top_down.net.1.bias"],
                         P["top_down.net.3.weight"], P["top_down.net.3.bias"])            # (:136)
        td = F.pad(td, (0, 0, 0, 1))                                                      # (:137)
        cons = _consensus(levels, consensus_self, mask)                                   # (:139)
        levels = (levels + bu + td + cons) / contrib[None, None, :, None]                 # (:141-142)
        hiddens.append(levels)                                                            # (:145)
    if return_all:
        return torch.stack(hiddens)                                                       # (:147-148)
    return levels                                                                         # (:150)
