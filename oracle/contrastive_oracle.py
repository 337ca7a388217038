"""fp64 reference of the column-contrastive loss (glom_pytorch_b200.column_contrastive_loss) by explicit formulas.

Per selected level, rows r = (b, i), R = B n:  a_r = za[b,i,l] / max(|za[b,i,l]|, 1e-12), b_r likewise,
s_rc = <a_r, b_c> / tau, cand(r) = {r} u {c : image(c) != image(r)},
    l_r = 1/2 [ (lse_(c in cand r) s_rc - s_rr) + (lse_(c in cand r) s_cr - s_rr) ],   loss = mean over levels and rows.
Gradients (R_tot = levels x R rows, G_rc = 1/2 [exp(s_rc - lse_r) + exp(s_rc - lse'_c)] on candidates, 0 elsewhere,
lse = row logsumexp, lse' = column logsumexp):
    dL/da_r = (sum_c G_rc b_c - b_r) / (tau R_tot),   dL/db_c = (sum_r G_rc a_r - a_c) / (tau R_tot),
    dL/dz = (da - a <a, da>) / |z|   (F.normalize; a clamped norm passes da / 1e-12 through).
Everything is row-chunked (``chunk`` rows of logits at a time), so R = 65 536 runs on a GPU in a few GB.
"""
import torch


def _unit(z):
    nrm = torch.linalg.vector_norm(z, dim=1, keepdim=True)
    inv = 1.0 / nrm.clamp_min(1e-12)
    return z * inv, inv, nrm


def _other_image_logits(x, y, idx, n, tau):
    """Logits of rows idx of x against all rows of y; entries of the row's own image (the diagonal included) at -inf."""
    s = (x[idx] @ y.T) / tau
    cols = torch.arange(y.shape[0], device=x.device)
    return s.masked_fill(idx[:, None] // n == cols[None, :] // n, float("-inf"))


def contrastive_reference(za, zb, levels=(-1,), temperature=0.1, *, grad_out=1.0, grad_rows=None, chunk=1024):
    """-> dict(loss (0-dim fp64), dza, dzb ((B, n, L, d) fp64) on za's device).

    Computed relative to the positive: X_r = sum over other-image c of exp(s_rc - s_rr) gives l_r = 1/2 [log1p X_r +
    log1p X'_r], lse_r = s_rr + log1p X_r and G_rr - 1 = -1/2 [X_r / (1 + X_r) + X'_r / (1 + X'_r)], so B = 1 (X = 0)
    gives exact zeros and aligned views (p_rr -> 1) lose no digits.
    grad_rows: None (all rows) or a 1-D index tensor of rows r = b n + i: gradients are computed for those rows only (at
    every selected level; other rows of the selected levels are NaN).  Unselected levels are exactly zero."""
    za = za.detach().double()
    zb = zb.detach().double()
    B, n, L, d = za.shape
    R = B * n
    sel = [l % L for l in levels]
    tau = float(temperature)
    rtot = len(sel) * R
    dev = za.device
    dza = torch.zeros_like(za)
    dzb = torch.zeros_like(zb)
    loss = torch.zeros((), dtype=torch.float64, device=dev)
    rows_needed = torch.arange(R, device=dev) if grad_rows is None else torch.as_tensor(grad_rows, device=dev).long()
    for l in sel:
        xa = za[:, :, l].reshape(R, d)
        xb = zb[:, :, l].reshape(R, d)
        a, inv_a, nrm_a = _unit(xa)
        b, inv_b, nrm_b = _unit(xb)
        s_rr = (a * b).sum(1) / tau
        x_a = torch.empty(R, dtype=torch.float64, device=dev)       # a -> b direction (row sums of S)
        x_b = torch.empty(R, dtype=torch.float64, device=dev)       # b -> a direction (column sums of S)
        for r0 in range(0, R, chunk):
            idx = torch.arange(r0, min(r0 + chunk, R), device=dev)
            x_a[idx] = torch.exp(torch.logsumexp(_other_image_logits(a, b, idx, n, tau) - s_rr[idx, None], dim=1))
            x_b[idx] = torch.exp(torch.logsumexp(_other_image_logits(b, a, idx, n, tau) - s_rr[idx, None], dim=1))
        loss = loss + (0.5 * (torch.log1p(x_a) + torch.log1p(x_b))).sum()
        lse_a, lse_b = s_rr + torch.log1p(x_a), s_rr + torch.log1p(x_b)
        dg = -0.5 * (x_a / (1 + x_a) + x_b / (1 + x_b))
        da = torch.full((R, d), float("nan"), dtype=torch.float64, device=dev)
        db = torch.full((R, d), float("nan"), dtype=torch.float64, device=dev)
        for i0 in range(0, rows_needed.numel(), chunk):
            idx = rows_needed[i0:i0 + chunk]
            # row r of dA: sum_c G_rc b_c + (G_rr - 1) b_r;  row c of dB: sum_r G_rc a_r + (G_cc - 1) a_c
            for x, y, lse_x, lse_y, out in ((a, b, lse_a, lse_b, da), (b, a, lse_b, lse_a, db)):
                s = _other_image_logits(x, y, idx, n, tau)
                g = 0.5 * (torch.exp(s - lse_x[idx, None]) + torch.exp(s - lse_y[None, :]))
                out[idx] = (g @ y + dg[idx, None] * y[idx]) / (tau * rtot)
        for u, inv, nrm, du, dz in ((a, inv_a, nrm_a, da, dza), (b, inv_b, nrm_b, db, dzb)):
            proj = du - u * (u * du).sum(1, keepdim=True)
            g = torch.where(nrm > 1e-12, inv * proj, du * inv)
            dz[:, :, l] = (grad_out * g).reshape(B, n, d)
    return dict(loss=loss / rtot, dza=dza, dzb=dzb)


def contrastive_naive(za, zb, levels=(-1,), temperature=0.1):
    """The definition written plainly (full R x R logits, F.normalize, torch autograd-able): the check on the chunked
    explicit formulas above."""
    B, n, L, d = za.shape
    R = B * n
    total = 0.0
    img = torch.arange(R, device=za.device) // n
    eye = torch.eye(R, dtype=torch.bool, device=za.device)
    cand = (img[:, None] != img[None, :]) | eye
    for l in levels:
        a = torch.nn.functional.normalize(za[:, :, l].reshape(R, d), dim=1)
        b = torch.nn.functional.normalize(zb[:, :, l].reshape(R, d), dim=1)
        s = (a @ b.T) / temperature
        sm = s.masked_fill(~cand, float("-inf"))
        pos = torch.diagonal(s)
        ell = 0.5 * ((torch.logsumexp(sm, 1) - pos) + (torch.logsumexp(sm.T, 1) - pos))
        total = total + ell.sum()
    return total / (len(levels) * R)
