"""Device time of column_contrastive_loss (fused tcgen05 kernels) against the same loss in eager torch under bf16 autocast,
and the loss's share of a configs[1] training step.  Prints one JSON line; needs a B200.

    python tools/contrastive_probe.py [--window 2.0]

Workloads (the card's name and power limit are read in the same call):
  * configs[1] shapes: za, zb (32, 256, 6, 512) fp32, levels (-2, -1), tau 0.1 -- 100 MB each, so the two inputs
    together exceed the 126 MB L2; and B = 256 (805 MB each).
  * forward = the loss alone (no autograd graph); fwd+bwd = the loss and both input gradients.
  * eager torch: the definition with an R x R logit matrix per level (F.normalize, matmul, mask, logsumexp) under
    torch.autocast(bfloat16); at B = 256 an out-of-memory error is reported as such.
  * training step: two noised views through Glom(512, 6, 224/14, bf16), 12 iterations, the loss on the final states,
    backward through everything; the share is the fused loss's fwd+bwd time over the step time.
Algorithmic FLOPs per level (R = B n): forward 2 * 2 R (R - n) d (two logit GEMMs over the candidate columns), backward
2 * 4 R (R - n) d (logits again + G B for each input).  Each timing warms up, then runs back-to-back calls for at least
``--window`` seconds between CUDA events; the median of three such windows is reported.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import glom_pytorch_b200 as G  # noqa: E402

DEV = "cuda:0"


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, window):
    """Median over three windows of the per-call device time (ms) of fn(), calls back to back."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); fn(); e.record(); torch.cuda.synchronize()
    reps = max(3, int(window * 1e3 / max(s.elapsed_time(e), 1e-3)))
    out = []
    for _ in range(3):
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        out.append(s.elapsed_time(e) / reps)
    return {"ms": statistics.median(out), "spread_ms": [min(out), max(out)], "calls_per_window": reps}


def eager_loss(za, zb, levels, tau):
    B, n, L, d = za.shape
    R = B * n
    img = torch.arange(R, device=za.device) // n
    cand = (img[:, None] != img[None, :]) | torch.eye(R, dtype=torch.bool, device=za.device)
    total = 0.0
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for l in levels:
            a = torch.nn.functional.normalize(za[:, :, l].reshape(R, d), dim=1)
            b = torch.nn.functional.normalize(zb[:, :, l].reshape(R, d), dim=1)
            s = (a @ b.T).float() / tau
            sm = s.masked_fill(~cand, float("-inf"))
            pos = torch.diagonal(s)
            total = total + (0.5 * ((torch.logsumexp(sm, 1) - pos) + (torch.logsumexp(sm.T, 1) - pos))).sum()
    return total / (len(levels) * R)


def loss_workload(B, n, L, d, levels, tau, window, eager):
    g = torch.Generator(device=DEV).manual_seed(B)
    za = torch.randn(B, n, L, d, device=DEV, generator=g).requires_grad_(True)
    zb = torch.randn(B, n, L, d, device=DEV, generator=g).requires_grad_(True)
    R = B * n
    fl_f = len(levels) * 2 * 2 * R * (R - n) * d
    fl_b = len(levels) * 2 * 4 * R * (R - n) * d
    res = {"shape": [B, n, L, d], "levels": list(levels), "tau": tau, "R": R,
           "flops_forward": fl_f, "flops_backward": fl_b}

    def fused_fwd():
        with torch.no_grad():
            G.column_contrastive_loss(za, zb, levels=levels, temperature=tau)

    def fused_fb():
        torch.autograd.grad(G.column_contrastive_loss(za, zb, levels=levels, temperature=tau), (za, zb))

    f = timed(fused_fwd, window)
    fb = timed(fused_fb, window)
    res["fused"] = {"forward": f, "fwd_bwd": fb,
                    "forward_tflops": fl_f / f["ms"] * 1e-9, "fwd_bwd_tflops": (fl_f + fl_b) / fb["ms"] * 1e-9}
    if eager:
        try:
            def eager_fwd():
                with torch.no_grad():
                    eager_loss(za, zb, levels, tau)

            def eager_fb():
                torch.autograd.grad(eager_loss(za, zb, levels, tau), (za, zb))
            torch.cuda.reset_peak_memory_stats()
            ef = timed(eager_fwd, window)
            efb = timed(eager_fb, window)
            res["eager_autocast"] = {"forward": ef, "fwd_bwd": efb,
                                     "peak_memory_gb": torch.cuda.max_memory_allocated() / 1e9,
                                     "fused_speedup_forward": ef["ms"] / f["ms"], "fused_speedup_fwd_bwd": efb["ms"] / fb["ms"]}
            with torch.no_grad():
                fused = G.column_contrastive_loss(za, zb, levels=levels, temperature=tau).item()
                res["eager_autocast"]["loss_eager_vs_fused"] = [eager_loss(za, zb, levels, tau).item(), fused]
        except torch.OutOfMemoryError as e:
            res["eager_autocast"] = {"error": "torch.OutOfMemoryError", "message": str(e).splitlines()[0][:300]}
        torch.cuda.empty_cache()
    return res


def train_step_share(window):
    B, d, L, isz, p, iters = 32, 512, 6, 224, 14, 12
    m = G.Glom(dim=d, levels=L, image_size=isz, patch_size=p, precision="bf16").to(DEV)
    g = torch.Generator(device=DEV).manual_seed(0)
    img = torch.randn(B, 3, isz, isz, device=DEV, generator=g)
    views = [img + 0.1 * torch.randn(img.shape, device=DEV, generator=g) for _ in range(2)]

    def step():
        m.zero_grad(set_to_none=True)
        za, zb = (m(v, iters=iters) for v in views)
        G.column_contrastive_loss(za, zb, levels=(-2, -1), temperature=0.1).backward()

    def step_without_loss():
        m.zero_grad(set_to_none=True)
        za, zb = (m(v, iters=iters) for v in views)
        (za.sum() + zb.sum()).backward()

    s = timed(step, window)
    s0 = timed(step_without_loss, window)
    return {"workload": "Glom(512, 6, 224/14, bf16), two views of 32 images, 12 iterations, loss on the final states, "
                        "levels (-2, -1), backward to the parameters",
            "step_ms": s, "step_without_loss_ms": s0, "loss_share_of_step": 1 - s0["ms"] / s["ms"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=2.0, help="seconds per timing window")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    out = {"card": card()}
    out["configs1"] = loss_workload(32, 256, 6, 512, (-2, -1), 0.1, args.window, eager=True)
    share = train_step_share(args.window)
    share["fused_loss_fwd_bwd_over_step"] = out["configs1"]["fused"]["fwd_bwd"]["ms"] / share["step_ms"]["ms"]
    out["configs1"]["share"] = share
    out["card_after"] = card()["nvidia_smi"]
    out["B256"] = loss_workload(256, 256, 6, 512, (-2, -1), 0.1, args.window, eager=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
