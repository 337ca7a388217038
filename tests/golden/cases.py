"""Golden-case table and input generator shared by make_golden.py (build container, imports
the reference) and the tests (any box; no reference needed).  numpy PCG64 only."""
import numpy as np

CASES = {
    # BASELINE.json configs[0]: dim=64 levels=3 image_size=28 patch_size=7 iters=2 batch=1 fp32
    "c1_return_all": dict(dim=64, levels=3, image_size=28, patch_size=7, batch=1, iters=2,
                          return_all=True),
    "c1_default_iters": dict(dim=64, levels=3, image_size=28, patch_size=7, batch=2,
                             iters=None, return_all=False),
    # mid case (SURVEY 7.1): d=128 L=4 N=64
    "mid_return_all": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2, iters=5,
                           return_all=True, unstored_from=(5, 0, 24, 0, 0)),
    "mid_consensus_self": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2,
                               iters=3, return_all=False, consensus_self=True),
    "mid_radius": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2, iters=3,
                       return_all=False, local_consensus_radius=1.5),
    "mid_radius_self": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=1, iters=2,
                            return_all=False, local_consensus_radius=2, consensus_self=True),
    # peaky attention: carried-in state scaled x20 (softmax far from uniform)
    "mid_peaky": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2, iters=3,
                      return_all=True, levels_scale=20.0),
    # non-square image, n < num_patches (SURVEY 8b): 16x32 with patch 4 -> n = 32 of 64
    "mid_nonsquare": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2, iters=3,
                          return_all=False, img_hw=(16, 32)),
    # 3-frame continuation (README.md:105-111; BASELINE config 5 shape, small dims)
    "mid_continuation": dict(dim=128, levels=4, image_size=32, patch_size=4, batch=2,
                             iters=[4, 3, 2], return_all=False, frames=3),
    # two levels (smallest legal L: top_down has L-1 = 1 group)
    "two_levels": dict(dim=64, levels=2, image_size=16, patch_size=4, batch=3, iters=4,
                       return_all=True),
    # iters = 0 returns S_0
    "zero_iters": dict(dim=64, levels=3, image_size=28, patch_size=7, batch=2, iters=0,
                       return_all=True),
}



def inputs(case, frame=0):
    rng = np.random.default_rng(1000 + frame)
    H, W = case.get("img_hw", (case["image_size"],) * 2)
    img = rng.standard_normal((case["batch"], 3, H, W)).astype(np.float32)
    levels = None
    if "levels_scale" in case:
        n = (H // case["patch_size"]) * (W // case["patch_size"])
        levels = (rng.standard_normal((case["batch"], n, case["levels"], case["dim"]))
                  * case["levels_scale"]).astype(np.float32)
    return img, levels


# ----------------------------------------------------------------------------- gradient fixtures (f2)
GRAD_CASES = {
    # BASELINE configs[0] shapes, default attention (diag fill), init_levels start, loss on every time step
    "grad_c1_all": dict(dim=64, levels=3, image_size=28, patch_size=7, batch=2, iters=2, return_all=True,
                        param_seed=11),
    # carried-in levels (gradient w.r.t. the input state), radius mask + consensus_self, loss on the last step only
    "grad_c1_masked": dict(dim=64, levels=3, image_size=28, patch_size=7, batch=2, iters=3, return_all=False,
                           param_seed=12, consensus_self=True, local_consensus_radius=1.5, with_levels=True),
}


def grad_inputs(case):
    rng = np.random.default_rng(2000 + case["param_seed"])
    B, L, d = case["batch"], case["levels"], case["dim"]
    n = (case["image_size"] // case["patch_size"]) ** 2
    img = rng.standard_normal((B, 3, case["image_size"], case["image_size"])).astype(np.float32)
    lv = rng.standard_normal((B, n, L, d)).astype(np.float32) if case.get("with_levels") else None
    shape = ((case["iters"] + 1,) if case["return_all"] else ()) + (B, n, L, d)
    cot = rng.standard_normal(shape).astype(np.float32)
    return img, lv, cot
