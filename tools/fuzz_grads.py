"""Randomised shape sweep of the engine's backward against the fp64 reference along the saved forward states.

    python tools/fuzz_grads.py [seed] [cases]

Uses the comparator of tests/test_backward_reference.py (``check`` at that file's thresholds for the path each case
takes), so the sweep and the suite judge a gradient the same way."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_backward_reference import (C, check, engine_and_reference, make_inputs, make_model, path,  # noqa: E402
                                     report, tolerances)

rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
N = int(sys.argv[2]) if len(sys.argv) > 2 else 14
bad = 0
for it in range(N):
    prec = "fp32" if rng.random() < 0.2 else "bf16"
    dim = int(rng.choice([192, 256, 512]))
    L = int(rng.integers(2, 5))
    p = 2
    side = int(rng.choice([2, 3, 8, 10, 11, 16, 18, 20, 26, 28]))     # 26, 28: n = 676 / 784 > 576 columns
    if side >= 26:
        dim = min(dim, 256)
    B = int(rng.integers(1, 4))
    T = int(rng.integers(1, 3))
    radius = float(rng.choice([1.5, 2.5])) if rng.random() < 0.3 else 0.0
    case = C(f"[{it}]", prec, dim, L, side * p, p, B, T, return_all=bool(rng.random() < 0.5),
             levels=bool(rng.random() < 0.5), consensus_self=bool(rng.random() < 0.3), radius=radius)
    seed = int(rng.integers(1 << 30))
    tag = (f"[{it}] {prec} d={dim} L={L} n={case['n']} rows={B * case['n']} B={B} T={T} all={case['return_all']} "
           f"lv={case['levels']} self={case['consensus_self']} radius={radius} [{path(case)}]")
    try:
        m, params = make_model(case, seed)
        got, ref = engine_and_reference(m, params, case, *make_inputs(case, seed))
    except Exception as e:
        print(f"{tag}: EXC {type(e).__name__}: {str(e)[:100]}", flush=True)
        bad += 1
        continue
    failures, worst = check(got, ref, L, dim, **tolerances(case))
    report(tag, worst)
    for f in failures[:5]:
        print("   ", f)
    bad += bool(failures)
print("FAILURES:", bad)
