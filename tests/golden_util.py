"""Load golden fixtures (reference outputs) and rebuild their seeded inputs/parameters."""
import os

import numpy as np

from cases import CASES, inputs  # tests/golden/cases.py (on sys.path via conftest)
from oracle.glom_oracle import synth_params

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Outputs(dict):
    """Reference outputs by key, at full shape.  A fixture may leave the tail (C order) of an output unstored (NaN in
    the file; case key ``unstored_from``, see make_golden.py).  Those entries are 0 here, and ``pick`` checks a full
    output's shape and finiteness and zeroes the same entries, so that both sides compare element for element."""

    def __init__(self, arrays):
        self.unstored = {k: np.isnan(v) for k, v in arrays.items() if np.isnan(v).any()}
        super().__init__({k: np.where(np.isnan(v), 0, v) for k, v in arrays.items()})

    def pick(self, key, arr):
        assert arr.shape == self[key].shape, (key, arr.shape, self[key].shape)
        assert np.isfinite(arr).all(), key
        mask = self.unstored.get(key)
        return arr if mask is None else np.where(mask, 0, arr)


def load(name):
    case = CASES[name]
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        outs = Outputs({k: z[k] for k in z.files})
    params = synth_params(case["dim"], case["levels"], case["image_size"], case["patch_size"],
                          seed=case.get("param_seed", 0))
    return case, params, outs


def model_kwargs(case):
    return dict(dim=case["dim"], levels=case["levels"], image_size=case["image_size"],
                patch_size=case["patch_size"], consensus_self=case.get("consensus_self", False),
                local_consensus_radius=case.get("local_consensus_radius", 0))


__all__ = ["CASES", "GOLDEN_DIR", "inputs", "load", "model_kwargs"]
