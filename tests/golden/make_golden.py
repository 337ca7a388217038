"""Generate the golden fixtures in this directory from the LIVE reference.

Run in the build container only (it imports /root/reference, which does not exist on the
GPU box):

    python tests/golden/make_golden.py

Each case: parameters from ``oracle.glom_oracle.synth_params`` (numpy PCG64, so the test
can rebuild the identical weights without torch's RNG), loaded into the unmodified
reference ``Glom`` through ``load_state_dict``; inputs from numpy PCG64; the reference is run
in fp32 on CPU under ``torch.no_grad()``.  Only inputs' seeds and the reference OUTPUTS are
stored (float32, compressed), keeping fixtures small.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.environ.get("GLOM_REF_PATH", "/root/reference"))

from glom_pytorch import Glom as RefGlom  # noqa: E402  (the reference)
from oracle.glom_oracle import synth_params  # noqa: E402
sys.path.insert(0, HERE)
from cases import CASES, inputs  # noqa: E402

def build(case):
    kw = dict(dim=case["dim"], levels=case["levels"], image_size=case["image_size"],
              patch_size=case["patch_size"],
              consensus_self=case.get("consensus_self", False),
              local_consensus_radius=case.get("local_consensus_radius", 0))
    model = RefGlom(**kw).eval()
    params = synth_params(case["dim"], case["levels"], case["image_size"], case["patch_size"],
                          seed=case.get("param_seed", 0))
    sd = {k: torch.from_numpy(v) for k, v in params.items()}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(m == "attention.non_local_mask" for m in missing), missing
    return model


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    index = {}
    for name, case in CASES.items():
        model = build(case)
        outs = {}
        with torch.no_grad():
            if case.get("frames"):
                levels = None
                for f in range(case["frames"]):
                    img, _ = inputs(case, f)
                    levels = model(torch.from_numpy(img), iters=case["iters"][f], levels=levels)
                    outs[f"out{f}"] = levels.numpy().astype(np.float32)
            else:
                img, lv = inputs(case)
                out = model(torch.from_numpy(img), iters=case["iters"],
                            levels=None if lv is None else torch.from_numpy(lv),
                            return_all=case["return_all"])
                outs["out0"] = out.numpy().astype(np.float32)
        if case.get("unstored_from"):
            # keeps the fixture under 1 MB: out0 is stored up to the index `unstored_from` (C order) and NaN from there
            # on (compressed to nothing), so the file keeps the output's full shape
            outs["out0"].flat[np.ravel_multi_index(case["unstored_from"], outs["out0"].shape):] = np.nan
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **outs)
        index[name] = dict(case=case, shapes={k: list(v.shape) for k, v in outs.items()})
        print(name, {k: v.shape for k, v in outs.items()})
    with open(os.path.join(HERE, "index.json"), "w") as f:
        json.dump(dict(reference_commit="f30f62165d0c9f9ccdc0330b0005c35ffaaa1635",
                       torch=torch.__version__, cases=index), f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
