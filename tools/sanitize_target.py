"""Small workload for compute-sanitizer that touches every tensor-core kernel of the forward: the three-kernel step,
the consensus kernel with a radius mask, the tokeniser, the island analytics and one backward."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import glom_pytorch_b200 as G

torch.manual_seed(0)
m = G.Glom(dim=256, levels=3, image_size=32, patch_size=4, local_consensus_radius=2).cuda().eval()
img = torch.randn(5, 3, 32, 32, device="cuda")           # 320 rows: a partial 256-row pair tile
with torch.no_grad():
    a = m(img, iters=3, return_all=True)
    isl = G.islands(a, threshold=0.5)
torch.cuda.synchronize()
if len(sys.argv) > 1 and sys.argv[1] == "bwd":
    m.train()
    x = img[:2].clone().requires_grad_(True)
    m(x, iters=2, return_all=True)[1:].square().mean().backward()
    torch.cuda.synchronize()
print("sanitize target ok", float(a.abs().max()), int(isl.num_islands.sum()))
