"""Small workload for compute-sanitizer that touches every tensor-core kernel of the forward: the three-kernel step,
the consensus kernel with a radius mask, the tokeniser, the island analytics and one backward.  `contrastive`: only the
column-contrastive loss's forward and backward at a ragged shape (n = 196: images straddle the 128-row tiles)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import glom_pytorch_b200 as G

torch.manual_seed(0)
if len(sys.argv) > 1 and sys.argv[1] == "contrastive":
    za = torch.randn(3, 196, 3, 192, device="cuda", requires_grad=True)
    zb = torch.randn(3, 196, 3, 192, device="cuda", requires_grad=True)
    loss = G.column_contrastive_loss(za, zb, levels=(0, 2), temperature=0.1)
    loss.backward()
    torch.cuda.synchronize()
    print("sanitize target ok", loss.item(), za.grad.abs().max().item(), zb.grad.abs().max().item())
    sys.exit(0)
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
