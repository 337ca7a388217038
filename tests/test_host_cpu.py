"""CPU-side tests: the C-ABI library loads and exports every symbol the header declares, host
logic (layout sizes, argument errors), drop-in surface, and the batch-sharding logic under gloo."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import glom_pytorch_b200 as G
from glom_pytorch_b200 import _native
from glom_pytorch_b200.sharding import shard_range

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "glom_b200.h")).read()
    declared = set(re.findall(r"GLOM_B200_API\s+[\w\s\*]+?\b(glom_b200_\w+)\s*\(", hdr))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    lib = ctypes.CDLL(G.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.glom_b200_abi_version() == 1


def test_layout_sizes_without_gpu():
    cfg = _native.make_cfg(512, 6, 256, False, 0, 0, "bf16")
    pw = _native.packed_weight_bytes(cfg)
    G_, d, L = 11, 512, 6
    assert pw >= (G_ * 4 * d * d + L * d * 8 * d) * 2 + (G_ * 4 * d + L * d) * 4
    ws = _native.workspace_bytes(cfg, 32, 12, False)
    rows = 32 * 256
    assert ws >= rows * G_ * 4 * d * 2 + rows * L * d * 4
    ws_all = _native.workspace_bytes(cfg, 32, 12, True)
    assert ws - ws_all >= rows * L * d * 4 - 4096      # return_all needs no private fp32 slab
    off, nb = _native.workspace_offset(cfg, 32, 12, False, 0)
    assert nb == rows * G_ * 4 * d * 2 and off % 1024 == 0


@pytest.mark.parametrize("kw,msg", [
    (dict(dim=512, levels=1), "levels"),
    (dict(dim=70, levels=3), "dim"),
    (dict(dim=96, levels=3, precision="bf16"), "64"),
])
def test_bad_config_is_an_error_not_a_fallback(kw, msg):
    cfg = _native.make_cfg(kw.get("dim"), kw.get("levels"), 16, False, 0, 0, kw.get("precision", "fp32"))
    with pytest.raises(_native.GlomB200Error, match=msg):
        _native.packed_weight_bytes(cfg)


def test_forward_on_cpu_tensor_raises():
    m = G.Glom(dim=64, levels=3, image_size=28, patch_size=7)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 3, 28, 28))


def test_state_dict_surface_matches_reference_layout():
    m = G.Glom(dim=64, levels=3, image_size=28, patch_size=7, local_consensus_radius=1.5)
    sd = m.state_dict()
    want = {
        "init_levels": (3, 64), "image_to_tokens.1.weight": (64, 147), "image_to_tokens.1.bias": (64,),
        "pos_emb.weight": (16, 64), "bottom_up.net.1.weight": (768, 64, 1), "bottom_up.net.1.bias": (768,),
        "bottom_up.net.3.weight": (192, 256, 1), "bottom_up.net.3.bias": (192,),
        "top_down.net.1.weight": (512, 64, 1), "top_down.net.1.bias": (512,),
        "top_down.net.3.weight": (128, 256, 1), "top_down.net.3.bias": (128,),
        "attention.non_local_mask": (1, 16, 16),
    }
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    assert m.levels == 3


def test_radius_mask_params_follow_the_buffer():
    from oracle.glom_oracle import radius_mask
    for side, r in [(4, 1.5), (4, 1), (8, 2), (8, 2.9), (6, 10)]:
        m = G.Glom(dim=64, levels=2, image_size=side * 4, patch_size=4, local_consensus_radius=r)
        assert np.array_equal(m.attention.non_local_mask[0].numpy(), radius_mask(side, r))
        s, d2 = m.attention.mask_params(side * side)
        hh, ww = np.meshgrid(np.arange(side), np.arange(side), indexing="ij")
        co = np.stack([hh.ravel(), ww.ravel()], -1)
        dd = ((co[:, None] - co[None]) ** 2).sum(-1)
        assert s == side and np.array_equal(dd > d2, radius_mask(side, r))


def test_shard_range_covers_batch():
    for batch in (1, 7, 32, 256):
        for world in (1, 2, 3, 8):
            spans = [shard_range(batch, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == batch
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from golden_util import inputs, load
    from oracle import glom_oracle as O
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    case, params, outs = load("mid_consensus_self")
    img, _ = inputs(case)
    s, e = shard_range(img.shape[0], rank, world)
    mine = O.glom_forward(params, img[s:e], patch_size=case["patch_size"], iters=case["iters"],
                          consensus_self=True, dtype=np.float32)
    t = torch.from_numpy(np.ascontiguousarray(mine))
    gathered = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(gathered, t)                      # off the timed path; only to check the partition
    elapsed = torch.tensor([1.0 + rank])
    dist.all_reduce(elapsed, op=dist.ReduceOp.MAX)    # bench.py's max-over-ranks timing reduction
    if rank == 0:
        full = torch.cat(gathered).numpy()
        q.put((float(np.abs(full - outs["out0"]).max()), float(elapsed.item())))
    dist.barrier()
    dist.destroy_process_group()


def test_batch_sharding_two_ranks_gloo():
    """world_size 2 on gloo: each rank updates its own images with no data-path collective; the
    concatenation equals the unsharded reference output (golden)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    err, tmax = q.get(timeout=120)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert err <= 1e-4 and tmax == 2.0


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    from glom_pytorch_b200.dp import allreduce_gradients, broadcast_parameters
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(100 + rank)                       # deliberately different init per rank
    m = G.Glom(dim=64, levels=3, image_size=28, patch_size=7)
    broadcast_parameters(m, src=0)
    ref = [p.detach().clone() for p in m.parameters()]
    gens = torch.Generator().manual_seed(7)
    for i, p in enumerate(m.parameters()):              # rank r holds gradient (r + 1) * base_i; init_levels has none on rank 1
        base = torch.randn(p.shape, generator=gens)
        p.grad = None if (rank == 1 and i == 0) else (rank + 1) * base
    calls = allreduce_gradients(m, bucket_bytes=64 << 10)
    gens = torch.Generator().manual_seed(7)
    err = 0.0
    for i, p in enumerate(m.parameters()):
        base = torch.randn(p.shape, generator=gens)
        want = base * (1.0 / 2.0 if i == 0 else 1.5)    # mean of (1, 2) * base; param 0: (1, 0) * base
        err = max(err, float((p.grad - want).abs().max()))
    same = all(torch.equal(a, b) for a, b in zip(ref, [p.detach() for p in m.parameters()]))
    t = torch.tensor([float(ref[3].sum())])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t2 = torch.tensor([float(ref[3].sum())])
    dist.all_reduce(t2, op=dist.ReduceOp.MIN)
    if rank == 0:
        q.put((err, calls, same, float(t.item() - t2.item())))
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_gradient_allreduce_two_ranks_gloo():
    """SURVEY 8e / 8f-2: the only collective of the path -- bucketed gradient averaging over the ranks (NCCL on the
    box, gloo here), incl. a parameter that has no gradient on one rank, and the setup-time parameter broadcast."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    err, calls, same, spread = q.get(timeout=180)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert err <= 1e-6 and calls >= 2 and same and spread == 0.0
