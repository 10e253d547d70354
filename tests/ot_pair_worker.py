"""Worker of tests/test_multi_gpu_ot.py (torchrun, one process per GPU over NCCL; with --shared-gpu every process on
cuda:0 over gloo, whose all-reduce takes CUDA tensors — the same union protocol on a box with one GPU).

sharded   granules dealt over the ranks with the last rank holding none (synthesize_sharded(group=), targets="ot"):
          coefficients bit-identical on every rank and to one process's synthesize_sharded over every granule.
s2 bands  one zone 11 target cut into row bands (dist.shard_rows), one band per rank through
          synthesize_slab_on_s2_grid(allreduce=True): coefficients bit-identical to one synthesize_on_s2_grid call.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hsr_b200 import dist as hdist  # noqa: E402
from hsr_b200 import synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer, s2_target  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

PIX = 0.000542232520256367
GLT_GT = (-118.30, PIX, 0.0, 34.20, 0.0, -PIX)
S2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)


def same_on_every_rank(t, world):
    g = [None] * world
    dist.all_gather_object(g, t.detach().cpu().numpy().tobytes())
    return all(x == g[0] for x in g)


def granule(ps, i, device):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    Hr, Wr = 30 + 2 * i, 28
    raw = torch.from_numpy(synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=400 + i, good=good)).to(device)
    gx, gy = (torch.from_numpy(a).to(device) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    g = {"raw": raw, "glt_x": gx, "glt_y": gy}
    if i % 2:
        g["target"] = s2_target(GLT_GT, tuple(gx.shape), S2)
        x = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K,) + g["target"].shape, device=device),
                                     g["target"]).bands
    else:
        x = ps.bands_from_raw(raw, gx, gy)[0]
    g["s2_ref"] = synthetic.s2_reference_torch(torch.nan_to_num(x), seed=500 + i)
    return g


def sharded(rank, world, device):
    alone = [dist.new_group([r]) for r in range(world)]                # every rank creates every group, in order
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    for stretch in (None, (2, 98)):
        ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=4, device=device, stretch=stretch, stretch_scope="fit",
                             targets="ot", n_samples=1500)
        n = 2 * (world - 1)
        gs = [granule(ps, i, device) for i in range(n)]
        mine = [i for i in range(n) if i // 2 == rank]                # two per rank; rank world - 1 holds none
        assert (len(mine) == 0) == (rank == world - 1)
        res = ps.synthesize_sharded([gs[i] for i in mine], group=None)
        whole = ps.synthesize_sharded(gs, group=alone[rank])            # one process over every granule
        torch.cuda.synchronize()
        for r in res:
            assert torch.equal(r.coeffs.view(torch.int64), whole[0].coeffs.view(torch.int64)), "sharded != union"
        c = res[0].coeffs if res else whole[0].coeffs
        assert same_on_every_rank(c, world), "ranks solved different systems"


def s2_bands(rank, world, device):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    Hr, Wr = 200, 180
    raw = torch.from_numpy(synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=9, good=good)).to(device)
    gx, gy = (torch.from_numpy(a).to(device) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    target = s2_target(GLT_GT, tuple(gx.shape), S2)
    Hd, Wd = target.shape
    for stretch in (None, (2, 98)):
        ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=4, device=device, stretch=stretch, stretch_scope="fit",
                             targets="ot")
        full0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K, Hd, Wd), device=device), target)
        s2 = synthetic.s2_reference_torch(torch.nan_to_num(full0.bands), seed=13)
        full = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
        t0, t1 = hdist.shard_rows(Hd, rank, world)
        res = ps.synthesize_slab_on_s2_grid(raw, gx, gy, s2[:, t0:t1].contiguous(), target, (t0, t1), allreduce=True)
        torch.cuda.synchronize()
        assert torch.equal(res.coeffs.view(torch.int64), full.coeffs.view(torch.int64)), "bands != one call"
        assert same_on_every_rank(res.coeffs, world)


def main():
    if "--shared-gpu" in sys.argv:
        device = torch.device("cuda", 0)
        torch.cuda.set_device(device)
        dist.init_process_group("gloo")
        rank, world = dist.get_rank(), dist.get_world_size()
    else:
        rank, world, device = hdist.init_from_env()
    sharded(rank, world, device)
    s2_bands(rank, world, device)
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print("multi-gpu ot pair OK", world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
