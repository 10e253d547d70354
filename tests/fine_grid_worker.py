"""Worker of tests/test_multi_gpu_fine.py (torchrun, one process per GPU).  Granules on their own S2 targets are dealt
to the ranks (the last rank holds none), one global fit with stretch_scope="fit" (synthesize_sharded), then
matched_fine(group=) at factor 6.  Checked on every rank: the 10 m limits are the same on every rank and bit-identical
to np.percentile of the concatenation of every rank's fine planes (kernels.bilinear_upsample) under their masks; the
planes are those of kernels.bilinear_apply with those limits.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hsr_b200 import dist as hdist  # noqa: E402
from hsr_b200 import kernels, synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer, s2_target  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

PIX = 0.000542232520256367
GEOMS = [((-118.30, PIX, 0.0, 34.20, 0.0, -PIX),
          hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)),
         ((18.40, PIX, 0.0, -33.90, 0.0, -PIX),
          hwarp.S2Grid(epsg=32734, x0=256590.0, y0=6248900.0, dx=10.0, dy=10.0, width=10980, height=10980))]
F = 6
Q = (2, 98)


def gather_np(a):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, a)
    return out


def main():
    rank, world, device = hdist.init_from_env()
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device=device, stretch=Q, stretch_scope="fit")
    granules = []
    if rank < world - 1:                                    # the last rank holds no granule
        for j in range(2):
            Hr, Wr = 36, 30
            raw = torch.from_numpy(synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=500 + 2 * rank + j,
                                                                 good=good)).to(device)
            gx, gy = (torch.from_numpy(a).to(device) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
            glt_gt, s2g = GEOMS[(rank + j) % 2]
            target = s2_target(glt_gt, gx.shape, s2g)
            x0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K,) + target.shape, device=device), target)
            s2 = synthetic.s2_reference_torch(torch.nan_to_num(x0.bands), seed=600 + rank)
            granules.append({"raw": raw, "glt_x": gx, "glt_y": gy, "s2_ref": s2, "target": target})
    res = ps.synthesize_sharded(granules, group=dist.group.WORLD)
    fine = ps.matched_fine(res, F, group=dist.group.WORLD)
    assert len(fine) == len(res)
    # the concatenation of every rank's fine planes under their masks
    mine = [kernels.bilinear_upsample(r.bands, F).cpu().numpy().reshape(ps.K, -1)[:, fr.mask.cpu().numpy().reshape(-1)]
            for r, fr in zip(res, fine)]
    parts = gather_np(mine)
    cat = np.concatenate([p for rp in parts for p in rp], axis=1)
    want = np.stack([np.percentile(cat[k], Q) for k in range(ps.K)])
    for fr in fine:
        got = fr.x_limits.cpu().numpy().reshape(ps.K, 2)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (got, want)
        assert fr.s2_window is not None and fr.factor == F
    # the same limits on every rank, also on the rank without a granule (it joined the reduce)
    lim = fine[0].x_limits if fine else None
    all_lims = gather_np(None if lim is None else lim.cpu().numpy())
    ref = [a for a in all_lims if a is not None]
    assert len(ref) == world - 1 and all(np.array_equal(a.view(np.int64), ref[0].view(np.int64)) for a in ref)
    for r, fr in zip(res, fine):
        out, m = kernels.bilinear_apply(r.bands, F, r.coeffs, x_stretch=fr.x_limits)
        assert torch.equal(m, fr.mask) and torch.equal(out.view(torch.int32), fr.matched.view(torch.int32))
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print("multi-gpu fine grid OK", world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
