"""Worker of tests/test_multi_gpu_s2_grid.py (torchrun, one process per GPU): BASELINE.json configs[3] and configs[4] on
the Sentinel-2 grid, at sizes the numpy oracle finishes in seconds.

configs[3]  one granule per rank on its own S2 target (ranks alternate zone 11 N and zone 34 S), one global fit through
            synthesize_on_s2_grid(exchange=) and (allreduce=True).  Checked on every rank: coefficients equal on every
            rank and within 1e-4 of oracle.poly.polyfit_paired over the concatenated masked planes of every rank.
configs[4]  a mosaic (raw in HOST memory) onto a zone 11 target cut into row bands (dist.shard_rows), each rank staging
            only the ortho and raw rows its band reads (synthesize_slab_on_s2_grid).  Checked: the band's planes /
            masks equal the un-sharded run's rows bit for bit, moments and coefficients match the un-sharded fit, a
            rank stages fewer raw rows than the mosaic has, and with stretch_scope="fit" the limits agree on every rank.
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
from oracle import poly as opoly  # noqa: E402

DEG = 2
PIX = 0.000542232520256367
GEOMS = [((-118.30, PIX, 0.0, 34.20, 0.0, -PIX),
          hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)),
         ((18.40, PIX, 0.0, -33.90, 0.0, -PIX),             # S2 origin ~3 km north-west of the ortho corner
          hwarp.S2Grid(epsg=32734, x0=256590.0, y0=6248900.0, dx=10.0, dy=10.0, width=10980, height=10980))]


def gather_np(a):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, a)
    return out


def config3(rank, world, device, px):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=DEG, device=device)
    Hr, Wr = 40, 34
    raw = torch.from_numpy(synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=200 + rank, good=good)).to(device)
    gx, gy = (torch.from_numpy(a).to(device) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    glt_gt, s2g = GEOMS[rank % 2]
    target = s2_target(glt_gt, gx.shape, s2g)
    x0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K,) + target.shape, device=device), target)
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(x0.bands), seed=300 + rank)
    m = x0.fit_mask.cpu().numpy().reshape(-1)
    parts = gather_np((x0.bands.cpu().numpy().reshape(ps.K, -1)[:, m], s2.cpu().numpy().reshape(ps.K, -1)[:, m]))
    xcat = np.concatenate([p[0] for p in parts], axis=1)
    ycat = np.concatenate([p[1] for p in parts], axis=1)
    want = opoly.polyfit_paired(xcat, ycat, np.ones(xcat.shape[1], bool), DEG, min_count=200)
    for path in ("peer", "nccl"):
        kw = {"exchange": px} if path == "peer" else {"allreduce": True}
        r = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target, **kw)
        torch.cuda.synchronize()
        if path == "peer":
            px.check()
        assert torch.equal(r.bands.contiguous().view(torch.int32), x0.bands.contiguous().view(torch.int32))
        c = r.coeffs
        err = float(np.max(np.abs(c.cpu().numpy() - want).max(1) / np.abs(want).max(1)))
        assert err < 1e-4, f"{path}: global coefficients off by {err:.2e}"
        g = [torch.empty_like(c) for _ in range(world)]
        dist.all_gather(g, c.contiguous())
        assert all(torch.equal(x, g[0]) for x in g), f"{path}: ranks solved different systems"
    return True


def config4(rank, world, device, px):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    Hr, Wr = 300, 300
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=7, good=good)
    gxn, gyn = synthetic.rotation_glt(Hr, Wr, 25.0)
    gxn, gyn = synthetic.inject_glt_defects(gxn, gyn, Hr, Wr, seed=3, n_oob=16, n_neg=16)
    gx, gy = torch.from_numpy(gxn).to(device), torch.from_numpy(gyn).to(device)
    glt_gt, s2g = GEOMS[0]
    target = s2_target(glt_gt, gx.shape, s2g)
    Hd, Wd = target.shape
    raw_host = torch.from_numpy(raw).pin_memory()
    rawd = torch.from_numpy(raw).to(device)
    for stretch in (None, (2, 98)):
        ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=DEG, device=device, stretch=stretch,
                             stretch_scope="fit")
        b0 = ps.synthesize_on_s2_grid(rawd, gx, gy, torch.zeros((ps.K, Hd, Wd), device=device), target).bands
        s2 = synthetic.s2_reference_torch(torch.nan_to_num(b0), seed=11)
        full = ps.synthesize_on_s2_grid(rawd, gx, gy, s2, target)          # one process, the whole target
        t0, t1 = hdist.shard_rows(Hd, rank, world)
        assert t1 > t0
        res = ps.synthesize_slab_on_s2_grid(raw_host, gx, gy, s2[:, t0:t1].contiguous(), target, (t0, t1),
                                            exchange=px)
        torch.cuda.synchronize()
        px.check()
        lo, hi = res.raw_rows
        if world > 1:
            assert hi - lo < Hr, f"band staged all {Hr} raw rows"
        assert torch.equal(res.bands.contiguous().view(torch.int32), full.bands[:, t0:t1].contiguous().view(torch.int32))
        assert torch.equal(res.valid, full.valid[t0:t1]) and torch.equal(res.fit_mask, full.fit_mask[t0:t1])
        if stretch is None:
            torch.testing.assert_close(res.moments, full.moments, rtol=1e-12, atol=0)
            torch.testing.assert_close(res.coeffs, full.coeffs, rtol=1e-8, atol=1e-11)
        else:
            for lim in (res.x_limits, res.y_limits):
                g = [torch.empty_like(lim) for _ in range(world)]
                dist.all_gather(g, lim.contiguous())
                assert all(torch.equal(x, g[0]) for x in g), "ranks stretched with different limits"
            assert torch.equal(res.x_limits, full.x_limits) and torch.equal(res.y_limits, full.y_limits)
    return True


def main():
    rank, world, device = hdist.init_from_env()
    px = hdist.PeerExchange(device=device, timeout_ms=20000)
    config3(rank, world, device, px)
    config4(rank, world, device, px)
    dist.barrier()
    torch.cuda.synchronize()
    px.close()
    if rank == 0:
        print("multi-gpu s2 grid OK", world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
