"""Worker of tests/test_multi_gpu_global_stretch.py (torchrun, one process per GPU): the percentile stretch over a global
fit (PairSynthesizer(stretch=(2, 98), stretch_scope="fit")) in BASELINE.json configs[3] and configs[4].

configs[3]  16 synthetic granules dealt round-robin, ONE global fit through dist.PeerExchange and through NCCL: the
            stretch limits equal np.percentile over ALL granules bit for bit on every rank, the coefficients and the
            rank's matched planes meet the oracle's bars on the stretched concatenation.  Then an uneven deal (3
            granules: ranks with none) completes without a hang and gives the limits of those 3.
configs[4]  a mosaic cut into row slabs (raw in host memory, per-slab staging) with a global fit through the peer
            exchange and through allreduce=True: limits bit-identical to the un-sharded single-image run, coefficients
            within rtol 1e-8, matched planes within 2.4e-7 of it.
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
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402
from oracle import color as ocolor  # noqa: E402
from oracle import glt as oglt  # noqa: E402
from oracle import poly as opoly  # noqa: E402
from oracle import srf as osrf  # noqa: E402

N_GRANULES = 16
SEED0 = 300
DEG = 2
STRETCH = (2, 98)


def synthesizer(device):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    return PairSynthesizer(w, synthetic_s2_srf(), good, deg=DEG, stretch=STRETCH, stretch_scope="fit", device=device)


def stretch_np(x, lim):
    lo, hi = lim[:, 0:1], lim[:, 1:2]
    with np.errstate(invalid="ignore"):
        return np.clip((x.reshape(x.shape[0], -1) - lo) / (hi - lo + 1e-12), 0, 1).astype(np.float32).reshape(x.shape)


def same_on_every_rank(t, world):
    if world == 1:
        return True
    gathered = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(gathered, t.contiguous())
    return all(torch.equal(g.view(torch.int64), gathered[0].view(torch.int64)) for g in gathered)


def config3(rank, world, device, px):
    ps = synthesizer(device)
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    Hr, Wr = 40, 34
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gxd, gyd = torch.from_numpy(gx).to(device), torch.from_numpy(gy).to(device)
    every = []
    for i in range(N_GRANULES):
        raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=SEED0 + i, good=good)
        ortho, valid, _ = oglt.glt_ortho(raw, gx, gy)
        ref = osrf.pseudo_s2_srf_integral(ortho, w, table, good)
        x = np.stack([ref[b] for b in ps.band_names]).astype(np.float32)
        every.append((raw, x, synthetic.s2_reference_np(x, seed=SEED0 + 1000 + i), opoly.fit_mask(x, valid, 0, 0.0)))
    K = ps.K

    def oracle(idx, bands):
        """Limits and fit over the granules idx; the limits are exact functions of the planes the device produced
        (``bands``: every granule's, gathered from all ranks), the mask is the oracle's."""
        xc = np.concatenate([bands[i].reshape(K, -1) for i in idx], axis=1)
        yc = np.concatenate([every[i][2].reshape(K, -1) for i in idx], axis=1)
        mc = np.concatenate([every[i][3].reshape(-1) for i in idx])
        xl, yl = ocolor.shared_percentile_limits(xc.T, mc), ocolor.shared_percentile_limits(yc.T, mc)
        return xl, yl, opoly.polyfit_paired(stretch_np(xc, xl), stretch_np(yc, yl), mc, DEG, min_count=200)

    def check(res, mine, want, what):
        xl, yl, coeffs = want
        for r, i in zip(res, mine):
            assert np.array_equal(r.x_limits.cpu().numpy().reshape(K, 2).view(np.int64), xl.view(np.int64)), what
            assert np.array_equal(r.y_limits.cpu().numpy().reshape(K, 2).view(np.int64), yl.view(np.int64)), what
            c = r.coeffs.cpu().numpy()
            err = float(np.max(np.abs(c - coeffs).max(1) / np.abs(coeffs).max(1)))
            assert err < 1e-4, f"{what}: coefficients off by {err:.2e}"
            matched = opoly.apply_poly_planes(stretch_np(r.bands.cpu().numpy(), xl), coeffs, every[i][3])
            assert np.max(np.abs(r.matched.cpu().numpy() - matched)) < 1e-4, what

    mine = hdist.shard_units(N_GRANULES, rank, world)
    granules = [{"raw": torch.from_numpy(every[i][0]).to(device), "glt_x": gxd, "glt_y": gyd,
                 "s2_ref": torch.from_numpy(every[i][2]).to(device)} for i in mine]
    # every granule's device planes, from the rank that owns it (the SRF is per granule, rank-independent)
    own = [ps.bands_from_raw(g["raw"], gxd, gyd)[0].cpu().numpy() for g in granules]
    gathered = [dict(zip(mine, own))] * world
    if world > 1:
        dist.all_gather_object(gathered, gathered[0])
    bands = {i: b for d in gathered for i, b in d.items()}
    want = oracle(range(N_GRANULES), bands)
    for path in ("peer", "nccl"):
        res = ps.synthesize_sharded(granules, exchange=px if path == "peer" else None)
        torch.cuda.synchronize()
        if path == "peer":
            px.check()
        assert len(res) == len(mine)
        check(res, mine, want, path)
        assert same_on_every_rank(res[0].x_limits, world) and same_on_every_rank(res[0].y_limits, world), path
    # uneven deal: 3 granules, so with 4 or 8 ranks some rank holds none and still takes part in every reduction
    few_idx = [i for i in mine if i < 3]
    res = ps.synthesize_sharded([g for g, i in zip(granules, mine) if i < 3], exchange=px)
    torch.cuda.synchronize()
    px.check()
    assert len(res) == len(few_idx)
    check(res, few_idx, oracle(range(3), bands), "uneven deal")


def config4(rank, world, device, px):
    ps = synthesizer(device)
    good = synthetic.good_band_mask(synthetic.emit_wavelengths())
    Hr, Wr = 300, 300
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=17, good=good)
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=5, n_oob=16, n_neg=16)
    Ho, Wo = gx.shape
    gxd, gyd = torch.from_numpy(gx).to(device), torch.from_numpy(gy).to(device)
    rawd = torch.from_numpy(raw).to(device)
    s2 = synthetic.s2_reference_torch(ps.bands_from_raw(rawd, gxd, gyd)[0], seed=19)
    full = ps.synthesize(rawd, gxd, gyd, s2)            # the un-sharded single-image run
    torch.cuda.synchronize()
    del rawd
    raw_host = torch.from_numpy(raw).pin_memory()
    r0, r1 = hdist.shard_rows(Ho, rank, world, align=8)
    for path in ("peer", "allreduce"):
        kw = {"exchange": px} if path == "peer" else {"allreduce": True}
        res = ps.synthesize_slab(raw_host, gxd[r0:r1], gyd[r0:r1], s2[:, r0:r1], **kw)
        torch.cuda.synchronize()
        if path == "peer":
            px.check()
        assert torch.equal(res.x_limits.view(torch.int64), full.x_limits.view(torch.int64)), path
        assert torch.equal(res.y_limits.view(torch.int64), full.y_limits.view(torch.int64)), path
        torch.testing.assert_close(res.coeffs, full.coeffs, rtol=1e-8, atol=1e-11)
        assert (res.matched - full.matched[:, r0:r1]).abs().max().item() <= 2.4e-7, path


def main():
    rank, world, device = hdist.init_from_env()
    px = hdist.PeerExchange(device=device, timeout_ms=20000)
    config3(rank, world, device, px)
    config4(rank, world, device, px)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    px.close()
    if rank == 0:
        print("global stretch OK", world)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
