"""Timing of the pair on the Sentinel-2 grid (PairSynthesizer.synthesize_on_s2_grid) on the granule workload: raw
1280 x 1242 x 285, 25 degree GLT (ortho 1685 x 1667), the zone 11 60 m target of profiles/prof_warp.py (1215 x 959).
Per stage (glt_srf, coords, warp_planes, fit, solve / apply), the whole call with and without the cached coordinates,
and the chained GPU path on the same inputs (glt_ortho -> warp of 285 bands -> srf_integrate -> fit -> solve / apply),
the two alternated in one run.  Algorithmic bytes over time against the HBM copy bandwidth measured in the same run.
CUDA events, warmed up; card name and power limit printed first.
    python profiles/prof_s2_grid.py [reps]"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import kernels, synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("card:", smi[0] if smi else torch.cuda.get_device_name(dev))


def timed(fn, r=reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(r):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / r


src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
dst = torch.empty_like(src)
hbm = 2 * src.numel() * 4 / timed(lambda: dst.copy_(src), 10) / 1e6
print(f"HBM copy bandwidth (measured, 4 GiB d2d): {hbm:.0f} GB/s")
del src, dst

Hr, Wr, B = 1280, 1242, 285
w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, dev, good=good)
gx, gy = (torch.from_numpy(a).to(dev) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
src_gt = (-118.60, 0.000542232520256367, 0.0, 34.90, 0.0, -0.000542232520256367)
s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
target = hwarp.s2_target(src_gt, gx.shape, s2g)
Ho, Wo = gx.shape
Hd, Wd = target.shape
No, Nd = Ho * Wo, Hd * Wd
ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device=dev)
K = ps.K
print(f"ortho {Ho}x{Wo} -> utm {Hd}x{Wd}, scales {target.scales[0]:.4f} {target.scales[1]:.4f}, K = {K}")

# preallocated buffers: the timed region allocates nothing it does not have to
srcp = kernels.alloc_planes(K, (Ho, Wo), dev)
valid_o = torch.empty((Ho, Wo), dtype=torch.bool, device=dev)
bands = kernels.alloc_planes(K, (Hd, Wd), dev)
matched = kernels.alloc_planes(K, (Hd, Wd), dev)
dvalid = torch.empty((Hd, Wd), dtype=torch.bool, device=dev)
fm = torch.empty((Hd, Wd), dtype=torch.bool, device=dev)
coords = target.coords(dev)
ps.bands_from_raw(raw, gx, gy, bands_out=srcp, valid_out=valid_o)
kernels.warp_planes(srcp, valid_o, coords, target.scales, kernel="cubic", fill_out=ps.fill_out, out=bands,
                    valid_out=dvalid, fit_mask_out=fm)
s2 = synthetic.s2_reference_torch(torch.nan_to_num(bands), seed=1)
mom, fmf, _, _ = ps.fit(bands, s2, dvalid, fm)

t_srf = timed(lambda: ps.bands_from_raw(raw, gx, gy, bands_out=srcp, valid_out=valid_o, want_diag=False))
t_coords = timed(lambda: kernels.warp_coords(src_gt, target.dst_gt, target.shape, utm_zone=11, device=dev))
t_warp = timed(lambda: kernels.warp_planes(srcp, valid_o, coords, target.scales, kernel="cubic", fill_out=ps.fill_out,
                                           out=bands, valid_out=dvalid, fit_mask_out=fm))
t_fit = timed(lambda: ps.fit(bands, s2, dvalid, fm))
t_apply = timed(lambda: kernels.poly_solve_apply(bands, mom, fmf, 2, min_count=ps.min_count, out=matched))
wp_bytes = K * No * 4 + No + 16 * Nd + K * Nd * 4 + 2 * Nd
print(f"stage glt_srf          {t_srf:8.3f} ms")
print(f"stage coords           {t_coords:8.3f} ms   (skipped when cached)")
print(f"stage warp_planes      {t_warp:8.3f} ms   {wp_bytes / 1e9:.3f} GB algorithmic -> "
      f"{wp_bytes / t_warp / 1e6:.0f} GB/s = {wp_bytes / t_warp / 1e6 / hbm:.2f} of measured HBM")
print(f"stage fit              {t_fit:8.3f} ms")
print(f"stage solve/apply      {t_apply:8.3f} ms")


def plane_path():
    return ps.synthesize_on_s2_grid(raw, gx, gy, s2, target, bands_out=bands, matched_out=matched)


def plane_path_uncached():
    target._coords.clear()
    return plane_path()


P = kernels.padded_bands(B)
obuf = torch.empty((Ho, Wo, P), dtype=torch.float32, device=dev)
wbuf = torch.empty((Hd, Wd, P), dtype=torch.float32, device=dev)
cb = kernels.alloc_planes(K, (Hd, Wd), dev)
cfm = torch.empty((Hd, Wd), dtype=torch.bool, device=dev)


def chained_path():
    _, v, _ = kernels.glt_ortho(raw, gx, gy, out=obuf, out_pix_stride=P, want_diag=False)
    warped = kernels.warp(obuf[:, :, :B], src_gt, target.dst_gt, target.shape, utm_zone=11, scales=target.scales,
                          nodata=-9999.0, out=wbuf[:, :, :B])
    kernels.srf_integrate(warped, ps.W, cb, fit_mask_out=cfm, gate_k=0, gate_gt=0.0)
    cov = warped[..., 0] != -9999.0
    m, f, _, _ = ps.fit(cb, s2, cov, cfm & cov)
    return kernels.poly_solve_apply(cb, m, f, 2, min_count=ps.min_count, out=matched)


rows = {"synthesize_on_s2_grid (cached coords)": [], "synthesize_on_s2_grid (coords each call)": [],
        "chained glt_ortho -> warp -> srf_integrate -> fit -> apply": []}
for _ in range(3):                                   # alternate the variants: shared hosts drift
    rows["synthesize_on_s2_grid (cached coords)"].append(timed(plane_path))
    rows["synthesize_on_s2_grid (coords each call)"].append(timed(plane_path_uncached))
    rows["chained glt_ortho -> warp -> srf_integrate -> fit -> apply"].append(timed(chained_path))
for name, ts in rows.items():
    print(f"{name:60s} " + " ".join(f"{t:7.3f}" for t in ts) + f"  ms (median {sorted(ts)[1]:.3f})")
a = sorted(rows["synthesize_on_s2_grid (cached coords)"])[1]
c = sorted(rows["chained glt_ortho -> warp -> srf_integrate -> fit -> apply"])[1]
print(f"plane path / chained path: {a / c:.3f} ({c / a:.1f}x faster)")
