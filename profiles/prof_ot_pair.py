"""Timing of OT-target colour matching in the pair pipeline (PairSynthesizer(targets="ot")) on the granule workload of
profiles/prof_s2_grid.py: raw 1280 x 1242 x 285, 25 degree GLT, the zone 11 60 m target (1215 x 959), deg 4 with the
(2, 98) stretch, at K = 3 (B4, B3, B2, the reference script's case) and K = 12.  In one run:
  (a) synthesize_on_s2_grid with targets="paired" against targets="ot" (whole call, end to end);
  (b) the OT tail split into its stages, each on its own: planar pair compaction (+ the count download), the host
      draw (numpy Generator.choice), the planar gather, the Sinkhorn (with its iteration count) and the moments +
      solve / apply;
  (c) a 64-granule sharded OT fit on one GPU (the granule above 64 times: 64 units, one union draw).
CUDA events, warmed up; card name and power limit first.
    python profiles/prof_ot_pair.py [reps]"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import kernels, synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("card:", smi[0] if smi else torch.cuda.get_device_name(dev))


def timed(fn, r=reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(r):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / r


def host_timed(fn, r=reps):
    fn()
    t0 = time.perf_counter()
    for _ in range(r):
        fn()
    return (time.perf_counter() - t0) / r * 1e3


Hr, Wr, B = 1280, 1242, 285
w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, dev, good=good)
gx, gy = (torch.from_numpy(a).to(dev) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
src_gt = (-118.60, 0.000542232520256367, 0.0, 34.90, 0.0, -0.000542232520256367)
s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
target = hwarp.s2_target(src_gt, gx.shape, s2g)
Hd, Wd = target.shape
print(f"granule {Hr} x {Wr} x {B} -> zone 11 60 m target {Hd} x {Wd}, deg 4, stretch (2, 98), n_samples 5000")

table = synthetic_s2_srf()
for K, srf in ((3, {b: table[b] for b in ("B4", "B3", "B2")}), (12, table)):
    kw = dict(deg=4, device=dev, stretch=(2, 98), gate_band="B2")
    paired = PairSynthesizer(w, srf, good, **kw)
    ot = PairSynthesizer(w, srf, good, targets="ot", **kw)
    assert ot.K == K
    b0 = paired.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((K, Hd, Wd), device=dev), target).bands
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(b0), seed=1)
    t_p = timed(lambda: paired.synthesize_on_s2_grid(raw, gx, gy, s2, target))
    t_o = timed(lambda: ot.synthesize_on_s2_grid(raw, gx, gy, s2, target))
    res = ot.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    print(f"K = {K:2d}: synthesize_on_s2_grid paired {t_p:7.3f} ms, ot {t_o:7.3f} ms "
          f"(Sinkhorn iterations {int(res.ot_info[0])}, err {res.ot_info[1]:.2e})")

    # the OT tail, stage by stage, on this result's planes
    bands, m, xl, yl = res.bands, res.fit_mask, res.x_limits, res.y_limits
    lists = {}

    def compact():
        lists["l"] = kernels.compact_planes_pair(bands, s2, m, x_stretch=xl, y_stretch=yl)
        lists["n"] = torch.cat([lists["l"][1], lists["l"][3]]).tolist()
    t_c = host_timed(compact)
    nx, ny = lists["n"]
    sel = {}

    def draw():
        rng = np.random.default_rng(0)
        sel["x"] = rng.choice(nx, size=min(5000, nx), replace=False).astype(np.int64)
        sel["y"] = rng.choice(ny, size=min(5000, ny), replace=False).astype(np.int64)
    t_d = host_timed(draw)
    sx, sy = torch.from_numpy(sel["x"]).to(dev), torch.from_numpy(sel["y"]).to(dev)
    ix, _, iy, _ = lists["l"]
    XY = {}

    def gather():
        XY["X"] = kernels.gather_planes_f64(bands, ix, sx, stretch=xl)
        XY["Y"] = kernels.gather_planes_f64(s2, iy, sy, stretch=yl)
    t_g = timed(gather)
    t_s = timed(lambda: XY.__setitem__("yb", kernels.sinkhorn_barycentric(XY["X"], XY["Y"], 0.05, 300, 1e-6)))
    it = int(XY["yb"][1][0].item())

    def solve_apply():
        mom = kernels.polyfit_moments_f64(XY["X"], XY["yb"][0], 4)
        kernels.poly_solve_apply(bands, mom, m, 4, min_count=0, x_stretch=xl)
    t_a = timed(solve_apply)
    print(f"         OT tail: compaction + counts {t_c:.3f} ms (host clock, incl. download), draw {t_d:.3f} ms (host), "
          f"gather {t_g:.3f} ms, Sinkhorn {t_s:.3f} ms ({it} iterations, {t_s / max(it, 1) * 1e3:.1f} us each), "
          f"moments + solve / apply {t_a:.3f} ms")
    del paired, ot, res, lists, XY

# 64 granules, one union, one GPU
ps = PairSynthesizer(w, table, good, deg=4, device=dev, stretch=(2, 98), stretch_scope="fit", targets="ot")
b0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K, Hd, Wd), device=dev), target).bands
s2 = synthetic.s2_reference_torch(torch.nan_to_num(b0), seed=1)
g = {"raw": raw, "glt_x": gx, "glt_y": gy, "s2_ref": s2, "target": target}
granules = [g] * 64
t64 = timed(lambda: ps.synthesize_sharded(granules), r=max(reps // 5, 1))
r64 = ps.synthesize_sharded(granules)
paired64 = PairSynthesizer(w, table, good, deg=4, device=dev, stretch=(2, 98), stretch_scope="fit")
tp64 = timed(lambda: paired64.synthesize_sharded(granules), r=max(reps // 5, 1))
print(f"64-granule sharded fit, K = 12, one GPU: ot {t64:.1f} ms ({t64 / 64:.2f} ms per granule, Sinkhorn iterations "
      f"{int(r64[0].ot_info[0])}), paired {tp64:.1f} ms ({tp64 / 64:.2f} ms per granule)")
