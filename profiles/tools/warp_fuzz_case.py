"""Re-run one geometry of tests/test_gpu_fuzz.py::test_warp_random_geometries_with_coordinate_workspace and show the worst element.
   python profiles/tools/warp_fuzz_case.py SEED [SEED ...]"""
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hsr_b200 import kernels                                  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp                  # noqa: E402
from oracle import warp as owarp                              # noqa: E402


def case(seed):
    rng = np.random.default_rng(5000 + seed)
    ND = -9999.0
    bands = int(rng.choice([1, 3, 4, 7, 12, 129, 285]))
    Hs, Ws = int(rng.integers(6, 40)), int(rng.integers(6, 40))
    Hd, Wd = int(rng.integers(1, 22)), int(rng.integers(1, 22))
    src = rng.random((Hs, Ws, bands)).astype(np.float32)
    mode = rng.integers(0, 4)
    if mode >= 1:
        yy, xx = np.mgrid[0:Hs, 0:Ws]
        src[(yy * rng.uniform(-1, 1) + xx * rng.uniform(-1, 1)) > rng.uniform(0, 10)] = ND
    if mode >= 2:
        src[rng.random(src.shape) < 0.01] = ND
        src[rng.integers(0, Hs), rng.integers(0, Ws), rng.integers(0, bands)] = np.nan
        src[rng.integers(0, Hs), rng.integers(0, Ws), rng.integers(0, bands)] = np.inf
    nodata = None if mode == 3 and rng.random() < 0.5 else ND
    sgt = (1000.0, 10.0, 0.0, 5000.0, 0.0, -10.0)
    th = rng.uniform(0, 2 * np.pi) if rng.random() < 0.5 else rng.uniform(-0.05, 0.05)
    fx, fy = rng.uniform(0.35, 2.5, size=2)
    cx, cy = 1000.0 + rng.uniform(0.2, 0.8) * Ws * 10.0, 5000.0 - rng.uniform(0.2, 0.8) * Hs * 10.0
    a, b_, d_, e = 10 * fx * np.cos(th), 10 * fy * np.sin(th), 10 * fx * np.sin(th), -10 * fy * np.cos(th)
    dgt = (cx - a * Wd / 2 - b_ * Hd / 2, a, b_, cy - d_ * Wd / 2 - e * Hd / 2, d_, e)
    kernel = "cubic" if rng.random() < 0.7 else "bilinear"
    scales = hwarp.warp_scales(dgt, sgt, (Hd, Wd)) if rng.random() < 0.8 else (1.0, 1.0)
    r0 = 2 if kernel == "cubic" else 1
    if max(np.ceil(r0 / min(scales[0], 1.0)), np.ceil(r0 / min(scales[1], 1.0))) > 8:
        scales = (1.0, 1.0)
    want = owarp.warp(src, sgt, dgt, Hd, Wd, utm=False, nodata=nodata, kernel=kernel, scales=scales)
    if rng.random() < 0.5:
        P = kernels.padded_bands(bands)
        buf = torch.full((Hs, Ws, P), 55.0, dtype=torch.float32, device="cuda")
        buf[..., :bands] = torch.from_numpy(src).cuda()
        s = buf[..., :bands]
    else:
        s = torch.from_numpy(src).cuda()
    out = None if rng.random() < 0.5 else torch.empty((Hd, Wd, bands), dtype=torch.float32, device="cuda")
    got = kernels.warp(s, sgt, dgt, (Hd, Wd), scales=scales, kernel=kernel, nodata=nodata, out=out).cpu().numpy()
    ok = np.isfinite(want)
    err = np.where(ok, np.abs(got.astype(np.float64) - want), 0.0)
    bar = 1e-5 * np.maximum(np.abs(want), 1.0) * 4 + 1e-6
    bad = ok & (err > bar)
    print(f"seed {seed}: bands {bands} src {Hs}x{Ws} dst {Hd}x{Wd} mode {int(mode)} nodata {nodata} kernel {kernel} scales "
          f"{scales[0]:.3f} {scales[1]:.3f} records {'padded' if s.stride(1) != bands else 'dense'}: {int(bad.sum())} elements over the bar")
    for r, c, b in list(zip(*np.nonzero(bad)))[:6]:
        sx, sy = owarp.dst_to_src(c, r, dgt, sgt, 0, False, False)
        ix, iy = int(math.floor(sx - 0.5)), int(math.floor(sy - 0.5))
        win = src[max(iy - 7, 0):iy + 9, max(ix - 7, 0):ix + 9, b]
        print(f"   px ({r},{c}) band {b}: got {got[r, c, b]!r} want {want[r, c, b]!r} err {err[r, c, b]:.3e}; src centre ({sx:.2f},{sy:.2f}); "
              f"window values min {np.nanmin(win):.4g} max {np.nanmax(win[np.isfinite(win)]):.4g}, nodata in window {int((win == -9999.0).sum())}, non-finite {int((~np.isfinite(win)).sum())}")


for sd in sys.argv[1:]:
    case(int(sd))
