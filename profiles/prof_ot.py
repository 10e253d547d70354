"""Timing of the OT target stage (fit_ot_poly_rgb, s2_emit/poly_regression.py:16-62) at the reference's sizes:
5000 x 5000 samples, reg 0.05, <= 300 iterations, on a granule-sized RGB pair.
    python profiles/prof_ot.py
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hsr_b200 import kernels  # noqa: E402
from hsr_b200.s2_emit import poly_regression  # noqa: E402

dev = torch.device("cuda", 0)
H, W = 1685, 1667
g = torch.Generator(device=dev).manual_seed(0)
src = torch.rand((H, W, 3), generator=g, device=dev) ** 1.5 * torch.tensor([0.9, 0.7, 0.5], device=dev)
ref = (0.8 * src ** 2 + 0.15 * src + 0.02 + 0.02 * torch.randn((H, W, 3), generator=g, device=dev)).clamp(0, 1)
mask = torch.rand((H, W), generator=g, device=dev) < 0.566


def timed(name, fn, reps=3, nbytes=None):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / reps * 1e3
    extra = f"   {nbytes / ms / 1e6:8.1f} GB/s" if nbytes else ""
    print(f"{name:60s} {ms:9.3f} ms{extra}")
    return out


c, info = timed("fit_ot_poly_rgb (5000 samples, deg 4, reference defaults)",
                lambda: poly_regression.fit_ot_poly_rgb(src, ref, mask, deg=4, return_info=True))
print("   info:", info)
X = torch.rand((5000, 3), generator=g, device=dev, dtype=torch.float64)
Y = torch.rand((5000, 3), generator=g, device=dev, dtype=torch.float64) ** 2
for iters in (300,):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernels.sinkhorn_barycentric(X, Y, 0.05, iters, 0.0)
    torch.cuda.synchronize()
    e0.record()
    _, inf = kernels.sinkhorn_barycentric(X, Y, 0.05, iters, 0.0)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    passes = 1                                                     # sweeps of K per iteration
    nbytes = 5000 * 5000 * 8 * (passes * iters + 3)
    print(f"sinkhorn 5000x5000, {iters} iterations (stopThr 0)              {ms:9.3f} ms   {nbytes / ms / 1e6:8.1f} GB/s of K traffic"
          f"   ({ms / iters * 1e3:.1f} us / iteration, {passes} sweep(s) of K each)")
idx, cnt = timed("compact_finite_rows (2.8 Mpx x 3)", lambda: kernels.compact_finite_rows(src.reshape(-1, 3), mask.reshape(-1)),
                 nbytes=H * W * 13 + 4 * int(mask.sum()))
