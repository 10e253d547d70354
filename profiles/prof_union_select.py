"""Timing of the union percentile select (kernels.masked_percentiles_union: 4 radix passes, histograms summed over
units) for a granule-size K = 12 (x, y) pair split into 1, 4 and 16 units on one GPU, next to the one-pass select
(kernels.masked_percentiles) on the same pixels; per-pass bytes over time against the HBM bandwidth measured in the same
run (a device-to-device copy).  CUDA events; card name and power limit printed first.
    python profiles/prof_union_select.py [reps]"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import kernels  # noqa: E402

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


# HBM bandwidth: copy of a 4 GiB buffer (read + write), far larger than the 126 MB L2
src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
dst = torch.empty_like(src)
ms = timed(lambda: dst.copy_(src), 10)
hbm = 2 * src.numel() * 4 / ms / 1e6
print(f"HBM copy bandwidth (measured, 4 GiB d2d): {hbm:.0f} GB/s")
del src, dst

K, n = 12, 1685 * 1667
g = torch.Generator(device=dev).manual_seed(0)
mask = torch.rand(n, generator=g, device=dev) < 0.566
x = kernels.alloc_planes(K, (n,), dev)
y = kernels.alloc_planes(K, (n,), dev)
x.copy_((torch.rand((K, n), generator=g, device=dev) ** 2 * 0.8).clamp_(0.08, 1.0) - 0.08)   # image-like, 10 % zeros
y.copy_(torch.rand((K, n), generator=g, device=dev) * 0.5 + 0.1)
ms_one = timed(lambda: kernels.masked_percentiles(x, mask, [2, 98], y=y))
ox, oy = kernels.masked_percentiles(x, mask, [2, 98], y=y)
print(f"one-pass select, K = {K} pair, n = {n}: {ms_one * 1e3:.1f} us")
pass_bytes = 2 * K * n * 4 + n             # both plane sets + the mask once per pass (its re-reads hit L2)
for units in (1, 4, 16):
    b = [n * i // units // 4 * 4 for i in range(units)] + [n]     # 16-byte aligned unit starts
    parts = [(x[:, b[i]:b[i + 1]], y[:, b[i]:b[i + 1]], mask[b[i]:b[i + 1]]) for i in range(units)]
    ms_u = timed(lambda: kernels.masked_percentiles_union(parts, [2, 98]))
    ux, uy = kernels.masked_percentiles_union(parts, [2, 98])
    same = torch.equal(ux.view(torch.int64), ox.view(torch.int64)) and torch.equal(uy.view(torch.int64), oy.view(torch.int64))
    gbs = 4 * pass_bytes / ms_u / 1e6
    print(f"union select, {units:2d} unit(s): {ms_u * 1e3:.1f} us ({ms_u / ms_one:.2f} x one-pass), "
          f"{pass_bytes / 1e6:.0f} MB per pass x 4 -> {gbs:.0f} GB/s = {gbs / hbm:.2f} of measured HBM; "
          f"bit-identical to one-pass: {same}")
