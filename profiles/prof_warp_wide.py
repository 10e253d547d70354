"""Timing of the general grid warp (hsr_warp_f32) on inputs whose filter is wider than the quad and lane kernels hold
(radius > 4), the inputs that take the exact pass.  CUDA events, warm-up, medians.
  (a) a 12-band 10980 x 10980 S2-like stack (a corner of fill) -> a 60 m grid shifted by a third of a pixel, bilinear
      (radius 6);
  (b) the 1685 x 1667 x 285 granule ortho cube of prof_warp.py (records padded to 288) -> a same-CRS grid 3.4x
      coarser, cubic (radius 7);
  (c) the same cube with x scale 0.4 and y scale 1, cubic (radii 5 x 2).
Each output is also checked against oracle/warp.py on a crop across the edge of the data.
    python profiles/prof_warp_wide.py [--reps N] [--lib PATH] [--dump DIR]
    python profiles/prof_warp_wide.py --compare DIR_A DIR_B
--lib times another build of libhsr_b200.so (another commit's, for a before / after comparison); --dump saves the
outputs (.npy) so that --compare can set two builds side by side on the timed inputs."""
import argparse
import ctypes
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ND = -9999.0
RTOL, ATOL = 1e-5, 1e-6
CASES = ("a_s2_bilinear_r6", "b_cube_cubic_r7", "c_cube_cubic_r5x2")


def oracle_crop(src, sgt, dgt, out, kernel, scales):
    """Max error over the bar of an 8 x 8 crop of `out` against oracle/warp.py.  The crop straddles the first change of
    coverage (the edge of the data) along the middle row or row Hd / 8; the source is cut with a margin wider than the
    filter."""
    from oracle import warp as owarp
    Hd, Wd = out.shape[:2]
    r, c = Hd // 2, Wd // 2
    for rr in (Hd // 2, Hd // 8):
        cov = (out[rr, :, 0] != ND).cpu().numpy()
        flips = np.nonzero(cov[1:] != cov[:-1])[0]
        if flips.size:
            r, c = rr, int(flips[0])
            break
    r0, c0 = max(r - 4, 0), max(c - 4, 0)
    h, w = min(8, Hd - r0), min(8, Wd - c0)
    Hs, Ws = src.shape[:2]
    rad = math.ceil(2 / min(scales[0], scales[1], 1.0)) + 2
    xa, xb = (dgt[0] + c0 * dgt[1] - sgt[0]) / sgt[1], (dgt[0] + (c0 + w) * dgt[1] - sgt[0]) / sgt[1]
    ya, yb = (dgt[3] + r0 * dgt[5] - sgt[3]) / sgt[5], (dgt[3] + (r0 + h) * dgt[5] - sgt[3]) / sgt[5]
    x0, x1 = max(int(math.floor(xa)) - rad, 0), min(int(math.ceil(xb)) + rad, Ws)
    y0, y1 = max(int(math.floor(ya)) - rad, 0), min(int(math.ceil(yb)) + rad, Hs)
    s = src[y0:y1, x0:x1].cpu().numpy()
    csgt = (sgt[0] + x0 * sgt[1], sgt[1], 0.0, sgt[3] + y0 * sgt[5], 0.0, sgt[5])
    cdgt = (dgt[0] + c0 * dgt[1], dgt[1], 0.0, dgt[3] + r0 * dgt[5], 0.0, dgt[5])
    want = owarp.warp(s, csgt, cdgt, h, w, utm=False, nodata=ND, kernel=kernel, scales=scales)
    got = out[r0:r0 + h, c0:c0 + w].cpu().numpy().astype(np.float64)
    same = np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got == ND, want == ND)
    ok = np.isfinite(want) & (want != ND)
    worst = float((np.abs(got[ok] - want[ok]) / (RTOL * np.abs(want[ok]) + ATOL)).max()) if ok.any() else 0.0
    return f"oracle crop {h}x{w} at ({r0},{c0}): patterns {'equal' if same else 'DIFFER'}, {int(ok.sum())} values, " \
           f"max err / bar {worst:.3f}"


def compare(dir_a, dir_b):
    for name in CASES:
        a = np.load(os.path.join(dir_a, name + ".npy"), mmap_mode="r")
        b = np.load(os.path.join(dir_b, name + ".npy"), mmap_mode="r")
        assert a.shape == b.shape, (name, a.shape, b.shape)
        worst, over, nan_diff, nd_diff = 0.0, 0, 0, 0
        for r in range(0, a.shape[0], 64):
            x, y = np.asarray(a[r:r + 64], np.float64), np.asarray(b[r:r + 64], np.float64)
            nan_diff += int((np.isnan(x) != np.isnan(y)).sum())
            nd_diff += int(((x == ND) != (y == ND)).sum())
            ok = np.isfinite(x) & np.isfinite(y)
            err = np.abs(x[ok] - y[ok])
            bar = RTOL * np.abs(x[ok]) + ATOL
            over += int((err > bar).sum())
            if err.size:
                worst = max(worst, float((err / bar).max()))
        print(f"{name:20s} {a.shape}: NaN pattern differs at {nan_diff}, nodata pattern at {nd_diff}, "
              f"max |a - b| / (1e-5 |a| + 1e-6) = {worst:.3f}, elements over that bar: {over}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--lib")
    ap.add_argument("--dump")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
        return

    import torch

    from hsr_b200 import _lib, kernels, synthetic
    from hsr_b200.EMIT_data import warp as hwarp

    if args.lib:
        _lib.LIB_PATH = os.path.abspath(args.lib)
        _lib.ABI_VERSION = ctypes.CDLL(_lib.LIB_PATH).hsr_version()     # another commit's build may carry an older ABI
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    print(f"library {os.path.relpath(_lib.LIB_PATH, root)} (ABI {_lib.lib().hsr_version()}) on {torch.cuda.get_device_name()}")

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    def run(name, src, sgt, dgt, shape, kernel):
        scales = hwarp.warp_scales(dgt, sgt, shape)
        B = src.shape[2]
        out = torch.empty((shape[0], shape[1], kernels.padded_bands(B)), dtype=torch.float32, device="cuda")[:, :, :B]
        ms = timed(lambda: kernels.warp(src, sgt, dgt, shape, scales=scales, kernel=kernel, nodata=ND, out=out))
        r0 = 2 if kernel == "cubic" else 1
        radii = [math.ceil(r0 / min(s, 1.0)) for s in scales]
        print(f"{name:20s} {src.shape[0]}x{src.shape[1]}x{B} -> {shape[0]}x{shape[1]} {kernel} radii {radii[0]}x{radii[1]}: "
              f"{ms:8.3f} ms  ({shape[0] * shape[1] / ms / 1e3:.1f} Mpix/s)  {oracle_crop(src, sgt, dgt, out, kernel, scales)}",
              flush=True)
        if args.dump:
            os.makedirs(args.dump, exist_ok=True)
            np.save(os.path.join(args.dump, name + ".npy"), out.cpu().numpy())

    # (a) S2-like stack: 10 m pixels, a triangle of fill in one corner (the edge of an orbit)
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 10980
    s2 = torch.rand((n, n, 12), generator=g, device="cuda").mul_(0.9).add_(0.05)
    idx = torch.arange(n, device="cuda")
    s2[(idx[:, None] + idx[None, :]) < 3000] = ND
    sgt = (300000.0, 10.0, 0.0, 3900000.0, 0.0, -10.0)
    run(CASES[0], s2, sgt, (300020.0, 60.0, 0.0, 3899980.0, 0.0, -60.0), (1829, 1829), "bilinear")
    del s2, idx
    torch.cuda.empty_cache()

    # (b), (c): the granule ortho cube (GLT fill outside the rotated swath), on a metric same-CRS grid
    Hr, Wr, B = 1280, 1242, 285
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, "cuda")
    gx, gy = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    buf = torch.empty((gx.shape[0], gx.shape[1], kernels.padded_bands(B)), dtype=torch.float32, device="cuda")
    _, valid, _ = kernels.glt_ortho(raw, gx, gy, out=buf, out_pix_stride=buf.shape[2])
    del raw
    Ho, Wo = valid.shape
    cube = buf[:, :, :B]
    sgt = (500000.0, 60.0, 0.0, 4000000.0, 0.0, -60.0)
    run(CASES[1], cube, sgt, (500000.0, 204.0, 0.0, 4000000.0, 0.0, -204.0), (int(Ho / 3.4), int(Wo / 3.4)), "cubic")
    run(CASES[2], cube, sgt, (500000.0, 150.0, 0.0, 4000000.0, 0.0, -60.0), (Ho, int(Wo / 2.5)), "cubic")


if __name__ == "__main__":
    main()
