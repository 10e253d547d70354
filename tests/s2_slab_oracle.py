"""numpy model of the row-slab bookkeeping on the Sentinel-2 grid (tests/test_s2_grid_slab_model.py,
tests/test_gpu_s2_grid_slabs.py): which ortho rows a band of target rows reads through the plane warp's filter
(hsr_warp_src_row_range), which raw rows those ortho rows reference (hsr_glt_row_range), and the rows that actually
carry a non-zero tap (the tap loop of hsr_warp_planes_f32 / s2_grid_oracle.warp_conditioned)."""
from __future__ import annotations

import math

import numpy as np

from oracle import warp as owarp


def plane_radius(scales, kernel):
    """(rx, ry, fx, fy) of the plane warp: radius ceil(r / scale) below scale 1, argument scaled by min(scale, 1)."""
    r0 = 2 if kernel == "cubic" else 1
    xs, ys = scales
    rx = r0 if xs >= 1.0 else int(math.ceil(r0 / xs))
    ry = r0 if ys >= 1.0 else int(math.ceil(r0 / ys))
    return rx, ry, min(xs, 1.0), min(ys, 1.0)


def src_row_range(coords, Hs, Ws, scales, kernel):
    """coords [..., 2] (x, y) -> (lo, hi) source rows, or None when no pixel centre is inside the Hs x Ws source."""
    _, ry, _, _ = plane_radius(scales, kernel)
    px, py = coords[..., 0].reshape(-1), coords[..., 1].reshape(-1)
    inside = (px >= 0.0) & (px < Ws) & (py >= 0.0) & (py < Hs)
    if not inside.any():
        return None
    y0 = np.floor(py[inside] - 0.5).astype(np.int64) + 1 - ry
    return int(max(0, y0.min())), int(min(Hs, (y0 + 2 * ry).max()))


def tap_rows(coords, Hs, Ws, scales, kernel):
    """Set of source rows that carry a tap of non-zero fp32-rounded weight for some pixel of coords [..., 2]."""
    rx, ry, fx, fy = plane_radius(scales, kernel)
    wfun = owarp.cubic_weight if kernel == "cubic" else owarp.bilinear_weight
    rows = set()
    for sx, sy in coords.reshape(-1, 2):
        if not (0.0 <= sx < Ws and 0.0 <= sy < Hs):
            continue
        ix, iy = int(math.floor(sx - 0.5)), int(math.floor(sy - 0.5))
        ddx, ddy = sx - 0.5 - ix, sy - 0.5 - iy
        for j in range(1 - ry, ry + 1):
            yy = iy + j
            if yy < 0 or yy >= Hs or yy in rows:
                continue
            wy = wfun((j - ddy) * fy)
            for i in range(1 - rx, rx + 1):
                xx = ix + i
                if 0 <= xx < Ws and float(np.float32(wy * wfun((i - ddx) * fx))) != 0.0:
                    rows.add(yy)
                    break
    return rows


def glt_raw_rows(gx, gy, Hr, Wr):
    """(lo, hi) raw rows the valid, in-bounds entries of GLT planes reference (hsr_glt_row_range), None if none."""
    gx, gy = np.asarray(gx, np.int64), np.asarray(gy, np.int64)
    ok = (gx != 0) & (gy != 0) & (gx - 1 >= 0) & (gx - 1 < Wr) & (gy - 1 >= 0) & (gy - 1 < Hr)
    if not ok.any():
        return None
    return int((gy[ok] - 1).min()), int((gy[ok] - 1).max()) + 1


def centres(target, rows=None):
    """[rows, Wd, 2] f64 source coordinates of the target's pixel centres on the host (EMIT_data.warp.dst_to_src)."""
    from hsr_b200.EMIT_data import warp as hwarp

    Hd, Wd = target.shape
    r0, r1 = rows if rows is not None else (0, Hd)
    rr, cc = np.meshgrid(np.arange(r0, r1, dtype=np.float64), np.arange(Wd, dtype=np.float64), indexing="ij")
    sx, sy = hwarp.dst_to_src(cc + 0.5, rr + 0.5, target.dst_gt, target.src_gt, target.zone, target.south)
    return np.stack([sx, sy], axis=-1)


def uneven_bands(Hd, n, seed=0):
    """n contiguous, non-empty [t0, t1) bands of uneven height covering [0, Hd)."""
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.choice(np.arange(1, Hd), size=n - 1, replace=False))
    edges = [0, *[int(c) for c in cuts], Hd]
    return [(edges[i], edges[i + 1]) for i in range(n)]
