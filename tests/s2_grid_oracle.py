"""Reference pieces for the pair on the Sentinel-2 grid (tests/test_s2_grid_model.py, tests/test_gpu_s2_grid.py).

``warp_conditioned`` is the tap loop of ``oracle.warp.warp`` (same weights, the same fp32 rounding of the tap weight,
zero weights skipped, taps outside the source skipped, centre outside the source or weight sum < 1e-6 uncovered)
kept in fp64 end to end, with tap validity either per band (value != nodata, as gdalwarp) or per source pixel
(``src_valid``, as ``hsr_warp_planes_f32``).  Next to the result it returns the conditioning figure of each output

    C_k(d) = sum_t |w_t| |v_tk| / |sum_t w_t|

which bounds how far fp rounding of the inputs can move the renormalised sum.  Near the swath edge GDAL's partial sums
can cancel (weight sums just above 1e-6), so no fixed relative bar holds there; a bar scaled by C does.

``reference_chain`` is the reference's order: ``oracle.glt`` -> ``oracle.warp`` (every band) -> ``oracle.srf``.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import glt as oglt
from oracle import srf as osrf
from oracle import warp as owarp

ND = -9999.0


def warp_conditioned(src, src_gt, dst_gt, Hd, Wd, *, scales, zone=0, south=False, utm=True, kernel="cubic",
                     src_valid=None, nodata=None, fill=np.nan):
    """src [Hs, Ws, B] (any float; used in fp64) -> (out [Hd, Wd, B] f64, covered [Hd, Wd, B] bool, C [Hd, Wd, B])."""
    src = np.asarray(src, dtype=np.float64)
    Hs, Ws, B = src.shape
    out = np.full((Hd, Wd, B), fill, dtype=np.float64)
    cond = np.zeros((Hd, Wd, B))
    covered = np.zeros((Hd, Wd, B), dtype=bool)
    xs, ys = scales
    wfun, r0 = (owarp.cubic_weight, 2) if kernel == "cubic" else (owarp.bilinear_weight, 1)
    fx, fy = min(xs, 1.0), min(ys, 1.0)
    rx, ry = (r0 if xs >= 1.0 else int(math.ceil(r0 / xs))), (r0 if ys >= 1.0 else int(math.ceil(r0 / ys)))
    for row in range(Hd):
        for col in range(Wd):
            sx, sy = owarp.dst_to_src(col, row, dst_gt, src_gt, zone, south, utm)
            if not (0.0 <= sx < Ws and 0.0 <= sy < Hs):
                continue
            ix, iy = int(math.floor(sx - 0.5)), int(math.floor(sy - 0.5))
            ddx, ddy = sx - 0.5 - ix, sy - 0.5 - iy
            acc, wsum, absacc = np.zeros(B), np.zeros(B), np.zeros(B)
            for j in range(1 - ry, ry + 1):
                yy = iy + j
                if yy < 0 or yy >= Hs:
                    continue
                wy = wfun((j - ddy) * fy)
                for i in range(1 - rx, rx + 1):
                    xx = ix + i
                    if xx < 0 or xx >= Ws:
                        continue
                    w = float(np.float32(wy * wfun((i - ddx) * fx)))
                    if w == 0.0:
                        continue
                    if src_valid is not None:
                        if not src_valid[yy, xx]:
                            continue
                        ok = np.ones(B, bool)
                    else:
                        ok = np.ones(B, bool) if nodata is None else (src[yy, xx] != nodata)
                    v = src[yy, xx]
                    acc += np.where(ok, w * v, 0.0)
                    wsum += np.where(ok, w, 0.0)
                    absacc += np.where(ok, abs(w) * np.abs(v), 0.0)
            good = wsum >= 1e-6
            covered[row, col] = good
            with np.errstate(invalid="ignore", divide="ignore"):
                out[row, col, good] = acc[good] / wsum[good]
                cond[row, col, good] = absacc[good] / np.abs(wsum[good])
    return out, covered, cond


def srf_planes(cube, emit_w, table, good, names):
    """[K, H, W] f64 pseudo-S2 planes of a [H, W, B] cube (oracle.srf, reference synth.py:9-45)."""
    d = osrf.pseudo_s2_srf_integral(cube, emit_w, table, good)
    return np.stack([d[n] for n in names])


def reference_chain(raw, gx, gy, glt_gt, target, emit_w, table, good, names, *, transpose_raw_yx=False):
    """The reference's order on the oracles: (planes [K, Hd, Wd] f64, covered [Hd, Wd] bool, ortho, valid)."""
    ortho, valid, _ = oglt.glt_ortho(raw, gx, gy, transpose_raw_yx=transpose_raw_yx)
    Hd, Wd = target.shape
    warped = owarp.warp(ortho, glt_gt, target.dst_gt, Hd, Wd, zone=target.zone, south=target.south, utm=True,
                        nodata=ND, dst_nodata=ND, kernel=target.kernel, scales=target.scales)
    return srf_planes(warped, emit_w, table, good, names), warped[..., 0] != ND, ortho, valid
