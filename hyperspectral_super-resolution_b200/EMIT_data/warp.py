"""The UTM warp of ``nc_to_envi`` without the ``gdalwarp`` subprocess (EMIT_data/emit_proj.py:876-940).

The reference projects the WGS-84 ortho cube onto the Sentinel-2 UTM grid with

    gdalwarp -t_srs <S2 CRS> -te <extent snapped to the S2 origin> -ts cols rows
             -srcnodata -9999 -dstnodata -9999 -r cubic -of ENVI src dst

after computing the snapped extent with ``_bounds_to_out_crs`` (:309-324), ``_intersect`` (:326-332) and
``_compute_te`` (:354-382).  Here the extent arithmetic is host numpy (it is four corner points) and the resampling
is one CUDA kernel (``hsr_warp_f32``); there is no CPU resampler.  Supported CRS pair: geographic WGS-84 source
(EPSG:4326, what the EMIT geotransform is) and WGS-84 / UTM destination (EPSG:326zz / 327zz, what Sentinel-2 tiles
are); or one shared CRS (affine only).  Parity with GDAL / PROJ is unpinned — see ``oracle/warp.py``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from .. import kernels
from .._host import is_numpy_like, to_device, to_host

NO_DATA_VALUE = -9999.0   # reference emit_proj.py:27

_A = 6378137.0
_F = 1.0 / 298.257223563
_K0 = 0.9996


def _kruger():
    n = _F / (2.0 - _F)
    p = [n ** k for k in range(7)]
    A = _A / (1.0 + n) * (1.0 + p[2] / 4.0 + p[4] / 64.0 + p[6] / 256.0)
    alpha = np.array([
        p[1] / 2 - 2 * p[2] / 3 + 5 * p[3] / 16 + 41 * p[4] / 180 - 127 * p[5] / 288 + 7891 * p[6] / 37800,
        13 * p[2] / 48 - 3 * p[3] / 5 + 557 * p[4] / 1440 + 281 * p[5] / 630 - 1983433 * p[6] / 1935360,
        61 * p[3] / 240 - 103 * p[4] / 140 + 15061 * p[5] / 26880 + 167603 * p[6] / 181440,
        49561 * p[4] / 161280 - 179 * p[5] / 168 + 6601661 * p[6] / 7257600,
        34729 * p[5] / 80640 - 3418889 * p[6] / 1995840,
        212378941 * p[6] / 319334400])
    beta = np.array([
        p[1] / 2 - 2 * p[2] / 3 + 37 * p[3] / 96 - p[4] / 360 - 81 * p[5] / 512 + 96199 * p[6] / 604800,
        p[2] / 48 + p[3] / 15 - 437 * p[4] / 1440 + 46 * p[5] / 105 - 1118711 * p[6] / 3870720,
        17 * p[3] / 480 - 37 * p[4] / 840 - 209 * p[5] / 4480 + 5569 * p[6] / 90720,
        4397 * p[4] / 161280 - 11 * p[5] / 504 - 830251 * p[6] / 7257600,
        4583 * p[5] / 161280 - 108847 * p[6] / 3991680,
        20648693 * p[6] / 638668800])
    return A, alpha, beta


_AK, _ALPHA, _BETA = _kruger()
_E = math.sqrt(_F * (2.0 - _F))
_J2 = 2.0 * np.arange(1, 7)


def epsg_to_utm(epsg: int) -> Tuple[int, bool]:
    """EPSG:326zz -> (zone, False), EPSG:327zz -> (zone, True)."""
    epsg = int(epsg)
    if 32601 <= epsg <= 32660:
        return epsg - 32600, False
    if 32701 <= epsg <= 32760:
        return epsg - 32700, True
    raise ValueError(f"EPSG:{epsg} is not a WGS-84 UTM zone (326xx / 327xx): only those are supported as warp target")


def _taup(tau):
    sigma = np.sinh(_E * np.arctanh(_E * tau / np.hypot(1.0, tau)))
    return tau * np.hypot(1.0, sigma) - sigma * np.hypot(1.0, tau)


def utm_forward(lon, lat, zone: int, south: bool = False):
    """lon / lat (degrees, arrays) -> easting / northing (metres) in WGS-84 UTM ``zone`` (Krueger series, n^6)."""
    lon, lat = np.asarray(lon, dtype=np.float64), np.asarray(lat, dtype=np.float64)
    lam = np.radians(lon - (-183.0 + 6.0 * zone))
    tp = _taup(np.tan(np.radians(lat)))
    xi = np.arctan2(tp, np.cos(lam))
    eta = np.arcsinh(np.sin(lam) / np.hypot(tp, np.cos(lam)))
    a = _J2.reshape((-1,) + (1,) * xi.ndim)
    al = _ALPHA.reshape(a.shape)
    x = eta + np.sum(al * np.cos(a * xi) * np.sinh(a * eta), axis=0)
    y = xi + np.sum(al * np.sin(a * xi) * np.cosh(a * eta), axis=0)
    return _K0 * _AK * x + 500000.0, _K0 * _AK * y + (10000000.0 if south else 0.0)


def utm_inverse(x, y, zone: int, south: bool = False):
    """easting / northing (metres, arrays) -> lon / lat (degrees)."""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    xi = (y - (10000000.0 if south else 0.0)) / (_K0 * _AK)
    eta = (x - 500000.0) / (_K0 * _AK)
    a = _J2.reshape((-1,) + (1,) * xi.ndim)
    be = _BETA.reshape(a.shape)
    xip = xi - np.sum(be * np.sin(a * xi) * np.cosh(a * eta), axis=0)
    etap = eta - np.sum(be * np.cos(a * xi) * np.sinh(a * eta), axis=0)
    tp = np.sin(xip) / np.hypot(np.sinh(etap), np.cos(xip))
    lam = np.arctan2(np.sinh(etap), np.cos(xip))
    tau = tp.copy()
    e2m = 1.0 - _E * _E
    for _ in range(4):
        ti = _taup(tau)
        tau = tau + (tp - ti) / np.hypot(1.0, ti) * (1.0 + e2m * tau * tau) / (e2m * np.hypot(1.0, tau))
    return np.degrees(lam) + (-183.0 + 6.0 * zone), np.degrees(np.arctan(tau))


@dataclass
class S2Grid:
    """Georeferencing of the Sentinel-2 raster ``nc_to_envi`` aligns to — what the reference reads from
    ``rasterio.open(s2_tif_path)`` (emit_proj.py:772-797): CRS, affine transform, size."""
    epsg: int
    x0: float          # transform.c: left edge
    y0: float          # transform.f: top edge
    dx: float          # |transform.a|
    dy: float          # |transform.e|
    width: int
    height: int

    @property
    def bounds(self):  # (left, bottom, right, top)
        return self.x0, self.y0 - self.height * self.dy, self.x0 + self.width * self.dx, self.y0

    @classmethod
    def from_raster(cls, path) -> "S2Grid":
        """Read the grid from a GeoTIFF with rasterio (lazy import, as in the reference)."""
        try:
            import rasterio
        except ImportError as e:
            raise ImportError("reading the Sentinel-2 grid from a file needs rasterio; pass an S2Grid (or a dict with "
                              "epsg / x0 / y0 / dx / dy / width / height) instead") from e
        with rasterio.open(path) as src:  # pragma: no cover  (rasterio is not installable in the build image)
            t = src.transform
            return cls(int(src.crs.to_epsg()), float(t.c), float(t.f), abs(float(t.a)), abs(float(t.e)),
                       int(src.width), int(src.height))

    @classmethod
    def coerce(cls, g) -> "S2Grid":
        if isinstance(g, cls):
            return g
        if isinstance(g, dict):
            return cls(**{k: g[k] for k in ("epsg", "x0", "y0", "dx", "dy", "width", "height")})
        return cls.from_raster(g)


def bounds_of(gt: Sequence[float], width: int, height: int):
    """``ds.bounds`` of a north-up raster: (left, bottom, right, top)."""
    return float(gt[0]), float(gt[3] + height * gt[5]), float(gt[0] + width * gt[1]), float(gt[3])


def _bounds_to_out_crs(src_bounds, zone: int, south: bool):
    """The four corners of the source in the target CRS (reference :309-324)."""
    l, b, r, t = src_bounds
    X, Y = utm_forward([l, l, r, r], [b, t, b, t], zone, south)
    return float(X.min()), float(Y.min()), float(X.max()), float(Y.max())


def _intersect(a, b):
    l, bb, r, t = max(a[0], b[0]), max(a[1], b[1]), min(a[2], b[2]), min(a[3], b[3])   # reference :326-332
    if r <= l or t <= bb:
        return None
    return l, bb, r, t


def compute_te(src_bounds, s2: S2Grid, xres: float = 60.0, yres: float = 60.0):
    """Target extent (left, bottom, right, top): source bounds in the S2 CRS, intersected with the S2 extent and snapped
    inwards to the grid anchored at the S2 origin with step (xres, yres)  (reference ``_compute_te`` :354-382)."""
    zone, south = epsg_to_utm(s2.epsg)
    inter = _intersect(_bounds_to_out_crs(src_bounds, zone, south), s2.bounds)
    if inter is None:
        raise ValueError("No overlap between EMIT source bounds and S2 extent in out_crs.")
    il, ib, ir, it = inter
    eps = 1e-9
    left = s2.x0 + math.ceil(((il - s2.x0) / xres) - eps) * xres
    right = s2.x0 + math.floor(((ir - s2.x0) / xres) + eps) * xres
    top = s2.y0 - math.ceil(((s2.y0 - it) / yres) - eps) * yres
    bottom = s2.y0 - math.floor(((s2.y0 - ib) / yres) + eps) * yres
    if right <= left or top <= bottom:
        raise ValueError(f"Snapped TE is invalid: {(left, bottom, right, top)}")
    return left, bottom, right, top


def target_grid(src_gt, src_shape, s2, xres: float = 60.0, yres: float = 60.0, *, check_ratio: bool = True):
    """(dst_gt, (rows, cols), aligned_extent record) of the warp ``nc_to_envi`` runs (reference :886-908, :794-797)."""
    s2 = S2Grid.coerce(s2)
    if check_ratio:
        for step, d, n in ((xres, s2.dx, "dx"), (yres, s2.dy, "dy")):
            if abs((step / d) - round(step / d)) > 1e-9:
                raise ValueError(f"emit_step={step} must be integer multiple of S2 {n}={d}")
    Hs, Ws = int(src_shape[0]), int(src_shape[1])
    left, bottom, right, top = compute_te(bounds_of(src_gt, Ws, Hs), s2, xres, yres)
    cols, rows = int(round((right - left) / xres)), int(round((top - bottom) / yres))
    if cols <= 0 or rows <= 0:
        raise ValueError(f"Bad target shape cols={cols}, rows={rows} from snapped extent.")
    dst_gt = (left, (right - left) / cols, 0.0, top, 0.0, -(top - bottom) / rows)       # what -te / -ts define
    rec = {"left": left, "bottom": bottom, "right": right, "top": top, "cols": cols, "rows": rows, "xres": xres,
           "yres": yres, "anchor_x0": s2.x0, "anchor_y0": s2.y0}
    return dst_gt, (rows, cols), rec


def dst_to_src(col, row, dst_gt, src_gt, zone: int = 0, south: bool = False):
    """Destination pixel-corner coordinates (col, row arrays) -> source pixel coordinates (host numpy; used for the
    scale estimate and footprints only — the kernel transforms every pixel itself)."""
    col, row = np.asarray(col, dtype=np.float64), np.asarray(row, dtype=np.float64)
    X = dst_gt[0] + col * dst_gt[1] + row * dst_gt[2]
    Y = dst_gt[3] + col * dst_gt[4] + row * dst_gt[5]
    if zone:
        X, Y = utm_inverse(X, Y, zone, south)
    det = src_gt[1] * src_gt[5] - src_gt[2] * src_gt[4]
    dx, dy = X - src_gt[0], Y - src_gt[3]
    return (src_gt[5] * dx - src_gt[2] * dy) / det, (-src_gt[4] * dx + src_gt[1] * dy) / det


def warp_scales(dst_gt, src_gt, dst_shape, zone: int = 0, south: bool = False, npts: int = 21):
    """(xscale, yscale): destination size / extent of its edges in source pixels (22 samples per edge), the per-axis
    ratio GDAL derives from its source window and uses to widen the filter when downsampling."""
    Hd, Wd = dst_shape
    t = np.arange(npts + 1) / npts
    c = np.concatenate([t * Wd, t * Wd, np.zeros_like(t), np.full_like(t, Wd)])
    r = np.concatenate([np.zeros_like(t), np.full_like(t, Hd), t * Hd, t * Hd])
    sx, sy = dst_to_src(c, r, dst_gt, src_gt, zone, south)
    return float(Wd / (sx.max() - sx.min())), float(Hd / (sy.max() - sy.min()))


def warp_to_grid(cube, src_gt, dst_gt, dst_shape, *, epsg: Optional[int] = None, kernel: str = "cubic",
                 nodata: Optional[float] = NO_DATA_VALUE, dst_nodata: Optional[float] = None, scales=None):
    """Resample the band-interleaved cube [Hs, Ws, B] (or a plane [Hs, Ws]) from the grid ``src_gt`` onto ``dst_gt`` /
    ``dst_shape``.  ``epsg``: the destination's UTM code when the source is geographic WGS-84 (None: same CRS).
    numpy in -> numpy out, CUDA tensor in -> CUDA tensor out."""
    numpy_in = is_numpy_like(cube)
    t = to_device(cube, torch.float32)
    plane = t.dim() == 2
    if plane:
        t = t.unsqueeze(-1)
    zone, south = epsg_to_utm(epsg) if epsg else (0, False)
    if scales is None:
        scales = warp_scales(dst_gt, src_gt, dst_shape, zone, south)
    out = kernels.warp(t, src_gt, dst_gt, dst_shape, utm_zone=zone, south=south, scales=scales, kernel=kernel,
                       nodata=nodata, dst_nodata=dst_nodata)
    if plane:
        out = out[..., 0]
    return to_host(out, np.float32) if numpy_in else out


def warp_to_s2_grid(cube, src_gt, s2, xres: float = 60.0, yres: float = 60.0, *, kernel: str = "cubic",
                    nodata: float = NO_DATA_VALUE):
    """``_run_gdalwarp`` of the reference (:876-940) on arrays: returns ``(warped, dst_gt, aligned_extent)``."""
    s2 = S2Grid.coerce(s2)
    shape = cube.shape
    dst_gt, dst_shape, rec = target_grid(src_gt, shape[:2], s2, xres, yres)
    out = warp_to_grid(cube, src_gt, dst_gt, dst_shape, epsg=s2.epsg, kernel=kernel, nodata=nodata, dst_nodata=nodata)
    return out, dst_gt, rec


warp_planes = kernels.warp_planes


@dataclass
class S2Target:
    """The Sentinel-2 grid a pair is synthesised on (``PairSynthesizer.synthesize_on_s2_grid``): the grid
    ``nc_to_envi`` warps the ortho cube onto, with what the plane warp needs to reach it.

    ``s2_window`` = (row, col): where the target's top-left pixel sits in the S2 grid counted in target pixels
    (xres / yres), so that ``s2_stack_at_target_res[:, row:row + shape[0], col:col + shape[1]]`` is the reference on
    the target grid.  :meth:`coords` runs the fp64 inverse transverse Mercator once per device and keeps the result,
    so repeated syntheses on one geometry skip it."""
    src_gt: Tuple[float, ...]
    dst_gt: Tuple[float, ...]
    shape: Tuple[int, int]
    rec: dict
    zone: int
    south: bool
    scales: Tuple[float, float]
    s2_window: Tuple[int, int]
    kernel: str = "cubic"
    _coords: dict = field(default_factory=dict, repr=False, compare=False)

    def coords(self, device=None, rows=None) -> torch.Tensor:
        """[Hd, Wd, 2] f64 source pixel coordinates of the target's pixel centres on ``device`` (cached).  ``rows`` =
        (r0, r1): only target rows [r0, r1), bit-identical to those rows of the whole grid and not cached (a rank of a
        mosaic transforms its own band; the whole target would be 16 bytes per pixel on every rank)."""
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if rows is not None:
            return kernels.warp_coords(self.src_gt, self.dst_gt, self.shape, utm_zone=self.zone, south=self.south,
                                       device=dev, rows=rows)
        c = self._coords.get(dev)
        if c is None:
            c = kernels.warp_coords(self.src_gt, self.dst_gt, self.shape, utm_zone=self.zone, south=self.south,
                                    device=dev)
            self._coords[dev] = c
        return c


def s2_target(glt_gt, ortho_shape, s2, xres: float = 60.0, yres: float = 60.0, kernel: str = "cubic") -> S2Target:
    """The S2 target of an ortho (GLT) grid with geotransform ``glt_gt`` and shape ``ortho_shape`` = (Ho, Wo): the
    snapped extent of ``target_grid`` (reference :354-382, :886-908), the UTM zone of the S2 CRS, the filter scales of
    ``warp_scales`` and the integer offset of the target in the S2 grid at (xres, yres).  Raises ``ValueError`` when
    the grids do not overlap, when xres / yres is not an integer multiple of the S2 pixel size, or for a kernel other
    than "cubic" / "bilinear"."""
    if kernel not in kernels.PLANE_WARP_KERNELS:
        raise ValueError(f"kernel must be one of {sorted(kernels.PLANE_WARP_KERNELS)}, got {kernel!r}")
    s2 = S2Grid.coerce(s2)
    zone, south = epsg_to_utm(s2.epsg)
    glt_gt = tuple(float(v) for v in glt_gt)
    dst_gt, shape, rec = target_grid(glt_gt, ortho_shape, s2, xres, yres)
    # compute_te snaps the extent to whole steps from the S2 origin: the offsets are integers up to rounding
    window = (int(round((s2.y0 - rec["top"]) / yres)), int(round((rec["left"] - s2.x0) / xres)))
    scales = warp_scales(dst_gt, glt_gt, shape, zone, south)
    return S2Target(glt_gt, tuple(dst_gt), tuple(shape), rec, zone, south, scales, window, kernel)
