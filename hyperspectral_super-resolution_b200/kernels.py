"""Tensor-level entry points of the hot path: torch CUDA tensors in, torch CUDA tensors out.

Every function here is a thin shim over one C-ABI call of ``libhsr_b200.so``
(``include/hsr_b200.h``): it validates dtype/device/layout, allocates the outputs with torch,
and launches on ``torch.cuda.current_stream()``.  Nothing is computed in Python and nothing
runs on the CPU; a non-CUDA tensor raises ``TypeError``.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib

NO_DATA_VALUE = -9999.0  # EMIT_data/emit_proj.py:27


# --------------------------------------------------------------------------------------- helpers
def _cuda(t, name: str, dtype: torch.dtype) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor on a CUDA device (got {type(t).__name__}); "
                        "use the hsr_b200.EMIT_data / hsr_b200.s2_emit wrappers for numpy input")
    if not t.is_cuda:
        raise TypeError(f"{name} must live on a CUDA device: hsr_b200 has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _pixel_major(t: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Return (tensor, pixel_stride) for a [..., B] cube whose leading dims are dense over a pixel pitch."""
    if t.dim() < 2:
        raise ValueError("cube must have at least 2 dims [..., bands]")
    B = t.shape[-1]
    if t.stride(-1) == 1 or B == 1:
        pitch = t.stride(-2) if t.shape[-2] > 1 else max(B, t.stride(-2))
        ok = pitch >= B
        expect = pitch
        for d in range(t.dim() - 2, -1, -1):
            if t.shape[d] > 1 and t.stride(d) != expect:
                ok = False
                break
            expect *= t.shape[d]
        if ok:
            return t, int(pitch)
    t = t.contiguous()
    return t, int(B)


def prepare_glt(glt_x, glt_y, device=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """GLT planes -> contiguous int32 CUDA planes, NaN -> 0 (EMIT_data/emit_proj.py:683-687)."""
    import numpy as np

    outs = []
    for g in (glt_x, glt_y):
        if isinstance(g, np.ndarray):
            g = torch.from_numpy(np.ascontiguousarray(g))
        if not isinstance(g, torch.Tensor):
            g = torch.as_tensor(g)
        if device is not None:
            g = g.to(device, non_blocking=True)
        if not g.is_cuda:
            raise TypeError("GLT planes must end up on a CUDA device (pass device=...)")
        if g.dtype.is_floating_point:
            g = torch.nan_to_num(g, nan=0.0).to(torch.int32)
        elif g.dtype != torch.int32:
            g = g.to(torch.int32)
        outs.append(g.contiguous())
    if outs[0].shape != outs[1].shape or outs[0].dim() != 2:
        raise ValueError(f"glt_x / glt_y must be 2-D planes of equal shape, got {outs[0].shape} and {outs[1].shape}")
    return outs[0], outs[1]


def _raw_geometry(raw: torch.Tensor, transpose_raw_yx: bool):
    plane = raw.dim() == 2
    r3 = raw.unsqueeze(-1) if plane else raw
    if r3.dim() != 3:
        raise ValueError(f"raw must be [H, W, B] or [H, W], got shape {tuple(raw.shape)}")
    r3, pitch = _pixel_major(r3)
    d0, d1, B = r3.shape
    raw_h, raw_w = (d1, d0) if transpose_raw_yx else (d0, d1)  # emit_proj.py:696
    return r3, pitch, int(raw_h), int(raw_w), int(B), plane


def _raw_view(d0: int, raw_h: int, raw_w: int, transpose: bool, raw_row0: int, raw_rows_total, tile_rows):
    """(ctypes RawView | None, raw_h, raw_w): ``raw`` holds only the slow-axis indices [raw_row0, raw_row0 + d0) of a
    cube with ``raw_rows_total`` of them (hsr_raw_view_t), and / or the grid is a stack of tiles ``tile_rows`` =
    (ortho rows, raw rows) per tile."""
    if raw_rows_total is None and not raw_row0 and tile_rows is None:
        return None, raw_h, raw_w
    v = _lib.RawView(0, 0, 0, 0)
    if raw_rows_total is not None or raw_row0:
        total = int(raw_rows_total) if raw_rows_total is not None else int(raw_row0) + d0
        v.row0, v.rows = int(raw_row0), d0
        if transpose:
            raw_w = total
        else:
            raw_h = total
    if tile_rows is not None:
        v.batch_out_rows, v.batch_raw_rows = int(tile_rows[0]), int(tile_rows[1])
    return v, raw_h, raw_w


def _view_diag(device, want: bool, view):
    return torch.zeros(4 if view is not None else 3, dtype=torch.int64, device=device) if want else None


PLANE_ALIGN = 32  # floats: planes start on 128-byte boundaries so that the plane kernels can use 16-byte accesses


def alloc_planes(K: int, spatial, device) -> torch.Tensor:
    """[K, *spatial] f32 planes whose plane stride is padded to a multiple of 32 floats (the ortho grid of a
    granule has an odd pixel count; dense planes would start 4-byte aligned only).  Each plane is contiguous."""
    n = 1
    for d in spatial:
        n *= int(d)
    stride = -(-max(n, 1) // PLANE_ALIGN) * PLANE_ALIGN
    buf = torch.empty((K, stride), dtype=torch.float32, device=device)
    return buf[:, :n].view((K,) + tuple(int(d) for d in spatial))


def _plane_stride(t: torch.Tensor, K: int, n: int, name: str) -> int:
    """Plane stride (elements) of a [K, ...] tensor whose planes are dense; raises if they are not."""
    if t.shape[0] != K or t.numel() != K * n:
        raise ValueError(f"{name} must hold {K} planes of {n} samples, got shape {tuple(t.shape)}")
    if n == 0:
        return 0
    inner = t[0]
    if not inner.is_contiguous():
        raise ValueError(f"{name}: every plane must be contiguous")
    stride = t.stride(0) if K > 1 else n
    if stride < n:
        raise ValueError(f"{name}: plane stride {stride} < plane size {n}")
    return int(stride)


# --------------------------------------------------------------------------------------- kernel 1
def glt_ortho(raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, *, fill: float = NO_DATA_VALUE,
              transpose_raw_yx: bool = False, out: Optional[torch.Tensor] = None,
              out_pix_stride: Optional[int] = None, want_valid: bool = True, want_diag: bool = True,
              raw_row0: int = 0, raw_rows_total: Optional[int] = None, tile_rows=None):
    """GLT-indexed ortho gather, bit-exact (EMIT_data/emit_proj.py:682-703,947-948,968-987).

    raw [Hr, Wr, B] (or a [Hr, Wr] plane) f32, glt_x / glt_y [Ho, Wo] int32 (1-based, 0 = nodata).
    Returns ``(ortho [Ho, Wo, B] f32, valid [Ho, Wo] bool | None, diag int64[3] | None)`` where
    diag = (valid_glt_count, valid_glt_inbounds_count, valid_glt_dropped_oob), still on the device.
    ``raw_row0`` / ``raw_rows_total``: ``raw`` is only the window of rows [raw_row0, raw_row0 + raw.shape[0]) of a
    cube of raw_rows_total rows (hsr_raw_view_t; diag then has a 4th entry, valid entries outside the window, which
    must be 0); ``tile_rows`` = (ortho rows, raw rows) per tile of a stacked tile batch.
    """
    _cuda(raw, "raw", torch.float32)
    gx = _cuda(glt_x, "glt_x", torch.int32)
    gy = _cuda(glt_y, "glt_y", torch.int32)
    if gx.shape != gy.shape or gx.dim() != 2:
        raise ValueError("glt_x / glt_y must be 2-D planes of equal shape")
    gx, gy = gx.contiguous(), gy.contiguous()
    r3, pitch, raw_h, raw_w, B, plane = _raw_geometry(raw, transpose_raw_yx)
    view, raw_h, raw_w = _raw_view(r3.shape[0], raw_h, raw_w, transpose_raw_yx, raw_row0, raw_rows_total, tile_rows)
    Ho, Wo = gx.shape
    with torch.cuda.device_of(r3):
        ops = int(out_pix_stride) if out_pix_stride else B
        if out is None:
            buf = torch.empty((Ho, Wo, ops), dtype=torch.float32, device=r3.device)
        else:
            buf = _cuda(out, "out", torch.float32)
            if not buf.is_contiguous() or buf.numel() < Ho * Wo * ops:
                raise ValueError("out must be a contiguous buffer of at least Ho*Wo*out_pix_stride floats")
        valid = torch.empty((Ho, Wo), dtype=torch.uint8, device=r3.device) if want_valid else None
        diag = _view_diag(r3.device, want_diag, view)
        _lib.check(_lib.lib().hsr_glt_ortho_f32(
            r3.data_ptr(), raw_h, raw_w, B, pitch, int(bool(transpose_raw_yx)), gx.data_ptr(), gy.data_ptr(),
            Ho, Wo, Wo, float(fill), buf.data_ptr(), ops, _ptr(valid), _ptr(diag),
            ctypes.byref(view) if view is not None else None, _stream()))
    ortho = buf if out is not None else (buf[..., :B] if ops != B else buf)
    if plane and out is None:
        ortho = ortho[..., 0]
    return ortho, (valid.view(torch.bool) if valid is not None else None), diag


def glt_row_range(glt_x: torch.Tensor, glt_y: torch.Tensor, raw_h: int, raw_w: int, *,
                  transpose_raw_yx: bool = False) -> torch.Tensor:
    """int64[2] on the device: [first, last + 1) raw row (raw column when transposed) that the valid, in-bounds
    entries of the GLT planes reference; (2^63 - 1 .. wrapped -1, 0) -> ``range[1] == 0`` when there is none
    (hsr_glt_row_range).  Works on any row slab of a GLT (pass contiguous row slices)."""
    gx = _cuda(glt_x, "glt_x", torch.int32)
    gy = _cuda(glt_y, "glt_y", torch.int32)
    if gx.shape != gy.shape or gx.dim() != 2:
        raise ValueError("glt_x / glt_y must be 2-D planes of equal shape")
    gx, gy = gx.contiguous(), gy.contiguous()
    Ho, Wo = gx.shape
    with torch.cuda.device_of(gx):
        rng = torch.tensor([-1, 0], dtype=torch.int64, device=gx.device)       # u64 max, 0
        _lib.check(_lib.lib().hsr_glt_row_range(gx.data_ptr(), gy.data_ptr(), Ho, Wo, Wo, int(raw_h), int(raw_w),
                                                int(bool(transpose_raw_yx)), rng.data_ptr(), _stream()))
    return rng


# --------------------------------------------------------------------------------------- kernel 2
def glt_srf(raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, W: torch.Tensor,
            fill_out: Optional[torch.Tensor] = None, *, fill: float = NO_DATA_VALUE,
            transpose_raw_yx: bool = False, materialize_ortho: bool = False,
            bands_out: Optional[torch.Tensor] = None, ortho_out: Optional[torch.Tensor] = None,
            want_valid: bool = True, want_diag: bool = True, fit_mask_out: Optional[torch.Tensor] = None,
            gate_k: int = -1, gate_gt: float = 0.0, raw_row0: int = 0, raw_rows_total: Optional[int] = None,
            tile_rows=None, valid_out: Optional[torch.Tensor] = None):
    """Fused GLT gather + SRF contraction: ``bands[k] = sum_b raw[gy, gx, b] * W[b, k]``.

    Replaces the gather of emit_proj.py:968-987 followed by s2_emit/synth.py:32-43 with the
    trapezoid weights folded into W (see ``hsr_b200.s2_emit.srf.srf_fold_weights``).
    ``fit_mask_out`` ([Ho, Wo] bool/u8): also emit the fit mask of poly_regression.py:106,
    ``valid & isfinite(bands).all(0) & (bands[gate_k] > gate_gt)``, while the planes are written.
    ``raw_row0`` / ``raw_rows_total`` / ``tile_rows``: as in :func:`glt_ortho` (hsr_raw_view_t).
    Returns ``(bands [K, Ho, Wo] f32, valid bool | None, diag | None, ortho [Ho, Wo, B] | None)``.
    """
    _cuda(raw, "raw", torch.float32)
    gx = _cuda(glt_x, "glt_x", torch.int32).contiguous()
    gy = _cuda(glt_y, "glt_y", torch.int32).contiguous()
    Wt = _cuda(W, "W", torch.float32).contiguous()
    if gx.shape != gy.shape or gx.dim() != 2:
        raise ValueError("glt_x / glt_y must be 2-D planes of equal shape")
    r3, pitch, raw_h, raw_w, B, _ = _raw_geometry(raw, transpose_raw_yx)
    view, raw_h, raw_w = _raw_view(r3.shape[0], raw_h, raw_w, transpose_raw_yx, raw_row0, raw_rows_total, tile_rows)
    if Wt.dim() != 2 or Wt.shape[0] != B:
        raise ValueError(f"W must be [bands={B}, K], got {tuple(Wt.shape)}")
    K = int(Wt.shape[1])
    Ho, Wo = gx.shape
    with torch.cuda.device_of(r3):
        if fill_out is None:
            fill_out = (Wt.double().sum(0) * float(fill)).float()
        fo = _cuda(fill_out, "fill_out", torch.float32).contiguous()
        if fo.numel() != K:
            raise ValueError("fill_out must have K entries")
        if bands_out is None:
            bands_out = alloc_planes(K, (Ho, Wo), r3.device)
        else:
            _cuda(bands_out, "bands_out", torch.float32)
        plane_stride = _plane_stride(bands_out, K, Ho * Wo, "bands_out")
        ortho = None
        if ortho_out is not None:
            ortho = _cuda(ortho_out, "ortho_out", torch.float32)
            if not ortho.is_contiguous() or ortho.numel() < Ho * Wo * B:
                raise ValueError("ortho_out must be a contiguous [Ho, Wo, B] buffer")
        elif materialize_ortho:
            ortho = torch.empty((Ho, Wo, B), dtype=torch.float32, device=r3.device)
        if valid_out is not None:           # caller-owned [Ho, Wo] bool / u8 (no allocation in a timed or captured region)
            valid = _mask_out(valid_out, Ho * Wo).view(Ho, Wo)
        else:
            valid = torch.empty((Ho, Wo), dtype=torch.uint8, device=r3.device) if want_valid else None
        diag = _view_diag(r3.device, want_diag, view)
        fm = _mask_out(fit_mask_out, Ho * Wo)
        _lib.check(_lib.lib().hsr_glt_srf_f32(
            r3.data_ptr(), raw_h, raw_w, B, pitch, int(bool(transpose_raw_yx)), gx.data_ptr(), gy.data_ptr(),
            Ho, Wo, Wo, float(fill), Wt.data_ptr(), fo.data_ptr(), K, bands_out.data_ptr(), plane_stride,
            _ptr(ortho), B, _ptr(valid), _ptr(diag), _ptr(fm), int(gate_k), float(gate_gt),
            ctypes.byref(view) if view is not None else None, _stream()))
    return bands_out, (valid.view(torch.bool) if valid is not None else None), diag, ortho


def _mask_out(t: Optional[torch.Tensor], n: int):
    """A caller-provided [n] bool/u8 output mask as a u8 view (None passes through)."""
    if t is None:
        return None
    m = t.view(torch.uint8) if t.dtype == torch.bool else t
    _cuda(m, "fit_mask_out", torch.uint8)
    if not m.is_contiguous() or m.numel() != n:
        raise ValueError(f"fit_mask_out must be a contiguous mask of {n} pixels")
    return m


def srf_integrate(cube: torch.Tensor, W: torch.Tensor, bands_out: Optional[torch.Tensor] = None, *,
                  fit_mask_out: Optional[torch.Tensor] = None, gate_k: int = -1, gate_gt: float = 0.0) -> torch.Tensor:
    """Un-fused SRF contraction of an ortho cube [..., B] -> [K, ...] (s2_emit/synth.py:32-43)."""
    _cuda(cube, "cube", torch.float32)
    Wt = _cuda(W, "W", torch.float32).contiguous()
    c, pitch = _pixel_major(cube)
    B = c.shape[-1]
    if Wt.dim() != 2 or Wt.shape[0] != B:
        raise ValueError(f"W must be [bands={B}, K], got {tuple(Wt.shape)}")
    K = int(Wt.shape[1])
    spatial = tuple(c.shape[:-1])
    n = 1
    for s in spatial:
        n *= s
    with torch.cuda.device_of(c):
        if bands_out is None:
            bands_out = alloc_planes(K, spatial, c.device)
        else:
            _cuda(bands_out, "bands_out", torch.float32)
        plane_stride = _plane_stride(bands_out, K, n, "bands_out")
        fm = _mask_out(fit_mask_out, n)
        _lib.check(_lib.lib().hsr_srf_f32(c.data_ptr(), n, B, pitch, Wt.data_ptr(), K, bands_out.data_ptr(),
                                          max(plane_stride, n), _ptr(fm), int(gate_k), float(gate_gt), _stream()))
    return bands_out


# --------------------------------------------------------------------------------------- kernel 3
def _series(t: torch.Tensor, name: str, layout: str):
    """(tensor, K, n, k_stride, n_stride) of K sample series held planar [K, ...] or interleaved [..., K]."""
    _cuda(t, name, torch.float32)
    if layout == "planar":
        K = t.shape[0]
        n = t.numel() // max(K, 1)
        dense_planes = K > 0 and n > 0 and t[0].is_contiguous() and (K == 1 or t.stride(0) >= n)
        if not dense_planes:
            t = t.contiguous()
        ks = int(t.stride(0)) if (K > 1 and n > 0) else int(n)
        return t, int(K), int(n), ks, 1
    t = t.contiguous()
    if layout == "interleaved":
        K = t.shape[-1]
        n = t.numel() // max(K, 1)
        return t, int(K), int(n), 1, int(K)
    raise ValueError("layout must be 'planar' or 'interleaved'")


def _mask_arg(mask, K: int, n: int, mask_rows: str = "auto"):
    """(mask tensor, div, mod): series k uses mask row (k // div) % mod (see include/hsr_b200.h)."""
    if mask is None:
        return None, 1, 1
    if mask.dtype == torch.bool:
        mask = mask.view(torch.uint8)
    _cuda(mask, "mask", torch.uint8)
    mask = mask.contiguous()
    if n == 0 or mask.numel() % max(n, 1) != 0:
        raise ValueError(f"mask with {mask.numel()} elements does not match n = {n}")
    rows = mask.numel() // n
    if rows == 1:
        return mask, 1, 1                      # one mask shared by all series
    if rows == K:
        return mask, 1, K                      # one mask per series
    if K % rows != 0:
        raise ValueError(f"mask with {rows} rows does not divide K = {K} series")
    if mask_rows == "inner":                   # series laid out [group][row]: row = k % rows
        return mask, 1, rows
    if mask_rows == "outer":                   # series laid out [row][group]: row = k // (K / rows)
        return mask, K // rows, rows
    raise ValueError("mask has one row per GROUP of series: pass mask_rows='inner' or 'outer'")


def poly_moments(x: torch.Tensor, y: torch.Tensor, mask: Optional[torch.Tensor], deg: int, *,
                 layout: str = "planar", mask_rows: str = "auto") -> torch.Tensor:
    """fp64 normal-equation moments [K, 3*deg+2] of K paired series (np.polyfit's X^T X / X^T y)."""
    xs, K, n, xks, xns = _series(x, "x", layout)
    ys, Ky, ny, yks, yns = _series(y, "y", layout)
    if (K, n) != (Ky, ny):
        raise ValueError(f"x and y disagree: {K}x{n} vs {Ky}x{ny}")
    m, mdiv, mmod = _mask_arg(mask, K, n, mask_rows)
    with torch.cuda.device_of(xs):
        ws = _lib.lib().hsr_workspace_bytes(_lib.HSR_OP_POLY_MOMENTS, n, K, int(deg))
        partial = torch.empty(max(ws // 8, 1), dtype=torch.float64, device=xs.device)
        moments = torch.empty((K, 3 * int(deg) + 2), dtype=torch.float64, device=xs.device)
        _lib.check(_lib.lib().hsr_poly_moments_f64(xs.data_ptr(), xks, xns, ys.data_ptr(), yks, yns, _ptr(m), mdiv,
                                                   mmod, n, K, int(deg), partial.data_ptr(), moments.data_ptr(), _stream()))
    return moments


def poly_solve(moments: torch.Tensor, deg: int, min_count: int = 0) -> torch.Tensor:
    """Solve the scaled normal equations: [K, 3*deg+2] moments -> [K, deg+1] coefficients, highest power first."""
    mo = _cuda(moments, "moments", torch.float64).contiguous()
    K = mo.shape[0]
    if mo.shape[1] != 3 * int(deg) + 2:
        raise ValueError(f"moments must be [K, {3 * int(deg) + 2}] for deg = {deg}")
    with torch.cuda.device_of(mo):
        coeffs = torch.empty((K, int(deg) + 1), dtype=torch.float64, device=mo.device)
        _lib.check(_lib.lib().hsr_poly_solve_f64(mo.data_ptr(), K, int(deg), int(min_count), coeffs.data_ptr(),
                                                 _stream()))
    return coeffs


def poly_fit(x: torch.Tensor, y: torch.Tensor, mask: Optional[torch.Tensor], deg: int, *, min_count: int = 0,
             layout: str = "planar", mask_rows: str = "auto", return_moments: bool = False):
    """Per-series least-squares polynomial (np.polyfit(x[mask], y[mask], deg) for every series).
    ``return_moments``: also the [K, 3*deg+2] moments (the host mirrors repair rank-deficient series from them)."""
    mom = poly_moments(x, y, mask, deg, layout=layout, mask_rows=mask_rows)
    co = poly_solve(mom, deg, min_count)
    return (co, mom) if return_moments else co


def poly_apply(x: torch.Tensor, coeffs: torch.Tensor, mask: Optional[torch.Tensor] = None, *,
               lo: float = 0.0, hi: float = 1.0, layout: str = "planar", mask_rows: str = "auto",
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Horner apply + mask + clip (s2_emit/poly_regression.py:65-84).  ``lo > hi`` disables the clip."""
    xs, K, n, xks, xns = _series(x, "x", layout)
    co = _cuda(coeffs, "coeffs", torch.float64).contiguous()
    if co.dim() != 2 or co.shape[0] != K:
        raise ValueError(f"coeffs must be [K={K}, deg+1], got {tuple(co.shape)}")
    deg = co.shape[1] - 1
    m, mdiv, mmod = _mask_arg(mask, K, n, mask_rows)
    with torch.cuda.device_of(xs):
        if out is None:
            out = alloc_planes(K, xs.shape[1:], xs.device) if layout == "planar" else torch.empty_like(xs)
        else:
            _cuda(out, "out", torch.float32)
            if out.shape != xs.shape:
                raise ValueError("out must have the shape of x")
        if layout == "planar":
            oks, ons = _plane_stride(out, K, n, "out"), 1
        else:
            if not out.is_contiguous():
                raise ValueError("out must be contiguous")
            oks, ons = xks, xns
        _lib.check(_lib.lib().hsr_poly_apply_f32(xs.data_ptr(), xks, xns, co.data_ptr(), _ptr(m), mdiv, mmod, n, K, deg,
                                                 float(lo), float(hi), out.data_ptr(), oks, ons, _stream()))
    return out


def _grouped(t: torch.Tensor, name: str, K: int, G: int, n: int):
    """(tensor, k_stride, g_stride) of a [K, G, n]-shaped view (any trailing dims flattened into n) whose
    innermost n samples are dense."""
    _cuda(t, name, torch.float32)
    if t.numel() != K * G * n:
        raise ValueError(f"{name} must hold {K} x {G} x {n} samples, got shape {tuple(t.shape)}")
    try:
        v = t.view(K, G, n)
    except RuntimeError:
        v = t.contiguous().view(K, G, n)
    if n > 1 and v.stride(2) != 1:
        v = v.contiguous()
    ks = int(v.stride(0)) if K > 1 else G * n
    gs = int(v.stride(1)) if G > 1 else n
    return v, ks, gs


def fit_mask(x: torch.Tensor, valid: Optional[torch.Tensor] = None, *, gate_k: int = 0,
             gate_gt: float = 0.0, y: Optional[torch.Tensor] = None, groups: int = 1) -> torch.Tensor:
    """mask = valid & isfinite(x).all(0) & (x[gate_k] > gate_gt) [& isfinite(y).all(0)]
    (s2_emit/poly_regression.py:106, :118).  x, y: [K, ...] planes of ``groups`` x n samples."""
    K = int(x.shape[0])
    G = int(groups)
    n = x.numel() // max(K * G, 1)
    xv, xks, xgs = _grouped(x, "x", K, G, n)
    yv, yks, ygs = (None, 0, 0)
    if y is not None:
        yv, yks, ygs = _grouped(y, "y", K, G, n)
    v = None
    if valid is not None:
        v = valid.view(torch.uint8) if valid.dtype == torch.bool else valid
        _cuda(v, "valid", torch.uint8)
        v = v.contiguous()
        if v.numel() != G * n:
            raise ValueError("valid must have one entry per pixel")
    with torch.cuda.device_of(xv):
        shape = tuple(x.shape[1:]) if G == 1 else (G, n)
        mask = torch.empty(shape, dtype=torch.uint8, device=xv.device)
        _lib.check(_lib.lib().hsr_fit_mask_u8(xv.data_ptr(), xks, xgs, _ptr(yv), yks, ygs, n, K, G, _ptr(v),
                                              int(gate_k), float(gate_gt), mask.data_ptr(), _stream()))
    return mask.view(torch.bool)


# --------------------------------------------------------------------------------------- fused fit / apply
def _stretch_arg(stretch, K: int, G: int, name: str):
    """[K, G, 2] f64 (lo, hi) per series or None."""
    if stretch is None:
        return None
    st = _cuda(stretch, name, torch.float64).contiguous()
    if st.numel() != K * G * 2:
        raise ValueError(f"{name} must be [K={K}, G={G}, 2] (lo, hi) pairs, got shape {tuple(st.shape)}")
    return st


def _exchange_arg(exchange, stage: int):
    """None or a ctypes pointer to an hsr_exchange_t (``hsr_b200.dist.PeerExchange.next()``).  ``stage`` 1 = the fit
    publishes, 2 = the solve/apply consumes: a descriptor must go through them in that order, once each."""
    if exchange is None:
        return None
    have = getattr(exchange, "_stage", None)
    if have is not None:
        if have != stage - 1:
            raise RuntimeError("peer exchange descriptor used out of order: fit_moments(exchange=d) must be followed by "
                               "exactly one poly_solve_apply(exchange=d)")
        exchange._stage = stage
    return ctypes.byref(exchange)


def fit_moments(x: torch.Tensor, y: torch.Tensor, valid: Optional[torch.Tensor], deg: int, *, groups: int = 1,
                gate_k: int = 0, gate_gt: float = 0.0, want_mask: bool = True, mask_given: bool = False,
                y_finite: bool = False, x_stretch: Optional[torch.Tensor] = None,
                y_stretch: Optional[torch.Tensor] = None, exchange=None):
    """Fit mask (unless given) + fp64 moments of the K*G series (poly_regression.py:106, :35-36, :58-60).

    x, y: [K, ...] planes holding ``groups`` independent groups of n samples each ([K, G, n] once flattened);
    valid: [G, n] bool/u8 or None.  ``mask_given``: ``valid`` already is the fit mask (returned unchanged);
    ``y_finite``: the computed mask also needs every y[k] finite (poly_regression.py:118);
    ``x_stretch`` / ``y_stretch``: [K, G, 2] f64 (lo, hi) percentile stretch applied on the fly (color.py:25-34).
    Returns ``(moments [K, G, 3*deg+2] f64, mask [G, n] bool | None)``.
    """
    K = int(x.shape[0])
    G = int(groups)
    n = x.numel() // max(K * G, 1)
    xv, xks, xgs = _grouped(x, "x", K, G, n)
    yv, yks, ygs = _grouped(y, "y", K, G, n)
    v = None
    if valid is not None:
        v = valid.view(torch.uint8) if valid.dtype == torch.bool else valid
        _cuda(v, "valid", torch.uint8)
        v = v.contiguous()
        if v.numel() != G * n:
            raise ValueError("valid must have one entry per (group, sample)")
    if mask_given and v is None:
        raise ValueError("mask_given=True needs the mask in `valid`")
    xst, yst = _stretch_arg(x_stretch, K, G, "x_stretch"), _stretch_arg(y_stretch, K, G, "y_stretch")
    flags = (_lib.HSR_FIT_MASK_GIVEN if mask_given else 0) | (_lib.HSR_FIT_Y_FINITE if y_finite else 0)
    with torch.cuda.device_of(xv):
        ws = _lib.lib().hsr_fit_moments_workspace_bytes(n, K, G, int(deg))
        partial = torch.empty(max(ws // 8, 1), dtype=torch.float64, device=xv.device)
        moments = torch.empty((K, G, 3 * int(deg) + 2), dtype=torch.float64, device=xv.device)
        mask = None
        if not mask_given:
            mask = torch.empty((G, n), dtype=torch.uint8, device=xv.device)
        _lib.check(_lib.lib().hsr_fit_moments_f64(xv.data_ptr(), xks, xgs, yv.data_ptr(), yks, ygs, _ptr(v), n, K, G,
                                                  int(deg), int(gate_k), float(gate_gt), flags, _ptr(xst), _ptr(yst),
                                                  _ptr(mask), partial.data_ptr(), moments.data_ptr(), _exchange_arg(exchange, 1),
                                                  _stream()))
    if mask_given:
        return moments, (v.view(torch.bool).view(G, n) if want_mask else None)
    return moments, (mask.view(torch.bool) if want_mask else None)


def moments_sum(per_unit, *, like: Optional[torch.Tensor] = None, exchange=None) -> torch.Tensor:
    """Fixed-order sum of this rank's per-unit moment matrices (a list of equal-shaped f64 CUDA tensors, or one
    stacked [U, ...] tensor) -> one matrix of that shape (hsr_moments_sum_f64).  ``exchange``: also publish the sums
    to the peers (takes the fit's turn of the descriptor).  An empty list needs ``like`` for the shape and gives zeros."""
    if isinstance(per_unit, torch.Tensor):
        stacked = _cuda(per_unit, "per_unit", torch.float64).contiguous()
        units, shape = int(stacked.shape[0]), tuple(stacked.shape[1:])
    else:
        per_unit = list(per_unit)
        units = len(per_unit)
        if units == 0:
            if like is None:
                raise ValueError("an empty unit list needs like= for the shape of the moments")
            stacked, shape = None, tuple(like.shape)
        else:
            shape = tuple(per_unit[0].shape)
            stacked = torch.stack([_cuda(m, "moments", torch.float64) for m in per_unit]).contiguous()
    dev_t = stacked if stacked is not None else like
    count = 1
    for d in shape:
        count *= int(d)
    with torch.cuda.device_of(dev_t):
        out = torch.empty(shape, dtype=torch.float64, device=dev_t.device)
        _lib.check(_lib.lib().hsr_moments_sum_f64(_ptr(stacked), units, count, out.data_ptr(), _exchange_arg(exchange, 1),
                                                  _stream()))
        if stacked is not None:
            stacked.record_stream(torch.cuda.current_stream())
    return out


def poly_solve_apply(x: torch.Tensor, moments: torch.Tensor, mask: Optional[torch.Tensor], deg: int, *,
                     groups: int = 1, min_count: int = 0, lo: float = 0.0, hi: float = 1.0,
                     out: Optional[torch.Tensor] = None, x_stretch: Optional[torch.Tensor] = None, exchange=None,
                     moments_out: Optional[torch.Tensor] = None):
    """Fused solve + apply: ``(coeffs [K, G, deg+1] f64, out like x)`` from ``moments [K, G, 3*deg+2]``;
    ``x_stretch`` [K, G, 2] f64 (lo, hi): x is percentile-stretched first (color.py:25-34).
    ``exchange`` (the struct given to ``fit_moments``): solve the rank-ordered SUM of every rank's moments instead
    (the all-reduce of the global fit, done in this kernel's prologue); ``moments_out`` [K, G, 3*deg+2] receives it."""
    K = int(x.shape[0])
    G = int(groups)
    n = x.numel() // max(K * G, 1)
    xv, xks, xgs = _grouped(x, "x", K, G, n)
    mo = _cuda(moments, "moments", torch.float64).contiguous()
    if mo.numel() != K * G * (3 * int(deg) + 2):
        raise ValueError(f"moments must be [K, G, {3 * int(deg) + 2}]")
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        _cuda(m, "mask", torch.uint8)
        m = m.contiguous()
        if m.numel() != G * n:
            raise ValueError("mask must have one entry per (group, sample)")
    with torch.cuda.device_of(xv):
        if out is None:
            out = alloc_planes(K, x.shape[1:], xv.device)
        ov, oks, ogs = _grouped(out, "out", K, G, n)
        if ov.data_ptr() != out.data_ptr():
            raise ValueError("out must be viewable as [K, G, n] with dense samples")
        coeffs = torch.empty((K, G, int(deg) + 1), dtype=torch.float64, device=xv.device)
        xst = _stretch_arg(x_stretch, K, G, "x_stretch")
        _lib.check(_lib.lib().hsr_poly_solve_apply_f32(xv.data_ptr(), xks, xgs, mo.data_ptr(), _ptr(m), n, K, G,
                                                       int(deg), int(min_count), float(lo), float(hi), _ptr(xst),
                                                       coeffs.data_ptr(), ov.data_ptr(), oks, ogs,
                                                       _exchange_arg(exchange, 2), _ptr(moments_out), _stream()))
    return coeffs, out


# --------------------------------------------------------------------------------------- percentile stretch
_Q_CACHE: dict = {}


def _percentile_fractions(q):
    import numpy as np

    qf = np.true_divide(np.asarray(q, dtype=np.float64).reshape(-1), 100)   # as np.percentile does
    if qf.size < 1 or qf.size > _lib.HSR_MAX_PERCENTILES:
        raise ValueError(f"between 1 and {_lib.HSR_MAX_PERCENTILES} percentiles per call")
    if not ((qf >= 0) & (qf <= 1)).all():
        raise ValueError("Percentiles must be in the range [0, 100]")
    return qf


def _fractions_on(qf, device) -> torch.Tensor:
    """The fractions on the device, uploaded once per (q, device)."""
    key = (tuple(qf.tolist()), device)
    qd = _Q_CACHE.get(key)
    if qd is None:
        qd = _Q_CACHE[key] = torch.from_numpy(qf).to(device)
    return qd


def masked_percentiles(x: torch.Tensor, mask: Optional[torch.Tensor], q, *, groups: int = 1,
                       y: Optional[torch.Tensor] = None, _workspace_out: Optional[list] = None):
    """``out[k, g, j] = np.percentile(x[k, g][mask[g]], q[j])`` — exact (sampled brackets, one streaming pass, radix
    select among the collected keys, numpy's "linear" interpolation: bit-identical float64), s2_emit/color.py:30-32.

    x: [K, ...] f32 planes of ``groups`` x n samples; mask: [G, n] bool/u8 or None; q: percentiles in
    [0, 100] (at most HSR_MAX_PERCENTILES).  Returns [K, G, Q] f64 on the device (NaN where a series has no
    masked sample or a NaN among them).  ``y``: a second plane set of x's shape (the reference image of the shared
    stretch) handled in the same three launches: returns ``(out_x, out_y)``.
    """
    K = int(x.shape[0])
    G = int(groups)
    n = x.numel() // max(K * G, 1)
    xv, xks, xgs = _grouped(x, "x", K, G, n)
    yv = None
    if y is not None:
        if int(y.shape[0]) != K or y.numel() != x.numel():
            raise ValueError("y must have the shape of x")
        yv, yks, ygs = _grouped(y, "y", K, G, n)
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        _cuda(m, "mask", torch.uint8)
        m = m.contiguous()
        if m.numel() != G * n:
            raise ValueError("mask must have one entry per (group, sample)")
    qf = _percentile_fractions(q)
    with torch.cuda.device_of(xv):
        qd = _fractions_on(qf, xv.device)
        ws =_lib.lib().hsr_percentiles_workspace_bytes(n, K, G, 2 if yv is not None else 1)
        work = torch.empty(ws + 256, dtype=torch.uint8, device=xv.device)
        off = (-work.data_ptr()) % 256
        out = torch.empty((K, G, qf.size), dtype=torch.float64, device=xv.device)
        if _workspace_out is not None:       # diagnostics (profiles/prof_select.py): the per-series state lives at its start
            _workspace_out.append(work[off:])
        if yv is None:
            _lib.check(_lib.lib().hsr_masked_percentiles_f64(xv.data_ptr(), xks, xgs, _ptr(m), n, K, G, qd.data_ptr(),
                                                             int(qf.size), work.data_ptr() + off, out.data_ptr(),
                                                             _stream()))
            return out
        out_y = torch.empty_like(out)
        _lib.check(_lib.lib().hsr_masked_percentiles_pair_f64(xv.data_ptr(), xks, xgs, yv.data_ptr(), yks, ygs, _ptr(m), n, K,
                                                              G, qd.data_ptr(), int(qf.size), work.data_ptr() + off,
                                                              out.data_ptr(), out_y.data_ptr(), _stream()))
    return out, out_y


def masked_percentiles_union(units, q, *, reduce=None, K: Optional[int] = None, pair: Optional[bool] = None,
                             device=None, factor: int = 1, _state_out: Optional[list] = None):
    """``out[k, 0, j] = np.percentile(concatenation over units of x[k][mask], q[j])`` — the exact percentiles of the
    UNION of several units (granules, slabs) and, through ``reduce``, of every process's units: a radix select by four
    8-bit passes whose per-pass histograms are summed over the units and then across processes (hsr_union_select_*).
    Only integer counts cross units and processes, so the result is bit-identical on every process and to numpy.

    units: a list of ``(x, mask)`` or ``(x, y, mask)``; x, y: [K, ...] f32 planes of one unit, mask: bool/u8 with one
    entry per sample, or None.  The list may be empty (a process that holds no unit still takes part in the
    reductions); then ``K``, ``pair`` and ``device`` give the shape.  ``reduce``: callable that sums an f64 CUDA tensor
    in place across processes, called once per pass; default ``dist.allreduce_moments`` on the default group (a no-op
    for one process).  Every process must make the call.  Returns [K, 1, Q] f64 (a pair for ``(x, y, mask)`` units;
    NaN where the union has no sample or a NaN among them).  ``_state_out``: diagnostics (tests) — receives the
    per-series select state after the last pass.

    ``factor > 1``: the samples of every unit's x planes [K, Hs, Ws] are those of ``bilinear_upsample(x, factor)``
    (same bits), formed on the fly from the coarse planes in each pass and never written
    (hsr_union_select_count_bilinear); the mask then has the fine shape [Hs*factor, Ws*factor], units are ``(x, mask)``
    and ``pair`` must be False."""
    from . import dist as hdist

    units = [tuple(u) for u in units]
    if units:
        arity = {len(u) for u in units}
        if len(arity) != 1 or arity.pop() not in (2, 3):
            raise ValueError("units must all be (x, mask) or all be (x, y, mask)")
        pair = len(units[0]) == 3
        K = int(units[0][0].shape[0])
        device = units[0][0].device
    elif K is None or pair is None or device is None:
        raise ValueError("an empty unit list needs K=, pair= and device=")
    K, pair, device = int(K), bool(pair), torch.device(device)
    f = _factor(factor)
    if f > 1 and pair:
        raise ValueError("factor > 1 takes (x, mask) units only (pair=False)")
    qf = _percentile_fractions(q)
    Q, S = int(qf.size), K * (2 if pair else 1)
    prepared = []
    for u in units:
        x, y, mask = (u[0], u[1], u[2]) if pair else (u[0], None, u[1])
        if int(x.shape[0]) != K or x.device != device:
            raise ValueError(f"every unit must hold K = {K} planes on {device}")
        if f > 1:
            xv, _, Hs, Ws, xks = _coarse_planes(x, "x")
            n = Hs * Ws * f * f
        else:
            n = x.numel() // max(K, 1)
            xv, xks, _ = _grouped(x, "x", K, 1, n)
        yv, yks = None, 0
        if y is not None:
            if int(y.shape[0]) != K or y.numel() != x.numel():
                raise ValueError("y must have the shape of x")
            yv, yks, _ = _grouped(y, "y", K, 1, n)
        m = None
        if mask is not None:
            m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
            m = _cuda(m, "mask", torch.uint8).contiguous()
            if m.numel() != n:
                raise ValueError("mask must have one entry per sample" + (" of the fine grid" if f > 1 else ""))
        prepared.append((xv, xks, yv, yks, m, n))
    reduce = reduce if reduce is not None else hdist.allreduce_moments
    lib = _lib.lib()
    with torch.cuda.device(device):
        qd = _fractions_on(qf, device)
        state, sp = _aligned_workspace(lib.hsr_union_select_state_bytes(Q, S), device)
        hist = torch.empty(lib.hsr_union_select_hist_doubles(Q, S), dtype=torch.float64, device=device)
        out = torch.empty((S, Q), dtype=torch.float64, device=device)
        _lib.check(lib.hsr_union_select_begin(qd.data_ptr(), Q, S, sp, hist.data_ptr(), _stream()))
        more, p = ctypes.c_int(1), 0
        while more.value:
            for xv, xks, yv, yks, m, n in prepared:
                if f > 1:
                    _lib.check(lib.hsr_union_select_count_bilinear(xv.data_ptr(), xks, xv.shape[1], xv.shape[2], f, _ptr(m),
                                                                   K, Q, p, sp, hist.data_ptr(), _stream()))
                    continue
                _lib.check(lib.hsr_union_select_count(xv.data_ptr(), xks, _ptr(yv), yks, _ptr(m), n, K, Q, p, sp,
                                                      hist.data_ptr(), _stream()))
            reduce(hist)
            _lib.check(lib.hsr_union_select_step(Q, S, p, sp, hist.data_ptr(), out.data_ptr(), ctypes.byref(more),
                                                 _stream()))
            p += 1
        if _state_out is not None:
            _state_out.append(state[sp - state.data_ptr():])
    out = out.view(S // K, K, 1, Q)
    return (out[0], out[1]) if pair else out[0]


def stretch_apply(x: torch.Tensor, lohi: torch.Tensor, *, groups: int = 1,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``out = float32(clip((float64(x) - lo) / (hi - lo + 1e-12), 0, 1))`` per series (color.py:33), bit-exact.
    x: [K, ...] planes; lohi: [K, G, 2] f64."""
    K = int(x.shape[0])
    G = int(groups)
    n = x.numel() // max(K * G, 1)
    xv, xks, xgs = _grouped(x, "x", K, G, n)
    st = _stretch_arg(lohi, K, G, "lohi")
    with torch.cuda.device_of(xv):
        if out is None:
            out = alloc_planes(K, x.shape[1:], xv.device)
        ov, oks, ogs = _grouped(out, "out", K, G, n)
        if ov.data_ptr() != out.data_ptr():
            raise ValueError("out must be viewable as [K, G, n] with dense samples")
        _lib.check(_lib.lib().hsr_stretch_f32(xv.data_ptr(), xks, xgs, st.data_ptr(), n, K, G, ov.data_ptr(), oks, ogs,
                                              _stream()))
    return out


def stretch_apply_f64(x: torch.Tensor, lohi: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``float64: clip((x - lo) / (hi - lo + 1e-12), 0, 1)``, NaN where ``mask`` is False (color.py:6-23).
    x: [K, ...] f32 planes; lohi: [K, 1, 2] f64; mask: one [n] mask shared by the planes, or None.  Returns [K, ...] f64."""
    K = int(x.shape[0])
    n = x.numel() // max(K, 1)
    xv, xks, xgs = _grouped(x, "x", K, 1, n)
    st = _stretch_arg(lohi, K, 1, "lohi")
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        m = _cuda(m, "mask", torch.uint8).contiguous()
        if m.numel() != n:
            raise ValueError("mask must have one entry per sample")
    with torch.cuda.device_of(xv):
        out = torch.empty((K,) + tuple(x.shape[1:]), dtype=torch.float64, device=xv.device)
        _lib.check(_lib.lib().hsr_stretch_f64(xv.data_ptr(), xks, xgs, st.data_ptr(), _ptr(m), n, K, 1, out.data_ptr(), n, n,
                                              _stream()))
    return out


def notnan_mask(x: torch.Tensor, base: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``~isnan(x)`` (``& base``) as a bool tensor of x's shape: the samples np.nanpercentile keeps."""
    xv = _cuda(x, "x", torch.float32).contiguous()
    b = None
    if base is not None:
        b = base.view(torch.uint8) if base.dtype == torch.bool else base
        b = _cuda(b, "base", torch.uint8).contiguous()
        if b.numel() != xv.numel():
            raise ValueError("base must have one entry per sample")
    with torch.cuda.device_of(xv):
        out = torch.empty(xv.shape, dtype=torch.uint8, device=xv.device)
        _lib.check(_lib.lib().hsr_notnan_mask_u8(xv.data_ptr(), _ptr(b), xv.numel(), out.data_ptr(), _stream()))
    return out.view(torch.bool)


def hist_match_channel(src: torch.Tensor, ref: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """One channel of histogram_match_rgb (s2_emit/color.py:36-61): masked ``src`` samples mapped through the source CDF
    and the inverse reference CDF (np.unique / np.cumsum / np.interp of the reference), then every pixel clipped to
    [0, 1].  src, ref: f32 of one shape; mask: bool of that shape.  The two sorts are ``torch.sort`` (a library sort is
    plumbing here, as cuBLAS would be); run detection, compaction, CDF look-ups and the interpolation are ours."""
    s = _cuda(src, "src", torch.float32).contiguous()
    r = _cuda(ref, "ref", torch.float32).contiguous()
    m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    m = _cuda(m, "mask", torch.uint8).contiguous()
    if s.shape != r.shape or m.numel() != s.numel():
        raise IndexError("boolean index did not match: src, ref and mask must have one shape")
    n = s.numel()
    lib = _lib.lib()
    with torch.cuda.device_of(s):
        sel = m.view(-1).view(torch.bool)
        s_sorted = torch.sort(s.view(-1)[sel]).values
        r_sorted = torch.sort(r.view(-1)[sel]).values
        ns = int(s_sorted.numel())
        if ns == 0:
            raise IndexError("index -1 is out of bounds for axis 0 with size 0")       # s_quant[-1] of nothing (:44)
        flags = torch.empty(ns, dtype=torch.uint8, device=s.device)
        _lib.check(lib.hsr_run_ends_u8(r_sorted.data_ptr(), ns, flags.data_ptr(), _stream()))
        ends, nu = compact_finite_rows(r_sorted.view(-1, 1), flags)
        nu = int(nu.item())
        if nu == 0:
            raise ValueError("histogram matching needs finite reference samples inside the mask")
        out = torch.empty_like(s)
        _lib.check(lib.hsr_hist_match_f32(s.data_ptr(), m.data_ptr(), n, s_sorted.data_ptr(), ns, r_sorted.data_ptr(), ns,
                                          ends.data_ptr(), nu, out.data_ptr(), _stream()))
    return out


# --------------------------------------------------------------------------------------- OT targets
def _aligned_workspace(nbytes: int, device) -> tuple:
    work = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
    return work, work.data_ptr() + ((-work.data_ptr()) % 256)


def compact_finite_rows(img: torch.Tensor, mask: Optional[torch.Tensor]):
    """Row-major indices of the rows of ``img`` [n, C] (f32) with ``mask`` set and every channel finite —
    ``img[mask]`` + the finite filter of s2_emit/poly_regression.py:33-36.
    Returns ``(idx int32 [n] (first ``count`` entries valid), count int64[1])``, both on the device."""
    x = _cuda(img, "img", torch.float32).contiguous()
    if x.dim() != 2:
        raise ValueError("img must be [n, C]")
    n, C = x.shape
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        _cuda(m, "mask", torch.uint8)
        m = m.contiguous()
        if m.numel() != n:
            raise ValueError("mask must have one entry per row")
    with torch.cuda.device_of(x):
        work, wptr = _aligned_workspace(_lib.lib().hsr_compact_workspace_bytes(n), x.device)
        idx = torch.empty(max(n, 1), dtype=torch.int32, device=x.device)
        count = torch.zeros(1, dtype=torch.int64, device=x.device)
        _lib.check(_lib.lib().hsr_compact_finite_rows(x.data_ptr(), _ptr(m), n, C, wptr, idx.data_ptr(),
                                                      count.data_ptr(), _stream()))
    return idx, count


def gather_rows_f64(img: torch.Tensor, idx: torch.Tensor, sel: torch.Tensor) -> torch.Tensor:
    """``out[r] = float64(img[idx[sel[r]]])`` — X_all[rng.choice(...)] (poly_regression.py:46-47)."""
    x = _cuda(img, "img", torch.float32).contiguous()
    ix = _cuda(idx, "idx", torch.int32).contiguous()
    se = _cuda(sel, "sel", torch.int64).contiguous()
    ns, C = se.numel(), x.shape[1]
    with torch.cuda.device_of(x):
        out = torch.empty((ns, C), dtype=torch.float64, device=x.device)
        _lib.check(_lib.lib().hsr_gather_rows_f64(x.data_ptr(), ix.data_ptr(), se.data_ptr(), ns, C, out.data_ptr(),
                                                  _stream()))
    return out


def compact_planes_pair(x: torch.Tensor, y: torch.Tensor, mask: Optional[torch.Tensor], *,
                        x_stretch: Optional[torch.Tensor] = None, y_stretch: Optional[torch.Tensor] = None):
    """The two row filters of s2_emit/poly_regression.py:33-36 on K planes (hsr_compact_planes_pair): ``idx_x`` holds
    the row-major indices of the pixels with ``mask`` set and all K planes of ``x`` finite, ``idx_y`` likewise for
    ``y``, independently.  x, y: [K, ...] f32 planes (padded or dense); mask: one entry per pixel, or None;
    ``x_stretch`` / ``y_stretch``: [K, 1, 2] f64 (lo, hi) — the planes are judged as the percentile stretch of
    color.py:33 leaves them.  Returns ``(idx_x int32 [n], count_x int64[1], idx_y, count_y)`` on the device (the first
    ``count`` entries of each list are valid)."""
    xs, K, n, xks, _ = _series(x, "x", "planar")
    ys, Ky, ny, yks, _ = _series(y, "y", "planar")
    if (K, n) != (Ky, ny):
        raise ValueError(f"x and y disagree: {K}x{n} vs {Ky}x{ny}")
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        m = _cuda(m, "mask", torch.uint8).contiguous()
        if m.numel() != n:
            raise ValueError("mask must have one entry per pixel")
    xst, yst = _stretch_arg(x_stretch, K, 1, "x_stretch"), _stretch_arg(y_stretch, K, 1, "y_stretch")
    lib = _lib.lib()
    with torch.cuda.device_of(xs):
        work, wptr = _aligned_workspace(lib.hsr_compact_planes_pair_workspace_bytes(n), xs.device)
        idx = torch.empty((2, max(n, 1)), dtype=torch.int32, device=xs.device)
        count = torch.zeros(2, dtype=torch.int64, device=xs.device)
        _lib.check(lib.hsr_compact_planes_pair(xs.data_ptr(), xks, _ptr(xst), ys.data_ptr(), yks, _ptr(yst), _ptr(m), n, K,
                                               wptr, idx[0].data_ptr(), count[0:1].data_ptr(), idx[1].data_ptr(),
                                               count[1:2].data_ptr(), _stream()))
        work.record_stream(torch.cuda.current_stream())
    return idx[0], count[0:1], idx[1], count[1:2]


def gather_planes_f64(planes: torch.Tensor, idx: torch.Tensor, sel: torch.Tensor, *,
                      stretch: Optional[torch.Tensor] = None, dst: Optional[torch.Tensor] = None,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Sample rows of K planes (hsr_gather_planes_f64): ``out[dst[r], k] = float64(s(planes[k, idx[sel[r]]]))``, ``s``
    the percentile stretch of color.py:33 with ``stretch`` [K, 1, 2] f64 (lo, hi) (bit-identical to
    ``stretch_apply``), or none.  Without ``dst`` row r is written to row r of a new [len(sel), K] f64 tensor; with it
    (int64, one per ``sel``, each in [0, rows); checked on the host, one synchronisation) into ``out`` [rows, K] f64,
    whose other rows keep what the caller put there."""
    xs, K, n, ks, _ = _series(planes, "planes", "planar")
    ix = _cuda(idx, "idx", torch.int32).contiguous()
    se = _cuda(sel, "sel", torch.int64).contiguous()
    ns = se.numel()
    st = _stretch_arg(stretch, K, 1, "stretch")
    ds = None
    if dst is not None:
        ds = _cuda(dst, "dst", torch.int64).contiguous()
        if ds.numel() != ns:
            raise ValueError("dst must hold one row per sel entry")
        if out is None:
            raise ValueError("dst= writes into a caller's out= buffer")
        if ns:
            lo, hi = (int(v) for v in torch.aminmax(ds))
            if lo < 0 or hi >= out.shape[0]:
                raise IndexError(f"dst holds rows in [{lo}, {hi}], out has {out.shape[0]} rows")
    with torch.cuda.device_of(xs):
        if out is None:
            out = torch.empty((ns, K), dtype=torch.float64, device=xs.device)
        _cuda(out, "out", torch.float64)
        if out.dim() != 2 or out.shape[1] != K or not out.is_contiguous() or (ds is None and out.shape[0] < ns):
            raise ValueError(f"out must be a contiguous [rows, K={K}] f64 tensor")
        _lib.check(_lib.lib().hsr_gather_planes_f64(xs.data_ptr(), ks, K, ix.data_ptr(), se.data_ptr(), _ptr(ds), ns,
                                                    _ptr(st), out.data_ptr(), _stream()))
    return out


def sinkhorn_barycentric(X: torch.Tensor, Y: torch.Tensor, reg: float = 0.05, numItermax: int = 300,
                         stopThr: float = 1e-6):
    """``Ybar = (P @ Y) / (P.sum(1) + 1e-32)``, ``P = ot.sinkhorn(1/ns, 1/nt, ot.dist(X, Y), reg, ...)``
    (poly_regression.py:49-56), fp64.  X [ns, C], Y [nt, C] f64, C <= 16 (hsr_sinkhorn_barycentric_k_f64; C <= 4 runs
    the kernels of hsr_sinkhorn_barycentric_f64, bit for bit).
    Returns ``(Ybar [ns, C] f64, info f64[4] = (iteration used, last error, iteration of that check, numerical flag))``."""
    Xd = _cuda(X, "X", torch.float64).contiguous()
    Yd = _cuda(Y, "Y", torch.float64).contiguous()
    if Xd.dim() != 2 or Yd.dim() != 2 or Xd.shape[1] != Yd.shape[1]:
        raise ValueError("X, Y must be [ns, C] and [nt, C]")
    ns, C = Xd.shape
    nt = Yd.shape[0]
    with torch.cuda.device_of(Xd):
        work, wptr = _aligned_workspace(_lib.lib().hsr_sinkhorn_workspace_bytes(ns, nt), Xd.device)
        ybar = torch.empty((ns, C), dtype=torch.float64, device=Xd.device)
        info = torch.zeros(4, dtype=torch.float64, device=Xd.device)
        _lib.check(_lib.lib().hsr_sinkhorn_barycentric_k_f64(Xd.data_ptr(), Yd.data_ptr(), ns, nt, C, float(reg),
                                                             int(numItermax), float(stopThr), wptr, ybar.data_ptr(),
                                                             info.data_ptr(), _stream()))
        work.record_stream(torch.cuda.current_stream())
    return ybar, info


def polyfit_moments_f64(x: torch.Tensor, y: torch.Tensor, deg: int) -> torch.Tensor:
    """The [S, 3*deg+2] fp64 normal-equation moments of the columns of two [n, S] f64 arrays
    (hsr_polyfit_moments_f64in; the layout ``poly_solve`` / ``poly_solve_apply`` take)."""
    xd = _cuda(x, "x", torch.float64).contiguous()
    yd = _cuda(y, "y", torch.float64).contiguous()
    if xd.shape != yd.shape or xd.dim() != 2:
        raise ValueError("x, y must be [n, S] of equal shape")
    n, S = xd.shape
    with torch.cuda.device_of(xd):
        mom = torch.empty((S, 3 * int(deg) + 2), dtype=torch.float64, device=xd.device)
        _lib.check(_lib.lib().hsr_polyfit_moments_f64in(xd.data_ptr(), yd.data_ptr(), n, S, int(deg), mom.data_ptr(),
                                                        _stream()))
    return mom


def polyfit_f64(x: torch.Tensor, y: torch.Tensor, deg: int, min_count: int = 0, return_moments: bool = False):
    """``coeffs[c] = np.polyfit(x[:, c], y[:, c], deg)`` for the columns of two [n, S] f64 arrays
    (poly_regression.py:58-60): fp64 moments + the warp solve."""
    mom = polyfit_moments_f64(x, y, deg)
    co = poly_solve(mom, deg, min_count)
    return (co, mom) if return_moments else co


def affine_fit(X: torch.Tensor, Ybar: torch.Tensor) -> torch.Tensor:
    """``W, *_ = np.linalg.lstsq([X 1], Ybar)`` (s2_emit/color.py:103-106): [(C+1), C] f64, rows 0..C-1 = A, row C = t."""
    Xd = _cuda(X, "X", torch.float64).contiguous()
    Yd = _cuda(Ybar, "Ybar", torch.float64).contiguous()
    if Xd.shape != Yd.shape or Xd.dim() != 2:
        raise ValueError("X, Ybar must be [ns, C] of equal shape")
    ns, C = Xd.shape
    with torch.cuda.device_of(Xd):
        W = torch.empty((C + 1, C), dtype=torch.float64, device=Xd.device)
        _lib.check(_lib.lib().hsr_affine_fit_f64(Xd.data_ptr(), Yd.data_ptr(), ns, C, W.data_ptr(), _stream()))
    return W


def affine_apply(rgb: torch.Tensor, W: torch.Tensor, mask: Optional[torch.Tensor] = None, *, lo: float = 0.0,
                 hi: float = 1.0) -> torch.Tensor:
    """``out = rgb.astype(f32); out[mask] = clip(out[mask] @ A + t, lo, hi)`` (s2_emit/color.py:108-115) on an
    interleaved [..., C] image; pixels outside the mask are copied unchanged."""
    x = _cuda(rgb, "rgb", torch.float32).contiguous()
    Wd = _cuda(W, "W", torch.float64).contiguous()
    C = x.shape[-1]
    if tuple(Wd.shape) != (C + 1, C):
        raise ValueError(f"W must be [{C + 1}, {C}]")
    n = x.numel() // C
    m = None
    if mask is not None:
        m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        m = _cuda(m, "mask", torch.uint8).contiguous()
        if m.numel() != n:
            raise IndexError("boolean index did not match: one mask entry per pixel expected")
    with torch.cuda.device_of(x):
        out = torch.empty_like(x)
        _lib.check(_lib.lib().hsr_affine_apply_f32(x.data_ptr(), Wd.data_ptr(), _ptr(m), n, C, float(lo), float(hi),
                                                   out.data_ptr(), _stream()))
    return out


# --------------------------------------------------------------------------------------- tiles
def black_mask(arr: torch.Tensor, nodata=None, masked_val: float = -0.01, nodata_atol: float = 1e-3,
               zero_atol: float = 1e-6, *, want_count: bool = False):
    """is_black_mask of tiles_helpers/utils.py:201-220 on band-sequential tiles: arr [B, H, W] or a batch
    [T, B, H, W] f32 -> bool [H, W] / [T, H, W] (and, with ``want_count``, int64 [T] black pixels per tile)."""
    import numpy as np

    a = _cuda(arr, "arr", torch.float32)
    batched = a.dim() == 4
    if a.dim() not in (3, 4):
        raise ValueError("arr must be (bands, H, W) or (T, bands, H, W)")
    a4 = a if batched else a.unsqueeze(0)
    if not (a4.stride(-1) == 1 and a4.stride(-2) == a4.shape[-1]):
        a4 = a4.contiguous()
    T, B, H, Wd = a4.shape
    n = H * Wd
    rtol = 1e-5                                                        # np.isclose default
    tol = lambda y: float(np.float32(float(nodata_atol) + rtol * abs(float(y))))   # noqa: E731
    nd = 0.0 if nodata is None else float(np.float32(nodata))
    with torch.cuda.device_of(a4):
        out = torch.empty((T, H, Wd), dtype=torch.uint8, device=a4.device)
        count = torch.zeros(T, dtype=torch.int64, device=a4.device) if want_count else None
        _lib.check(_lib.lib().hsr_black_mask_f32(
            a4.data_ptr(), int(a4.stride(0)) if T > 1 else B * n, int(a4.stride(1)) if B > 1 else n, n, B, T,
            int(nodata is not None), nd, tol(nodata) if nodata is not None else 0.0, float(np.float32(masked_val)),
            tol(masked_val), float(np.float32(zero_atol)), out.data_ptr(), _ptr(count), _stream()))
    mask = out.view(torch.bool)
    if not batched:
        mask = mask[0]
    return (mask, count) if want_count else mask


def quantize_u16(x: torch.Tensor, nodata=None, scale: float = 10000.0, nodata_u16: int = 65535) -> torch.Tensor:
    """EMIT tile -> uint16 of save_tile_pair (tiles_helpers/utils.py:362-373); returned as an int16-typed tensor's
    bit pattern is avoided: the result is a torch.uint16 tensor of x's shape."""
    import numpy as np

    a = _cuda(x, "x", torch.float32).contiguous()
    with torch.cuda.device_of(a):
        out = torch.empty(a.shape, dtype=torch.uint16, device=a.device)
        _lib.check(_lib.lib().hsr_quantize_u16_f32(a.data_ptr(), a.numel(), int(nodata is not None),
                                                   0.0 if nodata is None else float(np.float32(nodata)),
                                                   float(np.float32(scale)), int(nodata_u16), out.data_ptr(), _stream()))
    return out


def tile_sums(mask: torch.Tensor, tile_h: int, tile_w: int) -> torch.Tensor:
    """Set pixels of a [H, W] bool/u8 mask per non-overlapping tile -> int32-valued [nty, ntx] (uint32 storage)."""
    m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    _cuda(m, "mask", torch.uint8)
    m = m.contiguous()
    H, Wd = m.shape
    nty, ntx = H // int(tile_h), Wd // int(tile_w)
    with torch.cuda.device_of(m):
        out = torch.zeros((nty, ntx), dtype=torch.int32, device=m.device)
        _lib.check(_lib.lib().hsr_tile_sums_u8(m.data_ptr(), H, Wd, int(tile_h), int(tile_w), nty, ntx, out.data_ptr(),
                                               _stream()))
    return out


def glt_ortho_u16(raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, *, fill: float = NO_DATA_VALUE,
                  nodata=NO_DATA_VALUE, scale: float = 10000.0, nodata_u16: int = 65535, transpose_raw_yx: bool = False,
                  want_black: bool = True, masked_val: float = -0.01, nodata_atol: float = 1e-3, zero_atol: float = 1e-6,
                  want_valid: bool = True, want_diag: bool = True, raw_row0: int = 0,
                  raw_rows_total: Optional[int] = None, tile_rows=None):
    """Fused tile export: GLT gather + uint16 quantisation (tiles_helpers/utils.py:357-371) + is_black_mask (:201-220)
    in one pass over the raw cube; the fp32 ortho cube is never written.

    Returns ``(u16 [B, Ho, Wo] band-sequential torch.uint16, valid bool | None, black bool | None, diag | None)``;
    identical to ``quantize_u16(glt_ortho(...).permute(2, 0, 1), nodata, scale, nodata_u16)`` and
    ``black_mask(<that ortho cube>, nodata, masked_val, nodata_atol, zero_atol)``.
    """
    import numpy as np

    _cuda(raw, "raw", torch.float32)
    gx = _cuda(glt_x, "glt_x", torch.int32).contiguous()
    gy = _cuda(glt_y, "glt_y", torch.int32).contiguous()
    if gx.shape != gy.shape or gx.dim() != 2:
        raise ValueError("glt_x / glt_y must be 2-D planes of equal shape")
    r3, pitch, raw_h, raw_w, B, _ = _raw_geometry(raw, transpose_raw_yx)
    view, raw_h, raw_w = _raw_view(r3.shape[0], raw_h, raw_w, transpose_raw_yx, raw_row0, raw_rows_total, tile_rows)
    Ho, Wo = gx.shape
    rtol = 1e-5
    tol = lambda y: float(np.float32(float(nodata_atol) + rtol * abs(float(y))))   # noqa: E731
    with torch.cuda.device_of(r3):
        n = Ho * Wo
        stride = -(-max(n, 1) // 8) * 8                      # planes start on 16-byte boundaries
        buf = torch.empty((B, stride), dtype=torch.uint16, device=r3.device)
        valid = torch.empty((Ho, Wo), dtype=torch.uint8, device=r3.device) if want_valid else None
        black = torch.empty((Ho, Wo), dtype=torch.uint8, device=r3.device) if want_black else None
        diag = _view_diag(r3.device, want_diag, view)
        nd = 0.0 if nodata is None else float(np.float32(nodata))
        _lib.check(_lib.lib().hsr_glt_ortho_u16(
            r3.data_ptr(), raw_h, raw_w, B, pitch, int(bool(transpose_raw_yx)), gx.data_ptr(), gy.data_ptr(), Ho, Wo, Wo,
            float(fill), float(np.float32(scale)), int(nodata is not None), nd, int(nodata_u16), buf.data_ptr(), stride,
            _ptr(valid), _ptr(black), tol(nodata) if nodata is not None else 0.0, float(np.float32(masked_val)),
            tol(masked_val), float(np.float32(zero_atol)), _ptr(diag),
            ctypes.byref(view) if view is not None else None, _stream()))
    out = buf[:, :n].view(B, Ho, Wo)
    return (out, valid.view(torch.bool) if valid is not None else None,
            black.view(torch.bool) if black is not None else None, diag)


# --------------------------------------------------------------------------------------- resampling (aligned grids)
def block_average(src: torch.Tensor, factor: int, *, nodata=None, scale=None, out: Optional[torch.Tensor] = None):
    """"average" resampling of [C, Hs, Ws] planes (uint8 / uint16 / float32) onto the ``factor``-times coarser aligned
    grid: float32 [C, Hs // factor, Ws // factor] = mean of the valid pixels of every factor x factor block
    (``* scale`` afterwards) — downsample_s2_to_grid of the reference's notebook for snapped grids."""
    if not isinstance(src, torch.Tensor) or not src.is_cuda:
        raise TypeError("src must be a CUDA tensor: hsr_b200 has no CPU path")
    code = {torch.uint8: 0, torch.uint16: 1, torch.float32: 2}.get(src.dtype)
    if code is None:
        raise TypeError(f"src must be uint8, uint16 or float32, got {src.dtype}")
    if src.dim() != 3:
        raise ValueError("src must be [C, Hs, Ws]")
    s = src if src[0].is_contiguous() and (src.shape[0] == 1 or src.stride(0) >= src[0].numel()) else src.contiguous()
    C, Hs, Ws = s.shape
    f = int(factor)
    Hd, Wd = Hs // f, Ws // f
    with torch.cuda.device_of(s):
        if out is None:
            out = alloc_planes(C, (Hd, Wd), s.device)
        else:
            _cuda(out, "out", torch.float32)
        ps = _plane_stride(out, C, Hd * Wd, "out")
        _lib.check(_lib.lib().hsr_block_average_f32(s.data_ptr(), code, C, Hs, Ws, int(s.stride(0)) if C > 1 else Hs * Ws, f,
                                                    int(nodata is not None), 0.0 if nodata is None else float(nodata),
                                                    int(scale is not None), 1.0 if scale is None else float(scale),
                                                    out.data_ptr(), max(ps, Hd * Wd), _stream()))
    return out


def bilinear_upsample(src: torch.Tensor, factor: int, *, nodata=None, out: Optional[torch.Tensor] = None):
    """Bilinear resampling of [C, Hs, Ws] f32 planes onto the ``factor``-times finer aligned grid
    (reproject_stack_to_grid of the reference's notebook for snapped grids): f32 [C, Hs*factor, Ws*factor]."""
    s = _cuda(src, "src", torch.float32)
    if s.dim() != 3:
        raise ValueError("src must be [C, Hs, Ws]")
    if not (s[0].is_contiguous() and (s.shape[0] == 1 or s.stride(0) >= s[0].numel())):
        s = s.contiguous()
    C, Hs, Ws = s.shape
    f = int(factor)
    with torch.cuda.device_of(s):
        if out is None:
            out = alloc_planes(C, (Hs * f, Ws * f), s.device)
        else:
            _cuda(out, "out", torch.float32)
        ps = _plane_stride(out, C, Hs * f * Ws * f, "out")
        _lib.check(_lib.lib().hsr_bilinear_upsample_f32(s.data_ptr(), C, Hs, Ws, int(s.stride(0)) if C > 1 else Hs * Ws, f,
                                                        int(nodata is not None), 0.0 if nodata is None else float(nodata),
                                                        out.data_ptr(), max(ps, Hs * f * Ws * f), _stream()))
    return out


def _coarse_planes(src: torch.Tensor, name: str = "src"):
    """(planes, K, Hs, Ws, plane stride) of [K, Hs, Ws] f32 CUDA planes whose every plane is dense."""
    s = _cuda(src, name, torch.float32)
    if s.dim() != 3:
        raise ValueError(f"{name} must be [K, Hs, Ws], got shape {tuple(s.shape)}")
    if not (s[0].is_contiguous() and (s.shape[0] == 1 or s.stride(0) >= s[0].numel())):
        s = s.contiguous()
    K, Hs, Ws = (int(d) for d in s.shape)
    if not 1 <= K <= _lib.HSR_MAX_SRF_BANDS:
        raise ValueError(f"{name} must hold 1..{_lib.HSR_MAX_SRF_BANDS} planes, got {K}")
    return s, K, Hs, Ws, int(s.stride(0)) if K > 1 else Hs * Ws


def _factor(factor) -> int:
    f = int(factor)
    if f < 1 or f != factor:
        raise ValueError(f"factor must be an integer >= 1, got {factor!r}")
    return f


def bilinear_fine_mask(src: torch.Tensor, factor: int, *, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``mask10`` of s2_emit/poly_regression.py:159 without the fine planes: [Hs*factor, Ws*factor] bool =
    ``isfinite(bilinear_upsample(src, factor)).all(0)`` (no nodata, no gate), from the [K, Hs, Ws] f32 planes."""
    s, K, Hs, Ws, sps = _coarse_planes(src)
    f = _factor(factor)
    with torch.cuda.device_of(s):
        if out is None:
            out = torch.empty((Hs * f, Ws * f), dtype=torch.bool, device=s.device)
        elif out.dtype != torch.bool or tuple(out.shape) != (Hs * f, Ws * f) or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous [{Hs * f}, {Ws * f}] bool tensor")
        _lib.check(_lib.lib().hsr_bilinear_fine_mask_u8(s.data_ptr(), K, Hs, Ws, sps, f, _cuda(out.view(torch.uint8), "out", torch.uint8).data_ptr(),
                                                        _stream()))
    return out


def bilinear_apply(src: torch.Tensor, factor: int, coeffs: torch.Tensor, *, x_stretch: Optional[torch.Tensor] = None,
                   lo: float = 0.0, hi: float = 1.0, out: Optional[torch.Tensor] = None,
                   mask_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Colour-matched planes on the ``factor``-times finer grid in one pass (s2_emit/poly_regression.py:150-162 on K
    planes): ``x10 = bilinear_upsample(src, factor)``, ``mask10 = isfinite(x10).all(0)``, ``xs = x10`` stretched with
    ``x_stretch`` ([K, 1, 2] f64 (lo, hi), optional) on every pixel, ``(f32) polyval_f64(coeffs[k], xs)`` where mask10,
    then every pixel clipped to [lo, hi] (``lo > hi``: no clip).  Bit-identical to ``bilinear_upsample`` ->
    ``fit_mask(gate_k=-1)`` -> ``poly_solve_apply`` with the moments that gave ``coeffs``; the fine intermediates are
    never written.  Returns ``(out [K, Hs*factor, Ws*factor] f32 padded planes, mask10 [Hs*factor, Ws*factor] bool)``."""
    s, K, Hs, Ws, sps = _coarse_planes(src)
    f = _factor(factor)
    co = _cuda(coeffs, "coeffs", torch.float64).contiguous()
    if co.dim() != 2 or co.shape[0] != K or not 2 <= co.shape[1] <= _lib.HSR_MAX_POLY_DEG + 1:
        raise ValueError(f"coeffs must be [K={K}, deg+1] with 1 <= deg <= {_lib.HSR_MAX_POLY_DEG}, got {tuple(co.shape)}")
    deg = int(co.shape[1]) - 1
    xst = _stretch_arg(x_stretch, K, 1, "x_stretch")
    Hd, Wd = Hs * f, Ws * f
    with torch.cuda.device_of(s):
        if out is None:
            out = alloc_planes(K, (Hd, Wd), s.device)
        else:
            _cuda(out, "out", torch.float32)
            if tuple(out.shape) != (K, Hd, Wd):
                raise ValueError(f"out must be [{K}, {Hd}, {Wd}], got {tuple(out.shape)}")
        ops = _plane_stride(out, K, Hd * Wd, "out")
        if mask_out is None:
            mask_out = torch.empty((Hd, Wd), dtype=torch.bool, device=s.device)
        elif mask_out.dtype != torch.bool or tuple(mask_out.shape) != (Hd, Wd) or not mask_out.is_contiguous():
            raise ValueError(f"mask_out must be a contiguous [{Hd}, {Wd}] bool tensor")
        m = _cuda(mask_out.view(torch.uint8), "mask_out", torch.uint8)
        _lib.check(_lib.lib().hsr_bilinear_apply_f32(s.data_ptr(), K, Hs, Ws, sps, f, co.data_ptr(), deg, _ptr(xst),
                                                     float(lo), float(hi), out.data_ptr(), max(ops, Hd * Wd),
                                                     m.data_ptr(), _stream()))
    return out, mask_out


# --------------------------------------------------------------------------------------- general grid warp
WARP_KERNELS = {"nearest": 0, "bilinear": 1, "cubic": 2, "average": 3}


def _warp_geo(src_gt, dst_gt, utm_zone, south, scales):
    g = _lib.WarpGeo()
    for i in range(6):
        g.src_gt[i] = float(src_gt[i])
        g.dst_gt[i] = float(dst_gt[i])
    g.utm_zone = int(utm_zone)
    g.south = int(bool(south))
    g.xscale, g.yscale = (float(scales[0]), float(scales[1])) if scales is not None else (1.0, 1.0)
    return g


def padded_bands(bands: int) -> int:
    """Record length (floats) that puts every pixel of a band-interleaved cube on a 16-byte boundary."""
    return (int(bands) + 3) // 4 * 4


def warp(src: torch.Tensor, src_gt, dst_gt, dst_shape, *, utm_zone: int = 0, south: bool = False, scales=None,
         kernel: str = "cubic", nodata=None, dst_nodata=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Resample the band-interleaved cube ``src`` [Hs, Ws, B] f32 onto the grid ``dst_gt`` / ``dst_shape`` = (Hd, Wd):
    [Hd, Wd, B] f32 (``hsr_warp_f32``; gdalwarp of emit_proj.py:876-940).  ``src`` may be a view of a padded buffer
    (``src.stride(1) >= B``); ``out`` likewise — when it is not given it is allocated with records padded to a
    multiple of four floats (the fast path) and returned as the [Hd, Wd, B] view."""
    s = _cuda(src, "src", torch.float32)
    if s.dim() != 3:
        raise ValueError("src must be [Hs, Ws, B]")
    Hs, Ws, B = s.shape
    if not (s.stride(2) == 1 and s.stride(0) == Ws * s.stride(1) and s.stride(1) >= B):
        s = s.contiguous()
    Hd, Wd = int(dst_shape[0]), int(dst_shape[1])
    code = WARP_KERNELS.get(kernel)
    if code is None:
        raise ValueError(f"kernel must be one of {sorted(WARP_KERNELS)}, got {kernel!r}")
    fill = dst_nodata if dst_nodata is not None else (nodata if nodata is not None else 0.0)
    geo = _warp_geo(src_gt, dst_gt, utm_zone, south, scales)
    with torch.cuda.device_of(s):
        if out is None:
            out = torch.empty((Hd, Wd, padded_bands(B)), dtype=torch.float32, device=s.device)[:, :, :B]
        else:
            _cuda(out, "out", torch.float32)
            if tuple(out.shape) != (Hd, Wd, B) or out.stride(2) != 1 or out.stride(0) != Wd * out.stride(1):
                raise ValueError("out must be a [Hd, Wd, B] view with unit band stride and dense rows")
        wsb = int(_lib.lib().hsr_warp_workspace_bytes(Hd, Wd)) if code in (1, 2) else 0   # point kernels need none
        ws = torch.empty(wsb // 8, dtype=torch.float64, device=s.device) if wsb else None
        _lib.check(_lib.lib().hsr_warp_f32(s.data_ptr(), Hs, Ws, B, int(s.stride(1)), ctypes.addressof(geo), code,
                                           int(nodata is not None), 0.0 if nodata is None else float(nodata), float(fill),
                                           Hd, Wd, out.data_ptr(), int(out.stride(1)) if Hd * Wd else B, _ptr(ws), wsb,
                                           _stream()))
    return out


def warp_coords(src_gt, dst_gt, dst_shape, *, utm_zone: int = 0, south: bool = False, device=None,
                rows=None) -> torch.Tensor:
    """[Hd, Wd, 2] f64: source pixel coordinates (x, y) of every destination pixel centre (``hsr_warp_coords_f64``).
    ``rows`` = (r0, r1): only destination rows [r0, r1), [r1 - r0, Wd, 2], bit-identical to those rows of the whole
    grid (``hsr_warp_coords_rows_f64``)."""
    Hd, Wd = int(dst_shape[0]), int(dst_shape[1])
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    geo = _warp_geo(src_gt, dst_gt, utm_zone, south, None)
    if rows is not None:
        r0, r1 = int(rows[0]), int(rows[1])
        if not 0 <= r0 <= r1 <= Hd:
            raise ValueError(f"rows must satisfy 0 <= r0 <= r1 <= {Hd}, got {tuple(rows)}")
    with torch.cuda.device(dev):
        if rows is None:
            out = torch.empty((Hd, Wd, 2), dtype=torch.float64, device=dev)
            _lib.check(_lib.lib().hsr_warp_coords_f64(ctypes.addressof(geo), Hd, Wd, out.data_ptr(), _stream()))
        else:
            out = torch.empty((r1 - r0, Wd, 2), dtype=torch.float64, device=dev)
            if out.numel():                   # an empty tensor has no storage to point at
                _lib.check(_lib.lib().hsr_warp_coords_rows_f64(ctypes.addressof(geo), r0, r1 - r0, Wd, out.data_ptr(),
                                                               _stream()))
    return out


PLANE_WARP_KERNELS = {"bilinear": 1, "cubic": 2}


def _plane_kernel(kernel: str) -> int:
    code = PLANE_WARP_KERNELS.get(kernel)
    if code is None:
        raise ValueError(f"kernel must be one of {sorted(PLANE_WARP_KERNELS)} for a plane warp, got {kernel!r}")
    return code


def _coords_arg(coords) -> torch.Tensor:
    co = _cuda(coords, "coords", torch.float64)
    if co.dim() != 3 or co.shape[2] != 2 or not co.is_contiguous():
        raise ValueError(f"coords must be a contiguous [Hd, Wd, 2] tensor, got shape {tuple(co.shape)}")
    return co


def _scales_geo(scales):
    geo = _lib.WarpGeo()
    geo.xscale, geo.yscale = float(scales[0]), float(scales[1])
    return geo


def warp_src_row_range(coords: torch.Tensor, src_shape, scales, *, kernel: str) -> torch.Tensor:
    """int64[2] on the device: [first, last + 1) source row that :func:`warp_planes` reads through its filter for the
    pixels of ``coords`` [rows, Wd, 2] f64 (a band of :func:`warp_coords`) on a source of ``src_shape`` = (Hs, Ws);
    ``range[1] == 0`` when no pixel centre is inside the source (``hsr_warp_src_row_range``).  Conservative: zero
    weights and invalid source pixels are counted, so a window of these rows is never too small."""
    code = _plane_kernel(kernel)
    co = _coords_arg(coords)
    Hs, Ws = int(src_shape[0]), int(src_shape[1])
    geo = _scales_geo(scales)
    with torch.cuda.device_of(co):
        rng = torch.tensor([-1, 0], dtype=torch.int64, device=co.device)       # u64 max, 0
        _lib.check(_lib.lib().hsr_warp_src_row_range(co.data_ptr(), int(co.shape[0]), int(co.shape[1]), Hs, Ws,
                                                     ctypes.addressof(geo), code, rng.data_ptr(), _stream()))
    return rng


def warp_planes(planes: torch.Tensor, src_valid: torch.Tensor, coords: torch.Tensor, scales, *, kernel: str,
                fill_out: torch.Tensor, gate_k: int = 0, gate_gt: float = 0.0, out: Optional[torch.Tensor] = None,
                valid_out: Optional[torch.Tensor] = None, fit_mask_out: Optional[torch.Tensor] = None,
                src_row0: int = 0, src_rows_total: Optional[int] = None, outside: Optional[torch.Tensor] = None):
    """Warp K planar images ``planes`` [K, Hs, Ws] f32 (any plane stride, as ``alloc_planes`` pads them) onto the grid
    of ``coords`` [Hd, Wd, 2] f64 (:func:`warp_coords`) with the taps of :func:`warp` (``hsr_warp_planes_f32``).
    ``src_valid`` [Hs, Ws] bool/u8: source pixels whose taps may be used (the GLT valid mask); ``scales`` = (xscale,
    yscale) of ``EMIT_data.warp.warp_scales``; ``fill_out`` [K] f32: written where the destination is not covered.
    Returns ``(planes [K, Hd, Wd] f32, dst_valid [Hd, Wd] bool, fit_mask [Hd, Wd] bool)``, the fit mask being
    ``dst_valid & isfinite(planes).all(0) & (planes[gate_k] > gate_gt)`` (gate_k < 0: no gate).
    ``src_row0`` / ``src_rows_total``: ``planes`` and ``src_valid`` hold only source rows [src_row0, src_row0 + Hs) of
    a source of ``src_rows_total`` rows (``hsr_warp_planes_window_f32``; :func:`warp_src_row_range` sizes the window).
    Where the window holds every row a pixel's taps reach, the result is bit-identical to the warp of the whole source;
    the pixels that needed a row outside it are added to ``outside`` (int64[1] on the device), which must stay 0."""
    code = _plane_kernel(kernel)
    p = _cuda(planes, "planes", torch.float32)
    if p.dim() != 3:
        raise ValueError(f"planes must be [K, Hs, Ws], got shape {tuple(p.shape)}")
    K, Hs, Ws = (int(d) for d in p.shape)
    windowed = src_rows_total is not None or src_row0 != 0 or outside is not None
    ps = _plane_stride(p, K, Hs * Ws, "planes")
    sv = src_valid.view(torch.uint8) if src_valid.dtype == torch.bool else src_valid
    sv = _cuda(sv, "src_valid", torch.uint8).contiguous()
    if sv.numel() != Hs * Ws:
        raise ValueError(f"src_valid must have one entry per source pixel ({Hs} x {Ws}), got shape {tuple(sv.shape)}")
    co = _coords_arg(coords)
    Hd, Wd = int(co.shape[0]), int(co.shape[1])
    fo = _cuda(fill_out, "fill_out", torch.float32).contiguous()
    if fo.numel() != K:
        raise ValueError(f"fill_out must have K = {K} entries, got {fo.numel()}")
    if outside is not None:
        _cuda(outside, "outside", torch.int64)
        if outside.numel() != 1:
            raise ValueError("outside must be an int64[1] device tensor")
    geo = _scales_geo(scales)
    with torch.cuda.device_of(p):
        if out is None:
            out = alloc_planes(K, (Hd, Wd), p.device)
        else:
            _cuda(out, "out", torch.float32)
        ops = _plane_stride(out, K, Hd * Wd, "out")
        valid = (_mask_out(valid_out, Hd * Wd) if valid_out is not None
                 else torch.empty(Hd * Wd, dtype=torch.uint8, device=p.device))
        fm = (_mask_out(fit_mask_out, Hd * Wd) if fit_mask_out is not None
              else torch.empty(Hd * Wd, dtype=torch.uint8, device=p.device))
        if windowed:
            total = int(src_rows_total) if src_rows_total is not None else int(src_row0) + Hs
            _lib.check(_lib.lib().hsr_warp_planes_window_f32(
                p.data_ptr(), total, Ws, K, ps, sv.data_ptr(), int(src_row0), Hs, co.data_ptr(), ctypes.addressof(geo),
                code, fo.data_ptr(), int(gate_k), float(gate_gt), Hd, Wd, out.data_ptr(), ops, valid.data_ptr(),
                fm.data_ptr(), _ptr(outside), _stream()))
        else:
            _lib.check(_lib.lib().hsr_warp_planes_f32(p.data_ptr(), Hs, Ws, K, ps, sv.data_ptr(), co.data_ptr(),
                                                      ctypes.addressof(geo), code, fo.data_ptr(), int(gate_k),
                                                      float(gate_gt), Hd, Wd, out.data_ptr(), ops, valid.data_ptr(),
                                                      fm.data_ptr(), _stream()))
    return out, valid.view(torch.bool).view(Hd, Wd), fm.view(torch.bool).view(Hd, Wd)
