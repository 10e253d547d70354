"""Seeded randomised sweep of the GLT gather / fused SRF / tile export kernels against the oracle: shapes, band counts,
pixel strides, base alignments, GLT patterns and weight sparsity drawn at random (fixed seeds, so failures reproduce).
Bars as in test_gpu_parity.py: gather, masks, diagnostics and the uint16 export bit-exact; fused SRF bit-identical to the
un-fused kernel on the oracle's ortho cube and 1e-5 relative against a float64 contraction."""
import os

import numpy as np
import pytest
import torch

from hsr_b200 import kernels, synthetic
from oracle import glt as oglt
from oracle import tiles as otiles

pytestmark = pytest.mark.gpu


def bits(a):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def random_glt(rng, Hr, Wr, Ho, Wo):
    kind = rng.integers(0, 5)
    if kind == 0:                                               # uniformly random sources (no runs at all)
        gx = rng.integers(1, Wr + 1, size=(Ho, Wo))
        gy = rng.integers(1, Hr + 1, size=(Ho, Wo))
    elif kind == 1:                                             # affine map with random scale / rotation: runs + duplicates
        th, sc = rng.uniform(0, 2 * np.pi), rng.uniform(0.3, 2.5)
        yy, xx = np.mgrid[0:Ho, 0:Wo]
        sx = np.rint((xx - Wo / 2) * np.cos(th) * sc + (yy - Ho / 2) * np.sin(th) * sc + Wr / 2)
        sy = np.rint(-(xx - Wo / 2) * np.sin(th) * sc + (yy - Ho / 2) * np.cos(th) * sc + Hr / 2)
        ok = (sx >= 0) & (sx < Wr) & (sy >= 0) & (sy < Hr)
        gx, gy = np.where(ok, sx + 1, 0), np.where(ok, sy + 1, 0)
    elif kind == 2:                                             # linear scan of the raw grid from a random offset (long runs,
        q = (np.arange(Ho * Wo) + rng.integers(0, Hr * Wr)) % (Hr * Wr)     # wrapping rows and the end of the cube)
        gx, gy = (q % Wr + 1).reshape(Ho, Wo), (q // Wr + 1).reshape(Ho, Wo)
    elif kind == 3:                                             # descending scan
        q = (Hr * Wr - 1 - np.arange(Ho * Wo)) % (Hr * Wr)
        gx, gy = (q % Wr + 1).reshape(Ho, Wo), (q // Wr + 1).reshape(Ho, Wo)
    else:                                                       # everything invalid but a few pixels
        gx, gy = np.zeros((Ho, Wo), np.int64), np.zeros((Ho, Wo), np.int64)
        for _ in range(5):
            gx[rng.integers(0, Ho), rng.integers(0, Wo)] = rng.integers(1, Wr + 1)
        gy[gx != 0] = rng.integers(1, Hr + 1, size=int((gx != 0).sum()))
    gx, gy = gx.astype(np.int32), gy.astype(np.int32)
    n = Ho * Wo
    for val in (0, Wr + 1, Hr + 7, -3, -2147483648, 2147483647):       # holes, out of bounds, negative, int32 extremes
        k = rng.integers(0, max(2, n // 40))
        idx = rng.integers(0, n, size=k)
        (gx if rng.random() < 0.5 else gy).reshape(-1)[idx] = val
    gx.reshape(-1)[rng.integers(0, n)], gy.reshape(-1)[rng.integers(0, n)] = Wr, Hr      # the last raw pixel
    return gx, gy


@pytest.mark.parametrize("seed", range(int(os.environ.get("HSR_FUZZ_SEEDS", "24"))))     # HSR_FUZZ_SEEDS=400 for a long hunt
def test_gather_srf_export_random_configurations(seed):
    rng = np.random.default_rng(1000 + seed)
    bands = int(rng.choice([32, 33, 47, 64, 100, 128, 200, 285, 285, 285, 286, 287, 288, 330]))
    Hr, Wr = int(rng.integers(2, 60)), int(rng.integers(2, 60))
    Ho, Wo = int(rng.integers(1, 90)), int(rng.integers(1, 90))
    transpose = bool(rng.integers(0, 2))
    raw = synthetic.raw_cube_bits_np((Hr, Wr, bands), seed=seed)
    raw[rng.integers(0, Hr), rng.integers(0, Wr), rng.integers(0, bands)] = np.nan
    raw[Hr - 1, Wr - 1, bands - 1] = np.inf
    raw[0, 0, 0] = -np.inf
    gx, gy = random_glt(rng, Hr, Wr, Ho, Wo)
    phys = np.ascontiguousarray(raw.transpose(1, 0, 2)) if transpose else raw
    ref, vref, dref = oglt.glt_ortho(phys, gx, gy, transpose_raw_yx=transpose)

    # raw in a pitched buffer with a random pixel stride and a base that is only 4-byte aligned
    stride, off = bands + int(rng.integers(0, 9)), int(rng.integers(0, 4))
    d0, d1 = phys.shape[:2]
    buf = torch.full((d0 * d1 * stride + 8,), 123.0, dtype=torch.float32, device="cuda")
    view = buf[off:off + d0 * d1 * stride].view(d0, d1, stride)[..., :bands]
    view.copy_(dev(phys))
    ops = bands + int(rng.integers(0, 6))
    o, v, d = kernels.glt_ortho(view, dev(gx), dev(gy), transpose_raw_yx=transpose, out_pix_stride=ops)
    assert np.array_equal(bits(o), bits(ref)), (seed, bands, stride, off)
    assert np.array_equal(v.cpu().numpy(), vref)
    assert d.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]

    # fused gather + SRF: random sparse weights (zero columns, single-band columns, dense columns)
    K = int(rng.integers(1, 17))
    W = np.zeros((bands, K), np.float32)
    for k in range(K):
        mode = rng.integers(0, 4)
        if mode == 0:
            continue                                            # an all-zero response
        lo = int(rng.integers(0, bands))
        hi = lo + 1 if mode == 1 else int(rng.integers(lo + 1, bands + 1))
        W[lo:hi, k] = rng.normal(size=hi - lo).astype(np.float32) * (rng.random(hi - lo) < 0.9)
    fill_out = (W.astype(np.float64).sum(0) * -9999.0).astype(np.float32)
    fm = torch.zeros((Ho, Wo), dtype=torch.bool, device="cuda")
    b1, v1, _, _ = kernels.glt_srf(view, dev(gx), dev(gy), dev(W), dev(fill_out), transpose_raw_yx=transpose,
                                   fit_mask_out=fm, gate_k=0, gate_gt=0.0)
    assert np.array_equal(v1.cpu().numpy(), vref)
    b2 = kernels.srf_integrate(dev(ref), dev(W))                # un-fused kernel on the oracle's ortho cube
    assert np.array_equal(bits(b1)[:, vref], bits(b2)[:, vref]), (seed, bands, K)
    want = np.einsum("hwb,bk->khw", ref.astype(np.float64), W.astype(np.float64))
    got = b1.cpu().numpy().astype(np.float64)
    fin = np.isfinite(ref).all(-1) & vref                       # finite spectra: plain contraction
    scale = np.einsum("hwb,bk->khw", np.abs(np.where(np.isfinite(ref), ref, 0)).astype(np.float64), np.abs(W).astype(np.float64))
    assert np.all(np.abs(got - want)[:, fin] <= 1e-5 * scale[:, fin] + 1e-30)
    bad = ~np.isfinite(ref).all(-1) & vref                      # a NaN / Inf anywhere poisons every band (synth.py:41)
    assert not np.isfinite(got[:, bad]).any() or not bad.any()
    assert np.array_equal(got[:, ~vref], np.broadcast_to(fill_out[:, None].astype(np.float64), got[:, ~vref].shape))
    want_fm = vref & np.isfinite(got).all(0) & (got[0] > 0.0)
    assert np.array_equal(fm.cpu().numpy(), want_fm)

    # fused tile export: uint16 quantisation + black mask, band-sequential
    q16, vq, black, _ = kernels.glt_ortho_u16(view, dev(gx), dev(gy), transpose_raw_yx=transpose)
    wq = otiles.quantize_emit_u16(np.transpose(ref, (2, 0, 1)), nodata=-9999.0)
    assert np.array_equal(q16.view(torch.int16).cpu().numpy().view(np.uint16), wq), (seed, bands)
    assert np.array_equal(vq.cpu().numpy(), vref)
    assert np.array_equal(black.cpu().numpy(), otiles.is_black_mask(np.transpose(ref, (2, 0, 1)), nodata=-9999.0))


@pytest.mark.parametrize("seed", range(int(os.environ.get("HSR_FUZZ_WARP_SEEDS", "16"))))
def test_warp_random_geometries_with_coordinate_workspace(seed):
    """hsr_warp_f32 against oracle/warp.py on random same-CRS affine geometries (scale 0.35 .. 2.5 per axis, any rotation,
    partial overlap), band counts, record paddings, kernels and nodata patterns: every path of the kernels (staged lean /
    classified / global-memory taps, vector / scalar records, the exact pass of filters wider than 8 taps)."""
    from hsr_b200.EMIT_data import warp as hwarp
    from oracle import warp as owarp
    rng = np.random.default_rng(5000 + seed)
    ND = -9999.0
    bands = int(rng.choice([1, 3, 4, 7, 12, 129, 285]))
    Hs, Ws = int(rng.integers(6, 40)), int(rng.integers(6, 40))
    Hd, Wd = int(rng.integers(1, 22)), int(rng.integers(1, 22))
    src = rng.random((Hs, Ws, bands)).astype(np.float32)
    mode = rng.integers(0, 4)
    if mode >= 1:                                               # fill regions (every band nodata)
        yy, xx = np.mgrid[0:Hs, 0:Ws]
        src[(yy * rng.uniform(-1, 1) + xx * rng.uniform(-1, 1)) > rng.uniform(0, 10)] = ND
    if mode >= 2:                                               # band-specific nodata, non-finite samples
        src[rng.random(src.shape) < 0.01] = ND
        src[rng.integers(0, Hs), rng.integers(0, Ws), rng.integers(0, bands)] = np.nan
        src[rng.integers(0, Hs), rng.integers(0, Ws), rng.integers(0, bands)] = np.inf
    nodata = None if mode == 3 and rng.random() < 0.5 else ND
    sgt = (1000.0, 10.0, 0.0, 5000.0, 0.0, -10.0)
    th = rng.uniform(0, 2 * np.pi) if rng.random() < 0.5 else rng.uniform(-0.05, 0.05)
    fx, fy = rng.uniform(0.35, 2.5, size=2)                     # destination pixel size / source pixel size
    cx, cy = 1000.0 + rng.uniform(0.2, 0.8) * Ws * 10.0, 5000.0 - rng.uniform(0.2, 0.8) * Hs * 10.0
    a, b_, d_, e = 10 * fx * np.cos(th), 10 * fy * np.sin(th), 10 * fx * np.sin(th), -10 * fy * np.cos(th)
    dgt = (cx - a * Wd / 2 - b_ * Hd / 2, a, b_, cy - d_ * Wd / 2 - e * Hd / 2, d_, e)
    kernel = "cubic" if rng.random() < 0.7 else "bilinear"
    scales = hwarp.warp_scales(dgt, sgt, (Hd, Wd)) if rng.random() < 0.8 else (1.0, 1.0)
    r0 = 2 if kernel == "cubic" else 1
    if max(np.ceil(r0 / min(scales[0], 1.0)), np.ceil(r0 / min(scales[1], 1.0))) > 8:
        scales = (1.0, 1.0)                                     # beyond the 16-tap limit of the kernels
    want = owarp.warp(src, sgt, dgt, Hd, Wd, utm=False, nodata=nodata, kernel=kernel, scales=scales)
    if rng.random() < 0.5:                                      # padded records (vector path) or dense ones
        P = kernels.padded_bands(bands)
        buf = torch.full((Hs, Ws, P), 55.0, dtype=torch.float32, device="cuda")
        buf[..., :bands] = dev(src)
        s = buf[..., :bands]
    else:
        s = dev(src)
    out = None if rng.random() < 0.5 else torch.empty((Hd, Wd, bands), dtype=torch.float32, device="cuda")
    got = kernels.warp(s, sgt, dgt, (Hd, Wd), scales=scales, kernel=kernel, nodata=nodata, out=out).cpu().numpy()
    fill = ND if nodata is not None else 0.0
    assert np.array_equal(np.isnan(got), np.isnan(want)), seed
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf]), seed
    ok = np.isfinite(want)
    assert np.array_equal(got[ok] == fill, want[ok] == fill), seed
    # 1e-5 relative to the magnitude of the weighted terms (renormalised partial sums amplify rounding where the
    # accumulated weight is small: GDAL's rule, see oracle/warp.py) + 1e-6 absolute
    # ... + 4 ulp (fp32) of the largest sample that takes part: without a declared nodata value the -9999 fill IS data, and a
    # result of order 1 is then the difference of fp32 terms of order 1e4 (the oracle accumulates in float64, as GDAL does)
    part = np.isfinite(src) if nodata is None else np.isfinite(src) & (src != np.float32(ND))
    mag = float(np.abs(src[part]).max()) if part.any() else 0.0
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    assert np.all(err <= 1e-5 * np.maximum(np.abs(want[ok]), 1.0) * 4 + 1e-6 + 2.4e-7 * mag), (seed, float(err.max()))


@pytest.mark.parametrize("seed", range(int(os.environ.get("HSR_FUZZ_FIT_SEEDS", "16"))))
def test_fit_apply_percentiles_random_series(seed):
    """Polynomial fit / apply and the exact percentiles on random series: lengths that are no multiple of anything, 1..13
    series, degrees 1..4, shared / per-series masks of any density, non-finite samples, planar and interleaved layouts.
    Bars: coefficients 1e-4 relative against np.polyfit (float64), applied values 1e-4 absolute, percentiles bit-identical
    to np.percentile."""
    rng = np.random.default_rng(9000 + seed)
    K = int(rng.integers(1, 14))
    n = int(rng.choice([1, 7, 200, 201, 255, 1000, 4099, 65537, 100003]))
    deg = int(rng.integers(1, 5))
    x = rng.uniform(0.02, 0.9, size=(K, n)).astype(np.float32)
    true = rng.normal(size=(K, deg + 1)) * 0.5
    y = np.stack([np.polyval(true[k], x[k].astype(np.float64)) for k in range(K)]) + rng.normal(0, 0.01, size=(K, n))
    y = y.astype(np.float32)
    per_series = bool(rng.integers(0, 2)) and K > 1
    mask = rng.random((K if per_series else 1, n)) < rng.choice([0.05, 0.5, 0.95, 1.0])
    x[rng.integers(0, K), rng.integers(0, n)] = np.nan          # masked-in NaN / Inf are the caller's to exclude:
    y[rng.integers(0, K), rng.integers(0, n)] = np.inf          # np.polyfit would fail, so take them out of the mask
    finite = np.isfinite(x) & np.isfinite(y)
    mask = mask & (finite if per_series else finite.all(0, keepdims=True))
    xd, yd, md = dev(x), dev(y), dev(mask)
    interleaved = bool(rng.integers(0, 2)) and not per_series
    if interleaved:
        c = kernels.poly_fit(xd.t().contiguous(), yd.t().contiguous(), md.reshape(-1), deg, layout="interleaved")
    else:
        c = kernels.poly_fit(xd, yd, md if per_series else md.reshape(-1), deg)
    c = c.cpu().numpy()
    counts = mask.sum(1) if per_series else np.full(K, mask.sum())
    for k in range(K):
        mk = mask[k if per_series else 0]
        if counts[k] < 4 * (deg + 1):
            continue                                            # too few samples for a meaningful comparison
        ref = np.polyfit(x[k][mk].astype(np.float64), y[k][mk].astype(np.float64), deg)
        xs = np.linspace(x[k][mk].min(), x[k][mk].max(), 50)
        assert np.max(np.abs(np.polyval(c[k], xs) - np.polyval(ref, xs))) < 1e-4 * max(1.0, np.abs(np.polyval(ref, xs)).max()), (seed, k)
    # apply: float64 Horner where the mask is set, input elsewhere, everything clipped to [0, 1]
    coeffs = rng.normal(size=(K, deg + 1)) * 0.3
    xa = np.nan_to_num(x, nan=0.5)
    out = kernels.poly_apply(dev(xa), dev(coeffs), md if per_series else md.reshape(-1)).cpu().numpy().reshape(K, n)
    want = xa.astype(np.float32).copy()
    for k in range(K):
        mk = mask[k if per_series else 0]
        want[k][mk] = np.polyval(coeffs[k], xa[k][mk].astype(np.float64)).astype(np.float32)
    want = np.clip(want, 0, 1)
    assert np.max(np.abs(out - want)) < 1e-4
    # percentiles of the masked samples of every series: bit-identical to numpy
    if mask.any(1).all() and not per_series:
        q = sorted(rng.uniform(0, 100, size=2).tolist())
        got = kernels.masked_percentiles(dev(xa).reshape(K, n), md.reshape(1, n), q).cpu().numpy().reshape(K, 2)
        ref = np.stack([np.percentile(xa[k][mask[0]], q) for k in range(K)])
        assert np.array_equal(got.view(np.int64), ref.view(np.int64)), (seed, q)
