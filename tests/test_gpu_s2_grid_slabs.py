"""Row slabs and global fits on the Sentinel-2 grid on the GPU: coordinates of a band of target rows
(hsr_warp_coords_rows_f64), the source rows a band reads (hsr_warp_src_row_range) against the numpy model of
tests/s2_slab_oracle.py, the plane warp over a window of source rows (hsr_warp_planes_window_f32) against the warp of
the whole source, PairSynthesizer.synthesize_slab_on_s2_grid stitched against one synthesize_on_s2_grid call, and
synthesize_sharded with granules on S2 targets against the oracle's fit over the concatenation."""
import dataclasses
import math
import types

import numpy as np
import pytest
import torch

from hsr_b200 import _lib, kernels, synthetic
from hsr_b200.EMIT_data import warp as hwarp
from hsr_b200.pipeline import PairSynthesizer, s2_target
from hsr_b200.s2_emit.srf import synthetic_s2_srf
from oracle import poly as opoly

import s2_slab_oracle as sso

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

PIX = 0.000542232520256367
GLT_GT = (-118.30, PIX, 0.0, 34.20, 0.0, -PIX)
S2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)
GLT_GT_34S = (18.40, PIX, 0.0, -33.90, 0.0, -PIX)


def s2_grid_around(epsg, glt_gt):
    zone, south = hwarp.epsg_to_utm(epsg)
    X, Y = hwarp.utm_forward(glt_gt[0], glt_gt[3], zone, south)
    return hwarp.S2Grid(epsg=epsg, x0=math.floor((float(X) - 3000.0) / 60.0) * 60.0 + 30.0,
                        y0=math.floor((float(Y) + 3000.0) / 60.0) * 60.0 + 20.0, dx=10.0, dy=10.0, width=10980,
                        height=10980)


S2_34S = s2_grid_around(32734, GLT_GT_34S)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def bits(t):
    """int32 / int64 view of a tensor for bit-for-bit comparisons."""
    t = t.contiguous()
    return t.view(torch.int64) if t.dtype == torch.float64 else (t.view(torch.int32) if t.dtype == torch.float32 else t)


def grown(target, above):
    """The target with ``above`` extra rows on top: those rows have no pixel centre inside the source."""
    g = list(target.dst_gt)
    g[3] -= above * g[5]
    return dataclasses.replace(target, dst_gt=tuple(g), shape=(target.shape[0] + above, target.shape[1]), _coords={})


# ---------------------------------------------------------------------------------------------- coordinates of a band
@pytest.mark.parametrize("zone", ["11N", "34S"])
def test_coords_rows_bit_identical(zone):
    glt_gt, s2 = (GLT_GT, S2) if zone == "11N" else (GLT_GT_34S, S2_34S)
    t = hwarp.s2_target(glt_gt, (300, 260), s2)
    Hd, Wd = t.shape
    whole = t.coords()
    for r0, r1 in ((0, 7), (Hd // 3, Hd // 3 + 11), (Hd - 5, Hd), (Hd // 2, Hd // 2)):
        band = t.coords(rows=(r0, r1))
        assert band.shape == (r1 - r0, Wd, 2)
        assert torch.equal(bits(band), bits(whole[r0:r1]))
        band2 = kernels.warp_coords(t.src_gt, t.dst_gt, t.shape, utm_zone=t.zone, south=t.south, rows=(r0, r1))
        assert torch.equal(bits(band2), bits(band))
    assert t.coords() is whole                                    # a band is not cached in place of the whole grid


# ---------------------------------------------------------------------------------------------- source rows of a band
@pytest.mark.parametrize("kernel", ["cubic", "bilinear"])
@pytest.mark.parametrize("xres", [60.0, 120.0])
def test_src_row_range_vs_model(kernel, xres):
    Hs, Ws = 150, 140
    t = grown(hwarp.s2_target(GLT_GT, (Hs, Ws), S2, xres, xres, kernel=kernel), 4)
    assert xres == 60.0 or t.scales[1] < 1.0
    co = t.coords()
    for t0, t1 in [(0, 3)] + sso.uneven_bands(t.shape[0], 5, seed=int(xres)):
        band = co[t0:t1].contiguous()
        rng = kernels.warp_src_row_range(band, (Hs, Ws), t.scales, kernel=kernel).tolist()
        want = sso.src_row_range(host(band), Hs, Ws, t.scales, kernel)
        if want is None:
            assert rng[1] == 0 and (t0, t1) == (0, 3)
        else:
            assert tuple(rng) == want
    off = co[:2].clone()
    off[..., 1] += Hs + 50.0                                      # wholly below the source
    assert kernels.warp_src_row_range(off, (Hs, Ws), t.scales, kernel=kernel)[1].item() == 0


# ---------------------------------------------------------------------------------------------- the windowed warp
@pytest.mark.parametrize("kernel", ["cubic", "bilinear"])
@pytest.mark.parametrize("padded", [True, False])
@pytest.mark.parametrize("K", [1, 3, 12, 13])
def test_warp_planes_window(K, padded, kernel):
    rng = np.random.default_rng(K * 4 + padded * 2 + (kernel == "cubic"))
    Hs, Ws = 60, 52
    t = hwarp.s2_target(GLT_GT, (Hs, Ws), S2, kernel=kernel)
    Hd, Wd = t.shape
    valid = rng.random((Hs, Ws)) > 0.05
    fill_out = (-9999.0 * (0.5 + rng.random(K))).astype(np.float32)
    planes = (0.05 + 0.9 * rng.random((K, Hs, Ws))).astype(np.float32)
    planes[:, ~valid] = fill_out[:, None]
    planes[K - 1, 30, 20] = np.nan
    fo = dev(fill_out)
    src = dev(planes)
    sv = dev(valid)
    co = t.coords()
    kw = dict(kernel=kernel, fill_out=fo, gate_k=K - 1, gate_gt=0.3)
    whole = kernels.warp_planes(src, sv, co, t.scales, **kw)

    def window(band, o0, o1):
        if padded:
            w = kernels.alloc_planes(K, (o1 - o0, Ws), "cuda")
            w.copy_(src[:, o0:o1])
        else:
            w = src[:, o0:o1].contiguous()
        out = None if padded else torch.empty((K, band.shape[0], Wd), device="cuda")
        outside = torch.zeros(1, dtype=torch.int64, device="cuda")
        got = kernels.warp_planes(w, sv[o0:o1], band, t.scales, src_row0=o0, src_rows_total=Hs, outside=outside,
                                  out=out, **kw)
        return got, int(outside.item())

    for t0, t1 in sso.uneven_bands(Hd, 4, seed=K):
        band = co[t0:t1].contiguous()
        o0, o1 = kernels.warp_src_row_range(band, (Hs, Ws), t.scales, kernel=kernel).tolist()
        assert 0 <= o0 < o1 <= Hs
        (p, v, f), n_out = window(band, o0, o1)
        assert n_out == 0
        assert torch.equal(bits(p), bits(whole[0][:, t0:t1])), "planes differ from the whole-source warp"
        assert torch.equal(v, whole[1][t0:t1]) and torch.equal(f, whole[2][t0:t1])
        # the range is conservative (rows of zero weight included); the rows that carry a non-zero tap are the tight
        # window: it gives the same bits, and one row less at either end misses
        taps = sso.tap_rows(host(band), Hs, Ws, t.scales, kernel)
        a, b = min(taps), max(taps) + 1
        assert o0 <= a < b <= o1
        (p, v, f), n_out = window(band, a, b)
        assert n_out == 0 and torch.equal(bits(p), bits(whole[0][:, t0:t1]))
        assert window(band, a + 1, b)[1] > 0 and window(band, a, b - 1)[1] > 0
    # the window that is the whole source, through the window entry point
    (p, v, f), n_out = window(co, 0, Hs)
    assert n_out == 0 and torch.equal(bits(p), bits(whole[0])) and torch.equal(v, whole[1]) and torch.equal(f, whole[2])
    # a window of no rows: fill, nothing valid, nothing read
    empty = torch.empty((K, 0, Ws), device="cuda")
    p, v, f = kernels.warp_planes(empty, torch.empty((0, Ws), dtype=torch.bool, device="cuda"), co, t.scales,
                                  src_row0=7, src_rows_total=Hs, outside=torch.zeros(1, dtype=torch.int64,
                                                                                     device="cuda"), **kw)
    assert torch.equal(p, fo[:, None, None].expand(K, Hd, Wd)) and not v.any() and not f.any()


# ---------------------------------------------------------------------------------------------- slabs of a mosaic
def _small():
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    Hr, Wr = 40, 34
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=0, good=good)
    raw[11, 9, 40] = np.nan
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=1, hole_frac=0.01, n_oob=4, n_neg=4)
    return w, good, raw, gx, gy, s2_target(GLT_GT, gx.shape, S2)


def _run_slabs(ps, raw, gxd, gyd, s2, target, bands, Hr, **kw):
    out = []
    for t0, t1 in bands:
        r = ps.synthesize_slab_on_s2_grid(raw, gxd, gyd, s2[:, t0:t1].contiguous(), target, (t0, t1), **kw)
        assert r.grid is target and r.bands.shape == (ps.K, t1 - t0, target.shape[1])
        lo, hi = r.raw_rows
        assert hi - lo < Hr
        out.append(r)
    return out


def _check_stitched(res, full, bands):
    for name in ("bands", "valid", "fit_mask"):
        got = torch.cat([getattr(r, name) for r in res], dim=-2)
        assert torch.equal(bits(got), bits(getattr(full, name))), name


def test_slabs_small_bit_identical():
    w, good, raw, gx, gy, target = _small()
    target = grown(target, 6)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda")
    gxd, gyd = dev(gx), dev(gy)
    full0 = ps.synthesize_on_s2_grid(dev(raw), gxd, gyd, torch.zeros((ps.K,) + target.shape, device="cuda"), target)
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(full0.bands), seed=2)
    full = ps.synthesize_on_s2_grid(dev(raw), gxd, gyd, s2, target)
    Hd = target.shape[0]
    bands = [(0, 3)] + [(3 + a, 3 + b) for a, b in sso.uneven_bands(Hd - 3, 4, seed=0)]
    for raw_in in (torch.from_numpy(raw).pin_memory(), dev(raw)):
        res = _run_slabs(ps, raw_in, gxd, gyd, s2, target, bands, raw.shape[0])
        _check_stitched(res, full, bands)
        assert res[0].ortho_rows == (0, 0) and res[0].raw_rows == (0, 0) and not res[0].valid.any()
        assert all(r.ortho_rows[1] > r.ortho_rows[0] for r in res[1:])
        assert torch.equal(res[0].bands, ps.fill_out[:, None, None].expand_as(res[0].bands))


def test_slabs_shrunk_window_raises(monkeypatch):
    w, good, raw, gx, gy, target = _small()
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda")
    s2 = torch.rand((ps.K,) + target.shape, device="cuda")
    Hd = target.shape[0]
    args = (dev(raw), dev(gx), dev(gy), s2[:, Hd // 3:2 * Hd // 3].contiguous(), target, (Hd // 3, 2 * Hd // 3))
    ps.synthesize_slab_on_s2_grid(*args)
    real_src, real_glt = kernels.warp_src_row_range, kernels.glt_row_range

    def upper_half(r):                # the range with its first half cut away
        return torch.stack([(r[0] + r[1]) // 2, r[1]])

    monkeypatch.setattr(kernels, "warp_src_row_range", lambda *a, **k: upper_half(real_src(*a, **k)))
    with pytest.raises(RuntimeError, match="ortho rows"):
        ps.synthesize_slab_on_s2_grid(*args)
    monkeypatch.setattr(kernels, "warp_src_row_range", real_src)
    monkeypatch.setattr(kernels, "glt_row_range", lambda *a, **k: upper_half(real_glt(*a, **k)))
    with pytest.raises(RuntimeError, match="raw rows"):
        ps.synthesize_slab_on_s2_grid(*args)


def test_slabs_granule_bit_identical():
    """The 1280 x 1242 granule onto the 1215 x 959 zone 11 target of test_gpu_s2_grid.py, raw in pinned host memory."""
    Hr, Wr, B = 1280, 1242, 285
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    rawd = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, "cuda", good=good)
    gxd, gyd = (dev(a) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    src_gt = (-118.60, PIX, 0.0, 34.90, 0.0, -PIX)
    s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
    target = s2_target(src_gt, gxd.shape, s2g)
    assert target.shape == (1215, 959)
    target = grown(target, 5)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda")
    b0 = ps.synthesize_on_s2_grid(rawd, gxd, gyd, torch.zeros((ps.K,) + target.shape, device="cuda"), target).bands
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(b0), seed=1)
    full = ps.synthesize_on_s2_grid(rawd, gxd, gyd, s2, target)
    raw_host = rawd.cpu().pin_memory()
    del rawd
    Hd = target.shape[0]
    bands = [(0, 4)] + [(4 + a, 4 + b) for a, b in sso.uneven_bands(Hd - 4, 4, seed=3)]
    stage = torch.empty(Hr * Wr * B, dtype=torch.float32, device="cuda")
    res = _run_slabs(ps, raw_host, gxd, gyd, s2, target, bands, Hr, stage=stage)
    _check_stitched(res, full, bands)
    assert res[0].ortho_rows == (0, 0)


# ---------------------------------------------------------------------------------------------- many granules, S2 targets
def _granules(ps, w, good):
    out = []
    specs = [(GLT_GT, S2, "cubic", 21), ((-118.10, PIX, 0.0, 34.05, 0.0, -PIX), S2, "bilinear", 22),
             (GLT_GT_34S, S2_34S, "cubic", 23), (None, None, None, 24)]
    for glt_gt, s2g, kernel, seed in specs:
        Hr, Wr = 40, 34
        raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=good)
        gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
        g = {"raw": dev(raw), "glt_x": dev(gx), "glt_y": dev(gy)}
        if glt_gt is None:
            x = ps.bands_from_raw(g["raw"], g["glt_x"], g["glt_y"])[0]
        else:
            g["target"] = s2_target(glt_gt, gx.shape, s2g, kernel=kernel)
            x = ps.synthesize_on_s2_grid(g["raw"], g["glt_x"], g["glt_y"],
                                         torch.zeros((ps.K,) + g["target"].shape, device="cuda"), g["target"]).bands
        g["s2_ref"] = synthetic.s2_reference_torch(torch.nan_to_num(x), seed=seed + 100)
        out.append(g)
    return out


@pytest.mark.parametrize("stretch", [None, (2, 98)])
def test_sharded_with_s2_targets(stretch):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda", stretch=stretch,
                         stretch_scope="fit" if stretch else "granule")
    grans = _granules(ps, w, good)
    res = ps.synthesize_sharded(grans)
    torch.cuda.synchronize()
    single = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda")
    xs, ys = [], []
    for g, r in zip(grans, res):
        assert r.grid is g.get("target")
        if "target" in g:
            one = single.synthesize_on_s2_grid(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"], g["target"])
            assert r.bands.shape == (ps.K,) + g["target"].shape
        else:
            one = single.synthesize(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"])
        assert torch.equal(bits(r.bands), bits(one.bands)) and torch.equal(r.fit_mask, one.fit_mask)
        m = host(one.fit_mask).reshape(-1)
        xs.append(host(one.bands).reshape(ps.K, -1)[:, m])
        ys.append(host(g["s2_ref"]).reshape(ps.K, -1)[:, m])
    xcat, ycat = np.concatenate(xs, axis=1), np.concatenate(ys, axis=1)
    assert xcat.shape[1] > 1000
    if stretch is None:
        want = opoly.polyfit_paired(xcat, ycat, np.ones(xcat.shape[1], bool), 2, min_count=200)
        err = float(np.max(np.abs(host(res[0].coeffs) - want).max(1) / np.abs(want).max(1)))
        assert err < 1e-4, f"global coefficients off by {err:.2e}"
    else:
        for k in range(ps.K):
            assert np.array_equal(host(res[0].x_limits)[k, 0].view(np.int64),
                                  np.percentile(xcat[k], stretch).view(np.int64))
            assert np.array_equal(host(res[0].y_limits)[k, 0].view(np.int64),
                                  np.percentile(ycat[k], stretch).view(np.int64))
    for r in res[1:]:
        assert torch.equal(r.coeffs, res[0].coeffs)


# ---------------------------------------------------------------------------------------------- errors
def test_slab_errors():
    w, good, raw, gx, gy, target = _small()
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda")
    Hd, Wd = target.shape
    rawd, gxd, gyd = dev(raw), dev(gx), dev(gy)
    s2 = torch.zeros((ps.K, 5, Wd), device="cuda")
    for rows in ((5, 5), (-1, 4), (Hd - 2, Hd + 3), (6, 1)):
        with pytest.raises(ValueError, match="rows"):
            ps.synthesize_slab_on_s2_grid(rawd, gxd, gyd, s2, target, rows)
    with pytest.raises(ValueError, match="rows"):
        target.coords(rows=(0, Hd + 1))
    with pytest.raises(ValueError, match="s2_ref"):
        ps.synthesize_slab_on_s2_grid(rawd, gxd, gyd, s2, target, (0, 6))
    with pytest.raises(ValueError, match="s2_ref"):
        ps.synthesize_sharded([{"raw": rawd, "glt_x": gxd, "glt_y": gyd, "s2_ref": s2, "target": target}])
    with pytest.raises(_lib.HsrError):
        kernels.warp_planes(torch.rand((2, 4, gx.shape[1]), device="cuda"),
                            torch.ones((4, gx.shape[1]), dtype=torch.bool, device="cuda"), target.coords(),
                            target.scales, kernel="cubic", fill_out=torch.zeros(2, device="cuda"), src_row0=gx.shape[0] - 2,
                            src_rows_total=gx.shape[0])
    # a global fit with per-granule stretch limits
    psg = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device="cuda", stretch=(2, 98))
    two = types.SimpleNamespace(world=2)
    s2f = torch.zeros((ps.K, Hd, Wd), device="cuda")
    with pytest.raises(ValueError, match="global fit"):
        psg.synthesize_on_s2_grid(rawd, gxd, gyd, s2f, target, exchange=two)
    with pytest.raises(ValueError, match="global fit"):
        psg.synthesize_slab_on_s2_grid(rawd, gxd, gyd, s2f[:, :5].contiguous(), target, (0, 5), exchange=two)
    with pytest.raises(ValueError, match="global fit"):
        psg.synthesize_sharded([{"raw": rawd, "glt_x": gxd, "glt_y": gyd, "s2_ref": s2f, "target": target}])

