"""The pair on the Sentinel-2 grid on the GPU: hsr_warp_planes_f32 / kernels.warp_planes against the fp64 plane warp
of tests/s2_grid_oracle.py, PairSynthesizer.synthesize_on_s2_grid against the reference's order on the oracles
(glt -> warp of every band -> srf -> polyfit / apply) and, at granule size, against the chained GPU path
(glt_ortho -> warp -> srf_integrate -> fit / apply); the argument errors."""
import ctypes

import numpy as np
import pytest
import torch

from hsr_b200 import _lib, kernels, synthetic
from hsr_b200.EMIT_data import warp as hwarp
from hsr_b200.pipeline import PairSynthesizer, S2Target, s2_target
from hsr_b200.s2_emit.srf import synthetic_s2_srf
from oracle import color as ocolor
from oracle import glt as oglt
from oracle import poly as opoly

import s2_grid_oracle as sgo

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

ND = sgo.ND
COEF_RTOL = 1e-4
APPLY_ATOL = 1e-4
GLT_GT = (-118.30, 0.000542232520256367, 0.0, 34.20, 0.0, -0.000542232520256367)
S2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def coeff_err(got, ref):
    return float(np.max(np.abs(host(got) - ref).max(axis=-1) / np.abs(ref).max(axis=-1)))


def assert_planes(got, want, cov, C, fill_out):
    """The exactness bar: |got - want| <= 1e-5 C + 1e-7, identical NaN / +-Inf patterns, fill_out where uncovered."""
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern differs"
    assert np.array_equal(np.isposinf(got), np.isposinf(want)), "+Inf pattern differs"
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), "-Inf pattern differs"
    fin = np.isfinite(want) & cov[None]
    err = np.abs(got[fin].astype(np.float64) - want[fin])
    assert np.all(err <= 1e-5 * C[fin] + 1e-7), f"max err {err.max():.3e}"
    assert np.array_equal(got[:, ~cov], np.broadcast_to(np.asarray(fill_out, np.float32)[:, None], got[:, ~cov].shape))


# ---------------------------------------------------------------------------------------------- the kernel
@pytest.mark.parametrize("kernel", ["cubic", "bilinear"])
@pytest.mark.parametrize("padded", [True, False])
@pytest.mark.parametrize("K", [1, 3, 12, 13])
def test_warp_planes_vs_oracle(K, padded, kernel):
    rng = np.random.default_rng(K * 4 + padded * 2 + (kernel == "cubic"))
    Hs, Ws = 36, 40
    t = hwarp.s2_target(GLT_GT, (Hs, Ws), S2, kernel=kernel)
    Hd, Wd = t.shape
    valid = np.ones((Hs, Ws), bool)
    yy, xx = np.mgrid[0:Hs, 0:Ws]
    valid[(yy + 2 * xx) < 30] = False                            # a slanted fill region, like outside the swath
    valid[rng.random((Hs, Ws)) < 0.03] = False                   # GLT holes
    valid[20, 20] = valid[25, 12] = valid[12, 30] = True         # the non-finite samples below are GLT-valid
    fill_out = (-9999.0 * (0.5 + rng.random(K))).astype(np.float32)
    planes = (0.05 + 0.9 * rng.random((K, Hs, Ws))).astype(np.float32)
    planes[:, ~valid] = fill_out[:, None]                        # what glt_srf writes at GLT-invalid pixels
    planes[K - 1, 20, 20] = np.nan
    planes[0, 25, 12] = np.inf
    planes[K // 2, 12, 30] = -np.inf
    planes[:, 4, 35] = np.nan                                    # NaN under a skipped (invalid) tap: no effect
    valid[4, 35] = False
    want, cov, C = sgo.warp_conditioned(planes.transpose(1, 2, 0), GLT_GT, t.dst_gt, Hd, Wd, scales=t.scales,
                                        zone=11, kernel=kernel, src_valid=valid)
    want, cov, C = want.transpose(2, 0, 1), cov[..., 0], C.transpose(2, 0, 1)
    want[:, ~cov] = fill_out[:, None]
    if padded:
        src = kernels.alloc_planes(K, (Hs, Ws), "cuda")
        src.copy_(dev(planes))
        out = None
    else:
        src = dev(planes)
        out = torch.empty((K, Hd, Wd), dtype=torch.float32, device="cuda")
    gate_k, gate_gt = K - 1, 0.3
    got, dvalid, fm = kernels.warp_planes(src, dev(valid), t.coords(), t.scales, kernel=kernel, fill_out=dev(fill_out),
                                          gate_k=gate_k, gate_gt=gate_gt, out=out)
    if out is not None:
        assert got.data_ptr() == out.data_ptr()
    g = host(got)
    assert np.array_equal(host(dvalid), cov) and 0 < cov.sum() < cov.size
    assert_planes(g, want, cov, C, fill_out)
    assert np.isnan(want).any() and np.isinf(want).any()
    want32 = want.astype(np.float32)
    assert np.array_equal(host(fm), opoly.fit_mask(want32, cov, gate_k=gate_k, gate_gt=gate_gt))


# ---------------------------------------------------------------------------------------------- the pipeline, small
def _small_case(seed=0, Hr=40, Wr=34):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=good)
    raw[11, 9, 40] = np.nan
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=seed + 1, hole_frac=0.01, n_oob=4, n_neg=4)
    return w, good, raw, gx, gy


@pytest.mark.parametrize("mode", ["plain", "stretch", "y_finite"])
def test_synthesize_on_s2_grid_vs_oracle_chain(mode):
    w, good, raw, gx, gy = _small_case(seed=5)
    table = synthetic_s2_srf()
    kw = {"stretch": (2, 98)} if mode == "stretch" else ({"y_finite": True} if mode == "y_finite" else {})
    ps = PairSynthesizer(w, table, good, deg=2, device="cuda", **kw)
    target = s2_target(GLT_GT, gx.shape, S2)
    want, cov, ortho, valid = sgo.reference_chain(raw, gx, gy, GLT_GT, target, w, table, good, ps.band_names)
    planes = sgo.srf_planes(ortho, w, table, good, ps.band_names)
    _, _, C = sgo.warp_conditioned(planes.transpose(1, 2, 0), GLT_GT, target.dst_gt, *target.shape,
                                   scales=target.scales, zone=11, src_valid=valid)
    C = C.transpose(2, 0, 1)
    s2 = synthetic.s2_reference_np(np.nan_to_num(want, posinf=0.0, neginf=0.0).astype(np.float32), seed=2)
    fm0 = opoly.fit_mask(want.astype(np.float32), cov, gate_k=0, gate_gt=0.0)
    if mode == "y_finite":
        iy, ix = np.argwhere(fm0)[len(np.argwhere(fm0)) // 2]
        s2[3, iy, ix] = np.nan                                     # a non-finite reference pixel inside the fit mask
    res = ps.synthesize_on_s2_grid(dev(raw), dev(gx), dev(gy), dev(s2), target)
    assert res.grid is target and res.bands.shape == (ps.K,) + target.shape
    b = host(res.bands)
    assert np.array_equal(host(res.valid), cov)
    assert_planes(b, want, cov, C, host(ps.fill_out))
    _, _, diag = oglt.glt_ortho(raw, gx, gy)
    assert host(res.diag).tolist() == [diag["valid_glt_count"], diag["valid_glt_inbounds_count"],
                                       diag["valid_glt_dropped_oob"]]
    fm = opoly.fit_mask(b, cov, gate_k=0, gate_gt=0.0)
    if mode == "y_finite":
        fm &= np.isfinite(s2).all(0)
        assert fm.sum() < fm0.sum()
    assert np.array_equal(host(res.fit_mask), fm) and fm.sum() > 200
    if mode == "stretch":
        xi, yi = np.moveaxis(b, 0, -1), np.moveaxis(s2, 0, -1)     # limits are exact functions of the planes produced
        assert np.array_equal(host(res.x_limits).reshape(-1, 2), ocolor.shared_percentile_limits(xi, fm))
        assert np.array_equal(host(res.y_limits).reshape(-1, 2), ocolor.shared_percentile_limits(yi, fm))
        xn = ocolor.apply_shared_percentile_stretch(xi, fm)
        yn = ocolor.apply_shared_percentile_stretch(yi, fm)
        coeffs = opoly.fit_poly_rgb_paired(xn, yn, fm, 2)
        assert coeff_err(res.coeffs, coeffs) < COEF_RTOL
        wm = opoly.apply_poly_rgb(xn, coeffs, fm)
        gm = np.moveaxis(host(res.matched), 0, -1)
    else:
        xw = np.where(cov[None], want, b).astype(np.float32)      # the oracle chain's planes, fill_out where uncovered
        coeffs = opoly.polyfit_paired(xw, s2, fm, 2, min_count=200)
        assert coeff_err(res.coeffs, coeffs) < COEF_RTOL
        wm = opoly.apply_poly_planes(xw, coeffs, fm)
        gm = host(res.matched)
    ok = np.isfinite(wm)
    assert np.array_equal(np.isnan(gm), np.isnan(wm)) and np.max(np.abs(gm - wm)[ok]) <= APPLY_ATOL


# ---------------------------------------------------------------------------------------------- granule size
def test_granule_s2_grid_vs_chained_gpu_path():
    """Raw 1280 x 1242 x 285, 25 degree GLT, the zone 11 geometry of profiles/prof_warp.py: the plane path against
    glt_ortho -> warp (285 bands) -> srf_integrate -> the same fit / apply; two runs bit-identical."""
    Hr, Wr, B = 1280, 1242, 285
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, "cuda", good=good)
    gx, gy = (dev(a) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    src_gt = (-118.60, 0.000542232520256367, 0.0, 34.90, 0.0, -0.000542232520256367)
    s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
    target = s2_target(src_gt, gx.shape, s2g)
    assert target.shape == (1215, 959) and target.scales[0] < 1.0
    ps = PairSynthesizer(w, table, good, deg=2, device="cuda")
    # the chained path
    P = kernels.padded_bands(B)
    buf = torch.empty((gx.shape[0], gx.shape[1], P), dtype=torch.float32, device="cuda")
    _, valid_o, _ = kernels.glt_ortho(raw, gx, gy, out=buf, out_pix_stride=P)
    warped = kernels.warp(buf[:, :, :B], src_gt, target.dst_gt, target.shape, utm_zone=11, scales=target.scales,
                          nodata=ND)
    del buf
    cov_c = warped[..., 0] != ND
    fm_c = torch.empty(target.shape, dtype=torch.bool, device="cuda")
    bands_c = kernels.srf_integrate(warped, ps.W, fit_mask_out=fm_c, gate_k=0, gate_gt=0.0)
    del warped
    fm_c &= cov_c
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(bands_c), seed=1)
    res = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    res2 = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    torch.cuda.synchronize()
    for a, b2 in ((res.bands, res2.bands), (res.matched, res2.matched), (res.coeffs, res2.coeffs),
                  (res.fit_mask, res2.fit_mask), (res.valid, res2.valid)):
        assert torch.equal(a.contiguous().view(torch.uint8), b2.contiguous().view(torch.uint8))
    assert torch.equal(res.valid, cov_c)
    assert 0.3 < cov_c.float().mean().item() < 0.7
    interior = torch.nn.functional.max_pool2d((~cov_c).float()[None, None], 9, 1, 4)[0, 0] == 0
    assert 0.25 < interior.float().mean().item()
    bn, bc = res.bands[:, interior].double(), bands_c[:, interior].double()
    assert ((bn - bc).abs() <= 1e-5 * bc.abs() + 1e-7).all(), f"max err {(bn - bc).abs().max().item():.3e}"
    assert torch.equal(res.fit_mask[interior], fm_c[interior])
    # the same fit / apply on the chained planes
    for stretch in (None, (2, 98)):
        psx = PairSynthesizer(w, table, good, deg=2, device="cuda", stretch=stretch)
        mom, fm, xl, _ = psx.fit(bands_c, s2, cov_c, fm_c)
        coeffs_c, _ = kernels.poly_solve_apply(bands_c, mom, fm, 2, min_count=200, x_stretch=xl)
        r = res if stretch is None else psx.synthesize_on_s2_grid(raw, gx, gy, s2, target)
        assert coeff_err(r.coeffs, host(coeffs_c).reshape(ps.K, 3)) < COEF_RTOL


# ---------------------------------------------------------------------------------------------- errors
def test_s2_grid_errors():
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    ps = PairSynthesizer(w, table, good, deg=2, device="cuda")
    _, _, raw, gx, gy = _small_case()
    target = s2_target(GLT_GT, gx.shape, S2)
    assert isinstance(target, S2Target)
    Hd, Wd = target.shape
    K = ps.K
    planes = torch.rand((K, 20, 24), device="cuda")
    sv = torch.ones((20, 24), dtype=torch.bool, device="cuda")
    co = target.coords()
    assert target.coords() is co                                  # cached per device
    fo = ps.fill_out
    with pytest.raises(TypeError):
        kernels.warp_planes(planes.cpu(), sv, co, target.scales, kernel="cubic", fill_out=fo)
    with pytest.raises(TypeError):
        ps.synthesize_on_s2_grid(torch.from_numpy(raw), dev(gx), dev(gy), torch.zeros((K, Hd, Wd), device="cuda"),
                                 target)
    for k in ("nearest", "average", "lanczos"):
        with pytest.raises(ValueError):
            kernels.warp_planes(planes, sv, co, target.scales, kernel=k, fill_out=fo)
        with pytest.raises(ValueError):
            s2_target(GLT_GT, gx.shape, S2, kernel=k)
    with pytest.raises(ValueError, match="s2_ref"):
        ps.synthesize_on_s2_grid(dev(raw), dev(gx), dev(gy), torch.zeros((K, Hd + 1, Wd), device="cuda"), target)
    p17 = torch.rand((17, 20, 24), device="cuda")
    with pytest.raises(_lib.HsrError) as e:
        kernels.warp_planes(p17, sv, co, target.scales, kernel="cubic", fill_out=torch.zeros(17, device="cuda"))
    assert e.value.code == -1
    with pytest.raises(_lib.HsrError) as e:
        kernels.warp_planes(planes, sv, co, (0.2, 1.0), kernel="cubic", fill_out=fo)
    assert e.value.code == -1
    geo = _lib.WarpGeo()
    geo.xscale, geo.yscale = target.scales
    out = torch.empty((K, Hd, Wd), device="cuda")
    rc = _lib.lib().hsr_warp_planes_f32(planes.data_ptr(), 20, 24, K, 20 * 24, sv.data_ptr(), None,
                                        ctypes.addressof(geo), 2, fo.data_ptr(), 0, 0.0, Hd, Wd, out.data_ptr(), Hd * Wd,
                                        None, None, None)
    assert rc == -1
    torch.cuda.synchronize()
