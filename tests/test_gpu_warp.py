"""GPU parity of the general grid warp (``hsr_warp_f32`` / ``hsr_warp_coords_f64``; SURVEY 8f row 4: the gdalwarp
step of nc_to_envi, EMIT_data/emit_proj.py:876-940) against oracle/warp.py on small seeded cases, plus
size-independent properties at granule size.  Bars: source coordinates 1e-8 px (fp64 on both sides); resampled
values 1e-5 relative + 1e-6 absolute (fp32 accumulation of <= 64 fp32-weighted taps against the oracle's fp64);
nodata / NaN patterns identical.  Parity with GDAL / PROJ themselves is unpinned (oracle/warp.py header)."""
import ctypes

import numpy as np
import pytest
import torch

from hsr_b200 import kernels
from hsr_b200.EMIT_data import warp as hwarp
from oracle import warp as owarp

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
ND = -9999.0


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_warp_close(got, want):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern differs"
    assert np.array_equal(got == ND, want == ND), "nodata pattern differs"
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf]), "Inf pattern differs"
    ok = ~np.isnan(want) & ~inf
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    assert np.all(err <= RTOL * np.abs(want[ok]) + ATOL), f"max abs err {err.max():.3e}"


def emit_like_case(Hs=36, Ws=40, seed=0):
    """A small WGS-84 grid near 34 N / 118 W (UTM 11) and the snapped 60 m grid nc_to_envi would warp it onto."""
    src_gt = (-118.30, 0.000542232520256367, 0.0, 34.20, 0.0, -0.000542232520256367)
    s2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)
    dst_gt, shape, rec = hwarp.target_grid(src_gt, (Hs, Ws), s2)
    return src_gt, s2, dst_gt, shape


def test_coords_match_oracle_transformer():
    src_gt, s2, dst_gt, (Hd, Wd) = emit_like_case()
    got = kernels.warp_coords(src_gt, dst_gt, (Hd, Wd), utm_zone=11).cpu().numpy()
    for r in range(0, Hd, 5):
        for c in range(0, Wd, 3):
            ox, oy = owarp.dst_to_src(c, r, dst_gt, src_gt, 11, False, True)
            assert abs(got[r, c, 0] - ox) < 1e-8 and abs(got[r, c, 1] - oy) < 1e-8
    # southern hemisphere zone, and the affine-only mode
    sgt = (18.40, 0.0006, 0.0, -33.90, 0.0, -0.0006)
    dgt = (260000.0, 60.0, 0.0, 6250000.0, 0.0, -60.0)
    got = kernels.warp_coords(sgt, dgt, (7, 9), utm_zone=34, south=True).cpu().numpy()
    for r in range(7):
        for c in range(9):
            ox, oy = owarp.dst_to_src(c, r, dgt, sgt, 34, True, True)
            assert abs(got[r, c, 0] - ox) < 1e-8 and abs(got[r, c, 1] - oy) < 1e-8
    a = (100.0, 2.0, 0.1, 50.0, -0.2, -2.0)
    b = (101.0, 3.0, 0.0, 49.0, 0.0, -3.0)
    got = kernels.warp_coords(a, b, (5, 6)).cpu().numpy()
    for r in range(5):
        for c in range(6):
            ox, oy = owarp.dst_to_src(c, r, b, a, 0, False, False)
            assert abs(got[r, c, 0] - ox) < 1e-10 and abs(got[r, c, 1] - oy) < 1e-10


@pytest.mark.parametrize("bands,padded", [(285, True), (285, False), (37, False), (3, False), (8, True)])
def test_utm_cubic_warp_vs_oracle_with_coordinate_workspace(bands, padded):
    """The nc_to_envi geometry (lon / lat -> UTM 60 m, x-scale ~0.83 so the cubic filter is widened to 6 taps), with
    GLT-style fill pixels (every band nodata), band-specific nodata, NaN and Inf samples; vector and scalar paths."""
    rng = np.random.default_rng(bands)
    Hs, Ws = 36, 40
    src_gt, s2, dst_gt, (Hd, Wd) = emit_like_case(Hs, Ws)
    src = (0.05 + 0.9 * rng.random((Hs, Ws, bands))).astype(np.float32)
    yy, xx = np.mgrid[0:Hs, 0:Ws]
    src[(yy + 2 * xx) < 30] = ND                                   # a slanted fill region, like outside the swath
    src[rng.random((Hs, Ws)) < 0.03] = ND                          # GLT holes
    spots = rng.random((Hs, Ws, bands)) < 0.002
    src[spots] = ND                                                # band-specific nodata
    src[20, 20, bands // 2] = np.nan
    src[25, 10, 0] = np.inf
    scales = hwarp.warp_scales(dst_gt, src_gt, (Hd, Wd), 11, False)
    want = owarp.warp(src, src_gt, dst_gt, Hd, Wd, zone=11, utm=True, nodata=ND, scales=scales)
    if padded:
        P = kernels.padded_bands(bands)
        buf = torch.full((Hs, Ws, P), 7.0, dtype=torch.float32, device="cuda")
        buf[:, :, :bands] = dev(src)
        s = buf[:, :, :bands]
    else:
        s = dev(src)
    got = kernels.warp(s, src_gt, dst_gt, (Hd, Wd), utm_zone=11, scales=scales, nodata=ND)
    if not padded:                                                 # force the scalar path on the output side too
        out = torch.empty((Hd, Wd, bands), dtype=torch.float32, device="cuda")
        got = kernels.warp(s, src_gt, dst_gt, (Hd, Wd), utm_zone=11, scales=scales, nodata=ND, out=out)
    assert_warp_close(got, want)
    assert (want == ND).any() and (want != ND).any() and np.isnan(want).any()


def test_same_crs_bilinear_and_downsampling_vs_oracle():
    rng = np.random.default_rng(5)
    src = rng.random((30, 34, 12)).astype(np.float32)
    src[rng.random((30, 34)) < 0.05] = ND
    sgt = (500000.0, 10.0, 0.0, 4000000.0, 0.0, -10.0)
    for kernel, dgt, shape in (("bilinear", (500012.0, 4.0, 0.0, 3999991.0, 0.0, -4.0), (60, 70)),     # finer, shifted
                               ("cubic", (499990.0, 25.0, 0.0, 4000020.0, 0.0, -35.0), (10, 15)),      # coarser: wide filter
                               ("cubic", (500003.0, 10.0, 0.7, 3999998.0, -0.4, -10.0), (28, 30)),     # slight rotation
                               # 45 degrees and a 3.4x reduction: tap boxes too large to stage -> taps read from global memory
                               ("cubic", (500150.0, 7.0, 7.0, 4000000.0, 7.0, -7.0), (24, 20)),
                               ("cubic", (500000.0, 34.0, 0.0, 4000000.0, 0.0, -34.0), (8, 10)),
                               ("bilinear", (500000.0, 34.0, 0.0, 4000000.0, 0.0, -34.0), (8, 10))):
        scales = hwarp.warp_scales(dgt, sgt, shape)
        want = owarp.warp(src, sgt, dgt, shape[0], shape[1], utm=False, nodata=ND, kernel=kernel, scales=scales)
        got = hwarp.warp_to_grid(src, sgt, dgt, shape, kernel=kernel, nodata=ND, scales=scales)       # numpy in -> numpy out
        assert isinstance(got, np.ndarray)
        assert_warp_close(got, want)
    # filters wider than the quad and lane kernels hold (the exact pass): x scale 0.4 (cubic, radii 5 x 2) and a 6x
    # bilinear reduction (radius 6), on padded records (vector path) and on dense ones with a dense output (scalar path)
    sub = src[..., :11]
    for kernel, dgt, shape in (("cubic", (500003.0, 25.0, 0.0, 3999998.0, 0.0, -10.0), (28, 13)),
                               ("bilinear", (500007.0, 60.0, 0.0, 3999996.0, 0.0, -60.0), (5, 6))):
        scales = hwarp.warp_scales(dgt, sgt, shape)
        want = owarp.warp(sub, sgt, dgt, shape[0], shape[1], utm=False, nodata=ND, kernel=kernel, scales=scales)
        buf = torch.full((30, 34, kernels.padded_bands(11)), 7.0, dtype=torch.float32, device="cuda")
        buf[..., :11] = dev(sub)
        dense_out = torch.empty((shape[0], shape[1], 11), dtype=torch.float32, device="cuda")
        for s, out in ((buf[..., :11], None), (dev(sub), dense_out)):
            assert_warp_close(kernels.warp(s, sgt, dgt, shape, scales=scales, kernel=kernel, nodata=ND, out=out), want)
    # no nodata value given: every tap counts, the destination outside the source is 0
    want = owarp.warp(src, sgt, (499900.0, 10.0, 0.0, 4000000.0, 0.0, -10.0), 8, 20, utm=False, nodata=None)
    got = hwarp.warp_to_grid(src, sgt, (499900.0, 10.0, 0.0, 4000000.0, 0.0, -10.0), (8, 20), nodata=None)
    assert np.allclose(got, want, rtol=RTOL, atol=ATOL) and (got[:, :10] == 0).all()


@pytest.mark.parametrize("bands", [3, 20, 285])
def test_nearest_and_average_vs_oracle(bands):
    """kernel = "nearest" / "average" (rasterio.warp.reproject in s2_data/s2_utils.py:546-574 and the notebook's
    downsample_s2_to_grid on grids that are not snapped): lon / lat -> UTM and same-CRS geometries (finer, coarser,
    rotated, partly outside the source), nodata per band, NaN as an ordinary value.  Nearest copies samples: bit-exact.
    Average: fp64 sums on both sides, 1e-5 relative."""
    rng = np.random.default_rng(100 + bands)
    Hs, Ws = 30, 34
    src = (0.05 + 0.9 * rng.random((Hs, Ws, bands))).astype(np.float32)
    src[rng.random((Hs, Ws)) < 0.05] = ND
    src[rng.random((Hs, Ws, bands)) < 0.01] = ND
    src[11, 13, bands // 2] = np.nan
    sgt = (500000.0, 10.0, 0.0, 4000000.0, 0.0, -10.0)
    cases = [((500012.0, 4.0, 0.0, 3999991.0, 0.0, -4.0), (40, 50), 0),            # finer, shifted
             ((499990.0, 25.0, 0.0, 4000020.0, 0.0, -35.0), (10, 15), 0),          # coarser, sticks out of the source
             ((500003.0, 10.0, 0.7, 3999998.0, -0.4, -10.0), (28, 30), 0),         # slight rotation
             ((500000.0, 60.0, 0.0, 4000000.0, 0.0, -60.0), (5, 5), 0)]            # snapped 6 x 6 blocks
    usrc_gt, s2, udst_gt, ushape = emit_like_case(Hs, Ws)
    cases.append((udst_gt, ushape, 11))
    for dgt, shape, zone in cases:
        g = usrc_gt if zone else sgt
        for kernel in ("nearest", "average"):
            want = owarp.warp(src, g, dgt, shape[0], shape[1], zone=zone, utm=bool(zone), nodata=ND, kernel=kernel)
            got = kernels.warp(dev(src), g, dgt, shape, utm_zone=zone, nodata=ND, kernel=kernel)
            if kernel == "nearest":
                assert np.array_equal(got.cpu().numpy().view(np.int32), want.view(np.int32)), (dgt, kernel)
            else:
                assert_warp_close(got, want)
            assert (want != ND).any() and (kernel == "average" or (want == ND).any())
    # average on the snapped grid = the block mean of the aligned kernel (what the reference's geometry degenerates to)
    from oracle import resample as oresample
    clean = (0.05 + 0.9 * rng.random((Hs, 36, 4))).astype(np.float32)
    got = kernels.warp(dev(clean), sgt, (500000.0, 60.0, 0.0, 4000000.0, 0.0, -60.0), (5, 6), kernel="average").cpu().numpy()
    want = oresample.downsample_to_grid(np.transpose(clean, (2, 0, 1)), 6)
    assert np.allclose(np.transpose(got, (2, 0, 1)), want, rtol=1e-6, atol=1e-7)
    with pytest.raises(ValueError):
        kernels.warp(dev(clean), sgt, sgt, (5, 6), kernel="lanczos")


def test_warp_to_s2_grid_plane_and_errors():
    src_gt, s2, dst_gt, (Hd, Wd) = emit_like_case()
    rng = np.random.default_rng(2)
    plane = rng.random((36, 40)).astype(np.float32)                 # a LOC / OBS style plane
    out, gt2, rec = hwarp.warp_to_s2_grid(plane, src_gt, s2)
    assert out.shape == (Hd, Wd) and gt2 == pytest.approx(dst_gt) and rec["cols"] == Wd
    want = owarp.warp(plane[..., None], src_gt, dst_gt, Hd, Wd, zone=11, utm=True, nodata=ND,
                      scales=hwarp.warp_scales(dst_gt, src_gt, (Hd, Wd), 11, False))[..., 0]
    assert_warp_close(out, want)
    with pytest.raises(TypeError):
        kernels.warp(torch.zeros(4, 4, 3), src_gt, dst_gt, (2, 2))                     # CPU tensor: no CPU path
    with pytest.raises(ValueError):
        kernels.warp(torch.zeros(4, 4, 3, device="cuda"), src_gt, dst_gt, (2, 2), kernel="lanczos")
    from hsr_b200 import _lib
    with pytest.raises(_lib.HsrError):                                                   # scale needs > 16 taps
        kernels.warp(torch.zeros(4, 4, 3, device="cuda"), src_gt, dst_gt, (2, 2), scales=(0.1, 1.0))
    with pytest.raises(_lib.HsrError):                                                   # singular geotransform
        kernels.warp(torch.zeros(4, 4, 3, device="cuda"), (0, 0, 0, 0, 0, 0), dst_gt, (2, 2))
    s, d = torch.zeros(4, 4, 3, device="cuda"), torch.empty(2, 2, 3, device="cuda")
    geo = kernels._warp_geo(src_gt, dst_gt, 11, False, None)
    with pytest.raises(_lib.HsrError, match="workspace") as err:                          # cubic needs the coordinate workspace
        _lib.check(_lib.lib().hsr_warp_f32(s.data_ptr(), 4, 4, 3, 3, ctypes.addressof(geo), 2, 1, ND, ND, 2, 2,
                                           d.data_ptr(), 3, None, 0, None))
    assert err.value.code == -1                                                          # HSR_EINVAL


def test_full_granule_warp_properties():
    """Granule-sized (1685 x 1667 x 285, 3.2 GB) properties: (1) the same grid gives back the cube bit for bit;
    (2) a constant cube stays constant wherever the destination is covered, nodata elsewhere, with the covered
    footprint equal to the transformer's own; (3) fill pixels never leak: min over valid outputs >= min of inputs
    minus the cubic overshoot bound."""
    from hsr_b200 import synthetic
    Hr, Wr, B = 1280, 1242, 285
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, "cuda")
    gx, gy = (dev(a) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    P = kernels.padded_bands(B)
    buf = torch.empty((gx.shape[0], gx.shape[1], P), dtype=torch.float32, device="cuda")
    _, valid, _ = kernels.glt_ortho(raw, gx, gy, out=buf, out_pix_stride=P)
    del raw
    Ho, Wo = valid.shape
    ortho = buf[:, :, :B]
    src_gt = (-118.60, 0.000542232520256367, 0.0, 34.90, 0.0, -0.000542232520256367)
    pow2_gt = (1000.0, 0.5, 0.0, 2000.0, 0.0, -0.5)          # exactly representable: pixel centres map onto themselves
    same = kernels.warp(ortho, pow2_gt, pow2_gt, (Ho, Wo), nodata=ND)
    assert torch.equal(same.view(torch.int32), ortho.view(torch.int32))
    del same
    s2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
    dst_gt, (Hd, Wd), _ = hwarp.target_grid(src_gt, (Ho, Wo), s2)
    scales = hwarp.warp_scales(dst_gt, src_gt, (Hd, Wd), 11, False)
    out = kernels.warp(ortho, src_gt, dst_gt, (Hd, Wd), utm_zone=11, scales=scales, nodata=ND)
    covered = out[..., 0] != ND
    assert 0.3 < covered.float().mean().item() < 0.7
    lo, hi = ortho[valid].min().item(), ortho[valid].max().item()
    # away from the swath edge (9 x 9 covered neighbourhood: every tap valid) cubic overshoot is bounded; AT the edge the
    # renormalised partial sums of GDAL's rule may ring arbitrarily (weight sums just above 1e-6) - not asserted
    interior = torch.nn.functional.max_pool2d((~covered).float()[None, None], 9, 1, 4)[0, 0] == 0
    assert 0.25 < interior.float().mean().item()
    vals = out[interior]
    assert vals.min().item() >= lo - 0.5 * (hi - lo) and vals.max().item() <= hi + 0.5 * (hi - lo)
    assert torch.equal(covered, out[..., B - 1] != ND)                   # fill pixels are fill in every band
    ortho[valid] = 0.25                                                   # constant wherever there is data
    out2 = kernels.warp(ortho, src_gt, dst_gt, (Hd, Wd), utm_zone=11, scales=scales, nodata=ND)
    assert torch.equal(out2[..., 0] != ND, covered)
    assert (out2[covered] - 0.25).abs().max().item() < 1e-6


def test_notebook_resampling_names_on_grids():
    """downsample_s2_to_grid / reproject_stack_to_grid (Pairs_EMIT_S2_demo-2.ipynb cell 73) with grid descriptions instead
    of raster paths: snapped grids take the aligned kernels (bit-identical to them), shifted grids the general warp."""
    from hsr_b200.s2_emit import resample
    from oracle import resample as oresample
    rng = np.random.default_rng(3)
    s2 = rng.integers(0, 255, size=(4, 36, 48)).astype(np.uint8)
    fine = dict(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=48, height=36)
    coarse = dict(epsg=32611, x0=300000.0, y0=3900000.0, dx=60.0, dy=60.0, width=8, height=6)
    got = resample.downsample_s2_to_grid(s2, fine, coarse, band_indexes=[3, 2, 1], src_scale=1.0 / 255.0)
    want = oresample.downsample_to_grid(s2[[2, 1, 0]], 6, src_scale=1.0 / 255.0)
    assert got.shape == (3, 6, 8) and np.array_equal(got.view(np.int32), want.view(np.int32))
    planes = rng.random((3, 6, 8)).astype(np.float32)
    up = resample.reproject_stack_to_grid(planes, coarse, fine, "bilinear")
    assert up.shape == (3, 36, 48) and np.allclose(up, oresample.upsample_to_grid(planes, 6), rtol=0, atol=1e-6)
    # a grid shifted by a third of a pixel: the general kernel, checked against the warp oracle
    shifted = dict(fine, x0=300003.0, y0=3899996.0, width=40, height=30)
    got = resample.reproject_stack_to_grid(planes, coarse, shifted, "bilinear")
    gt = lambda g: (g["x0"], g["dx"], 0.0, g["y0"], 0.0, -g["dy"])            # noqa: E731
    scales = hwarp.warp_scales(gt(shifted), gt(coarse), (30, 40))
    want = owarp.warp(np.transpose(planes, (1, 2, 0)), gt(coarse), gt(shifted), 30, 40, utm=False, nodata=None,
                      kernel="bilinear", scales=scales)
    assert got.shape == (3, 30, 40) and np.allclose(got, np.transpose(want, (2, 0, 1)), rtol=RTOL, atol=ATOL)
    # 'average' on a non-snapped geometry: the general kernel (round 1 refused it)
    coarse_shifted = dict(coarse, x0=300007.0, y0=3899990.0, dx=50.0, dy=50.0, width=8, height=6)
    got = resample.downsample_s2_to_grid(s2, fine, coarse_shifted, band_indexes=[1, 4], src_scale=1.0 / 255.0)
    want = owarp.warp(np.transpose(s2[[0, 3]].astype(np.float32), (1, 2, 0)), gt(fine), gt(coarse_shifted), 6, 8, utm=False,
                      nodata=None, kernel="average")
    assert got.shape == (2, 6, 8) and np.allclose(got, np.transpose(want, (2, 0, 1)) / 255.0, rtol=RTOL, atol=ATOL)
    near = resample.reproject_stack_to_grid(planes, coarse, shifted, "nearest")
    want = owarp.warp(np.transpose(planes, (1, 2, 0)), gt(coarse), gt(shifted), 30, 40, utm=False, nodata=None, kernel="nearest")
    assert np.array_equal(near, np.transpose(want, (2, 0, 1)))
    with pytest.raises(NotImplementedError):
        resample.reproject_stack_to_grid(planes, coarse, dict(fine, epsg=32612))
