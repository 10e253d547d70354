"""CPU model of the pair on the Sentinel-2 grid (PairSynthesizer.synthesize_on_s2_grid): warping the K pseudo-S2
planes of the GLT-valid pixels equals warping the 285-band ortho cube and integrating the SRF over the result.

Both steps are linear and the warp's tap weights are the same for every band wherever a source pixel is all data or
all nodata (the GLT fill), so SRF(warp(cube)) = warp(SRF(cube)) with validity per pixel.  Checked here on the oracles
(oracle.glt / oracle.warp / oracle.srf against the fp64 plane warp of tests/s2_grid_oracle.py), and the one documented
deviation: a GLT-valid spectrum holding the nodata value in some of its bands."""
import math

import numpy as np
import pytest

from hsr_b200 import synthetic
from hsr_b200.EMIT_data import warp as hwarp
from hsr_b200.s2_emit.srf import srf_fold_weights, synthetic_s2_srf
from oracle import glt as oglt

import s2_grid_oracle as sgo

ND = sgo.ND
pytestmark = pytest.mark.filterwarnings("ignore::RuntimeWarning")      # NaN / Inf arithmetic of the cases
Hr, Wr = 14, 12

# (UTM EPSG, WGS-84 geotransform of the ortho grid): zone 11 north near 34 N, zone 34 south near 34 S
GEOMS = {
    "11N": (32611, (-118.30, 0.000542232520256367, 0.0, 34.20, 0.0, -0.000542232520256367)),
    "34S": (32734, (18.40, 0.000542232520256367, 0.0, -33.90, 0.0, -0.000542232520256367)),
}


def s2_grid_around(epsg, glt_gt, dx=10.0):
    """A 10 m S2 tile (109.8 km) whose origin lies ~3 km north-west of the ortho grid's corner."""
    zone, south = hwarp.epsg_to_utm(epsg)
    X, Y = hwarp.utm_forward(glt_gt[0], glt_gt[3], zone, south)
    x0 = math.floor((float(X) - 3000.0) / 60.0) * 60.0 + 30.0          # off the 60 m lattice of round numbers
    y0 = math.floor((float(Y) + 3000.0) / 60.0) * 60.0 + 20.0
    return hwarp.S2Grid(epsg=epsg, x0=x0, y0=y0, dx=dx, dy=dx, width=10980, height=10980)


def make_case(geom="11N", xres=60.0, kernel="cubic", seed=0, partial_nodata=False):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=good)
    raw[3, 4, 40] = np.nan                                       # one NaN band, one +Inf and one -Inf band
    raw[8, 6, 100] = np.inf
    raw[10, 3, 20] = -np.inf
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=seed + 1, hole_frac=0.03, n_oob=3, n_neg=3)
    if partial_nodata:
        raw[7, 5, 10:60] = ND                                    # a GLT-valid spectrum with nodata in 50 bands
    epsg, glt_gt = GEOMS[geom]
    ortho_shape = gx.shape
    s2 = s2_grid_around(epsg, glt_gt)
    target = hwarp.s2_target(glt_gt, ortho_shape, s2, xres, xres, kernel=kernel)
    W, names, _, fill_out = srf_fold_weights(w, table, good)
    return dict(raw=raw, gx=gx, gy=gy, glt_gt=glt_gt, target=target, w=w, good=good, table=table, names=names,
                fill_out=fill_out, s2=s2)


def plane_path(c):
    """SRF first (oracle.srf on the ortho cube, fp64), then the fp64 plane warp with per-pixel validity."""
    ortho, valid, _ = oglt.glt_ortho(c["raw"], c["gx"], c["gy"])
    planes = sgo.srf_planes(ortho, c["w"], c["table"], c["good"], c["names"])
    t = c["target"]
    out, cov, C = sgo.warp_conditioned(planes.transpose(1, 2, 0), c["glt_gt"], t.dst_gt, *t.shape, scales=t.scales,
                                       zone=t.zone, south=t.south, kernel=t.kernel, src_valid=valid)
    out = out.transpose(2, 0, 1)
    cov = cov[..., 0]
    out[:, ~cov] = c["fill_out"][:, None]
    return out, cov, C.transpose(2, 0, 1)


def assert_patterns_equal(got, want):
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern differs"
    assert np.array_equal(np.isposinf(got), np.isposinf(want)), "+Inf pattern differs"
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), "-Inf pattern differs"


CASES = [("11N", 60.0, "cubic"), ("11N", 60.0, "bilinear"), ("34S", 60.0, "cubic"), ("11N", 20.0, "cubic"),
         ("34S", 20.0, "bilinear")]


@pytest.mark.parametrize("geom,xres,kernel", CASES)
def test_plane_warp_commutes_with_srf_on_the_oracles(geom, xres, kernel):
    c = make_case(geom, xres, kernel)
    t = c["target"]
    assert (t.scales[0] < 1.0) == (xres == 60.0)                 # 60 m widens the filter, 20 m does not
    want, want_cov, _, _ = sgo.reference_chain(c["raw"], c["gx"], c["gy"], c["glt_gt"], t, c["w"], c["table"],
                                               c["good"], c["names"])
    got, cov, C = plane_path(c)
    assert np.array_equal(cov, want_cov), "coverage differs"
    assert 0 < cov.sum() < cov.size
    assert_patterns_equal(got, want)
    assert np.isnan(want).any() and np.isinf(want).any()
    fin = np.isfinite(want) & cov[None]
    err = np.abs(got[fin] - want[fin])
    assert np.all(err <= 1e-5 * C[fin] + 1e-7), f"max err {err.max():.3e}"
    unc = ~cov
    fo = c["fill_out"].astype(np.float64)[:, None]
    assert np.all(np.abs(want[:, unc] - fo) <= 1e-6 * np.abs(fo))  # the reference integrates the fill to fill_out


@pytest.mark.parametrize("geom,xres,kernel", CASES[:4])
def test_fp64_srf_first_equals_warp_first(geom, xres, kernel):
    """In fp64 the two orders agree to rounding: 1e-12 * C, identical NaN / Inf patterns and coverage."""
    c = make_case(geom, xres, kernel, seed=3)
    t = c["target"]
    ortho, valid, _ = oglt.glt_ortho(c["raw"], c["gx"], c["gy"])
    warped, cov_b, _ = sgo.warp_conditioned(ortho, c["glt_gt"], t.dst_gt, *t.shape, scales=t.scales, zone=t.zone,
                                            south=t.south, kernel=t.kernel, nodata=ND, fill=ND)
    want = sgo.srf_planes(warped, c["w"], c["table"], c["good"], c["names"])
    got, cov, C = plane_path(c)
    assert np.array_equal(cov_b.all(-1), cov) and np.array_equal(cov_b.any(-1), cov)
    assert_patterns_equal(got[:, cov], want[:, cov])
    fin = np.isfinite(want) & cov[None]
    err = np.abs(got[fin] - want[fin])
    assert np.all(err <= 1e-12 * C[fin]), f"max err / C {(err / C[fin]).max():.3e}"


def test_partial_nodata_spectrum_is_used_as_data():
    """The documented deviation: the reference skips a GLT-valid tap only in the bands that hold the nodata value, K
    planes cannot; the plane path uses the whole spectrum.  Destination pixels that tap it differ, the rest agree."""
    c = make_case("11N", 60.0, "cubic", partial_nodata=True)
    t = c["target"]
    want, want_cov, ortho, valid = sgo.reference_chain(c["raw"], c["gx"], c["gy"], c["glt_gt"], t, c["w"], c["table"],
                                                       c["good"], c["names"])
    got, cov, C = plane_path(c)
    assert np.array_equal(cov, want_cov)
    # destination pixels with a non-zero tap on the ortho pixels that carry the partial spectrum
    hit = np.zeros(ortho.shape[:2], bool)
    hit[(ortho[..., 10] == ND) & valid] = True
    assert hit.any()
    probe, _, _ = sgo.warp_conditioned(hit[..., None].astype(np.float64), c["glt_gt"], t.dst_gt, *t.shape,
                                       scales=t.scales, zone=t.zone, south=t.south, kernel=t.kernel, src_valid=valid,
                                       fill=0.0)
    touched = probe[..., 0] != 0.0
    assert touched.any()
    fin = np.isfinite(want) & np.isfinite(got) & cov[None]
    diff = np.abs(got - want)
    assert np.all(diff[fin & ~touched[None]] <= 1e-5 * C[fin & ~touched[None]] + 1e-7)
    assert diff[fin & touched[None]].max() > 1.0              # -9999 taken as data moves the touched pixels a lot


def test_s2_target_window_and_errors():
    c = make_case("11N", 60.0, "cubic")
    t, s2 = c["target"], c["s2"]
    row, col = t.s2_window
    assert isinstance(row, int) and isinstance(col, int)
    assert t.dst_gt[0] == pytest.approx(s2.x0 + col * 60.0, abs=1e-6)
    assert t.dst_gt[3] == pytest.approx(s2.y0 - row * 60.0, abs=1e-6)
    assert t.dst_gt[1] == 60.0 and t.dst_gt[5] == -60.0 and (t.zone, t.south) == (11, False)
    assert t.shape == (t.rec["rows"], t.rec["cols"])
    t20 = hwarp.s2_target(c["glt_gt"], c["gx"].shape, s2, 20.0, 20.0)
    assert t20.dst_gt[0] == pytest.approx(s2.x0 + t20.s2_window[1] * 20.0, abs=1e-6)
    assert t20.dst_gt[3] == pytest.approx(s2.y0 - t20.s2_window[0] * 20.0, abs=1e-6)
    ts = make_case("34S", 60.0, "cubic")["target"]
    assert (ts.zone, ts.south) == (34, True)
    far = hwarp.S2Grid(epsg=32611, x0=700000.0, y0=3000000.0, dx=10.0, dy=10.0, width=10980, height=10980)
    with pytest.raises(ValueError, match="No overlap"):
        hwarp.s2_target(c["glt_gt"], c["gx"].shape, far)
    with pytest.raises(ValueError, match="integer multiple"):
        hwarp.s2_target(c["glt_gt"], c["gx"].shape, s2, 25.0, 25.0)
    for k in ("nearest", "average", "lanczos"):
        with pytest.raises(ValueError, match="kernel"):
            hwarp.s2_target(c["glt_gt"], c["gx"].shape, s2, kernel=k)
