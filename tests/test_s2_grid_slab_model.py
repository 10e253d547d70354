"""CPU model of the row slabs on the Sentinel-2 grid (PairSynthesizer.synthesize_slab_on_s2_grid): the source rows a
band of target rows reads (tests/s2_slab_oracle.py, the rule of hsr_warp_src_row_range) hold every row that carries a
non-zero tap for the band, and the bookkeeping target band -> ortho rows -> raw rows (oracle/glt.py) reproduces the
band's planes from the staged rows alone."""
import dataclasses
import math

import numpy as np
import pytest

from hsr_b200 import synthetic
from hsr_b200.EMIT_data import warp as hwarp
from oracle import glt as oglt

import s2_grid_oracle as sgo
import s2_slab_oracle as sso

pytestmark = pytest.mark.filterwarnings("ignore::RuntimeWarning")
PIX = 0.000542232520256367


def random_target(rng, kernel):
    """An ortho grid of random size and place in zone 11 N or 34 S and its S2 target at a random resolution."""
    south = bool(rng.integers(2))
    epsg, lon0 = (32734, 21.0) if south else (32611, -117.0)
    lat = (-1.0 if south else 1.0) * rng.uniform(10.0, 60.0)
    lon = lon0 + rng.uniform(-2.5, 2.5)
    Ho, Wo = int(rng.integers(20, 60)), int(rng.integers(20, 60))
    glt_gt = (lon, PIX, 0.0, lat, 0.0, -PIX)
    zone, _ = hwarp.epsg_to_utm(epsg)
    X, Y = hwarp.utm_forward(lon, lat, zone, south)
    s2 = hwarp.S2Grid(epsg=epsg, x0=math.floor((float(X) - 3000.0) / 60.0) * 60.0,
                      y0=math.floor((float(Y) + 3000.0) / 60.0) * 60.0, dx=10.0, dy=10.0, width=10980, height=10980)
    xres = float(rng.choice([20.0, 60.0, 120.0]))
    return hwarp.s2_target(glt_gt, (Ho, Wo), s2, xres, xres, kernel=kernel), (Ho, Wo)


@pytest.mark.parametrize("kernel", ["cubic", "bilinear"])
def test_src_row_range_holds_every_tap_row(kernel):
    rng = np.random.default_rng(1 if kernel == "cubic" else 2)
    below_one = 0
    for _ in range(12):
        target, (Ho, Wo) = random_target(rng, kernel)
        below_one += target.scales[1] < 1.0
        Hd = target.shape[0]
        for t0, t1 in sso.uneven_bands(Hd, min(5, Hd), seed=int(rng.integers(1 << 30))):
            co = sso.centres(target, (t0, t1))
            rr = sso.src_row_range(co, Ho, Wo, target.scales, kernel)
            taps = sso.tap_rows(co, Ho, Wo, target.scales, kernel)
            if rr is None:
                assert not taps
                continue
            assert 0 <= rr[0] < rr[1] <= Ho
            assert all(rr[0] <= y < rr[1] for y in taps), (target.scales, (t0, t1), rr, sorted(taps))
        # a band moved wholly off the source: no centre inside, no range, no tap
        off = sso.centres(target, (0, 1)) + np.array([0.0, Ho + 50.0])
        assert sso.src_row_range(off, Ho, Wo, target.scales, kernel) is None
        assert not sso.tap_rows(off, Ho, Wo, target.scales, kernel)
    assert below_one > 0                                   # some geometries widen the filter


@pytest.mark.parametrize("geom", ["11N", "34S"])
def test_band_bookkeeping_reproduces_the_band(geom):
    """Target band -> ortho rows [o0, o1) -> raw rows [lo, hi): with every raw row outside [lo, hi) and every ortho
    row outside [o0, o1) replaced by garbage, the band's rows of the fp64 plane warp are unchanged, bit for bit."""
    Hr, Wr = 16, 14
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 6), seed=3, good=good[:6])
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=4, hole_frac=0.03, n_oob=3, n_neg=3)
    epsg, glt_gt = {"11N": (32611, (-118.30, PIX, 0.0, 34.20, 0.0, -PIX)),
                    "34S": (32734, (18.40, PIX, 0.0, -33.90, 0.0, -PIX))}[geom]
    zone, south = hwarp.epsg_to_utm(epsg)
    X, Y = hwarp.utm_forward(glt_gt[0], glt_gt[3], zone, south)
    s2 = hwarp.S2Grid(epsg=epsg, x0=math.floor((float(X) - 3000.0) / 60.0) * 60.0 + 30.0,
                      y0=math.floor((float(Y) + 3000.0) / 60.0) * 60.0 + 20.0, dx=10.0, dy=10.0, width=10980,
                      height=10980)
    target = hwarp.s2_target(glt_gt, gx.shape, s2, 60.0, 60.0)
    # three target rows above the source: the first band reads no source row
    dst_gt = list(target.dst_gt)
    dst_gt[3] -= 3 * dst_gt[5]
    target = dataclasses.replace(target, dst_gt=tuple(dst_gt), shape=(target.shape[0] + 3, target.shape[1]))
    Ho, Wo = gx.shape
    Hd, Wd = target.shape
    ortho, valid, _ = oglt.glt_ortho(raw, gx, gy)
    full, cov, _ = sgo.warp_conditioned(ortho, glt_gt, target.dst_gt, Hd, Wd, scales=target.scales, zone=zone,
                                        south=south, src_valid=valid)
    bands = [(0, 2)] + [(2 + a, 2 + b) for a, b in sso.uneven_bands(Hd - 2, 4, seed=5)]
    seen_empty = False
    for t0, t1 in bands:
        rr = sso.src_row_range(sso.centres(target, (t0, t1)), Ho, Wo, target.scales, "cubic")
        if rr is None:
            seen_empty = True
            assert not cov[t0:t1].any()
            continue
        o0, o1 = rr
        rw = sso.glt_raw_rows(gx[o0:o1], gy[o0:o1], Hr, Wr)
        assert rw is not None
        lo, hi = rw
        junk = np.full_like(raw, np.nan)
        junk[lo:hi] = raw[lo:hi]
        o_band, v_band, _ = oglt.glt_ortho(junk, gx[o0:o1], gy[o0:o1])
        assert np.array_equal(o_band.view(np.int32), ortho[o0:o1].view(np.int32))
        assert np.array_equal(v_band, valid[o0:o1])
        o_junk = np.full_like(ortho, np.inf)
        o_junk[o0:o1] = o_band
        v_junk = np.zeros_like(valid)
        v_junk[o0:o1] = v_band
        got, gcov, _ = sgo.warp_conditioned(o_junk, glt_gt, target.dst_gt, Hd, Wd, scales=target.scales, zone=zone,
                                            south=south, src_valid=v_junk)
        assert np.array_equal(gcov[t0:t1], cov[t0:t1])
        assert np.array_equal(got[t0:t1].view(np.int64), full[t0:t1].view(np.int64))
    assert seen_empty
