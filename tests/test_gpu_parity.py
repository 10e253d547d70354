"""Parity of the CUDA path (through the C ABI) against the oracle, the golden vectors produced by
the reference's own functions, and size-independent properties at BASELINE.json's full sizes.

Bars (BASELINE.json north_star): GLT gather + mask bit-exact; SRF bands 1e-5 relative (atol 1e-7
for |b| < 1e-2); fitted coefficients 1e-4 relative; applied values 1e-4 absolute.
"""
import warnings
from pathlib import Path

import numpy as np
import pytest
import torch

from hsr_b200 import kernels, synthetic
from hsr_b200.EMIT_data import emit_proj, emit_tools
from hsr_b200.pipeline import PairSynthesizer
from hsr_b200.s2_emit import poly_regression, srf, synth
from oracle import color as ocolor
from oracle import glt as oglt
from oracle import poly as opoly
from oracle import srf as osrf

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=RuntimeWarning)

DEV = "cuda"
SRF_RTOL, SRF_ATOL = 1e-5, 1e-7
COEF_RTOL = 1e-4
APPLY_ATOL = 1e-4


def bits(a):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def assert_srf_close(got, ref):
    got = got.detach().cpu().numpy().astype(np.float64) if isinstance(got, torch.Tensor) else np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), "NaN pattern differs"
    inf = np.isinf(ref)
    assert np.array_equal(got[inf], ref[inf]), "Inf pattern differs"
    ok = ~np.isnan(ref) & ~inf
    err = np.abs(got[ok] - ref[ok])
    tol = SRF_RTOL * np.abs(ref[ok]) + SRF_ATOL * (np.abs(ref[ok]) < 1e-2)
    assert np.all(err <= tol), f"max rel err {np.max(err / np.maximum(np.abs(ref[ok]), 1e-30)):.3e}"


def coeff_err(got, ref):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    return float(np.max(np.abs(got - ref).max(axis=-1) / np.abs(ref).max(axis=-1)))


# =============================================================================== kernel 1: GLT ortho
def test_glt_ortho_golden_apply_glt(golden):
    g = golden("glt_apply_glt.npz")
    raw, glt = g["raw"], g["glt"]
    gx, gy = kernels.prepare_glt(glt[..., 0], glt[..., 1], device=DEV)
    ortho, valid, diag = kernels.glt_ortho(dev(raw), gx, gy)
    assert np.array_equal(bits(ortho), bits(g["ortho"]))             # incl. NaN / Inf payloads
    assert np.array_equal(valid.cpu().numpy(), np.all(glt != 0, axis=-1))
    assert diag.tolist() == [int(valid.sum()), int(valid.sum()), 0]
    # reference call surface, numpy in / numpy out
    out = emit_tools.apply_glt(raw, glt)
    assert isinstance(out, np.ndarray) and out.dtype == np.float32
    assert np.array_equal(bits(out), bits(g["ortho"]))
    plane = emit_tools.apply_glt(raw[..., 40], glt)
    assert plane.shape == g["plane"].shape and np.array_equal(bits(plane), bits(g["plane"]))


@pytest.mark.parametrize("bands", [285, 32, 33, 64, 100, 7, 1, 3])
@pytest.mark.parametrize("transpose", [False, True])
def test_glt_ortho_defects_vs_oracle(bands, transpose):
    Hr, Wr = 61, 53
    raw = synthetic.raw_cube_bits_np((Hr, Wr, bands), seed=bands)
    raw[3, 4, 0] = np.nan
    raw[Hr - 1, Wr - 1, bands - 1] = -np.inf                      # last element of the allocation
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=1, hole_frac=0.01, n_oob=16, n_neg=16)
    gx[0, 0], gy[0, 0] = Wr, Hr                                   # last raw pixel (window would overrun)
    gx[0, 1], gy[0, 1] = 1, 1                                     # first raw pixel
    gx[0, 2], gy[0, 2] = Wr + 1, 1                                # one past the end in x
    gx[0, 3], gy[0, 3] = 1, Hr + 1                                # one past the end in y
    gx[0, 4], gy[0, 4] = -2147483648, 5                           # int32 minimum: (g - 1) wraps in numpy
    phys = np.ascontiguousarray(raw.transpose(1, 0, 2)) if transpose else raw
    ref, vref, dref = oglt.glt_ortho(phys, gx, gy, transpose_raw_yx=transpose)
    o, v, d = kernels.glt_ortho(dev(phys), dev(gx), dev(gy), transpose_raw_yx=transpose)
    assert np.array_equal(bits(o), bits(ref))
    assert np.array_equal(v.cpu().numpy(), vref)
    assert d.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    assert dref["valid_glt_dropped_oob"] > 0


@pytest.mark.parametrize("kind", ["identity", "upsample2", "upsample3x", "rowwrap", "reverse", "random", "angle3",
                                  "angle45", "angle80"])
@pytest.mark.parametrize("bands", [285, 40])
def test_glt_ortho_run_merging_shapes(kind, bands):
    """The producers merge lanes whose source pixels are equal or adjacent into one bulk copy: cover GLTs
    with long runs, duplicates (up-sampling GLTs), runs that wrap over the end of a raw row, descending
    and random sources."""
    Hr, Wr = 37, 41
    raw = synthetic.raw_cube_bits_np((Hr, Wr, bands), seed=17)
    rng = np.random.default_rng(5)
    if kind == "identity":
        gx, gy = synthetic.identity_glt(Hr, Wr, zero_frac=0.02, seed=3)
    elif kind == "upsample2":                                      # every source pixel 2 x 2 times
        yy, xx = np.meshgrid(np.arange(2 * Hr) // 2, np.arange(2 * Wr) // 2, indexing="ij")
        gx, gy = (xx + 1).astype(np.int32), (yy + 1).astype(np.int32)
    elif kind == "upsample3x":                                     # 3 x in x only, with holes
        yy, xx = np.meshgrid(np.arange(Hr), np.arange(3 * Wr) // 3, indexing="ij")
        gx, gy = (xx + 1).astype(np.int32), (yy + 1).astype(np.int32)
        gx[rng.random(gx.shape) < 0.05] = 0
    elif kind == "rowwrap":                                        # ortho width != raw width: runs wrap rows
        q = np.arange(Hr * Wr).reshape(Wr, Hr)                     # linear source order on a reshaped grid
        gx, gy = (q % Wr + 1).astype(np.int32), (q // Wr + 1).astype(np.int32)
    elif kind == "reverse":
        gx0, gy0 = synthetic.identity_glt(Hr, Wr, zero_frac=0.0)
        gx, gy = gx0[:, ::-1].copy(), gy0[::-1].copy()
    elif kind == "random":
        gx = rng.integers(0, Wr + 1, size=(50, 70)).astype(np.int32)
        gy = rng.integers(0, Hr + 1, size=(50, 70)).astype(np.int32)
    else:
        gx, gy = synthetic.rotation_glt(Hr, Wr, float(kind[5:]))
    ref, vref, dref = oglt.glt_ortho(raw, gx, gy)
    o, v, d = kernels.glt_ortho(dev(raw), dev(gx), dev(gy))
    assert np.array_equal(bits(o), bits(ref))
    assert np.array_equal(v.cpu().numpy(), vref)
    assert d.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    if bands == 285:                                               # the fused SRF consumer reads the same stages
        _, _, _, W, names, _, fill_out = _srf_setup(True)
        b1, _, _, _ = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out))
        b2 = kernels.srf_integrate(dev(ref), dev(W))
        assert np.array_equal(bits(b1)[:, vref], bits(b2)[:, vref])
        np.testing.assert_allclose(b1.cpu().numpy()[:, ~vref], b2.cpu().numpy()[:, ~vref], rtol=1e-6)


def test_glt_ortho_float_glt_with_nan_and_wrapper_diag():
    Hr, Wr, B = 20, 17, 285
    raw = synthetic.raw_cube_bits_np((Hr, Wr, B), seed=2)
    gx, gy = synthetic.rotation_glt(Hr, Wr, 40.0)
    gxf, gyf = gx.astype(np.float64), gy.astype(np.float64)
    gxf[gx == 0] = np.nan                                          # netCDF GLTs carry NaN for nodata
    gyf[::7, ::5] = np.nan
    ref, vref, dref = oglt.glt_ortho(raw, gxf, gyf)
    out, valid, info = emit_proj.glt_ortho(raw, gxf, gyf)
    assert isinstance(out, np.ndarray) and np.array_equal(bits(out), bits(ref))
    assert valid.dtype == bool and np.array_equal(valid, vref)
    assert info == dref


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_glt_ortho_misaligned_and_pitched_buffers(offset):
    Hr, Wr, B = 33, 29, 285
    raw = synthetic.raw_cube_bits_np((Hr, Wr, B), seed=9)
    gx, gy = synthetic.rotation_glt(Hr, Wr, 15.0)
    gx[1, 1], gy[1, 1] = 1, 1
    gx[1, 2], gy[1, 2] = Wr, Hr
    ref, vref, _ = oglt.glt_ortho(raw, gx, gy)
    # raw base only 4-byte aligned: a view `offset` floats into a larger buffer
    buf = torch.empty(raw.size + 8, dtype=torch.float32, device=DEV)
    view = buf[offset:offset + raw.size].view(Hr, Wr, B)
    view.copy_(dev(raw))
    o, v, _ = kernels.glt_ortho(view, dev(gx), dev(gy))
    assert np.array_equal(bits(o), bits(ref))
    # pitched raw (pixel stride 288 = 16-byte multiple) and pitched output
    pitched = torch.zeros((Hr, Wr, 288), dtype=torch.float32, device=DEV)
    pitched[..., :B] = dev(raw)
    o2, _, _ = kernels.glt_ortho(pitched[..., :B], dev(gx), dev(gy), out_pix_stride=288 + 4 * (offset - 1))
    assert o2.stride(1) == 288 + 4 * (offset - 1) and np.array_equal(bits(o2), bits(ref))
    # output base only 4-byte aligned
    Ho, Wo = gx.shape
    obuf = torch.full((Ho * Wo * B + 8,), 7.0, dtype=torch.float32, device=DEV)
    oview = obuf[offset:offset + Ho * Wo * B]
    kernels.glt_ortho(dev(raw), dev(gx), dev(gy), out=oview)
    assert np.array_equal(bits(oview.view(Ho, Wo, B)), bits(ref))
    assert obuf[:offset].eq(7.0).all() and obuf[offset + Ho * Wo * B:].eq(7.0).all()   # no stray writes


def test_glt_ortho_empty_and_all_fill():
    raw = dev(synthetic.raw_cube_bits_np((4, 5, 285), seed=1))
    z = torch.zeros((6, 7), dtype=torch.int32, device=DEV)
    o, v, d = kernels.glt_ortho(raw, z, z)
    assert o.eq(-9999.0).all() and not v.any() and d.tolist() == [0, 0, 0]
    e = torch.zeros((0, 7), dtype=torch.int32, device=DEV)
    o, v, d = kernels.glt_ortho(raw, e, e)
    assert o.shape == (0, 7, 285) and d.tolist() == [0, 0, 0]


def test_loc_obs_planes_vs_oracle():
    Hr, Wr = 40, 31
    rng = np.random.default_rng(4)
    planes = [rng.normal(size=(Hr, Wr)).astype(np.float32) for _ in range(3)]
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=3, n_oob=4, n_neg=4)
    outs = emit_proj.ortho_planes(planes, gx, gy)
    for pl, o in zip(planes, outs):
        assert np.array_equal(bits(o), bits(oglt.glt_plane(pl, gx, gy)))
    outs_t = emit_proj.ortho_planes([p.T.copy() for p in planes], gx, gy, transpose_raw_yx=True)
    for pl, o in zip(planes, outs_t):
        assert np.array_equal(bits(o), bits(oglt.glt_plane(pl.T.copy(), gx, gy, transpose_raw_yx=True)))


# =============================================================================== kernel 2: SRF
def _srf_setup(good_mask=True):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w) if good_mask else None
    table = srf.synthetic_s2_srf()
    W, names, none_bands, fill_out = srf.srf_fold_weights(w, table, good)
    return w, good, table, W, names, none_bands, fill_out


def test_srf_golden_through_reference_call_surface(golden):
    g = golden("srf_pseudo_s2.npz")
    names = [str(n) for n in g["names"]]
    table = {b: (g[f"lam_{b}"], g[f"rsp_{b}"]) for b in names}
    for tag, good in (("good", g["good"]), ("all", None)):
        out = synth.pseudo_s2_srf_integral(g["cube"], g["emit_w"], table, good)
        assert list(out) == names
        for b in names:
            if bool(g[f"none_{tag}_{b}"]):
                assert out[b] is None
            else:
                assert isinstance(out[b], np.ndarray) and out[b].dtype == np.float64
                assert_srf_close(out[b], g[f"out_{tag}_{b}"])
    out = synth.pseudo_s2_srf_integral(g["cube"], g["emit_w"], table, g["good"])
    rgb = synth.pseudo_s2_rgb(out)
    assert rgb.shape == g["rgb"].shape
    assert_srf_close(rgb, g["rgb"])
    # CUDA tensors in -> CUDA tensors out
    out_t = synth.pseudo_s2_srf_integral(dev(g["cube"]), g["emit_w"], table, g["good"])
    assert out_t["B2"].is_cuda and out_t["B10"] is None
    assert_srf_close(out_t["B8"], g["out_good_B8"])


@pytest.mark.parametrize("good_mask", [True, False])
def test_glt_srf_fused_vs_oracle(good_mask):
    w, good, table, W, names, none_bands, fill_out = _srf_setup(good_mask)
    Hr, Wr, B = 70, 45, 285
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, B), seed=6, good=good)
    rng = np.random.default_rng(8)
    for _ in range(12):                                            # non-finite samples, some in zero-weight bands
        raw[rng.integers(Hr), rng.integers(Wr), rng.integers(B)] = rng.choice([np.nan, np.inf, -np.inf])
    raw[5, 5, 0] = np.nan                                          # 381 nm: no S2 band has weight there
    raw[6, 6, 284] = np.inf
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=2, hole_frac=0.01, n_oob=8, n_neg=8)
    gx[0, 0], gy[0, 0] = Wr, Hr
    ortho_ref, vref, dref = oglt.glt_ortho(raw, gx, gy)
    ps = osrf.pseudo_s2_srf_integral(ortho_ref, w, table, good)
    ref = np.stack([ps[b] for b in names])
    bands, valid, diag, ortho = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out),
                                                materialize_ortho=True)
    assert np.array_equal(valid.cpu().numpy(), vref)
    assert np.array_equal(bits(ortho), bits(ortho_ref))
    assert diag.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    assert_srf_close(bands, ref)
    assert np.isnan(ref).any() and (ref[:, ~vref] < -9998).all()
    # without the ortho cube (the fused fast path) the planes are bit-identical
    b2, v2, _, o2 = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out))
    assert o2 is None and np.array_equal(bits(b2), bits(bands)) and v2.equal(valid)
    # un-fused kernel on the materialised cube agrees bit for bit with the fused one
    b3 = kernels.srf_integrate(ortho, dev(W))
    assert np.array_equal(bits(b3), bits(bands))
    # the fit mask emitted while the planes are written == fit_mask kernel == oracle rule on the planes,
    # for every gate band (incl. none) and in both the fused and the ortho-materialising variants
    got_planes = bands.cpu().numpy()
    for gate_k in (-1, 0, 3, len(names) - 1):
        for mat in (False, True):
            fm = torch.zeros(gx.shape, dtype=torch.bool, device=DEV)
            kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), materialize_ortho=mat,
                            fit_mask_out=fm, gate_k=gate_k, gate_gt=0.0)
            want = opoly.fit_mask(got_planes, vref, gate_k, 0.0)
            assert np.array_equal(fm.cpu().numpy(), want)
            assert fm.equal(kernels.fit_mask(bands, valid, gate_k=gate_k, gate_gt=0.0))
    assert want.any() and not want.all() and not want[np.isnan(got_planes).any(0)].any()
    fm3 = torch.zeros(gx.shape, dtype=torch.bool, device=DEV)
    kernels.srf_integrate(ortho, dev(W), fit_mask_out=fm3, gate_k=0, gate_gt=0.0)
    assert np.array_equal(fm3.cpu().numpy(), opoly.fit_mask(got_planes, None, 0, 0.0))


@pytest.mark.parametrize("pattern", ["all_nodata", "stripes", "sparse", "tail", "one_valid_per_tile"])
def test_glt_srf_nodata_tiles_finished_by_the_producer(pattern):
    """Whole 32-pixel tiles without a valid pixel never enter the stage ring of the fused kernel (the producer warp
    writes their fill planes, valid and fit-mask bytes itself): grids made of such tiles, alone and mixed with valid tiles
    in every order, must give exactly what the ring gives — compared with the ortho-materialising variant (every tile goes
    through the ring there) bit for bit and with the oracle."""
    w, good, table, W, names, none_bands, fill_out = _srf_setup(True)
    Hr, Wr, B = 40, 37, 285
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, B), seed=9, good=good)
    raw[3, 3, 100] = np.nan
    rng = np.random.default_rng(17)
    Ho, Wo = 61, 96                                                # 5856 px = 183 tiles; with "tail": 5857 -> a partial tile
    if pattern == "tail":
        Ho, Wo = 1, 5857
    n = Ho * Wo
    gx = rng.integers(1, Wr + 1, size=n).astype(np.int32)
    gy = rng.integers(1, Hr + 1, size=n).astype(np.int32)
    tile = np.arange(n) // 32
    if pattern == "all_nodata":
        gx[:] = 0
    elif pattern == "stripes":                                     # runs of 1, 2, 3, ... nodata tiles between valid ones
        k, t = 1, 0
        while t < tile.max() + 1:
            gx[(tile >= t + 1) & (tile < t + 1 + k)] = 0
            t += 1 + k
            k = k % 7 + 1
    elif pattern == "sparse":                                      # mostly nodata, isolated valid tiles
        gx[rng.random(tile.max() + 1)[tile] < 0.9] = 0
        gy[rng.random(n) < 0.05] = 0
    elif pattern == "tail":                                        # nodata everywhere but the first tiles; partial last tile nodata
        gx[64:] = 0
    else:                                                          # every tile keeps exactly one valid pixel: nothing is skipped
        keep = rng.integers(0, 32, size=tile.max() + 1)[tile] == (np.arange(n) % 32)
        gx[~keep] = 0
    gx, gy = gx.reshape(Ho, Wo), gy.reshape(Ho, Wo)
    ortho_ref, vref, dref = oglt.glt_ortho(raw, gx, gy)
    ps = osrf.pseudo_s2_srf_integral(ortho_ref, w, table, good)
    ref = np.stack([ps[b] for b in names])
    fm = torch.ones(gx.shape, dtype=torch.bool, device=DEV)
    bands, valid, diag, _ = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), fit_mask_out=fm, gate_k=0)
    fm2 = torch.ones(gx.shape, dtype=torch.bool, device=DEV)
    b2, v2, d2, _ = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), materialize_ortho=True,
                                    fit_mask_out=fm2, gate_k=0)
    assert np.array_equal(bits(bands), bits(b2)) and valid.equal(v2) and fm.equal(fm2) and diag.tolist() == d2.tolist()
    assert np.array_equal(valid.cpu().numpy(), vref)
    assert diag.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    assert_srf_close(bands, ref)
    assert np.array_equal(fm.cpu().numpy(), opoly.fit_mask(bands.cpu().numpy(), vref, 0, 0.0))
    if pattern == "all_nodata":
        assert not vref.any() and not fm.any()
    # twice in a row into the same buffers (stale stage contents, barrier phases start over)
    b3 = torch.full_like(bands, 7.0)
    kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), bands_out=b3, want_valid=False, want_diag=False)
    assert np.array_equal(bits(b3), bits(bands))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_glt_srf_nodata_tiles_long_sequences(seed):
    """The same property with MANY tiles per CTA (9375 tiles: ~13 uses of every stage of every CTA, so the stage barriers
    flip parity many times while the producers skip nodata tiles in runs of random length): the fused kernel — nodata
    tiles finished by the producers — against the ortho-materialising variant, where every tile goes through the ring,
    bit for bit; validity against the oracle rule."""
    w, good, table, W, names, none_bands, fill_out = _srf_setup(True)
    Hr, Wr, B = 64, 50, 285
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, B), seed=20 + seed, good=good)
    raw[7, 7, 11] = np.inf
    rng = np.random.default_rng(300 + seed)
    Ho, Wo = 300, 1000
    n = Ho * Wo
    gx = rng.integers(1, Wr + 1, size=n).astype(np.int32)
    gy = rng.integers(1, Hr + 1, size=n).astype(np.int32)
    ntile = n // 32
    dead = np.zeros(ntile, bool)
    t = 0
    while t < ntile:                                               # alternating runs of valid / nodata tiles, lengths 1 .. 40
        a, b = int(rng.integers(1, 41)), int(rng.integers(1, 41))
        dead[t + a:t + a + b] = True
        t += a + b
    if seed == 2:
        dead = rng.random(ntile) < 0.97                            # almost everything nodata: the producers race far ahead
    gx[np.repeat(dead, 32)] = 0
    gy[rng.random(n) < 0.02] = 0                                   # and scattered holes inside valid tiles
    gx, gy = gx.reshape(Ho, Wo), gy.reshape(Ho, Wo)
    vref = (gx != 0) & (gy != 0)
    fm = torch.ones(gx.shape, dtype=torch.bool, device=DEV)
    bands, valid, diag, _ = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), fit_mask_out=fm, gate_k=0)
    fm2 = torch.ones(gx.shape, dtype=torch.bool, device=DEV)
    b2, v2, d2, ortho = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), materialize_ortho=True,
                                        fit_mask_out=fm2, gate_k=0)
    assert np.array_equal(valid.cpu().numpy(), vref) and valid.equal(v2) and diag.tolist() == d2.tolist()
    assert np.array_equal(bits(bands), bits(b2)) and fm.equal(fm2)
    assert np.array_equal(bits(ortho), bits(oglt.glt_ortho(raw, gx, gy)[0]))
    assert diag.tolist()[0] == int(vref.sum())
    for _ in range(3):                                             # repeat launches: no state may leak from one to the next
        b3, _, _, _ = kernels.glt_srf(dev(raw), dev(gx), dev(gy), dev(W), dev(fill_out), want_valid=False, want_diag=False)
        assert np.array_equal(bits(b3), bits(bands))


@pytest.mark.parametrize("bands,K", [(285, 1), (285, 16), (64, 3), (33, 2), (5, 2), (300, 13)])
def test_srf_dense_weights_any_shape(bands, K):
    rng = np.random.default_rng(bands * 31 + K)
    cube = rng.uniform(0, 1, size=(37, 11, bands)).astype(np.float32)
    W = rng.uniform(0, 1, size=(bands, K)).astype(np.float32)
    W[:, 0] = 0.0
    W[bands // 2, 0] = 1.0                                          # a one-band response
    ref = cube.astype(np.float64) @ W.astype(np.float64)
    out = kernels.srf_integrate(dev(cube), dev(W))
    assert out.shape == (K, 37, 11)
    np.testing.assert_allclose(out.cpu().numpy(), np.moveaxis(ref, -1, 0), rtol=2e-5, atol=1e-6)
    with pytest.raises(Exception):
        kernels.srf_integrate(dev(cube), dev(np.zeros((bands, 17), np.float32)))


# =============================================================================== kernel 3: polyfit
@pytest.mark.parametrize("deg", [1, 2, 4])
def test_poly_fit_vs_np_polyfit(deg):
    rng = np.random.default_rng(deg)
    K, H, Wd = 5, 211, 173
    x = rng.uniform(0.0, 0.6, size=(K, H, Wd)).astype(np.float32)
    y = synthetic.s2_reference_np(x, seed=3)
    x[0, 0, 0] = np.nan
    y[1, 2, 3] = np.inf
    mask = rng.random((H, Wd)) < 0.8
    ref = opoly.polyfit_paired(x, y, mask, deg)
    got = kernels.poly_fit(dev(x), dev(y), dev(mask), deg)
    assert got.dtype == torch.float64 and coeff_err(got, ref) < COEF_RTOL
    xs = np.linspace(0, 1, 101)
    for k in range(K):                                             # fitted curves agree on [0, 1]
        assert np.max(np.abs(np.polyval(got[k].cpu().numpy(), xs) - np.polyval(ref[k], xs))) < 1e-4
    # per-series masks and no mask
    mk = rng.random((K, H, Wd)) < 0.5
    assert coeff_err(kernels.poly_fit(dev(x), dev(y), dev(mk), deg), opoly.polyfit_paired(x, y, mk, deg)) < COEF_RTOL
    assert coeff_err(kernels.poly_fit(dev(x), dev(y), None, deg), opoly.polyfit_paired(x, y, None, deg)) < COEF_RTOL
    # numpy wrapper
    c = poly_regression.poly_fit(x, y, mask, deg)
    assert isinstance(c, np.ndarray) and coeff_err(c, ref) < COEF_RTOL


def test_poly_fit_rank_deficient_bands_get_np_polyfit_answer_on_the_host():
    """A band with fewer distinct x than deg + 1 (a constant plane, a two-level plane): np.polyfit returns the minimum-norm
    solution with a RankWarning; the host mirrors do the same from the device moments (CUDA-tensor callers get NaN)."""
    import warnings

    from hsr_b200.s2_emit import poly_regression as pr
    rng = np.random.default_rng(4)
    H, W = 40, 50
    x = rng.random((3, H, W)).astype(np.float32)
    x[0] = 0.25                                                    # constant band
    x[1] = rng.choice(np.float32([0.5, 0.75]), size=(H, W))        # two levels, deg 2 needs three
    y = rng.random((3, H, W)).astype(np.float32)
    mask = rng.random((H, W)) < 0.8
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = np.stack([np.polyfit(x[k][mask].astype(np.float64), y[k][mask].astype(np.float64), 2) for k in range(3)])
    with pytest.warns(np.exceptions.RankWarning):
        got = pr.poly_fit(x, y, mask, 2)
    assert np.isfinite(got).all() and np.allclose(got, ref, rtol=1e-7, atol=1e-9)
    dev_out = pr.poly_fit(dev(x), dev(y), dev(mask), 2)            # device results: the raw solve (NaN or garbage on bands 0, 1)
    assert dev_out.is_cuda and torch.allclose(dev_out[2].cpu(), torch.from_numpy(ref[2]), rtol=1e-7, atol=1e-9)


def test_poly_moments_are_exact_sums_and_deterministic():
    rng = np.random.default_rng(0)
    K, n, deg = 3, 100_003, 2
    x = rng.uniform(0, 1, size=(K, n)).astype(np.float32)
    y = rng.uniform(0, 1, size=(K, n)).astype(np.float32)
    mask = rng.random(n) < 0.6
    m1 = kernels.poly_moments(dev(x), dev(y), dev(mask), deg)
    m2 = kernels.poly_moments(dev(x), dev(y), dev(mask), deg)
    assert m1.equal(m2)                                            # fixed reduction order
    xd, yd = x.astype(np.float64)[:, mask], y.astype(np.float64)[:, mask]
    ref = np.stack([np.concatenate([[np.sum(xd[k] ** j) for j in range(2 * deg + 1)],
                                    [np.sum(xd[k] ** j * yd[k]) for j in range(deg + 1)]]) for k in range(K)])
    np.testing.assert_allclose(m1.cpu().numpy(), ref, rtol=1e-12)
    assert m1[:, 0].tolist() == [float(mask.sum())] * K


def test_poly_identity_fallback_and_golden(golden):
    g = golden("poly_apply_fit.npz")
    img, yimg, mask = g["img"], g["yimg"], g["mask"]
    ident = poly_regression.fit_ot_poly_rgb(img, yimg, g["small_mask"], deg=2, targets="paired")
    assert np.array_equal(ident, g["ident"])
    for deg, key in ((2, "fit2"), (4, "fit4")):
        c = poly_regression.fit_ot_poly_rgb(img, yimg, mask, deg=deg, targets="paired")
        assert c.shape == (3, deg + 1) and coeff_err(c, g[key]) < COEF_RTOL


# =============================================================================== OT targets (fit_ot_poly_rgb)
def test_fit_ot_poly_rgb_golden_through_reference_call_surface(golden):
    """fit_ot_poly_rgb with its reference signature and defaults (targets = OT barycentric, poly_regression.py:16-62)
    against the coefficients the reference's own function produced (POT restated: parity unpinned there)."""
    g = golden("ot_fit.npz")
    for key in [k for k in g.files if k.startswith("coeffs_")]:
        _, d, n, sd = key.split("_")
        c, info = poly_regression.fit_ot_poly_rgb(g["src"], g["ref"], g["mask"], deg=int(d[1:]), n_samples=int(n[1:]),
                                                  seed=int(sd[1:]), return_info=True)
        assert c.dtype == np.float64 and c.shape == g[key].shape
        assert coeff_err(c, g[key]) < COEF_RTOL, (key, coeff_err(c, g[key]))
        assert info["numerical_error"] == 0 and info["err"] < 1e-6 and info["err_iteration"] % 10 == 0
        # fitted curves agree on [0, 1] (SURVEY 8c)
        xs = np.linspace(0, 1, 101)
        assert max(np.max(np.abs(np.polyval(c[k], xs) - np.polyval(g[key][k], xs))) for k in range(3)) < 1e-4
    assert np.array_equal(poly_regression.fit_ot_poly_rgb(g["src"], g["ref"], g["small"], deg=3), g["ident"])
    t = poly_regression.fit_ot_poly_rgb(dev(g["src"]), dev(g["ref"]), dev(g["mask"]), n_samples=600)
    assert t.is_cuda and coeff_err(t, g["coeffs_d2_n600_s0"]) < COEF_RTOL


def test_robust_norm_golden_bit_exact(golden):
    """robust_norm / robust_norm_rgb (s2_emit/color.py:6-23) against the reference's own outputs: float64, bit for bit
    (exact percentiles over the non-NaN / masked samples, the float64 stretch expression evaluated as numpy does)."""
    from hsr_b200.s2_emit import color
    g = golden("color_robust.npz")

    def same(a, b):
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        return a.dtype == np.float64 and a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))
    assert same(color.robust_norm(g["xn"]), g["rn"])
    assert same(color.robust_norm(g["xn"], 5, 90), g["rn_5_90"])
    assert same(color.robust_norm(g["img"]), g["rn_cube"])
    assert same(color.robust_norm_rgb(g["img"], g["mask"]), g["rgb"])
    assert same(color.robust_norm_rgb(g["img"], g["mask"], 1, 99), g["rgb_1_99"])
    t = color.robust_norm_rgb(dev(g["img"]), dev(g["mask"]))                      # CUDA in -> CUDA out
    assert t.is_cuda and same(t, g["rgb"])
    assert same(color.robust_norm(dev(g["xn"])), g["rn"])


def test_histogram_match_rgb_golden_bit_exact(golden):
    """histogram_match_rgb (s2_emit/color.py:36-63) against the reference's own output, bit for bit: source CDF by rank
    in the sorted samples, inverse reference CDF by np.interp's arithmetic over the distinct reference values."""
    from hsr_b200.s2_emit import color
    g = golden("color_histmatch.npz")
    got = color.histogram_match_rgb(g["src"], g["ref"], g["mask"])
    assert got.dtype == np.float32 and np.array_equal(bits(got), bits(g["out"]))
    assert np.array_equal(bits(color.histogram_match_rgb(g["src"], g["ref"], g["few"])), bits(g["out_few"]))
    t = color.histogram_match_rgb(dev(g["src"]), dev(g["ref"]), dev(g["mask"]))
    assert t.is_cuda and np.array_equal(bits(t), bits(g["out"]))
    with pytest.raises(IndexError):
        color.histogram_match_rgb(g["src"], g["ref"], np.zeros_like(g["mask"]))
    # a larger random case against the oracle (ties on both sides)
    from oracle import color as oc
    rng = np.random.default_rng(11)
    a = np.round(rng.random((211, 173, 3)) * 200).astype(np.float32) / 200
    b = (rng.random((211, 173, 3)) ** 2).astype(np.float32)
    mk = rng.random((211, 173)) < 0.5
    assert np.array_equal(bits(color.histogram_match_rgb(a, b, mk)), bits(oc.histogram_match_rgb(a, b, mk)))


def test_ot_match_rgb_golden_through_reference_call_surface(golden):
    """ot_match_rgb_sinkhorn_pot (s2_emit/color.py:63-116, reference signature) against what the reference's own function
    produced (POT restated: parity unpinned there).  Bar: 1e-5 absolute on [0, 1] values (fp64 Sinkhorn + normal-equation
    affine fit vs numpy's SVD lstsq), NaN pattern and the pixels outside the mask bit for bit."""
    from hsr_b200.s2_emit import color
    g = golden("color_ot_match.npz")
    cases = (("out_n400_s0", dict(n_samples=400, seed=0)), ("out_n100000_s2", dict(n_samples=100000, seed=2)),
             ("out_reg01_it20", dict(n_samples=300, reg=0.1, numItermax=20, stopThr=0.0, seed=5)))
    m = g["mask"]
    for key, kw in cases:
        got = color.ot_match_rgb_sinkhorn_pot(g["src"], g["ref"], m, **kw)
        want = g[key]
        assert got.dtype == np.float32 and got.shape == want.shape
        assert np.array_equal(np.isnan(got), np.isnan(want)), key
        assert np.array_equal(bits(got[~m]), bits(want[~m])), key
        ok = ~np.isnan(want)
        assert np.max(np.abs(got[ok] - want[ok])) < 1e-5, (key, np.max(np.abs(got[ok] - want[ok])))
    one = color.ot_match_rgb_sinkhorn_pot(g["src"], g["ref"], g["one"])
    assert np.array_equal(one, g["src"], equal_nan=True)
    t = color.ot_match_rgb_sinkhorn_pot(dev(g["src"]), dev(g["ref"]), dev(m), n_samples=400, seed=0)     # CUDA in -> CUDA out
    assert t.is_cuda and np.allclose(t.cpu().numpy(), g["out_n400_s0"], atol=1e-5, equal_nan=True)
    # the affine pair on its own: lstsq of an exactly affine relation recovers it
    rng = np.random.default_rng(3)
    X = rng.random((777, 3))
    A = rng.normal(size=(3, 3))
    tt = rng.normal(size=3)
    W = kernels.affine_fit(dev(X), dev(X @ A + tt)).cpu().numpy()
    assert np.allclose(W[:3], A, atol=1e-10) and np.allclose(W[3], tt, atol=1e-10)
    Wn, *_ = np.linalg.lstsq(np.c_[X, np.ones(777)], np.sin(X * 3), rcond=None)
    assert np.allclose(kernels.affine_fit(dev(X), dev(np.sin(X * 3))).cpu().numpy(), Wn, atol=1e-10)


def test_sinkhorn_barycentric_vs_oracle(golden):
    from oracle import ot as oot

    g = golden("ot_fit.npz")
    X, Y = g["X"], g["Y"]
    ybar, info = kernels.sinkhorn_barycentric(dev(X), dev(Y), 0.05, 300, 1e-6)
    np.testing.assert_allclose(ybar.cpu().numpy(), g["ybar"], rtol=0, atol=1e-11)
    _, ref_info = oot.sinkhorn_knopp(np.full(len(X), 1 / len(X)), np.full(len(Y), 1 / len(Y)), oot.dist(X, Y), 0.05, 300,
                                     1e-6, log=True)
    it, err, err_it, num = info.cpu().tolist()
    assert err_it == ref_info["niter"] and it == ref_info["niter"] + 1 and num == 0
    assert abs(err - ref_info["err"][-1]) <= 1e-9 * ref_info["err"][-1] + 1e-18
    # iteration cap without convergence: exactly numItermax updates
    ybar12, info12 = kernels.sinkhorn_barycentric(dev(X), dev(Y), 0.05, 12, 0.0)
    np.testing.assert_allclose(ybar12.cpu().numpy(), g["ybar_12it"], rtol=0, atol=1e-11)
    assert info12.cpu().tolist()[0] == 12
    # underflowing kernel matrix: POT rolls back to the initial scalings and stops
    with np.errstate(all="ignore"):
        want = oot.barycentric_targets(X * 1e3, Y * 1e3 + 7.0, 0.05, 50, 1e-9)
    got, info_bad = kernels.sinkhorn_barycentric(dev(X * 1e3), dev(Y * 1e3 + 7.0), 0.05, 50, 1e-9)
    assert info_bad.cpu().tolist()[3] == 1 and info_bad.cpu().tolist()[0] == 0
    assert np.array_equal(np.isfinite(got.cpu().numpy()), np.isfinite(want))
    # a mid-size problem (non-multiple-of-anything shapes, several column chunks)
    rng = np.random.default_rng(5)
    X2, Y2 = rng.random((1537, 3)), rng.random((1203, 3)) ** 2
    yb2, _ = kernels.sinkhorn_barycentric(dev(X2), dev(Y2), 0.05, 300, 1e-6)
    np.testing.assert_allclose(yb2.cpu().numpy(), oot.barycentric_targets(X2, Y2), rtol=0, atol=1e-10)


def test_compact_gather_and_f64_polyfit():
    rng = np.random.default_rng(9)
    n, C = 10007, 3
    img = rng.random((n, C)).astype(np.float32)
    img[rng.random(n) < 0.01, 1] = np.nan
    img[rng.random(n) < 0.01, 2] = np.inf
    mask = rng.random(n) < 0.7
    want = np.flatnonzero(mask & np.isfinite(img).all(1))
    idx, cnt = kernels.compact_finite_rows(dev(img), dev(mask))
    assert int(cnt.item()) == want.size and np.array_equal(idx[:want.size].cpu().numpy(), want)
    idx2, cnt2 = kernels.compact_finite_rows(dev(img), None)
    assert int(cnt2.item()) == np.isfinite(img).all(1).sum()
    sel = rng.choice(want.size, size=500, replace=False)
    got = kernels.gather_rows_f64(dev(img), idx, dev(sel.astype(np.int64)))
    assert np.array_equal(got.cpu().numpy(), img[want[sel]].astype(np.float64))
    x = rng.random((4000, 3))
    y = 0.3 * x ** 3 - 0.2 * x + 0.1 + rng.normal(0, 0.01, x.shape)
    for deg in (1, 2, 4):
        c = kernels.polyfit_f64(dev(x), dev(y), deg).cpu().numpy()
        ref = np.stack([np.polyfit(x[:, k], y[:, k], deg) for k in range(3)])
        assert coeff_err(c, ref) < 1e-8


def test_poly_apply_golden(golden):
    g = golden("poly_apply_fit.npz")
    img, mask = g["img"], g["mask"]
    for key, coeffs, m in (("out2_mask", g["coeffs2"], mask), ("out2_nomask", g["coeffs2"], None),
                           ("out4_mask", g["coeffs4"], mask)):
        out = poly_regression.apply_poly_rgb(img, coeffs, m)
        ref = g[key]
        assert out.dtype == np.float32 and out.shape == ref.shape
        assert np.array_equal(np.isnan(out), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert np.max(np.abs(out[ok] - ref[ok])) <= APPLY_ATOL
        assert np.mean(out[ok] == ref[ok]) > 0.999                # fp64 Horner -> same fp32 rounding
    # planar layout, clip disabled
    x = np.moveaxis(img, -1, 0).copy()
    out = kernels.poly_apply(dev(x), dev(g["coeffs2"]), dev(mask), lo=1.0, hi=0.0).cpu().numpy()
    ref = opoly.apply_poly_planes(x, g["coeffs2"], mask, lo=1.0, hi=0.0)
    ok = np.isfinite(ref)
    assert np.array_equal(np.isfinite(out), ok) and np.max(np.abs(out[ok] - ref[ok])) <= APPLY_ATOL
    assert out[ok].max() > 1.0


def test_fit_mask_vs_oracle():
    rng = np.random.default_rng(12)
    x = rng.normal(0.2, 0.3, size=(4, 50, 60)).astype(np.float32)
    x[1, 3, 3] = np.nan
    x[3, 4, 4] = np.inf
    valid = rng.random((50, 60)) < 0.7
    m = kernels.fit_mask(dev(x), dev(valid), gate_k=0, gate_gt=0.0)
    assert np.array_equal(m.cpu().numpy(), opoly.fit_mask(x, valid, 0, 0.0))
    m = kernels.fit_mask(dev(x), None, gate_k=-1)
    assert np.array_equal(m.cpu().numpy(), opoly.fit_mask(x, None, -1))
    # y given: every reference plane must be finite as well (poly_regression.py:118)
    y = np.random.default_rng(5).random(x.shape, dtype=np.float32)
    y[1, 3, 4] = np.nan
    y[0, 7, 7] = np.inf
    m = kernels.fit_mask(dev(x), dev(valid), gate_k=0, gate_gt=0.0, y=dev(y))
    assert np.array_equal(m.cpu().numpy(), opoly.fit_mask(x, valid, 0, 0.0) & np.isfinite(y).all(0))



@pytest.mark.parametrize("shape,groups", [((12, 53, 47), 1), ((12, 64, 64), 1), ((3, 6 * 40, 24), 6), ((16, 7, 5), 1)])
@pytest.mark.parametrize("deg", [1, 2, 4])
def test_fused_fit_moments_and_solve_apply(shape, groups, deg):
    """hsr_fit_moments_f64 == fit_mask + poly_moments, hsr_poly_solve_apply_f32 == poly_solve + poly_apply
    (odd plane sizes exercise the scalar-load paths, padded planes the 16-byte ones)."""
    rng = np.random.default_rng(shape[1] * 7 + deg)
    K = shape[0]
    x = rng.uniform(-0.1, 0.8, size=shape).astype(np.float32)
    c = rng.normal(0, 0.5, size=(K, deg + 1))
    y = np.stack([np.polyval(c[k], x[k].astype(np.float64)) for k in range(K)]) + rng.normal(0, 0.01, size=shape)
    y = y.astype(np.float32)
    x[0, 1, 2] = np.nan
    x[K - 1, 3, 1] = np.inf
    y[1, 2, 2] = np.nan                                            # drops the sample for band 1 only
    valid = rng.random(shape[1:]) < 0.8
    G = groups
    n = x[0].size // G
    for padded in (False, True):
        xt = kernels.alloc_planes(K, shape[1:], DEV) if padded else torch.empty(shape, dtype=torch.float32, device=DEV)
        yt = kernels.alloc_planes(K, shape[1:], DEV) if padded else torch.empty(shape, dtype=torch.float32, device=DEV)
        xt.copy_(dev(x))
        yt.copy_(dev(y))
        mom, fm = kernels.fit_moments(xt, yt, dev(valid), deg, groups=G, gate_k=0, gate_gt=0.0)
        fm_ref = opoly.fit_mask(x, valid, 0, 0.0)
        assert np.array_equal(fm.cpu().numpy().reshape(fm_ref.shape), fm_ref)
        # the un-fused kernels on the same series (one mask per group)
        xs, ys = dev(x).view(K * G, n), dev(y).view(K * G, n)
        mom_ref = kernels.poly_moments(xs, ys, dev(fm_ref).view(G, n), deg, mask_rows="inner")
        np.testing.assert_allclose(mom.cpu().numpy().reshape(K * G, -1), mom_ref.cpu().numpy(), rtol=1e-12, atol=0)
        assert mom.equal(kernels.fit_moments(xt, yt, dev(valid), deg, groups=G, gate_k=0)[0])   # deterministic
        coeffs, out = kernels.poly_solve_apply(xt, mom, fm, deg, groups=G, min_count=20)
        co_ref = kernels.poly_solve(mom.view(K * G, -1), deg, 20)
        assert coeffs.view(K * G, -1).equal(co_ref)
        out_ref = kernels.poly_apply(xs, co_ref, dev(fm_ref).view(G, n), mask_rows="inner")
        assert np.array_equal(bits(out).reshape(-1), bits(out_ref).reshape(-1))
        # against np.polyfit on the same masked samples
        ref = opoly.polyfit_paired(x.reshape(K * G, n), y.reshape(K * G, n),
                                   np.broadcast_to(fm_ref.reshape(1, G, n), (K, G, n)).reshape(K * G, n), deg,
                                   min_count=20)
        assert coeff_err(coeffs.view(K * G, -1), ref) < (COEF_RTOL if n * 0.5 > 200 or deg < 4 else 5e-3)

# =============================================================================== percentile stretch
def test_percentile_stretch_golden_through_reference_call_surface(golden):
    """hsr_b200.s2_emit.color.apply_shared_percentile_stretch == the reference's (s2_emit/color.py:25-34),
    bit for bit, on the golden inputs (ties, -0.0, +-Inf inside the mask, 3-sample mask, NaN -> NaN channel)."""
    from hsr_b200.s2_emit import color

    g = golden("color_stretch.npz")
    out = color.apply_shared_percentile_stretch(g["img"], g["mask"])
    assert out.dtype == np.float32 and np.array_equal(bits(out), bits(g["out"]))
    assert np.array_equal(bits(color.apply_shared_percentile_stretch(g["img"], g["mask"], 1, 99.5)), bits(g["out_1_995"]))
    assert np.array_equal(bits(color.apply_shared_percentile_stretch(g["img"], g["tiny_mask"])), bits(g["tiny"]))
    nout = color.apply_shared_percentile_stretch(g["nanimg"], g["nmask"])
    assert np.array_equal(nout, g["nout"], equal_nan=True)
    lim, _ = color.shared_percentile_limits(g["img"], g["mask"])
    assert np.array_equal(lim, g["limits"])                                  # float64, exact
    with pytest.raises(IndexError):
        color.apply_shared_percentile_stretch(g["img"], np.zeros_like(g["mask"]))
    t = color.apply_shared_percentile_stretch(dev(g["img"]), dev(g["mask"]))  # CUDA in -> CUDA out
    assert t.is_cuda and np.array_equal(bits(t), bits(g["out"]))


@pytest.mark.parametrize("n,groups", [(1, 1), (2, 1), (3, 1), (257, 1), (4099, 1), (64 * 64, 4), (300 * 300 + 7, 1),
                                      (10007, 3)])
def test_masked_percentiles_exact_vs_numpy(n, groups):
    rng = np.random.default_rng(n + groups)
    K = 3
    for kind in range(5):
        x = (rng.random((K, groups, n)) ** 2).astype(np.float32)
        if kind == 1:
            x = np.round(x * 20).astype(np.float32) / 20                       # ties, many equal to 0
        if kind == 2:
            x = rng.normal(0, 1e3, size=x.shape).astype(np.float32)             # negatives, wide range
            x[rng.random(x.shape) < 0.01] = np.inf
            x[rng.random(x.shape) < 0.01] = -np.inf
            x[rng.random(x.shape) < 0.02] = -0.0
        if kind == 3:
            x = (rng.integers(0, 2 ** 32, size=x.shape, dtype=np.uint64).astype(np.uint32)).view(np.float32)
            x[np.isnan(x)] = 1.0                                               # any finite / infinite bit pattern
        if kind == 4 and n > 3:
            x[1, 0, rng.integers(n)] = np.nan                                  # NaN poisons that series only
        mask = rng.random((groups, n)) < (0.6 if n > 3 else 2.0)
        mask[:, 0] = True
        for padded in (False, True):
            xt = kernels.alloc_planes(K, (groups, n), DEV) if padded else torch.empty(x.shape, dtype=torch.float32, device=DEV)
            xt.copy_(dev(x))
            for q in ([2, 98], [0, 100], [50, 99.9], [98, 2]):
                got = kernels.masked_percentiles(xt, dev(mask), q, groups=groups).cpu().numpy()
                for k in range(K):
                    for g_ in range(groups):
                        with np.errstate(invalid="ignore"):
                            want = np.percentile(x[k, g_][mask[g_]], q)
                        assert np.array_equal(got[k, g_], want, equal_nan=True), (kind, k, g_, q, got[k, g_], want)
            got = kernels.masked_percentiles(xt, None, [2, 98], groups=groups).cpu().numpy()   # no mask
            with np.errstate(invalid="ignore"):
                want = np.percentile(x, [2, 98], axis=-1).transpose(1, 2, 0)
            assert np.array_equal(got, want, equal_nan=True)
    empty = kernels.masked_percentiles(xt, dev(np.zeros((groups, n), bool)), [2, 98], groups=groups)
    assert torch.isnan(empty).all()


@pytest.mark.parametrize("deg", [2, 4])
def test_fit_and_apply_with_fused_stretch_vs_oracle(deg):
    """The script's order (poly_regression.py:106-139): mask -> shared percentile stretch of both images
    -> fit -> apply, with the stretch applied on the fly inside the moment and apply kernels."""
    rng = np.random.default_rng(17 + deg)
    K, H, Wd = 3, 83, 61
    x = (rng.random((K, H, Wd)) ** 2 * 0.5).astype(np.float32)
    cs = np.array([[-0.3, 1.1, 0.02], [0.25, 0.8, 0.0], [-0.1, 0.9, 0.05]])
    y = np.stack([np.polyval(cs[k], x[k].astype(np.float64)) for k in range(K)]) * 0.8
    y = (y + rng.normal(0, 0.004, y.shape)).astype(np.float32)
    x[0, 5, 5] = np.nan
    y[2, 9, 9] = np.inf
    valid = rng.random((H, Wd)) < 0.85
    fm = opoly.fit_mask(x, valid, 0, 0.0) & np.isfinite(y).all(0)               # :106, :118
    xi, yi = np.moveaxis(x, 0, -1), np.moveaxis(y, 0, -1)
    with np.errstate(invalid="ignore"):
        xn = ocolor.apply_shared_percentile_stretch(xi, fm)                      # :126-127
        yn = ocolor.apply_shared_percentile_stretch(yi, fm)
    want_c = opoly.fit_poly_rgb_paired(xn, yn, fm, deg)
    want_out = opoly.apply_poly_rgb(xn, want_c, fm)
    xt, yt = kernels.alloc_planes(K, (H, Wd), DEV), kernels.alloc_planes(K, (H, Wd), DEV)
    xt.copy_(dev(x))
    yt.copy_(dev(y))
    m = kernels.fit_mask(xt, dev(valid), gate_k=0, gate_gt=0.0, y=yt)
    assert np.array_equal(m.cpu().numpy(), fm)
    xl = kernels.masked_percentiles(xt, m, [2, 98])
    yl = kernels.masked_percentiles(yt, m, [2, 98])
    assert np.array_equal(xl.cpu().numpy().reshape(K, 2), ocolor.shared_percentile_limits(xi, fm))
    assert np.array_equal(bits(kernels.stretch_apply(xt, xl)), bits(np.moveaxis(xn, -1, 0)))
    mom, _ = kernels.fit_moments(xt, yt, m, deg, mask_given=True, x_stretch=xl, y_stretch=yl)
    # moments of the stretched planes, computed from materialised stretched planes, agree bit for bit
    mom2, _ = kernels.fit_moments(kernels.stretch_apply(xt, xl), kernels.stretch_apply(yt, yl), m, deg, mask_given=True)
    assert mom.equal(mom2)
    coeffs, out = kernels.poly_solve_apply(xt, mom, m, deg, min_count=200, x_stretch=xl)
    assert coeff_err(coeffs.view(K, -1), want_c) < COEF_RTOL
    got = out.cpu().numpy()
    assert np.max(np.abs(np.moveaxis(got, 0, -1) - want_out)[np.isfinite(want_out)]) <= APPLY_ATOL
    assert np.array_equal(np.isnan(np.moveaxis(got, 0, -1)), np.isnan(want_out))


# =============================================================================== tiles_helpers
def test_tiles_black_mask_quantize_and_window_walk(golden):
    from hsr_b200 import tiles_helpers
    from oracle import tiles as otiles

    g = golden("tiles.npz")
    tile = g["tile"]
    assert np.array_equal(tiles_helpers.is_black_mask(tile, nodata=-9999.0), g["black_nd"])
    assert np.array_equal(tiles_helpers.is_black_mask(tile), g["black_none"])
    assert np.array_equal(tiles_helpers.is_black_mask(tile, nodata=0.5, masked_val=0.25, nodata_atol=0.3, zero_atol=0.05),
                          g["black_custom"])
    rng = np.random.default_rng(4)
    for shape in ((5, 4, 64, 64), (3, 285, 17, 13), (2, 1, 7, 5)):                    # batches, odd sizes
        T, B, H, Wd = shape
        a = rng.uniform(-0.02, 0.5, size=shape).astype(np.float32)
        kind = rng.integers(0, 5, size=(T, H, Wd))
        a[np.broadcast_to((kind == 1)[:, None], shape)] = -9999.0
        a[np.broadcast_to((kind == 2)[:, None], shape)] = np.float32(-0.01)
        a[np.broadcast_to((kind == 3)[:, None], shape)] = 0.0
        a[:, B // 2][kind == 4] = 0.25                                                # kind 4: not black
        a += (rng.random(shape) < 0.3) * np.float32(2e-7)
        m, cnt = kernels.black_mask(dev(a), -9999.0, want_count=True)
        want = np.stack([otiles.is_black_mask(a[t], nodata=-9999.0) for t in range(T)])
        assert np.array_equal(m.cpu().numpy(), want) and cnt.tolist() == want.reshape(T, -1).sum(1).tolist()
    # quantisation: random + special values, bit-exact
    x = rng.uniform(-0.05, 7.0, size=100003).astype(np.float32)
    x[:14] = [0.0, 0.12345, 1.0, 6.5534, 6.5535, 7.0, -0.01, -9999.0, np.nan, np.inf, 0.00005, 0.00015, 3e5, -3e5]
    x[14:1000] = (rng.integers(0, 65536, 986) + 0.5).astype(np.float32) / np.float32(10000.0)   # near ties
    for nodata in (-9999.0, None):
        got = tiles_helpers.quantize_emit_u16(x, nodata=nodata)
        assert got.dtype == np.uint16 and np.array_equal(got, otiles.quantize_emit_u16(x, nodata=nodata))
    got = tiles_helpers.quantize_emit_u16(x.reshape(-1)[1:], nodata=-9999.0, emit_scale=1000.0, emit_nodata_u16=255)
    assert np.array_equal(got, otiles.quantize_emit_u16(x[1:], nodata=-9999.0, emit_scale=1000.0, emit_nodata_u16=255))
    # the window walk of find_valid_paired_tiles on in-memory rasters
    emit = rng.uniform(0.01, 0.5, size=(6, 47, 58)).astype(np.float32)
    s2 = rng.uniform(100, 5000, size=(4, 47 * 3, 58 * 3 - 5)).astype(np.float32)       # last tile column falls off S2
    emit[:, :12, :12] = -9999.0
    emit[:, 20:23, 30] = np.float32(-0.01)
    s2[:, 60:65, 40:50] = 0.0
    for frac, cap in ((0.0, None), (0.05, None), (1.0, 5)):
        a = tiles_helpers.find_valid_paired_tiles_arrays(emit, s2, 10, 3, frac, cap, emit_nodata=-9999.0)
        b = otiles.find_valid_paired_tiles_arrays(emit, s2, 10, 3, frac, cap, emit_nodata=-9999.0)
        assert a == b and (cap is None or len(a) == cap)
    sub, idx = tiles_helpers.subsample_bands(dev(np.arange(285 * 6, dtype=np.float32).reshape(285, 2, 3)), 32)
    assert np.array_equal(idx, g["idx_285_32"]) and sub.shape == (32, 2, 3) and float(sub[5, 0, 0]) == idx[5] * 6


@pytest.mark.parametrize("kind", ["rotation", "identity", "upsample"])
@pytest.mark.parametrize("nodata", [-9999.0, None])
def test_fused_tile_export_equals_gather_quantize_black(kind, nodata):
    """hsr_glt_ortho_u16 == hsr_glt_ortho_f32 -> hsr_quantize_u16_f32 / hsr_black_mask_f32 (and the oracle), bit for bit."""
    from oracle import tiles as otiles

    rng = np.random.default_rng(11)
    Hr, Wr, B = 61, 47, 285
    raw = rng.uniform(-0.02, 0.9, size=(Hr, Wr, B)).astype(np.float32)
    raw[5:9, 5:9, :] = np.float32(-0.01)                 # EMIT masked reflectance
    raw[12:15, 20:25, :] = 0.0                           # true black
    raw[30, 30, :] = -9999.0                             # nodata inside the raw cube
    raw[31, 31, 7] = np.nan
    raw[32, 32, 100] = np.inf
    raw[33, 33, :] = 7.5                                 # above the uint16 range
    raw[34, 34, 3] = 3e5                                 # product beyond int32
    raw[35, 35, :] = np.float32(-0.0104)                 # ~ masked value within tolerance
    if kind == "rotation":
        gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
        gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=3, hole_frac=0.01, n_oob=4, n_neg=4)
    elif kind == "identity":
        gx, gy = synthetic.identity_glt(Hr, Wr, 0.02, seed=4)
    else:
        yy, xx = np.mgrid[0:Hr * 2, 0:Wr * 3]
        gx, gy = (xx // 3 + 1).astype(np.int32), (yy // 2 + 1).astype(np.int32)
    ortho, vref, dref = oglt.glt_ortho(raw, gx, gy)
    bsq = np.ascontiguousarray(np.moveaxis(ortho, -1, 0))
    q, valid, black, diag = kernels.glt_ortho_u16(dev(raw), dev(gx), dev(gy), nodata=nodata)
    assert q.dtype == torch.uint16 and tuple(q.shape) == bsq.shape
    got = q.cpu().view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(got, otiles.quantize_emit_u16(bsq, nodata=nodata))
    assert np.array_equal(valid.cpu().numpy(), vref)
    assert np.array_equal(black.cpu().numpy(), otiles.is_black_mask(bsq, nodata=nodata))
    assert diag.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    # the un-fused kernels agree as well
    o2, _, _ = kernels.glt_ortho(dev(raw), dev(gx), dev(gy))
    cube = o2.permute(2, 0, 1).contiguous()
    assert torch.equal(kernels.quantize_u16(cube, nodata).view(torch.int16), q.contiguous().view(torch.int16))
    assert torch.equal(kernels.black_mask(cube, nodata), black)
    q2 = kernels.glt_ortho_u16(dev(raw), dev(gx), dev(gy), nodata=nodata, scale=1000.0, nodata_u16=255, want_black=False)[0]
    assert np.array_equal(q2.cpu().view(torch.int16).numpy().view(np.uint16),
                          otiles.quantize_emit_u16(bsq, nodata=nodata, emit_scale=1000.0, emit_nodata_u16=255))


def test_block_average_downsample_vs_oracle():
    """S2 10 m -> 60 m "average" on aligned grids (notebook cell 73 / poly_regression.py:110-116): block mean in float64,
    nodata excluded, empty blocks 0, then * src_scale — against oracle/resample.py, bit for bit (parity with GDAL unpinned)."""
    from hsr_b200.s2_emit import resample
    from oracle import resample as oresample

    rng = np.random.default_rng(21)
    u8 = rng.integers(0, 256, size=(3, 6 * 37 + 4, 6 * 29 + 1), dtype=np.uint8)          # TCI-like, ragged edges dropped
    got = resample.downsample_to_grid(u8, 6, src_scale=1.0 / 255.0)
    assert got.dtype == np.float32 and got.shape == (3, 37, 29)
    assert np.array_equal(bits(got), bits(oresample.downsample_to_grid(u8, 6, src_scale=1.0 / 255.0)))
    u16 = rng.integers(0, 12000, size=(10, 6 * 20, 6 * 33), dtype=np.uint16)
    u16[:, :12, :18] = 0                                                                 # nodata blocks (all) and partial ones
    u16[:, 30:33, 40:45] = 0
    for nodata in (0, None):
        got = resample.downsample_to_grid(u16, 6, nodata=nodata)
        assert np.array_equal(bits(got), bits(oresample.downsample_to_grid(u16, 6, nodata=nodata)))
    assert (got[:, :2, :3] == 0).all()
    f32 = rng.normal(0, 1, size=(2, 50, 70)).astype(np.float32)
    f32[0, 3, 3] = np.nan
    for f in (1, 2, 5, 7):
        got = resample.downsample_to_grid(f32, f, src_scale=0.5)
        assert np.array_equal(bits(got), bits(oresample.downsample_to_grid(f32, f, src_scale=0.5)))
    t = kernels.block_average(dev(u16.view(np.int16)).view(torch.uint16), 6, nodata=0)      # CUDA in -> CUDA out
    assert t.is_cuda and np.array_equal(bits(t), bits(oresample.downsample_to_grid(u16, 6, nodata=0)))


def test_bilinear_upsample_vs_oracle():
    """pseudo-S2 planes 60 m -> 10 m, bilinear on aligned grids (notebook cell 73 / poly_regression.py:150-156)
    against oracle/resample.py (parity with GDAL unpinned): exact at block centres of constants, renormalised at the
    borders and around nodata / NaN."""
    from hsr_b200.s2_emit import resample
    from oracle import resample as oresample

    rng = np.random.default_rng(23)
    a = rng.random((3, 23, 31)).astype(np.float32)
    a[1, 5, 5] = np.nan
    a[2, 10:12, 7:9] = -9999.0
    for f, nodata in ((6, None), (6, -9999.0), (1, None), (3, -9999.0)):
        got = resample.upsample_to_grid(a, f, nodata=nodata)
        want = oresample.upsample_to_grid(a, f, nodata=nodata)
        assert got.shape == (3, 23 * f, 31 * f) and got.dtype == np.float32
        ok = np.isfinite(want)
        assert np.array_equal(np.isnan(got), np.isnan(want)) and np.max(np.abs(got[ok] - want[ok])) <= 1e-6
    const = np.full((1, 4, 5), 0.37, np.float32)
    assert np.allclose(resample.upsample_to_grid(const, 6), 0.37, atol=1e-7)
    ramp = np.broadcast_to(np.arange(8, dtype=np.float32)[None, None, :], (1, 3, 8)).copy()
    up = resample.upsample_to_grid(ramp, 2)[0, 0]
    assert np.allclose(up[1:-1], (np.arange(16)[1:-1] + 0.5) / 2 - 0.5, atol=1e-6) and up[0] == 0 and up[-1] == 7
    assert np.array_equal(resample.upsample_to_grid(a, 1), np.nan_to_num(a, nan=0.0))      # factor 1: identity, NaN -> 0


def test_reference_script_sequence_end_to_end():
    """The reference's pair-synthesis script (s2_emit/poly_regression.py:97-162) as one call, every stage on the GPU,
    against the same sequence composed from the oracle: SRF -> mask -> S2 average to 60 m -> shared percentile stretch
    -> OT-target polynomial fit -> apply -> bilinear to 10 m -> stretch -> apply."""
    from hsr_b200.s2_emit import match_pair_rgb
    from oracle import ot as oot
    from oracle import resample as oresample

    rng = np.random.default_rng(31)
    H, Wd, f = 48, 56, 6
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = srf.synthetic_s2_srf()
    R = synthetic.raw_cube_spectra_np((H, Wd, 285), seed=5, good=good)
    R[:4, :, :] = -9999.0                                   # fill rows: rejected by emit[B2] > 0
    R[10, 10, 50] = np.nan
    base = np.kron(rng.random((3, H, Wd)), np.ones((1, f, f)))
    s2 = np.clip(255 * (0.15 + 0.7 * base + 0.03 * rng.normal(size=base.shape)), 0, 255).astype(np.uint8)
    got = match_pair_rgb(R, w, table, good, s2, factor=f, deg=2, n_samples=500, seed=0)
    # ---- the oracle composition, line by line
    ps = osrf.pseudo_s2_srf_integral(R, w, table, good)
    emit_sim = np.stack([ps[b] for b in ("B2", "B3", "B4")], axis=0).astype(np.float32)
    with np.errstate(invalid="ignore"):
        valid60 = np.isfinite(emit_sim).all(axis=0) & (emit_sim[0] > 0)
    s2_60 = oresample.downsample_to_grid(s2, f, src_scale=1.0 / 255.0)
    valid60 = valid60 & np.isfinite(s2_60).all(axis=0)
    assert valid60.any() and not valid60[:4].any() and not valid60[10, 10]
    assert np.array_equal(got["valid60"], valid60) and np.array_equal(bits(got["s2_real_60m"]), bits(s2_60))
    assert_srf_close(got["emit_sim_60m"], emit_sim)
    # from here on the GPU planes are the inputs (the stretch is an exact function of them)
    esim = got["emit_sim_60m"]
    emit_rgb = np.transpose(esim[[2, 1, 0]], (1, 2, 0))
    s2_rgb = np.transpose(s2_60, (1, 2, 0))
    with np.errstate(invalid="ignore"):
        emit_rgb_n = ocolor.apply_shared_percentile_stretch(emit_rgb, valid60)
        s2_rgb_n = ocolor.apply_shared_percentile_stretch(s2_rgb, valid60)
    assert np.array_equal(got["emit_rgb_n"], emit_rgb_n, equal_nan=True) and np.array_equal(bits(got["s2_rgb_n"]), bits(s2_rgb_n))
    coeffs = oot.fit_ot_poly_rgb(emit_rgb_n, s2_rgb_n, valid60, deg=2, n_samples=500, seed=0)
    assert coeff_err(got["coeffs"], coeffs) < COEF_RTOL
    m60 = opoly.apply_poly_rgb(emit_rgb_n, coeffs, valid60)
    ok = np.isfinite(m60)
    assert np.array_equal(np.isnan(got["matched_60m"]), np.isnan(m60)) and np.max(np.abs(got["matched_60m"] - m60)[ok]) <= APPLY_ATOL
    up = oresample.upsample_to_grid(esim, f)
    ok = np.isfinite(up)
    assert np.max(np.abs(got["emit_sim_10m"] - up)[ok]) <= 1e-6 * max(1.0, float(np.abs(up[ok]).max()))
    mask10 = np.isfinite(got["emit_sim_10m"]).all(axis=0)
    assert np.array_equal(got["mask10"], mask10)
    rgb10 = np.transpose(got["emit_sim_10m"][[2, 1, 0]], (1, 2, 0))
    with np.errstate(invalid="ignore"):
        rgb10_n = ocolor.apply_shared_percentile_stretch(rgb10, mask10)
    m10 = opoly.apply_poly_rgb(rgb10_n, np.asarray(got["coeffs"]), mask10)
    assert np.max(np.abs(got["matched_10m"] - m10)) <= APPLY_ATOL and got["matched_10m"].shape == (H * f, Wd * f, 3)


# =============================================================================== the fused pass
def _small_granule(seed=0, Hr=90, Wr=71):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=good)
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=seed + 1, hole_frac=0.002, n_oob=4, n_neg=4)
    return w, good, raw, gx, gy


def _oracle_pass(raw, gx, gy, w, good, table, s2, deg, min_count=200):
    ortho, valid, _ = oglt.glt_ortho(raw, gx, gy)
    ps = osrf.pseudo_s2_srf_integral(ortho, w, table, good)
    names = [b for b in table if ps[b] is not None]
    x = np.stack([ps[b] for b in names]).astype(np.float32)
    fm = opoly.fit_mask(x, valid, 0, 0.0)
    coeffs = opoly.polyfit_paired(x, s2, fm, deg, min_count=min_count)
    matched = opoly.apply_poly_planes(x, coeffs, fm)
    return x, valid, fm, coeffs, matched


def test_pair_synthesis_granule_vs_oracle():
    w, good, raw, gx, gy = _small_granule()
    table = srf.synthetic_s2_srf()
    ps = PairSynthesizer(w, table, good, deg=2, device=DEV)
    assert ps.band_names == [b for b in srf.S2_BANDS_13 if b != "B10"]
    bands0, _, _, _ = ps.bands_from_raw(dev(raw), dev(gx), dev(gy))
    s2 = synthetic.s2_reference_np(np.nan_to_num(bands0.cpu().numpy()), seed=1)
    res = ps.synthesize(dev(raw), dev(gx), dev(gy), dev(s2))
    x, valid, fm, coeffs, matched = _oracle_pass(raw, gx, gy, w, good, table, s2, 2)
    assert np.array_equal(res.valid.cpu().numpy(), valid)
    assert_srf_close(res.bands, x)
    assert np.array_equal(res.fit_mask.cpu().numpy(), fm)
    assert coeff_err(res.coeffs, coeffs) < COEF_RTOL
    got = res.matched.cpu().numpy()
    # unmasked fill pixels are clipped to 0 like any other pixel (poly_regression.py:84)
    assert np.max(np.abs(got - matched)) <= APPLY_ATOL
    assert (got[:, ~valid] == 0).all()


def test_pair_synthesis_with_stretch_vs_oracle():
    """PairSynthesizer(stretch=(2, 98), y_finite=True): the order of the reference's script,
    poly_regression.py:104-139, on all K planes."""
    w, good, raw, gx, gy = _small_granule(seed=3)
    table = srf.synthetic_s2_srf()
    ps = PairSynthesizer(w, table, good, deg=2, stretch=(2, 98), y_finite=True, device=DEV)
    bands0, _, _, _ = ps.bands_from_raw(dev(raw), dev(gx), dev(gy))
    s2 = synthetic.s2_reference_np(np.nan_to_num(bands0.cpu().numpy()), seed=1)
    x, valid, fm0, _, _ = _oracle_pass(raw, gx, gy, w, good, table, s2, 2)
    iy, ix = np.argwhere(fm0)[len(np.argwhere(fm0)) // 2]
    s2[4, iy, ix] = np.nan                              # a non-finite reference pixel inside the fit mask
    res = ps.synthesize(dev(raw), dev(gx), dev(gy), dev(s2))
    fm = fm0 & np.isfinite(s2).all(0)
    assert np.array_equal(res.fit_mask.cpu().numpy(), fm) and fm0.sum() > fm.sum()
    xg = res.bands.cpu().numpy()                       # stretch limits are exact functions of the planes we produced
    xi, yi = np.moveaxis(xg, 0, -1), np.moveaxis(s2, 0, -1)
    assert np.array_equal(res.x_limits.cpu().numpy().reshape(-1, 2), ocolor.shared_percentile_limits(xi, fm))
    assert np.array_equal(res.y_limits.cpu().numpy().reshape(-1, 2), ocolor.shared_percentile_limits(yi, fm))
    with np.errstate(invalid="ignore"):
        xn = ocolor.apply_shared_percentile_stretch(xi, fm)
        yn = ocolor.apply_shared_percentile_stretch(yi, fm)
    coeffs = opoly.fit_poly_rgb_paired(xn, yn, fm, 2)
    assert coeff_err(res.coeffs, coeffs) < COEF_RTOL
    want = opoly.apply_poly_rgb(xn, coeffs, fm)
    got = np.moveaxis(res.matched.cpu().numpy(), 0, -1)
    ok = np.isfinite(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.max(np.abs(got - want)[ok]) <= APPLY_ATOL


def test_host_granule_stream_equals_direct_pass():
    """HostGranuleStream (pinned host buffers, three streams, two slots) returns exactly what synthesize()
    returns for every granule, in submission order, also when slots are reused."""
    from hsr_b200.pipeline import HostGranuleStream

    table = srf.synthetic_s2_srf()
    gran = []
    for seed in range(5):
        w, good, raw, gx, gy = _small_granule(seed=seed)
        gran.append((raw, gx, gy))
    ps = PairSynthesizer(w, table, good, deg=2, device=DEV)
    Ho, Wo = gran[0][1].shape
    hs = HostGranuleStream(ps, gran[0][0].shape, (Ho, Wo), depth=2)
    outs, want = [], []
    for raw, gx, gy in gran:
        bands0, _, _, _ = ps.bands_from_raw(dev(raw), dev(gx), dev(gy))
        s2 = synthetic.s2_reference_np(np.nan_to_num(bands0.cpu().numpy()), seed=1)
        want.append(ps.synthesize(dev(raw), dev(gx), dev(gy), dev(s2)))
        out = hs.host_buffers()
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()  # noqa: E731
        hs.submit(pin(raw), pin(gx), pin(gy), pin(s2), out)
        outs.append(out)
    hs.drain()
    torch.cuda.synchronize()
    for out, res in zip(outs, want):
        assert np.array_equal(out["valid"].numpy(), res.valid.cpu().numpy())
        assert np.array_equal(out["coeffs"].numpy(), res.coeffs.cpu().numpy())
        got = out["matched"][:, :Ho * Wo].reshape(ps.K, Ho, Wo)
        assert np.array_equal(bits(got), bits(res.matched))


def test_pair_synthesis_tiles_vs_oracle():
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = srf.synthetic_s2_srf()
    T, h = 5, 24
    ps = PairSynthesizer(w, table, good, deg=2, min_count=50, device=DEV)
    raws = np.stack([synthetic.raw_cube_spectra_np((h, h, 285), seed=20 + t, good=good) for t in range(T)])
    glts = [synthetic.identity_glt(h, h, 0.02, seed=2 + t) for t in range(T)]
    gx = np.stack([g[0] for g in glts])
    gy = np.stack([g[1] for g in glts])
    gy[1, 0, 0] = h + 3                                            # out of ITS tile: dropped, must not read tile 2
    s2 = np.empty((12, T, h, h), np.float32)
    per_tile = []
    for t in range(T):
        ortho, valid, _ = oglt.glt_ortho(raws[t], gx[t], gy[t])
        psr = osrf.pseudo_s2_srf_integral(ortho, w, table, good)
        x = np.stack([psr[b] for b in ps.band_names]).astype(np.float32)
        s2[:, t] = synthetic.s2_reference_np(x, seed=50 + t)
        fm = opoly.fit_mask(x, valid, 0, 0.0)
        coeffs = opoly.polyfit_paired(x, s2[:, t], fm, 2, min_count=50)
        per_tile.append((x, valid, fm, coeffs, opoly.apply_poly_planes(x, coeffs, fm)))
    res = ps.synthesize_tiles(dev(raws), dev(gx), dev(gy), dev(s2))
    for t, (x, valid, fm, coeffs, matched) in enumerate(per_tile):
        assert np.array_equal(res.valid[t].cpu().numpy(), valid)
        assert_srf_close(res.bands[:, t], x)
        assert np.array_equal(res.fit_mask[t].cpu().numpy(), fm)
        assert coeff_err(res.coeffs[:, t], coeffs) < COEF_RTOL
        assert np.max(np.abs(res.matched[:, t].cpu().numpy() - matched)) <= APPLY_ATOL
    assert not res.valid[1, 0, 0]


def test_pair_synthesis_sharded_equals_single_global_fit():
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = srf.synthetic_s2_srf()
    ps = PairSynthesizer(w, table, good, deg=2, device=DEV)
    granules = []
    for s in range(3):
        _, _, raw, gx, gy = _small_granule(seed=100 + s, Hr=48, Wr=40)
        b, _, _, _ = ps.bands_from_raw(dev(raw), dev(gx), dev(gy))
        s2 = synthetic.s2_reference_torch(b, seed=s)
        granules.append({"raw": dev(raw), "glt_x": dev(gx), "glt_y": dev(gy), "s2_ref": s2})
    res = ps.synthesize_sharded(granules)
    xs = np.concatenate([r.bands.cpu().numpy().reshape(12, -1) for r in res], axis=1)
    ys = np.concatenate([g["s2_ref"].cpu().numpy().reshape(12, -1) for g in granules], axis=1)
    ms = np.concatenate([r.fit_mask.cpu().numpy().reshape(-1) for r in res])
    ref = opoly.polyfit_paired(xs, ys, ms, 2)
    assert coeff_err(res[0].coeffs, ref) < COEF_RTOL
    assert all(r.coeffs.equal(res[0].coeffs) for r in res)


# =============================================================================== full size properties
def test_full_granule_properties():
    """BASELINE config 1/2 at full size: 1280 x 1242 x 285 raw, 25-degree GLT -> 1685 x 1667 ortho."""
    Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, DEV, good)
    gx_np, gy_np = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx_np, gy_np = synthetic.inject_glt_defects(gx_np, gy_np, Hr, Wr)
    gx, gy = dev(gx_np), dev(gy_np)
    Ho, Wo = gx_np.shape
    assert (Ho, Wo) == (1685, 1667)
    ortho, valid, diag = kernels.glt_ortho(raw, gx, gy)
    # (a) bit-exact against an independent gather (torch advanced indexing) on the same device
    _, _, vref, dref = oglt.glt_validity(oglt.glt_to_int32(gx_np, gy_np), Hr, Wr)
    assert np.array_equal(valid.cpu().numpy(), vref)
    assert diag.tolist() == [dref["valid_glt_count"], dref["valid_glt_inbounds_count"], dref["valid_glt_dropped_oob"]]
    vt = valid
    src = raw[(gy[vt] - 1).long(), (gx[vt] - 1).long()]
    assert torch.equal(ortho[vt].view(torch.int32), src.view(torch.int32))
    assert ortho[~vt].eq(-9999.0).all()
    del src
    # (b) idempotence / determinism
    ortho2, _, _ = kernels.glt_ortho(raw, gx, gy)
    assert torch.equal(ortho.view(torch.int32), ortho2.view(torch.int32))
    del ortho2
    # (c) fused SRF == un-fused SRF of the materialised cube, and linear in the weights
    table = srf.synthetic_s2_srf()
    W, names, _, fill_out = srf.srf_fold_weights(w, table, good)
    Wd, fo = dev(W), dev(fill_out)
    bands, v2, _, _ = kernels.glt_srf(raw, gx, gy, Wd, fo)
    assert v2.equal(valid)
    unf = kernels.srf_integrate(ortho, Wd)
    assert torch.equal(bands.view(torch.int32), unf.view(torch.int32))
    del unf
    half, _, _, _ = kernels.glt_srf(raw, gx, gy, Wd * 0.5, fo * 0.5)
    assert torch.equal(half.view(torch.int32), (bands * 0.5).view(torch.int32))   # scaling by 2^-1 is exact
    # (d) against float64 matmul on a strip of rows
    rows = slice(800, 816)
    ref = (ortho[rows].double() @ Wd.double()).permute(2, 0, 1)
    got = bands[:, rows].double()
    vm = valid[rows]
    rel = ((got - ref).abs() / ref.abs().clamp_min(1e-2))[:, vm]
    assert rel.max().item() < 1e-5
    # (e) polynomial fit recovers the planted coefficients; apply is idempotent under identity coefficients
    s2 = synthetic.s2_reference_torch(bands, seed=1)
    fm = kernels.fit_mask(bands, valid)
    coeffs = kernels.poly_fit(bands, s2, fm, 2)
    planted = torch.tensor([[-0.3 + 0.02 * k, 1.1, 0.02] for k in range(len(names))], dtype=torch.float64)
    assert (coeffs.cpu() - planted).abs().max().item() < 2e-3     # noise 0.005 over ~1.6 M samples
    ident = torch.zeros_like(coeffs)
    ident[:, -2] = 1.0
    same = kernels.poly_apply(bands, ident, fm, lo=1.0, hi=0.0)
    assert torch.equal(same[:, fm].view(torch.int32), bands[:, fm].view(torch.int32))


def _free_gb():
    free, _ = torch.cuda.mem_get_info()
    return free / 2 ** 30


def test_full_tile_batch_properties():
    """BASELINE config 3 at full size: 512 paired 256 x 256 x 285 tiles (38 GB of raw tiles) through ortho + SRF +
    per-tile fit + apply in one launch per stage.  Properties: a sub-batch run alone gives bit-identical planes and
    masks and the same fit to rounding (tiles are independent; the reduction tree depends on how many blocks a
    series gets, so the fp64 sums agree to ~1e-15, not bit for bit); planted per-tile polynomials are recovered."""
    T, h, B = 512, 256, 285
    if _free_gb() < 60:
        pytest.skip("needs ~50 GB of free HBM")
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    ps = PairSynthesizer(w, srf.synthetic_s2_srf(), good, deg=2, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    raw = torch.empty((T, h, h, B), dtype=torch.float32, device=DEV)
    for t0 in range(0, T, 64):                                     # albedo x smooth spectrum + noise, 64 tiles at a time
        a = torch.rand((64, h, h, 1), generator=g, device=DEV) * 0.7 + 0.05
        raw[t0:t0 + 64] = a * (0.6 + 0.4 * torch.sin(0.02 * torch.arange(B, device=DEV))) \
            + 0.02 * (torch.rand((64, h, h, B), generator=g, device=DEV) - 0.5)
        del a
    ii = torch.arange(h, device=DEV, dtype=torch.int32)
    gy = (ii.view(1, h, 1) + 1).expand(T, h, h).contiguous()
    gx = (ii.view(1, 1, h) + 1).expand(T, h, h).contiguous()
    holes = torch.rand((T, h, h), generator=g, device=DEV) < 0.02
    gx[holes] = 0
    bands0 = ps.bands_from_raw(raw.view(T * h, h, B), gx.view(T * h, h),
                               torch.where(gy > 0, gy + (torch.arange(T, device=DEV, dtype=torch.int32) * h).view(T, 1, 1), gy)
                               .view(T * h, h))[0].view(ps.K, T, h, h)
    tile_c = torch.linspace(0.8, 1.2, T, device=DEV).view(1, T, 1, 1)
    s2 = (tile_c * bands0 + 0.01 * (torch.arange(ps.K, device=DEV).view(-1, 1, 1, 1) + 1)).contiguous()
    del bands0
    res = ps.synthesize_tiles(raw, gx, gy, s2)
    torch.cuda.synchronize()
    assert res.valid.shape == (T, h, h) and torch.equal(res.valid, ~holes)
    assert torch.equal(res.fit_mask, res.valid & (res.bands[0] > 0) & torch.isfinite(res.bands).all(0))
    c = res.coeffs.cpu().numpy()                                   # [K, T, 3]: y = c_t x + 0.01 (k + 1) exactly
    want1 = np.broadcast_to(np.linspace(0.8, 1.2, T, dtype=np.float32).astype(np.float64)[None, :], c.shape[:2])
    assert np.max(np.abs(c[..., 0])) < 1e-3 and np.max(np.abs(c[..., 1] - want1)) < 1e-3
    assert np.max(np.abs(c[..., 2] - 0.01 * (np.arange(ps.K)[:, None] + 1))) < 1e-3
    sel = slice(300, 308)                                          # a sub-batch alone: bit-identical
    sub = ps.synthesize_tiles(raw[sel], gx[sel], gy[sel], s2[:, sel].contiguous())
    assert torch.equal(sub.bands.view(torch.int32), res.bands[:, sel].view(torch.int32))
    assert torch.equal(sub.fit_mask, res.fit_mask[sel])
    assert torch.equal(sub.moments[..., 0], res.moments[:, sel][..., 0])                  # counts are exact
    torch.testing.assert_close(sub.moments, res.moments[:, sel], rtol=1e-13, atol=0)
    torch.testing.assert_close(sub.coeffs, res.coeffs[:, sel], rtol=1e-9, atol=1e-12)
    assert (sub.matched - res.matched[:, sel]).abs().max().item() <= 1.2e-7


def test_full_mosaic_slab_sharding_properties():
    """BASELINE config 5 at full size: 8192 x 8192 ortho grid over a 6164 x 6164 x 285 raw mosaic (43 GB), fused
    gather + SRF.  Properties: the 8 row slabs a rank would own (dist.shard_rows) reproduce the un-sharded planes,
    masks and diagnostics bit for bit; a strip agrees with a float64 matmul of gathered spectra."""
    from hsr_b200 import dist as hdist

    if _free_gb() < 70:
        pytest.skip("needs ~55 GB of free HBM")
    Ho = Wo = 8192
    Hr = Wr = 6164
    B = 285
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    W, names, _, fill_out = srf.srf_fold_weights(w, srf.synthetic_s2_srf(), good)
    Wd, fo = dev(W), dev(fill_out)
    g = torch.Generator(device=DEV).manual_seed(5)
    raw = torch.empty((Hr, Wr, B), dtype=torch.float32, device=DEV)
    for r0 in range(0, Hr, 512):
        r1 = min(Hr, r0 + 512)
        raw[r0:r1] = torch.rand((r1 - r0, Wr, B), generator=g, device=DEV) * 0.6
    # 25-degree nearest-neighbour rotation GLT, built on the device (SURVEY 8d)
    th = np.deg2rad(25.0)
    yy = torch.arange(Ho, device=DEV, dtype=torch.float64).view(-1, 1) - (Ho - 1) / 2
    xx = torch.arange(Wo, device=DEV, dtype=torch.float64).view(1, -1) - (Wo - 1) / 2
    rx = torch.round(xx * np.cos(th) + yy * np.sin(th) + (Wr - 1) / 2).to(torch.int64)
    ry = torch.round(-xx * np.sin(th) + yy * np.cos(th) + (Hr - 1) / 2).to(torch.int64)
    inside = (rx >= 0) & (rx < Wr) & (ry >= 0) & (ry < Hr)
    gx = torch.where(inside, rx + 1, torch.zeros_like(rx)).to(torch.int32)
    gy = torch.where(inside, ry + 1, torch.zeros_like(ry)).to(torch.int32)
    del rx, ry, xx, yy
    assert 0.5 < inside.float().mean().item() < 0.6
    bands, valid, diag, _ = kernels.glt_srf(raw, gx, gy, Wd, fo)
    torch.cuda.synchronize()
    assert torch.equal(valid, inside) and diag.tolist() == [int(inside.sum()), int(inside.sum()), 0]
    K = len(names)
    total = torch.zeros(3, dtype=torch.int64, device=DEV)
    for rank in range(8):
        r0, r1 = hdist.shard_rows(Ho, rank, 8)
        assert (r0, r1) == (1024 * rank, 1024 * (rank + 1))
        b, v, d, _ = kernels.glt_srf(raw, gx[r0:r1], gy[r0:r1], Wd, fo)
        assert torch.equal(b.view(torch.int32), bands[:, r0:r1].view(torch.int32)) and torch.equal(v, valid[r0:r1])
        total += d
    assert torch.equal(total, diag)
    rows = slice(4000, 4008)
    vm = valid[rows]
    src = raw[(gy[rows][vm] - 1).long(), (gx[rows][vm] - 1).long()].double() @ Wd.double()      # [n, K]
    got = bands[:, rows][:, vm].double().t()
    assert ((got - src).abs() / src.abs().clamp_min(1e-2)).max().item() < 1e-5
    assert torch.equal(bands[:, rows][:, ~vm], fo.view(K, 1).expand(K, int((~vm).sum())))


def test_abi_argument_errors_are_codes_not_crashes():
    """Every C entry point validates its arguments: a negative HSR_E* code + hsr_last_error(), no launch, no crash."""
    from hsr_b200 import _lib

    lib = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    raw = torch.zeros((4, 4, 285), device=DEV)
    g = torch.ones((4, 4), dtype=torch.int32, device=DEV)
    out = torch.zeros((4, 4, 285), device=DEV)
    W = torch.zeros((285, 3), device=DEV)
    f64 = torch.zeros(64, dtype=torch.float64, device=DEV)
    u8 = torch.zeros(64, dtype=torch.uint8, device=DEV)

    def expect(code, rc, frag):
        assert rc == code, (rc, lib.hsr_last_error())
        assert frag in lib.hsr_last_error().decode()

    p = lambda t: t.data_ptr()  # noqa: E731
    expect(-1, lib.hsr_glt_ortho_f32(None, 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None, None, st), "null")
    expect(-1, lib.hsr_glt_ortho_f32(p(raw), 4, 4, 285, 200, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None, None, st),
           "raw_pix_stride")
    expect(-2, lib.hsr_glt_ortho_f32(p(raw) + 2, 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None, None, st),
           "aligned")
    expect(-3, lib.hsr_glt_ortho_f32(p(raw), 1 << 20, 1 << 20, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None,
                                     None, None, st), "2^31")
    expect(-3, lib.hsr_glt_srf_f32(p(raw), 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(W), p(W), 17, p(out), 16, None,
                                   285, None, None, None, -1, 0.0, None, st), "K = 17")
    expect(-1, lib.hsr_glt_srf_f32(p(raw), 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(W), p(W), 3, p(out), 8, None,
                                   285, None, None, None, -1, 0.0, None, st), "bands_plane_stride")
    import ctypes
    view = _lib.RawView(2, 3, 0, 0)                                 # rows [2, 5) of a 4-row cube
    expect(-1, lib.hsr_glt_ortho_f32(p(raw), 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None,
                                     ctypes.byref(view), st), "raw view")
    view = _lib.RawView(0, 0, 3, 3)                                 # 4 ortho rows are not whole 3-row tiles
    expect(-1, lib.hsr_glt_ortho_f32(p(raw), 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None,
                                     ctypes.byref(view), st), "tile batch")
    view = _lib.RawView(0, 0, 2, 2)
    expect(-1, lib.hsr_glt_ortho_f32(p(raw), 4, 4, 285, 285, 1, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None,
                                     ctypes.byref(view), st), "transpose")
    expect(-3, lib.hsr_poly_moments_f64(p(out), 16, 1, p(out), 16, 1, None, 1, 1, 16, 3, 9, p(f64), p(f64), st), "deg = 9")
    expect(-1, lib.hsr_fit_moments_f64(p(out), 16, 16, p(out), 16, 16, None, 16, 3, 1, 2, 0, 0.0, 1, None, None, None,
                                       p(f64), p(f64), None, st), "HSR_FIT_MASK_GIVEN")
    expect(-1, lib.hsr_fit_moments_f64(p(out), 16, 16, p(out), 16, 16, None, 16, 3, 1, 2, 5, 0.0, 0, None, None, p(u8),
                                       p(f64), p(f64), None, st), "gate_k")
    import ctypes
    bad_ex = _lib.Exchange(p(f64), p(f64), 17, 0, 1)                # more ranks than a peer block has slots
    expect(-3, lib.hsr_fit_moments_f64(p(out), 16, 16, p(out), 16, 16, p(u8), 16, 3, 1, 2, 0, 0.0, 1, None, None, None,
                                       p(f64), p(f64), ctypes.byref(bad_ex), st), "exchange")
    bad_ex = _lib.Exchange(None, p(f64), 2, 0, 0)                   # no peer table
    expect(-1, lib.hsr_poly_solve_apply_f32(p(out), 16, 16, p(f64), None, 16, 3, 1, 2, 0, 0.0, 1.0, None, p(f64), p(out), 16,
                                            16, ctypes.byref(bad_ex), None, st), "exchange")
    expect(-1, lib.hsr_block_average_f32(p(u8), 3, 1, 8, 8, 64, 2, 0, 0.0, 0, 1.0, p(out), 16, st), "src_dtype")
    wsp = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    expect(-3, lib.hsr_masked_percentiles_f64(p(out), 16, 16, None, 16, 3, 1, p(f64), 3, p(wsp), p(f64), st), "Q = 3")
    expect(-3, lib.hsr_masked_percentiles_f64(p(out), 16, 16, None, 1 << 32, 3, 1, p(f64), 2, p(wsp), p(f64), st), "2^32")
    expect(-1, lib.hsr_masked_percentiles_pair_f64(p(out), 16, 16, p(out), 16, 16, None, 16, 3, 1, p(f64), 2, p(wsp), p(f64),
                                                   None, st), "together")
    expect(-3, lib.hsr_sinkhorn_barycentric_f64(p(f64), p(f64), 4, 4, 5, 0.05, 10, 1e-6, p(f64), p(f64), None, st), "C = 5")
    expect(-1, lib.hsr_sinkhorn_barycentric_f64(p(f64), p(f64), 4, 4, 3, 0.0, 10, 1e-6, p(f64), p(f64), None, st), "reg")
    expect(-3, lib.hsr_quantize_u16_f32(p(out), 16, 0, 0.0, 1e4, 70000, p(u8), st), "nodata_u16")
    expect(-1, lib.hsr_tile_sums_u8(p(u8), 8, 8, 4, 4, 3, 2, p(f64), st), "do not fit")
    torch.cuda.synchronize()                                       # nothing was launched, nothing is broken
    assert lib.hsr_glt_ortho_f32(p(raw), 4, 4, 285, 285, 0, p(g), p(g), 4, 4, 4, -9999.0, p(out), 285, None, None, None, st) == 0
    torch.cuda.synchronize()
    with pytest.raises(_lib.HsrError, match="K = 17"):
        kernels.glt_srf(raw, g, g, torch.zeros((285, 17), device=DEV))


# =============================================================================== file-level driver (nc_to_envi)
class _FakeVar:
    def __init__(self, arr, dims=None):
        self.arr, self.dimensions, self.shape = arr, dims, arr.shape

    def __getitem__(self, idx):
        return self.arr[idx]

    def set_auto_maskandscale(self, flag):
        self.masked = flag


class _FakeGroup:
    def __init__(self, **vars_):
        self.variables = {k: _FakeVar(v) for k, v in vars_.items()}


class _FakeNC:
    """The slice of the netCDF4.Dataset API that nc_to_envi uses (EMIT_data/emit_proj.py:607-687)."""

    def __init__(self, name, cube, dims, glt_x, glt_y, w, gt, extra_loc=None):
        self.variables = {name: _FakeVar(cube, dims)}
        self.groups = {"sensor_band_parameters": _FakeGroup(wavelengths=w, fwhm=np.full_like(w, 7.4)),
                       "location": _FakeGroup(glt_x=glt_x, glt_y=glt_y, **(extra_loc or {}))}
        self._attrs = {"geotransform": gt, "time_coverage_start": "2023-08-19T11:01:26+0000"}
        self.closed = False

    def ncattrs(self):
        return list(self._attrs)

    def getncattr(self, k):
        return self._attrs[k]

    def close(self):
        self.closed = True


@pytest.mark.parametrize("transposed", [False, True])
def test_nc_to_envi_driver_with_reference_signature(tmp_path, monkeypatch, transposed):
    """nc_to_envi / convert_emit_nc_to_envi (reference signatures, emit_proj.py:563-578, :1303-1314) on a fake netCDF
    dataset: the ENVI cube on disk is the oracle's ortho cube bit for bit (band-interleaved-by-line), LOC / OBS planes
    follow, outputs are skipped when they exist, the GLT diagnostics land in `info`."""
    from hsr_b200.EMIT_data import nc_export

    Hr, Wr, B = 40, 33, 285
    w = synthetic.emit_wavelengths()
    raw = synthetic.raw_cube_bits_np((Hr, Wr, B), seed=3, good=synthetic.good_band_mask(w))
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=2, n_oob=3, n_neg=3)
    gxf, gyf = gx.astype(np.float64), gy.astype(np.float64)
    gxf[0, 0] = np.nan                                            # float GLT with NaN, as in the product
    lon, lat = np.random.default_rng(0).random((2, Hr, Wr)).astype(np.float32)
    obs = np.random.default_rng(1).random((Hr, Wr, 3)).astype(np.float32)
    cube_file = np.transpose(raw, (1, 0, 2)) if transposed else raw
    dims = ("crosstrack", "downtrack", "bands") if transposed else ("downtrack", "crosstrack", "bands")
    extra = {"lon": lon.T if transposed else lon, "lat": lat.T if transposed else lat}
    gt = [10.0, 0.000542, 0.0, 45.0, 0.0, -0.000542]
    opened = []

    def fake_open(path):
        if "OBS" in str(path):
            ds = _FakeNC("obs", np.transpose(obs, (1, 0, 2)) if transposed else obs, dims, gxf, gyf, w, gt)
        else:
            ds = _FakeNC("reflectance", np.ascontiguousarray(cube_file), dims, gxf, gyf, w, gt, extra)
        opened.append(ds)
        return ds, "fake"

    monkeypatch.setattr(nc_export, "open_any_nc", fake_open)
    out, info = nc_export.nc_to_envi(str(tmp_path / "EMIT_L2A_RFL_001_x.nc"), str(tmp_path / "out"), str(tmp_path / "tmp"),
                                     obs_file=str(tmp_path / "EMIT_OBS.nc"), export_loc=True, return_info=True,
                                     save_info_path=tmp_path / "info.json")
    want, vref, dref = oglt.glt_ortho(raw, np.nan_to_num(gxf).astype(np.int32), gy)
    Ho, Wo = gx.shape
    disk = np.fromfile(out, dtype="<f4").reshape(Ho, B, Wo)                       # BIL
    assert np.array_equal(np.transpose(disk, (0, 2, 1)).view(np.int32), want.view(np.int32))
    hdr = open(str(out) + ".hdr").read()
    assert "interleave = bil" in hdr and f"samples = {Wo}" in hdr and f"bands = {B}" in hdr and "data ignore value = -9999.0" in hdr
    assert info["glt_diag"] == {"raw_shape_yx": [Hr, Wr], **dref} and info["transpose_raw_yx"] == transposed
    assert info["product"] == "L2A_RFL" and info["tag"] == "L2A_RFL_001_x" and all(d.closed for d in opened)
    assert (tmp_path / "info.json").exists()
    locd = np.fromfile(info["outputs"]["loc_gcs"], dtype="<f4").reshape(Ho, 2, Wo)
    assert np.array_equal(locd[:, 0][vref], lon[gy[vref] - 1, np.nan_to_num(gxf).astype(np.int32)[vref] - 1])
    assert (locd[:, 1][~vref] == -9999.0).all()
    obsd = np.fromfile(info["outputs"]["obs_gcs"], dtype="<f4").reshape(Ho, 3, Wo)
    assert np.array_equal(obsd[:, 2][vref], obs[..., 2][gy[vref] - 1, np.nan_to_num(gxf).astype(np.int32)[vref] - 1])
    # second call: everything exists -> skipped; overwrite=True redoes it
    _, info2 = nc_export.nc_to_envi(str(tmp_path / "EMIT_L2A_RFL_001_x.nc"), str(tmp_path / "out"), str(tmp_path / "tmp"),
                                    export_loc=True, return_info=True)
    assert info2["skipped"] == {"data": "exists", "loc": "exists"}
    out3 = nc_export.convert_emit_nc_to_envi([tmp_path / "EMIT_L2A_RFL_001_x.nc"], None, tmp_path / "conv", overwrite=True,
                                             export_loc=False)
    assert np.array_equal(np.fromfile(out3, dtype="<f4"), disk.reshape(-1), equal_nan=True)
    if not transposed:
        # the UTM step (reference _run_gdalwarp, :876-940) on the GPU: data, LOC and OBS onto the snapped S2 60 m grid
        from hsr_b200.EMIT_data import warp as hwarp
        from oracle import warp as owarp
        s2 = {"epsg": 32632, "x0": 570000.0, "y0": 4990020.0, "dx": 10.0, "dy": 10.0, "width": 3000, "height": 3000}
        out4, info4 = nc_export.nc_to_envi(str(tmp_path / "EMIT_L2A_RFL_001_x.nc"), str(tmp_path / "out"), str(tmp_path / "tmp"),
                                           obs_file=str(tmp_path / "EMIT_OBS.nc"), export_loc=True, s2_tif_path=s2,
                                           return_info=True)
        assert out4.name == "L2A_RFL_001_x.bin" and info4["outputs"]["data_envi_hdr"].endswith("L2A_RFL_001_x.hdr")
        dst_gt, (Hd, Wd), rec = hwarp.target_grid(gt, (Ho, Wo), hwarp.S2Grid.coerce(s2))
        assert info4["commands"][-1]["aligned_extent"] == rec and (rec["left"] - 570000.0) % 60.0 == 0.0
        scales = hwarp.warp_scales(dst_gt, gt, (Hd, Wd), 32, False)
        wantu = owarp.warp(want, gt, dst_gt, Hd, Wd, zone=32, utm=True, nodata=-9999.0, scales=scales)
        gotu = np.transpose(np.fromfile(out4, dtype="<f4").reshape(Hd, B, Wd), (0, 2, 1))
        assert np.array_equal(gotu == -9999.0, wantu == -9999.0) and (wantu != -9999.0).any()
        ok = wantu != -9999.0
        assert np.allclose(gotu[ok], wantu[ok], rtol=1e-5, atol=1e-6)
        hdru = open(info4["outputs"]["data_envi_hdr"]).read()
        assert "map info = { UTM , 1 , 1 ," in hdru and ", 32 , North , WGS-84 , units=Meters }" in hdru and "wavelength = {" in hdru
        obsu = np.fromfile(info4["outputs"]["obs_envi_bin"], dtype="<f4").reshape(Hd, 3, Wd)
        wobs = owarp.warp(np.transpose(obsd, (0, 2, 1)), gt, dst_gt, Hd, Wd, zone=32, utm=True, nodata=-9999.0, scales=scales)
        assert np.allclose(np.transpose(obsu, (0, 2, 1)), wobs, rtol=1e-5, atol=1e-6)
        assert Path(info4["outputs"]["loc_envi_bin"]).exists()
        _, info5 = nc_export.nc_to_envi(str(tmp_path / "EMIT_L2A_RFL_001_x.nc"), str(tmp_path / "out"), str(tmp_path / "tmp"),
                                        s2_tif_path=s2, return_info=True)
        assert info5["skipped"] == {"data": "exists", "data_utm": "exists", "geotiffs": "gdal_translate not installed"}
        _, info6 = nc_export.nc_to_envi(str(tmp_path / "EMIT_L2A_RFL_001_x.nc"), str(tmp_path / "out"), str(tmp_path / "tmp"),
                                        s2_tif_path=str(tmp_path / "s2.tif"), return_info=True)       # a path needs rasterio
        assert "rasterio" in info6["skipped"].get("warp", "rasterio")
        # the reference's public entry point with an S2 grid (its only supported path, emit_proj.py:1303-1356): returns
        # "<tag>.bin" whose header is "<tag>.hdr" (with_suffix, :1353), not "<tag>.bin.hdr"
        out7, info7 = nc_export.convert_emit_nc_to_envi([tmp_path / "EMIT_L2A_RFL_001_x.nc"], s2, tmp_path / "conv_s2",
                                                        export_loc=False, return_info=True)
        assert out7.name == "L2A_RFL_001_x.bin" and out7.with_suffix(".hdr").exists()
        assert np.array_equal(np.fromfile(out7, dtype="<f4"), np.fromfile(out4, dtype="<f4"), equal_nan=True)
        out8 = nc_export.convert_emit_nc_to_envi([tmp_path / "EMIT_L2A_RFL_001_x.nc"], hwarp.S2Grid.coerce(s2),
                                                 tmp_path / "conv_s2")                      # second call: skip-if-exists
        assert out8 == out7
    gt[2] = 1e-6
    with pytest.raises(ValueError, match="Rotated/sheared geotransform"):
        nc_export.nc_to_envi(str(tmp_path / "EMIT_rot.nc"), str(tmp_path / "o2"), str(tmp_path / "t2"))
