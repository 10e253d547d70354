"""OT-target colour matching in the pair pipeline (PairSynthesizer(targets="ot")): the planar pair compaction against
np.flatnonzero, the planar gather against stretch_apply + gather_rows_f64, the Sinkhorn entry for C <= 16 against the
C <= 4 entry and oracle/ot.py, synthesize / synthesize_on_s2_grid / synthesize_sharded against fit_ot_poly_rgb's
composition on the stacked planes, the reference script (match_pair_rgb) on an identity GLT, the identity branches and
the errors."""
import ctypes

import numpy as np
import pytest
import torch

from hsr_b200 import _lib, kernels, synthetic
from hsr_b200.EMIT_data import warp as hwarp
from hsr_b200.pipeline import HostGranuleStream, PairSynthesizer, s2_target
from hsr_b200.s2_emit import fit_ot_poly_rgb
from hsr_b200.s2_emit.srf import synthetic_s2_srf
from oracle import ot as oot

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

APPLY_ATOL = 1e-4
GLT_GT = (-118.30, 0.000542232520256367, 0.0, 34.20, 0.0, -0.000542232520256367)
S2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)
RGB = ("B4", "B3", "B2")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view({4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def planes(rng, K, H, W, padded):
    x = rng.random((K, H, W)).astype(np.float32) * 2 - 0.5
    if padded:
        t = kernels.alloc_planes(K, (H, W), "cuda")
        t.copy_(dev(x))
        return t
    return dev(x)


# ---------------------------------------------------------------------------------------------- 1. compaction
@pytest.mark.parametrize("padded", [True, False])
@pytest.mark.parametrize("K", [1, 3, 12, 16])
def test_compact_planes_pair_vs_flatnonzero(K, padded):
    rng = np.random.default_rng(K)
    H, W = 37, 53
    x, y = planes(rng, K, H, W, padded), planes(rng, K, H, W, padded)
    kx, ky = K - 1, K // 2
    x[kx].view(-1)[rng.choice(H * W, 40, replace=False)] = float("nan")          # one plane only of X
    y[ky].view(-1)[rng.choice(H * W, 30, replace=False)] = float("inf")
    y[ky].view(-1)[rng.choice(H * W, 30, replace=False)] = float("-inf")
    y[0].view(-1)[rng.choice(H * W, 20, replace=False)] = float("nan")
    mask = dev(rng.random((H, W)) < 0.7)
    xh, yh, mh = host(x).reshape(K, -1), host(y).reshape(K, -1), host(mask).reshape(-1)
    for m, mm in ((mask, mh), (None, np.ones_like(mh)), (torch.zeros_like(mask), np.zeros_like(mh))):
        ix, cx, iy, cy = kernels.compact_planes_pair(x, y, m)
        want_x = np.flatnonzero(mm & np.isfinite(xh).all(0))
        want_y = np.flatnonzero(mm & np.isfinite(yh).all(0))
        assert int(cx) == want_x.size and int(cy) == want_y.size
        assert np.array_equal(host(ix)[:want_x.size], want_x) and np.array_equal(host(iy)[:want_y.size], want_y)
    # with a stretch a row is judged on its stretched values: +-Inf are clipped into [0, 1], NaN stays
    lim = torch.stack([torch.full((K,), -0.1), torch.full((K,), 0.9)], -1).to(torch.float64).cuda().view(K, 1, 2)
    xs, ys = host(kernels.stretch_apply(x, lim)).reshape(K, -1), host(kernels.stretch_apply(y, lim)).reshape(K, -1)
    ix, cx, iy, cy = kernels.compact_planes_pair(x, y, mask, x_stretch=lim, y_stretch=lim)
    want_x, want_y = np.flatnonzero(mh & np.isfinite(xs).all(0)), np.flatnonzero(mh & np.isfinite(ys).all(0))
    assert np.array_equal(host(ix)[:int(cx)], want_x) and np.array_equal(host(iy)[:int(cy)], want_y)
    assert want_y.size > np.flatnonzero(mh & np.isfinite(yh).all(0)).size


def test_compact_planes_pair_empty():
    x = torch.empty((3, 0), dtype=torch.float32, device="cuda")
    ix, cx, iy, cy = kernels.compact_planes_pair(x, x, None)
    assert int(cx) == 0 and int(cy) == 0


# ---------------------------------------------------------------------------------------------- 2. gather
@pytest.mark.parametrize("K", [3, 12])
def test_gather_planes_vs_stretch_and_gather_rows(K):
    rng = np.random.default_rng(40 + K)
    H, W = 41, 29
    x = planes(rng, K, H, W, True)
    x[1, 3, 4] = -0.0
    lim = dev(np.stack([rng.random(K) * 0.2 - 0.3, 0.5 + rng.random(K)], -1).reshape(K, 1, 2))
    idx = dev(rng.permutation(H * W)[:700].astype(np.int32))
    sel = dev(rng.choice(700, 300, replace=False).astype(np.int64))
    for st in (None, lim):
        got = host(kernels.gather_planes_f64(x, idx, sel, stretch=st))
        xs = x if st is None else kernels.stretch_apply(x, st)
        want = host(xs).reshape(K, -1)[:, host(idx)[host(sel)]].T.astype(np.float64)
        assert np.array_equal(bits(got), bits(want))
        if K <= 4:
            inter = xs.reshape(K, -1).t().contiguous()
            assert np.array_equal(bits(got), bits(host(kernels.gather_rows_f64(inter, idx, sel))))
    # dst: rows land where dst says; the others keep the caller's -0.0
    out = torch.full((500, K), -0.0, dtype=torch.float64, device="cuda")
    dst = dev(rng.choice(500, 300, replace=False).astype(np.int64))
    kernels.gather_planes_f64(x, idx, sel, stretch=lim, dst=dst, out=out)
    o = host(out)
    want = host(kernels.stretch_apply(x, lim)).reshape(K, -1)[:, host(idx)[host(sel)]].T.astype(np.float64)
    assert np.array_equal(bits(o[host(dst)]), bits(want))
    rest = np.setdiff1d(np.arange(500), host(dst))
    assert np.all(bits(o[rest]) == np.uint64(0x8000000000000000))
    for bad in (500, -1):                                    # a dst row outside out is refused before any launch
        d = dst.clone()
        d[7] = bad
        with pytest.raises(IndexError):
            kernels.gather_planes_f64(x, idx, sel, dst=d, out=out)


# ---------------------------------------------------------------------------------------------- 3. wide Sinkhorn
def sinkhorn_old_entry(X, Y, reg, it, thr):
    ns, C = X.shape
    nt = Y.shape[0]
    lib = _lib.lib()
    work = torch.empty(lib.hsr_sinkhorn_workspace_bytes(ns, nt) + 256, dtype=torch.uint8, device="cuda")
    wptr = work.data_ptr() + (-work.data_ptr()) % 256
    ybar = torch.empty((ns, C), dtype=torch.float64, device="cuda")
    info = torch.zeros(4, dtype=torch.float64, device="cuda")
    _lib.check(lib.hsr_sinkhorn_barycentric_f64(X.data_ptr(), Y.data_ptr(), ns, nt, C, reg, it, thr, wptr,
                                                ybar.data_ptr(), info.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return ybar, info


@pytest.mark.parametrize("C", [1, 3, 4])
def test_wide_entry_bit_identical_for_narrow_c(C):
    rng = np.random.default_rng(C)
    for ns, nt in ((400, 300), (333, 301)):                 # fused (even nt) and un-fused (odd nt) paths
        X, Y = dev(rng.random((ns, C))), dev(rng.random((nt, C)) ** 2)
        a, ia = sinkhorn_old_entry(X, Y, 0.05, 300, 1e-6)
        b, ib = kernels.sinkhorn_barycentric(X, Y, 0.05, 300, 1e-6)
        assert torch.equal(a.view(torch.int64), b.view(torch.int64)) and torch.equal(ia, ib)


@pytest.mark.parametrize("C", [5, 12, 16])
def test_wide_sinkhorn_vs_oracle(C):
    rng = np.random.default_rng(50 + C)
    for ns, nt in ((600, 500), (517, 443)):                 # fused (even nt) and un-fused (odd nt) paths
        X, Y = rng.random((ns, C)), rng.random((nt, C)) ** 2
        ybar, info = kernels.sinkhorn_barycentric(dev(X), dev(Y), 0.05, 300, 1e-6)
        np.testing.assert_allclose(host(ybar), oot.barycentric_targets(X, Y, 0.05, 300, 1e-6), rtol=0, atol=1e-11)
        assert host(info).tolist()[3] == 0


def test_wide_sinkhorn_limits():
    X = torch.rand((8, 17), dtype=torch.float64, device="cuda")
    with pytest.raises(_lib.HsrError):
        kernels.sinkhorn_barycentric(X, X)
    with pytest.raises(_lib.HsrError):
        sinkhorn_old_entry(X[:, :5].contiguous(), X[:, :5].contiguous(), 0.05, 10, 1e-6)


# ---------------------------------------------------------------------------------------------- 4. the pipeline
def reference_coeffs(units, deg, xl=None, yl=None, min_count=200, n_samples=5000, reg=0.05, numItermax=300,
                     stopThr=1e-6, seed=0):
    """fit_ot_poly_rgb's recipe on the concatenation of the units' planes stacked as (n, K) (stretched with the given
    limits by kernels.stretch_apply): numpy filters and draw, then the library's Sinkhorn and fp64 polyfit."""
    xs, ys = [], []
    for bands, s2, mask in units:
        K = bands.shape[0]
        b = bands if xl is None else kernels.stretch_apply(bands, xl)
        y = s2 if yl is None else kernels.stretch_apply(s2, yl)
        m = host(mask).reshape(-1)
        xs.append(host(b).reshape(K, -1)[:, m].T)
        ys.append(host(y).reshape(K, -1)[:, m].T)
    X_all, Y_all = np.concatenate(xs).astype(np.float64), np.concatenate(ys).astype(np.float64)
    X_all, Y_all = X_all[np.isfinite(X_all).all(1)], Y_all[np.isfinite(Y_all).all(1)]
    K = X_all.shape[1]
    if len(X_all) < min_count or len(Y_all) < min_count:
        c = np.zeros((K, deg + 1))
        c[:, -2] = 1.0
        return c
    rng = np.random.default_rng(seed)
    X = X_all[rng.choice(len(X_all), min(n_samples, len(X_all)), replace=False)]
    Y = Y_all[rng.choice(len(Y_all), min(n_samples, len(Y_all)), replace=False)]
    ybar, _ = kernels.sinkhorn_barycentric(dev(X), dev(Y), reg, numItermax, stopThr)
    return host(kernels.polyfit_f64(dev(X), ybar, deg))


def _case(seed=0, Hr=40, Wr=34):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=good)
    raw[11, 9, 40] = np.nan
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=seed + 1, hole_frac=0.01, n_oob=4, n_neg=4)
    return w, good, dev(raw), dev(gx), dev(gy)


def _s2_for(ps, raw, gx, gy, target=None, seed=4, nan_frac=0.0):
    if target is None:
        b0 = ps.synthesize(raw, gx, gy, torch.zeros((ps.K,) + tuple(gx.shape), device="cuda")).bands
    else:
        b0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K,) + target.shape, device="cuda"), target).bands
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(b0), seed=seed)
    if nan_frac:
        g = torch.Generator(device="cuda").manual_seed(seed)
        s2[1][torch.rand(s2.shape[1:], device="cuda", generator=g) < nan_frac] = float("nan")
    return s2


@pytest.mark.parametrize("y_finite", [False, True])
@pytest.mark.parametrize("stretch", [None, (2, 98)])
@pytest.mark.parametrize("rgb", [True, False])
def test_synthesize_ot_vs_fit_ot_poly_rgb(rgb, stretch, y_finite):
    w, good, raw, gx, gy = _case(seed=3)
    table = synthetic_s2_srf()
    srf = {b: table[b] for b in RGB} if rgb else table
    ps = PairSynthesizer(w, srf, good, deg=4, device="cuda", stretch=stretch, y_finite=y_finite, targets="ot",
                         n_samples=700, gate_band="B2")
    assert ps.K == (3 if rgb else 12)
    # NaN reference pixels leave the Y rows; with a stretch but without y_finite they would also make the percentile
    # limits NaN (np.percentile of data holding NaN), so they are left out there
    s2 = _s2_for(ps, raw, gx, gy, nan_frac=0.05 if stretch is None or y_finite else 0.0)
    res = ps.synthesize(raw, gx, gy, s2)
    want = reference_coeffs([(res.bands, s2, res.fit_mask)], 4, res.x_limits, res.y_limits, n_samples=700)
    assert np.array_equal(bits(host(res.coeffs)), bits(want))
    assert res.ot_info is not None and res.ot_info[0] > 0 and res.ot_info[3] == 0
    if rgb:
        xs = res.bands if stretch is None else kernels.stretch_apply(res.bands, res.x_limits)
        ys = s2 if stretch is None else kernels.stretch_apply(s2, res.y_limits)
        got = fit_ot_poly_rgb(xs.permute(1, 2, 0), ys.permute(1, 2, 0), res.fit_mask, deg=4, n_samples=700,
                              return_info=True)
        assert np.array_equal(bits(host(res.coeffs)), bits(host(got[0])))
        assert tuple(got[1].values()) == res.ot_info
    # the apply is poly_solve_apply of the result's coefficients under the fit mask, with the stretch on the fly
    _, want_m = kernels.poly_solve_apply(res.bands, res.moments, res.fit_mask, 4, min_count=0, x_stretch=res.x_limits)
    assert torch.equal(res.matched.view(torch.int32), want_m.view(torch.int32))
    again = ps.synthesize(raw, gx, gy, s2)
    assert torch.equal(again.coeffs.view(torch.int64), res.coeffs.view(torch.int64))
    assert torch.equal(again.matched.view(torch.int32), res.matched.view(torch.int32))


@pytest.mark.parametrize("stretch", [None, (2, 98)])
def test_synthesize_on_s2_grid_ot(stretch):
    w, good, raw, gx, gy = _case(seed=5)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=4, device="cuda", stretch=stretch, targets="ot")
    target = s2_target(GLT_GT, tuple(gx.shape), S2)
    s2 = _s2_for(ps, raw, gx, gy, target, seed=6)
    res = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    assert res.grid is target
    want = reference_coeffs([(res.bands, s2, res.fit_mask)], 4, res.x_limits, res.y_limits)
    assert np.array_equal(bits(host(res.coeffs)), bits(want))
    paired = PairSynthesizer(w, synthetic_s2_srf(), good, deg=4, device="cuda", stretch=stretch)
    p = paired.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    assert torch.equal(p.bands.view(torch.int32), res.bands.view(torch.int32)) and torch.equal(p.fit_mask, res.fit_mask)
    assert p.ot_info is None


def _granules(ps):
    gs = []
    for i, seed in enumerate((11, 12, 13, 14)):
        w, good, raw, gx, gy = _case(seed=seed, Hr=30 + 4 * i, Wr=28)
        if i == 2:                                           # a granule whose GLT maps nothing: a unit with no rows
            gx, gy = torch.zeros_like(gx), torch.zeros_like(gy)
        g = {"raw": raw, "glt_x": gx, "glt_y": gy}
        if i == 3:
            g["target"] = s2_target(GLT_GT, tuple(gx.shape), S2)
        g["s2_ref"] = _s2_for(ps, raw, gx, gy, g.get("target"), seed=seed + 50)
        gs.append(g)
    return gs


@pytest.mark.parametrize("stretch", [None, (2, 98)])
def test_sharded_ot_equals_concatenation(stretch):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=4, device="cuda", stretch=stretch, stretch_scope="fit",
                         targets="ot", n_samples=900, seed=7)
    gs = _granules(ps)
    res = ps.synthesize_sharded(gs)
    assert len(res) == 4 and int(res[2].fit_mask.sum()) == 0
    want = reference_coeffs([(r.bands, g["s2_ref"], r.fit_mask) for r, g in zip(res, gs)], 4, res[0].x_limits,
                            res[0].y_limits, n_samples=900, seed=7)
    for r in res:
        assert np.array_equal(bits(host(r.coeffs)), bits(want))
    assert res[3].grid is gs[3]["target"]
    # the union's identity rule: every granule is below min_count, the union is not
    counts = [int(r.fit_mask.sum()) for r in res]
    mc = max(counts) + 1
    assert sum(counts) >= mc
    ps.min_count = mc
    res2 = ps.synthesize_sharded(gs)
    want2 = reference_coeffs([(r.bands, g["s2_ref"], r.fit_mask) for r, g in zip(res2, gs)], 4, res2[0].x_limits,
                             res2[0].y_limits, min_count=mc, n_samples=900, seed=7)
    assert np.array_equal(bits(host(res2[0].coeffs)), bits(want2)) and res2[0].ot_info is not None


def test_identity_branches():
    w, good, raw, gx, gy = _case(seed=8)
    ident = np.zeros((12, 3))
    ident[:, -2] = 1.0
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, device="cuda", targets="ot", min_count=10 ** 9)
    s2 = _s2_for(ps, raw, gx, gy)
    r = ps.synthesize(raw, gx, gy, s2)                       # nx below min_count
    assert np.array_equal(host(r.coeffs), ident) and r.ot_info is None
    _, want = kernels.poly_solve_apply(r.bands, torch.zeros_like(r.moments), r.fit_mask, 2, min_count=1)
    assert torch.equal(r.matched.view(torch.int32), want.view(torch.int32))
    ps = PairSynthesizer(w, synthetic_s2_srf(), good, device="cuda", targets="ot")
    s2y = s2.clone()
    s2y[0].view(-1)[100:] = float("nan")                     # ny = at most 100 < 200, nx is not
    r = ps.synthesize(raw, gx, gy, s2y)
    assert int(r.fit_mask.sum()) >= 200
    assert np.array_equal(host(r.coeffs), ident) and r.ot_info is None


# ---------------------------------------------------------------------------------------------- 5. the reference script
def test_script_configuration_vs_match_pair_rgb():
    """match_pair_rgb (the reference script, s2_emit/poly_regression.py:86-162) against the pipeline on an identity GLT
    with the script's settings: srf_dict B4, B3, B2, gate B2, stretch (2, 98), y_finite, deg 4."""
    from hsr_b200.s2_emit import match_pair_rgb

    rng = np.random.default_rng(77)
    H, Wd, f = 48, 40, 6
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    R = synthetic.raw_cube_spectra_np((H, Wd, 285), seed=9, good=good)
    R[10, 10, 50] = np.nan
    base = np.kron(rng.random((3, H, Wd)), np.ones((1, f, f)))
    s2 = np.clip(255 * (0.15 + 0.7 * base + 0.03 * rng.normal(size=base.shape)), 0, 255).astype(np.uint8)
    got = match_pair_rgb(R, w, table, good, s2, factor=f, deg=4, n_samples=5000, seed=0)
    ps = PairSynthesizer(w, {b: table[b] for b in RGB}, good, deg=4, device="cuda", gate_band="B2", stretch=(2, 98),
                         y_finite=True, targets="ot")
    yy, xx = np.meshgrid(np.arange(H, dtype=np.int32), np.arange(Wd, dtype=np.int32), indexing="ij")
    res = ps.synthesize(dev(R), dev(xx + 1), dev(yy + 1), dev(got["s2_real_60m"]))
    assert np.array_equal(bits(host(res.bands)), bits(got["emit_sim_60m"][[2, 1, 0]]))
    assert np.array_equal(host(res.fit_mask), got["valid60"])
    assert np.array_equal(bits(host(res.coeffs)), bits(got["coeffs"]))
    # matched: the fused apply stretches on the fly (stretch1, a * rcp with one Newton step) where the script applies to
    # the stretched image (true division); the two differ by one float32 ulp in about one sample in 2^29
    fine = ps.matched_fine(res, f)
    assert np.array_equal(host(fine.mask), got["mask10"])
    for gm, want in ((host(res.matched), got["matched_60m"]), (host(fine.matched), got["matched_10m"])):
        gm = np.moveaxis(gm, 0, -1)
        assert np.array_equal(np.isnan(gm), np.isnan(want))          # the NaN raw pixel stays NaN (np.clip keeps it)
        ok = ~np.isnan(want)
        assert np.max(np.abs(gm - want)[ok]) <= APPLY_ATOL


# ---------------------------------------------------------------------------------------------- 6. errors
def test_ot_errors():
    w, good, raw, gx, gy = _case(seed=2)
    table = synthetic_s2_srf()
    for kw in ({"targets": "sinkhorn"}, {"targets": "ot", "n_samples": 0}, {"targets": "ot", "n_samples": 2.5},
               {"targets": "ot", "reg": 0.0}, {"targets": "ot", "reg": float("nan")}, {"targets": "ot", "numItermax": -1},
               {"targets": "ot", "stopThr": float("nan")}, {"targets": "ot", "seed": "seed"}):
        with pytest.raises(ValueError):
            PairSynthesizer(w, table, good, device="cuda", **kw)
    ps = PairSynthesizer(w, table, good, device="cuda", targets="ot")
    s2 = torch.rand((ps.K,) + tuple(gx.shape), device="cuda")
    fake_exchange = ctypes.c_int(0)
    with pytest.raises(ValueError, match="exchange"):
        ps.synthesize(raw, gx, gy, s2, exchange=fake_exchange)
    with pytest.raises(ValueError, match="exchange"):
        ps.synthesize_sharded([], exchange=fake_exchange)
    target = s2_target(GLT_GT, tuple(gx.shape), S2)
    with pytest.raises(ValueError, match="exchange"):
        ps.synthesize_on_s2_grid(raw, gx, gy, torch.rand((ps.K,) + target.shape, device="cuda"), target,
                                 exchange=fake_exchange)
    T, h, ww = 2, 16, 16
    with pytest.raises(ValueError, match="tile"):
        ps.synthesize_tiles(torch.rand((T, h, ww, 285), device="cuda"), torch.ones((T, h, ww), dtype=torch.int32,
                            device="cuda"), torch.ones((T, h, ww), dtype=torch.int32, device="cuda"),
                            torch.rand((ps.K, T, h, ww), device="cuda"))
    with pytest.raises(ValueError, match="HostGranuleStream"):
        HostGranuleStream(ps, raw_shape=tuple(raw.shape), ortho_shape=tuple(gx.shape))
