"""The exact percentile select over a UNION of units (kernels.masked_percentiles_union) and the global-fit stretch built
on it (PairSynthesizer(stretch_scope="fit")): bit-identical to np.percentile of the concatenated masked samples."""
import numpy as np
import pytest
import torch

from hsr_b200 import kernels, synthetic
from hsr_b200.pipeline import PairSynthesizer
from hsr_b200.s2_emit.srf import synthetic_s2_srf
from oracle import color as ocolor
from oracle import glt as oglt
from oracle import poly as opoly
from oracle import srf as osrf
from test_union_select_model import union_model

DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None
STATE = np.dtype([("rank", "<u8", 4), ("prefix", "<u4", 4), ("gamma", "<f8", 2), ("dead", "<u4"), ("ticket", "<u4")])


def _bits_equal(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    ok = ~np.isnan(want)
    assert np.array_equal(got[ok].view(np.int64), want[ok].view(np.int64)), (got, want)


def _uneven_units(K, rng):
    """(x, y, mask) units of uneven sizes: an empty unit, an all-false mask, a unit holding the only NaN (plane 3 of x,
    masked), constant planes (plane 5 of x and y everywhere), ties from clipping."""
    units = []
    for n, kind in ((5000, "plain"), (0, "empty"), (3001, "nomask"), (777, "nan"), (12345, "plain"), (1, "plain")):
        x = np.clip(rng.random((K, n)) ** 1.5 * 1.1 - 0.05, 0, 1).astype(np.float32)
        y = np.clip(rng.normal(0.3, 0.1, (K, n)), 0, 1).astype(np.float32)
        x[5], y[5] = 0.25, 0.5
        m = rng.random(n) < 0.8
        if kind == "nomask":
            m[:] = False
            x[:] = np.nan                                # never seen: outside the mask
        if kind == "nan" and m.any():
            x[3, np.argmax(m)] = np.nan
        units.append((x, y, m))
    return units


def _concat(units, which):
    return [np.concatenate([u[which][k][u[2]] for u in units]) for k in range(units[0][0].shape[0])]


@pytest.mark.gpu
def test_union_select_uneven_units_bit_identical_to_numpy():
    K = 12
    rng = np.random.default_rng(0)
    units = _uneven_units(K, rng)
    dev = [(torch.from_numpy(x).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(m).to(DEV)) for x, y, m in units]
    for q in ((2, 98), (0, 100), (50,)):
        state = []
        xl, yl = kernels.masked_percentiles_union(dev, q, _state_out=state)
        assert xl.shape == (K, 1, len(q)) and xl.dtype == torch.float64
        xs, ys = _concat(units, 0), _concat(units, 1)
        for k in range(K):
            _bits_equal(xl[k, 0].cpu().numpy(), np.percentile(xs[k], q))
            _bits_equal(yl[k, 0].cpu().numpy(), np.percentile(ys[k], q))
        assert np.isnan(xl[3].cpu().numpy()).all() and not np.isnan(yl[3].cpu().numpy()).any()
        # the device's final per-target state is the model's (series s: x planes, then y planes)
        st = np.frombuffer(state[0].cpu().numpy()[256:256 + 2 * K * STATE.itemsize].tobytes(), dtype=STATE)
        for s, v in enumerate(xs + ys):
            trace = []
            want = union_model([v], q, trace)
            if np.isnan(want).all():
                assert st["dead"][s] == 1
                continue
            T = 2 * len(q)
            assert st["dead"][s] == 0
            assert list(st["prefix"][s][:T]) == trace[-1][0] and list(st["rank"][s][:T]) == trace[-1][1]


@pytest.mark.gpu
def test_union_select_x_only_and_empty_list():
    rng = np.random.default_rng(1)
    parts = [rng.random((3, n)).astype(np.float32) for n in (10, 4096, 333)]
    dev = [(torch.from_numpy(p).to(DEV), None) for p in parts]
    got = kernels.masked_percentiles_union(dev, (2, 98)).cpu().numpy()
    cat = np.concatenate(parts, axis=1)
    for k in range(3):
        _bits_equal(got[k, 0], np.percentile(cat[k], (2, 98)))
    empty = kernels.masked_percentiles_union([], (2, 98), K=4, pair=True, device=DEV)
    assert all(t.shape == (4, 1, 2) and torch.isnan(t).all() for t in empty)
    with pytest.raises(ValueError, match="K=, pair= and device="):
        kernels.masked_percentiles_union([], (2, 98))
    with pytest.raises(ValueError, match="range"):
        kernels.masked_percentiles_union(dev, (2, 101))


@pytest.mark.gpu
def test_union_select_on_one_unit_equals_the_one_pass_select():
    """The two paths the pipeline chooses between (one unit on one process: the one-pass select) agree bit for bit."""
    rng = np.random.default_rng(2)
    K, n = 12, 200_003
    x = torch.from_numpy(np.clip(rng.random((K, n)) * 1.2 - 0.1, 0, 1).astype(np.float32)).to(DEV)
    y = torch.from_numpy(rng.random((K, n)).astype(np.float32)).to(DEV)
    m = torch.from_numpy(rng.random(n) < 0.7).to(DEV)
    for q in ((2, 98), (0, 100), (25,)):
        ux, uy = kernels.masked_percentiles_union([(x, y, m)], q)
        ox, oy = kernels.masked_percentiles(x, m, q, y=y)
        assert torch.equal(ux.view(torch.int64), ox.view(torch.int64))
        assert torch.equal(uy.view(torch.int64), oy.view(torch.int64))


@pytest.mark.gpu
def test_union_count_beyond_2_pow_32():
    """One unit of ~2^31 samples passed three times: 6.4e9 samples in the union, above the 32-bit range.  Values are
    v[i] = i mod 4096, so the sorted union is known in closed form and the oracle needs no sort."""
    n, M = (1 << 31) - 8, 4096
    if torch.cuda.get_device_properties(DEV).total_memory < 3 * n * 4:
        pytest.skip("needs ~26 GB of device memory")
    x = (torch.arange(n, device=DEV, dtype=torch.int64) % M).to(torch.float32).view(1, n)
    q = (2, 50, 98)
    got = [kernels.masked_percentiles_union([(x, None)] * 3, (qq,)).item() for qq in q]
    del x
    torch.cuda.empty_cache()
    counts = 3 * np.array([n // M + (c < n % M) for c in range(M)], dtype=np.int64)
    cum = np.cumsum(counts)
    N = int(cum[-1])
    assert N > (1 << 32)
    for qq, g in zip(q, got):
        vi = (N - 1) * np.true_divide(np.float64(qq), 100)
        prev = np.floor(vi)
        r0 = int(prev)
        a = np.float32(np.searchsorted(cum, r0, side="right"))
        b = np.float32(np.searchsorted(cum, r0 + 1, side="right"))
        gamma = vi - prev
        diff = np.float64(b - a)
        want = np.float64(b) - diff * (1 - gamma) if gamma >= 0.5 else np.float64(a) + diff * gamma
        _bits_equal(g, want)


def _granules(n_gran, Hr=40, Wr=34, seed0=100):
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = synthetic_s2_srf()
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    out = []
    names = PairSynthesizer(w, table, good, device=DEV).band_names
    for i in range(n_gran):
        raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed0 + i, good=good)
        ortho, valid, _ = oglt.glt_ortho(raw, gx, gy)
        ref = osrf.pseudo_s2_srf_integral(ortho, w, table, good)
        x = np.stack([ref[b] for b in names]).astype(np.float32)
        s2 = synthetic.s2_reference_np(x, seed=seed0 + 1000 + i)
        out.append((raw, x, s2, opoly.fit_mask(x, valid, 0, 0.0)))
    return w, good, table, gx, gy, out


def _stretch_np(x, lim):
    """color.py:33 with given (lo, hi) per plane: float64 arithmetic, stored as float32."""
    lo, hi = lim[:, 0:1], lim[:, 1:2]
    with np.errstate(invalid="ignore"):
        return np.clip((x.reshape(x.shape[0], -1) - lo) / (hi - lo + 1e-12), 0, 1).astype(np.float32).reshape(x.shape)


@pytest.mark.gpu
def test_sharded_fit_scope_stretch_matches_the_concatenation():
    w, good, table, gx, gy, gran = _granules(5)
    ps = PairSynthesizer(w, table, good, deg=2, stretch=(2, 98), stretch_scope="fit", device=DEV)
    K = ps.K
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    res = ps.synthesize_sharded([{"raw": t(r), "glt_x": t(gx), "glt_y": t(gy), "s2_ref": t(s2)} for r, _, s2, _ in gran])
    torch.cuda.synchronize()
    # the limits are exact functions of the planes the device produced (its SRF differs from the oracle's in the last
    # bits); the mask is the oracle's
    xcat = np.concatenate([r.bands.cpu().numpy().reshape(K, -1) for r in res], axis=1)
    ycat = np.concatenate([g[2].reshape(K, -1) for g in gran], axis=1)
    mcat = np.concatenate([g[3].reshape(-1) for g in gran])
    xlim = ocolor.shared_percentile_limits(xcat.T, mcat)
    ylim = ocolor.shared_percentile_limits(ycat.T, mcat)
    for r, g in zip(res, gran):
        assert r.x_limits.shape == (K, 1, 2)
        assert np.array_equal(r.x_limits.cpu().numpy().reshape(K, 2).view(np.int64), xlim.view(np.int64))
        assert np.array_equal(r.y_limits.cpu().numpy().reshape(K, 2).view(np.int64), ylim.view(np.int64))
        assert np.array_equal(r.fit_mask.cpu().numpy(), g[3])
    want = opoly.polyfit_paired(_stretch_np(xcat, xlim), _stretch_np(ycat, ylim), mcat, 2,
                                min_count=200)
    for r, g in zip(res, gran):
        c = r.coeffs.cpu().numpy()
        assert np.max(np.abs(c - want).max(1) / np.abs(want).max(1)) < 1e-4
        matched = opoly.apply_poly_planes(_stretch_np(r.bands.cpu().numpy(), xlim), want, g[3])
        assert np.max(np.abs(r.matched.cpu().numpy() - matched)) < 1e-4
    # no granule on this (only) process: nothing to apply, no error
    assert ps.synthesize_sharded([]) == []


@pytest.mark.gpu
def test_single_granule_same_under_both_scopes():
    w, good, table, gx, gy, gran = _granules(1, Hr=64, Wr=48, seed0=7)
    raw, _, s2, _ = gran[0]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    out = []
    for scope in ("granule", "fit"):
        ps = PairSynthesizer(w, table, good, deg=2, stretch=(2, 98), stretch_scope=scope, y_finite=True, device=DEV)
        out.append(ps.synthesize(t(raw), t(gx), t(gy), t(s2)))
        one = ps.synthesize_sharded([{"raw": t(raw), "glt_x": t(gx), "glt_y": t(gy), "s2_ref": t(s2)}]) \
            if scope == "fit" else None
    a, b = out
    for f in ("x_limits", "y_limits", "coeffs", "matched", "fit_mask", "moments"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert torch.equal(one[0].x_limits, a.x_limits) and torch.equal(one[0].coeffs, a.coeffs)
    # the union select on the same unit gives the same limits (the path the one-granule fit does not take)
    ux, uy = kernels.masked_percentiles_union([(a.bands, t(s2), a.fit_mask)], (2, 98))
    assert torch.equal(ux.view(torch.int64), a.x_limits.view(torch.int64))
    assert torch.equal(uy.view(torch.int64), a.y_limits.view(torch.int64))


def test_invalid_stretch_scope_raises():
    w = synthetic.emit_wavelengths()
    with pytest.raises(ValueError, match="stretch_scope"):
        PairSynthesizer(w, synthetic_s2_srf(), synthetic.good_band_mask(w), stretch=(2, 98), stretch_scope="global")
