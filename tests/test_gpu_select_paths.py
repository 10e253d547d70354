"""Every route of the exact masked percentiles (csrc/select.cu, DESIGN 4.4): bracket misses, candidate overflow, wide
brackets, full per-block candidate buffers, the slow classification path and the whole-series fallback, alone and in
the pair API, through kernels.masked_percentiles and the public surfaces that reach it.

The sampled brackets only decide the speed; the results must be np.percentile's in every case.  Image-like data never
leaves the fast routes, so the inputs here are built to force each route, and each test asserts from the select
workspace that its route really fired.  A numpy model of the per-series bookkeeping (select_model) pins every field of
the workspace state: a wrong count that still ends in the right value (more series sent to the slow fallback) fails
here too.

Bars: percentiles bit-identical to np.percentile of x[k, g][mask[g]] (int64 view; +0 and -0 count as equal, since the
kernel folds -0 onto +0 and which zero numpy returns for a +-0 tie depends on its partition order; NaN where numpy
gives NaN); workspace state equal to the model field for field; stretched planes bit-identical to the oracle's.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from hsr_b200 import kernels
from oracle import color as ocolor

DEV = "cuda"

# constants of csrc/select.cu
SEL_SAMPLE = 8192          # samples per series in the bracket search
SEL_WIDE = 64              # fewer masked samples in the sample: the bracket is the whole key range
SEL_CAP_MIN, SEL_CAP_MAX = 4096, 49152
SEL_BLOCK_BUF = 1024       # candidates a collect block stages per bracket before appending straight to the list
COLLECT_SAMPLES_PER_BLOCK = 256 * 16
# struct SelSeries, one per series, set-major, at the start of the workspace
SEL_SERIES = np.dtype([("klo", "<u4", 2), ("khi", "<u4", 2), ("ncand", "<u4", 2), ("fell_back", "<u4"), ("pad", "<u4"),
                       ("lt", "<u8", 2), ("eqlo", "<u8", 2), ("eqhi", "<u8", 2), ("count", "<u8"), ("nan", "<u8")])
assert SEL_SERIES.itemsize == 96


# =============================================================================== model of the select bookkeeping
def sel_keys(x):
    """key_of / key_bits: the order-preserving u32 image of fp32 with -0 folded onto +0, and the NaN flags."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).copy()
    u[(u & 0x7FFFFFFF) == 0] = 0
    return np.where(u >> 31 == 1, ~u, u | 0x80000000).astype(np.uint32), np.isnan(x)


def sel_capacity(n):
    return min(max(n // 16, SEL_CAP_MIN), SEL_CAP_MAX, n) if n > 0 else SEL_CAP_MIN


def fma(a, b, c):
    """a * b + c rounded once (Fraction -> float rounds to nearest even)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def select_model(x, mask, q):
    """The SelSeries state (and the route of every rank) that select_sample / select_collect / select_finish leave for
    one series x [n] f32 under mask [n] bool (None: every sample), q in percent.  Everything but the order of the
    candidate list is a deterministic function of (x, mask, q)."""
    n = x.size
    key, nan = sel_keys(x)
    sel = np.ones(n, bool) if mask is None else np.asarray(mask, bool)
    m = min(n, SEL_SAMPLE)
    idx = np.array([j * n // m for j in range(m)], dtype=np.int64)       # the kernel's 128-bit j * n / m
    idx = idx[sel[idx] & ~nan[idx]]
    sk = np.sort(key[idx])
    mv = sk.size
    wide = mv < SEL_WIDE
    kk = key[sel & ~nan]
    st = dict(count=int(sel.sum()), nan=int((sel & nan).sum()), cap=sel_capacity(n), wide=wide, fell_back=0,
              klo=[], khi=[], ncand=[], lt=[], eqlo=[], eqhi=[], route=[])
    for qq in np.true_divide(np.asarray(q, dtype=np.float64), 100):
        qq = float(qq)
        klo, khi = 0, 0xFFFFFFFF
        if not wide:
            c = qq * (mv - 1)
            sd = math.sqrt(mv * qq * (1.0 - qq))
            mg = fma(5.0, sd, 3.0)          # nvcc contracts 5.0 * sd + 3.0 into one DFMA (c -/+ mg stay separate)
            lo, hi = max(math.floor(c - mg), 0), min(math.ceil(c + mg), mv - 1)
            if lo > 0:                      # a bracket reaching the sample's extremes is opened to the key range's ends
                klo = int(sk[lo])
            if hi < mv - 1:
                khi = int(sk[hi])
        lt, eqlo = int((kk < klo).sum()), int((kk == klo).sum())
        ncand = int(((kk > klo) & (kk < khi)).sum())
        eqhi = int((kk == khi).sum()) if khi != klo else 0
        for f, v in (("klo", klo), ("khi", khi), ("ncand", ncand), ("lt", lt), ("eqlo", eqlo), ("eqhi", eqhi)):
            st[f].append(v)
        if st["count"] == 0 or st["nan"]:   # NaN result, the finish kernel stops before routing
            st["route"].append(None)
            continue
        N = st["count"]
        vi = (N - 1) * qq                   # numpy's linear ranks
        r0 = math.floor(vi)
        r0, r1 = (N - 1, N - 1) if vi >= N - 1 else (r0, r0 + 1)

        def where(r):
            if r < lt:
                return "miss"
            r -= lt
            if r < eqlo:
                return "klo"
            r -= eqlo
            if r < ncand:
                return "cand" if ncand <= st["cap"] else "overflow"
            return "khi" if r - ncand < eqhi else "miss"
        route = (where(r0), where(r1))
        st["route"].append(route)
        st["fell_back"] += any(h in ("miss", "overflow") for h in route)
    return st


def assert_state(row, mdl, Q, what):
    for f in ("klo", "khi", "ncand", "lt", "eqlo", "eqhi"):
        assert np.array_equal(row[f][:Q], mdl[f]), (what, f, row[f][:Q], mdl[f])
    for f in ("fell_back", "count", "nan"):
        assert int(row[f]) == mdl[f], (what, f, int(row[f]), mdl[f])


def assert_same_percentiles(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, got, want)
    ok = ~np.isnan(want)
    g, w = np.where(got == 0, 0.0, got)[ok], np.where(want == 0, 0.0, want)[ok]      # +-0 -> +0
    assert np.array_equal(g.view(np.int64), w.view(np.int64)), (what, got, want)


def numpy_percentiles(vals, q):
    if vals.size == 0:
        return np.full(len(q), np.nan)
    with np.errstate(invalid="ignore"):
        return np.percentile(vals, q)


def run_select(x, mask, q, y=None, padded=False):
    """masked_percentiles of x (and the pair y) [K, G, n] f32 under mask [G, n] (or None); every percentile checked
    against np.percentile and the state of every series against select_model.  Returns (state [S], models [S])."""
    K, G, n = x.shape
    sets = [x] if y is None else [x, y]
    planes = []
    for a in sets:
        t = kernels.alloc_planes(K, (G, n), DEV) if padded else torch.empty(a.shape, dtype=torch.float32, device=DEV)
        t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        planes.append(t)
    mt = None if mask is None else torch.from_numpy(np.ascontiguousarray(mask)).to(DEV)
    ws = []
    out = kernels.masked_percentiles(planes[0], mt, q, groups=G, y=planes[1] if y is not None else None,
                                     _workspace_out=ws)
    outs = [o.cpu().numpy() for o in ([out] if y is None else out)]
    state = ws[0][:len(sets) * K * G * SEL_SERIES.itemsize].cpu().numpy().view(SEL_SERIES)
    models = []
    for i, a in enumerate(sets):
        for k in range(K):
            for g in range(G):
                mg = None if mask is None else mask[g]
                what = (i, k, g, q)
                assert_same_percentiles(outs[i][k, g], numpy_percentiles(a[k, g] if mg is None else a[k, g][mg], q), what)
                mdl = select_model(a[k, g], mg, q)
                assert_state(state[(i * K + k) * G + g], mdl, len(q), what)
                models.append(mdl)
    return state, models


def collect_blocks(n, S, sms):
    """Blocks per series of select_collect_kernel (masked_percentiles_impl's launch rule)."""
    return min(-(-n // COLLECT_SAMPLES_PER_BLOCK), max(8 * sms // S, 1))


# =============================================================================== constructions, one per route
def miss_planes(rng, K=2, G=1):
    """Only the sampled positions shifted up by 1: every bracket lies above its target ranks (a miss)."""
    n = 16 * SEL_SAMPLE
    x = rng.random((K, G, n), dtype=np.float32)
    x[..., ::16] += 1
    return x, None


def overflow_planes(rng, K=2, G=1):
    """Sampled positions uniform in [0, 1), every other sample just above 0.02: all of them inside the 2 % bracket."""
    n = 16 * SEL_SAMPLE
    x = (0.02 + 1e-5 * rng.random((K, G, n))).astype(np.float32)
    x[..., ::16] = rng.random((K, G, n // 16), dtype=np.float32)
    return x, None


def wide_overflow_planes(rng, K=2, G=1):
    """The mask excludes exactly the sampled positions: no masked sample, so every masked key is a candidate."""
    n = 1 << 20
    mask = np.ones((G, n), bool)
    mask[:, ::n // SEL_SAMPLE] = False
    return rng.random((K, G, n), dtype=np.float32), mask


def wide_planes(rng, K=2, G=1):
    """A sparse swath (~2 %) that misses the sampled positions: a wide bracket whose candidates fit the capacity."""
    n = 1 << 16
    mask = rng.random((G, n)) < 0.02
    mask[:, ::n // SEL_SAMPLE] = False
    return rng.random((K, G, n), dtype=np.float32), mask


def full_buffer_planes(rng, K=10, G=4):
    """30 000 unsampled samples per series moved into the 2 % bracket: ~1470 candidates per collect block (29 blocks per
    series on 148 SMs), more than a block's staging buffer holds."""
    n = 96 * SEL_SAMPLE
    x = rng.random((K, G, n), dtype=np.float32)
    unsampled = np.flatnonzero(np.arange(n) % 96 != 0)
    for s in x.reshape(K * G, n):
        s[rng.choice(unsampled, 30000, replace=False)] = 0.02 + 1e-5 * rng.random(30000)
    return x, None


def image_like(rng, K, G, n):
    return (rng.random((K, G, n)) ** 2).astype(np.float32)


def routes(models, b):
    return [m["route"][b] for m in models]


# =============================================================================== CPU: the constructions do what they say
def test_model_routes_every_construction():
    """Without a GPU: each construction of this file reaches the route it is meant to force, by the model's count."""
    rng = np.random.default_rng(0)
    x, mask = miss_planes(rng, K=1)
    m = select_model(x[0, 0], None, [2, 98])
    assert m["route"] == [("miss", "miss")] * 2 and m["fell_back"] == 2

    x, mask = overflow_planes(rng, K=1)
    m = select_model(x[0, 0], None, [2, 98])
    assert m["route"][0] == ("overflow", "overflow") and m["ncand"][0] > m["cap"] == 8192
    assert "miss" in m["route"][1] and m["fell_back"] == 2

    x, mask = wide_overflow_planes(rng, K=1)
    m = select_model(x[0, 0], mask[0], [2, 98])
    assert m["wide"] and min(m["ncand"]) > m["cap"] == SEL_CAP_MAX and m["fell_back"] == 2

    x, mask = wide_planes(rng, K=1)
    m = select_model(x[0, 0], mask[0], [2, 98])
    assert m["wide"] and 0 < m["ncand"][0] <= m["cap"] == SEL_CAP_MIN
    assert m["route"] == [("cand", "cand")] * 2 and m["fell_back"] == 0

    x, mask = full_buffer_planes(rng, K=2, G=1)
    blocks = collect_blocks(x.shape[-1], 40, 148)
    assert blocks == 29
    for s in x.reshape(2, -1):
        m = select_model(s, None, [2, 98])
        assert m["route"][0] == ("cand", "cand") and m["fell_back"] == 0
        assert m["ncand"][0] <= m["cap"] == SEL_CAP_MAX and m["ncand"][0] / blocks > 1.25 * SEL_BLOCK_BUF

    x = image_like(rng, 1, 1, 1685 * 1667)                   # the model keeps image-like data on the fast routes
    m = select_model(x[0, 0], rng.random(x.shape[-1]) < 0.566, [2, 98])
    assert m["route"] == [("cand", "cand")] * 2 and 0 < max(m["ncand"]) <= m["cap"]


# =============================================================================== GPU: each route, state against the model
@pytest.mark.gpu
def test_bracket_miss_falls_back_to_whole_series():
    state, models = run_select(*miss_planes(np.random.default_rng(1), K=2, G=2), [2, 98])
    assert (state["fell_back"] == 2).all()
    assert all(r == ("miss", "miss") for r in routes(models, 0) + routes(models, 1))


@pytest.mark.gpu
def test_candidate_overflow_falls_back():
    state, models = run_select(*overflow_planes(np.random.default_rng(2), K=3), [2, 98])
    assert (state["ncand"][:, 0] > sel_capacity(16 * SEL_SAMPLE)).all() and (state["fell_back"] == 2).all()
    assert all(r == ("overflow", "overflow") for r in routes(models, 0))


@pytest.mark.gpu
def test_wide_bracket_overflow_falls_back():
    """No masked sample in the sample (periodic mask aligned with it): bracket [0, 2^32), ~1 M candidates."""
    state, models = run_select(*wide_overflow_planes(np.random.default_rng(3)), [2, 98])
    assert all(m["wide"] for m in models)
    assert (state["klo"] == 0).all() and (state["khi"] == 0xFFFFFFFF).all()
    assert (state["ncand"] > SEL_CAP_MAX).all() and (state["fell_back"] == 2).all()


@pytest.mark.gpu
def test_wide_bracket_within_capacity_selects_candidates():
    """Wide bracket, candidates within the capacity: the finish kernel's 32-bit multiselect over the list."""
    state, models = run_select(*wide_planes(np.random.default_rng(4), K=3, G=2), [2, 98])
    assert all(m["wide"] for m in models)
    assert (state["khi"] == 0xFFFFFFFF).all() and (state["ncand"] <= SEL_CAP_MIN).all() and (state["ncand"] > 0).all()
    assert (state["fell_back"] == 0).all() and all(r == ("cand", "cand") for r in routes(models, 0) + routes(models, 1))


@pytest.mark.gpu
def test_full_block_buffer_appends_to_the_list():
    """More candidates of one bracket in one collect block than its staging buffer holds: the rest are appended
    straight to the series' list, interleaved with the other blocks' staged flushes."""
    K, G = 10, 4
    x, mask = full_buffer_planes(np.random.default_rng(5), K, G)
    state, models = run_select(x, mask, [2, 98])
    blocks = collect_blocks(x.shape[-1], K * G, torch.cuda.get_device_properties(0).multi_processor_count)
    nc = state["ncand"][:, 0]
    assert (nc <= SEL_CAP_MAX).all() and (nc / blocks > 1.25 * SEL_BLOCK_BUF).all(), (nc.min(), blocks)
    assert (state["fell_back"] == 0).all() and all(r == ("cand", "cand") for r in routes(models, 0))


@pytest.mark.gpu
@pytest.mark.parametrize("q", [[50], [2], [98, 2], [50, 50], [0, 100], [2, 98]])
def test_percentile_layouts_with_forced_fallback(q):
    """One percentile, descending or equal percentiles (every masked sample takes the slow classification path) and the
    0 / 100 extremes, on planes that fall back next to an ordinary plane of the same call."""
    rng = np.random.default_rng(6)
    x, _ = miss_planes(rng, K=3)
    x[0] = image_like(rng, 1, 1, x.shape[-1])
    state, models = run_select(x, None, q)
    assert state["fell_back"][0] == 0 and (state["fell_back"][1:] >= 1).all()


@pytest.mark.gpu
def test_nan_and_empty_series_beside_fallbacks():
    """A NaN among the masked samples (in the sample, or not) and a group without a masked sample give NaN, and leave
    the series beside them that fall back untouched."""
    rng = np.random.default_rng(7)
    x, _ = miss_planes(rng, K=3, G=2)
    n = x.shape[-1]
    x[1, 0, 16 * 5] = np.nan                                 # a sampled position
    x[2, 0, 7] = np.nan                                      # an unsampled one
    mask = np.ones((2, n), bool)
    mask[1] = False                                          # group 1 selects nothing
    state, models = run_select(x, mask, [2, 98])
    fb, nan, count = (state[f].reshape(3, 2) for f in ("fell_back", "nan", "count"))
    assert fb[0, 0] == 2 and fb[1, 0] == 0 and fb[2, 0] == 0 and (fb[:, 1] == 0).all()
    assert nan[1, 0] == 1 and nan[2, 0] == 1 and (count[:, 1] == 0).all()


@pytest.mark.gpu
def test_pair_api_falls_back_in_the_second_set_only():
    """The pair API with G > 1: only the y planes (set 1) fall back, so the fallback's set / series indexing of the
    planes and of the outputs is checked against set 0 that does not."""
    rng = np.random.default_rng(8)
    K, G, n = 2, 3, 16 * SEL_SAMPLE
    x = image_like(rng, K, G, n)
    y = image_like(rng, K, G, n)
    y[..., ::16] += 1
    mask = rng.random((G, n)) < 0.9
    state, _ = run_select(x, mask, [2, 98], y=y)
    assert (state["fell_back"][:K * G] == 0).all() and (state["fell_back"][K * G:] == 2).all()


@pytest.mark.gpu
@pytest.mark.parametrize("padded", [False, True])
@pytest.mark.parametrize("n,groups", [(1, 1), (2, 1), (3, 1), (257, 1), (4099, 1), (64 * 64, 4), (300 * 300 + 7, 1),
                                      (10007, 3)])
def test_state_on_image_like_inputs(n, groups, padded):
    """The bookkeeping of the fast routes, which the benchmark times: state equal to the model, no fallback."""
    rng = np.random.default_rng(n + groups)
    x = image_like(rng, 3, groups, n)
    mask = rng.random((groups, n)) < (0.6 if n > 3 else 2.0)
    mask[:, 0] = True
    state, _ = run_select(x, mask, [2, 98], padded=padded)
    assert (state["fell_back"] == 0).all()


# =============================================================================== GPU: public surfaces with a fallback
def _stretch_image(rng):
    H, W = 256, 512                                          # H * W = 16 * 8192: the sample takes every 16th pixel
    img = (rng.random((H, W, 3)) ** 2).astype(np.float32)
    img.reshape(-1, 3)[::16, 1:] += 1                        # channels 1 and 2 miss their brackets
    return img, rng.random((H, W)) < 0.9


@pytest.mark.gpu
def test_color_surfaces_with_forced_fallback():
    from hsr_b200.s2_emit import color

    img, mask = _stretch_image(np.random.default_rng(9))
    state, _ = run_select(np.ascontiguousarray(np.moveaxis(img, -1, 0)).reshape(3, 1, -1), mask.reshape(1, -1), [2, 98])
    assert list(state["fell_back"]) == [0, 2, 2]
    lim, _ = color.shared_percentile_limits(img, mask)
    assert np.array_equal(lim.view(np.int64), ocolor.shared_percentile_limits(img, mask).view(np.int64))
    out = color.apply_shared_percentile_stretch(img, mask)
    assert np.array_equal(out.view(np.int32), ocolor.apply_shared_percentile_stretch(img, mask).view(np.int32))
    rn = color.robust_norm_rgb(img, mask)
    assert rn.dtype == np.float64 and np.array_equal(rn.view(np.int64), ocolor.robust_norm_rgb(img, mask).view(np.int64))


@pytest.mark.gpu
def test_pair_synthesizer_fit_with_forced_fallback():
    """PairSynthesizer(stretch=(2, 98)).fit: the S2 reference planes fall back, the synthesised bands do not."""
    from hsr_b200 import synthetic
    from hsr_b200.pipeline import PairSynthesizer
    from hsr_b200.s2_emit import srf

    w = synthetic.emit_wavelengths()
    ps = PairSynthesizer(w, srf.synthetic_s2_srf(), synthetic.good_band_mask(w), deg=2, stretch=(2, 98), device=DEV)
    rng = np.random.default_rng(10)
    K, H, W = ps.K, 256, 512
    x = (rng.random((K, H, W)) ** 2).astype(np.float32)
    y = (rng.random((K, H, W)) ** 2).astype(np.float32)
    y.reshape(K, -1)[:, ::16] += 1
    fm = rng.random((H, W)) < 0.9
    xt, yt = kernels.alloc_planes(K, (H, W), DEV), kernels.alloc_planes(K, (H, W), DEV)
    xt.copy_(torch.from_numpy(x))
    yt.copy_(torch.from_numpy(y))
    fmt = torch.from_numpy(fm).to(DEV)
    ws = []
    kernels.masked_percentiles(xt, fmt, [2, 98], y=yt, _workspace_out=ws)
    fell_back = ws[0][:2 * K * SEL_SERIES.itemsize].cpu().numpy().view(SEL_SERIES)["fell_back"]
    assert (fell_back[:K] == 0).all() and (fell_back[K:] == 2).all()
    _, _, xl, yl = ps.fit(xt, yt, torch.ones((H, W), dtype=torch.bool, device=DEV), fmt)
    for got, planes in ((xl, x), (yl, y)):
        want = ocolor.shared_percentile_limits(np.moveaxis(planes, 0, -1), fm)
        assert np.array_equal(got.cpu().numpy().reshape(K, 2).view(np.int64), want.view(np.int64))
