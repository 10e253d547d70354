"""A numpy model of the union percentile select (hsr_union_select_*, kernels.masked_percentiles_union): four radix
passes of 8 bits over the order-preserving u32 keys, each pass's histograms summed over the units, one step per pass
that picks every target's digit.  Applied to the histograms of random unit splits it must give np.percentile of the
concatenation exactly; tests/test_gpu_union_select.py checks the device state against it."""
import numpy as np
import pytest


def keys_of(v):
    """(keys of the non-NaN samples, NaN count): -0 folded onto +0, negative floats bit-inverted (select.cu key_of)."""
    v = np.asarray(v, dtype=np.float32).reshape(-1)
    nan = int(np.isnan(v).sum())
    u = v[~np.isnan(v)].view(np.uint32).copy()
    u[(u << np.uint32(1)) == 0] = 0
    neg = (u & np.uint32(0x80000000)) != 0
    return np.where(neg, ~u, u | np.uint32(0x80000000)).astype(np.uint32), nan


def value_of(key):
    key = np.uint32(key)
    u = key & np.uint32(0x7FFFFFFF) if key & np.uint32(0x80000000) else ~key
    return np.array([u], dtype=np.uint32).view(np.float32)[0]


def numpy_ranks(n, q):
    vi = float(n - 1) * q
    prev = np.floor(vi)
    r0, r1 = int(prev), int(prev) + 1
    if vi >= n - 1:
        r0 = r1 = n - 1
        prev = -1.0
    if vi < 0:
        r0 = r1 = 0
        prev = 0.0
    return r0, r1, vi - prev


def numpy_lerp(ka, kb, gamma):
    a, b = value_of(ka), value_of(kb)
    diff = np.float64(np.float32(b) - np.float32(a))
    if gamma >= 0.5:
        return np.float64(b) - diff * (1.0 - gamma)
    return np.float64(a) + diff * gamma


def count(keys, nan, p, prefix):
    """One unit's histograms of pass p: [1, 256] + NaN count in pass 0, [T, 256] of the targets' prefixes after it."""
    shift = 24 - 8 * p
    digit = (keys >> np.uint32(shift)) & np.uint32(255)
    if p == 0:
        return np.bincount(digit, minlength=256)[None].astype(np.int64), nan
    hi = keys >> np.uint32(shift + 8)
    return np.stack([np.bincount(digit[hi == pre], minlength=256) for pre in prefix]).astype(np.int64), 0


def union_model(units, q_percent, trace=None):
    """units: list of 1-D float32 arrays (each unit's masked samples).  Returns the percentiles of the union; ``trace``
    (a list) receives (prefix, rank) of every target after each pass."""
    qf = np.true_divide(np.asarray(q_percent, dtype=np.float64).reshape(-1), 100)
    T = 2 * qf.size
    per_unit = [keys_of(u) for u in units]
    prefix, rank, gamma, dead = [0] * T, [0] * T, [0.0] * qf.size, False
    for p in range(4):
        hist = np.zeros((1 if p == 0 else T, 256), dtype=np.int64)
        nan = 0
        for keys, un in per_unit:           # any order: integer sums
            h, c = count(keys, un, p, prefix)
            hist += h
            nan += c
        if p == 0:
            n = int(hist.sum())
            if n == 0 or nan:
                dead = True
                break
            for j, qq in enumerate(qf):
                rank[2 * j], rank[2 * j + 1], gamma[j] = numpy_ranks(n, qq)
        for t in range(T):
            h = hist[0 if p == 0 else t]
            cum = np.cumsum(h)
            d = int(np.searchsorted(cum, rank[t], side="right"))
            rank[t] -= int(cum[d] - h[d])
            prefix[t] = (prefix[t] << 8) | d if p else d
        if trace is not None:
            trace.append((list(prefix), list(rank)))
    if dead:
        return np.full(qf.size, np.nan)
    return np.array([numpy_lerp(prefix[2 * j], prefix[2 * j + 1], gamma[j]) for j in range(qf.size)])


def _same(got, want):
    """Equal as numbers (numpy may return -0.0 where the folded key gives +0.0), NaN where numpy has NaN."""
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    ok = ~np.isnan(want)
    assert np.array_equal(got[ok], want[ok]), (got, want)


def _split(v, rng, parts):
    cuts = np.sort(rng.integers(0, v.size + 1, size=parts - 1))
    return np.split(v, cuts)


@pytest.mark.parametrize("seed", range(6))
def test_random_splits_reproduce_numpy(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 5000))
    v = rng.random(n).astype(np.float32) ** 2
    v[rng.random(n) < 0.2] = 0.0                         # a clipped image's exact zeros
    for q in ((2, 98), (0, 100), (50,), (98, 2), (37.5, 37.5)):
        for parts in (1, 2, 5, 16):
            units = _split(rng.permutation(v), rng, parts)
            _same(union_model(units, q), np.percentile(v, q))


def test_ties_across_digit_boundaries_and_signed_zero():
    # values whose keys differ only in one byte at each digit position, many repeats, +-0 and negatives
    base = np.float32(0.5).view(np.uint32)
    near = np.array([base + d for d in (0, 1, 255, 256, 257, 65535, 65536, 1 << 24)], dtype=np.uint32).view(np.float32)
    v = np.concatenate([np.repeat(near, 7), np.array([0.0, -0.0, -0.0, -1.5, -1e-30, 1e-30], dtype=np.float32)])
    rng = np.random.default_rng(3)
    for q in ((2, 98), (0, 100), (10, 90), (50, 51)):
        for parts in (2, 3, 7):
            _same(union_model(_split(rng.permutation(v), rng, parts), q), np.percentile(v, q))


def test_nan_in_one_unit_only_and_empty_union():
    a = np.array([0.1, 0.2, 0.3], dtype=np.float32)
    b = np.array([0.4, np.nan], dtype=np.float32)
    got = union_model([a, np.zeros(0, np.float32), b], (2, 98))
    assert np.isnan(got).all() and np.isnan(np.percentile(np.concatenate([a, b]), (2, 98))).all()
    assert np.isnan(union_model([], (2, 98))).all()
    assert np.isnan(union_model([np.zeros(0, np.float32)] * 3, (2, 98))).all()


@pytest.mark.parametrize("n", [1, 2])
def test_one_and_two_samples_split_over_two_units(n):
    v = np.array([0.75, 0.25], dtype=np.float32)[:n]
    for split in range(n + 1):
        for q in ((0, 100), (2, 98), (50,)):
            _same(union_model([v[:split], v[split:]], q), np.percentile(v, q))


def test_constant_planes_and_trace():
    v = np.full(1000, 0.3, dtype=np.float32)
    trace = []
    got = union_model([v[:10], v[10:]], (2, 98), trace)
    _same(got, np.percentile(v, (2, 98)))
    key = int(keys_of(v[:1])[0][0])
    assert trace[-1][0] == [key] * 4                      # every target ends on the one key
    assert [len(t[0]) for t in trace] == [4] * 4
