"""The union bookkeeping of an OT fit over several units and ranks (PairSynthesizer(targets="ot")), modelled in numpy:
every rank draws the same samples over the union counts, writes the rows its units own (pipeline.ot_owned_rows) into
buffers prefilled with -0.0, and a SUM over the ranks' buffers in any order reproduces X_all[sel] of the concatenation
bit for bit."""
import numpy as np
import pytest

from hsr_b200.pipeline import ot_owned_rows


def _split(rng, world, max_units=4, max_rows=60):
    """Per rank a list of per-unit row counts: empty units, and one rank (when world > 1) that holds no unit."""
    out = []
    empty_rank = int(rng.integers(world)) if world > 1 else -1
    for r in range(world):
        if r == empty_rank:
            out.append([])
            continue
        n = int(rng.integers(1, max_units + 1))
        out.append([int(rng.integers(0, max_rows)) if rng.random() > 0.25 else 0 for _ in range(n)])
    return out


def _rows(rng, n, K):
    """Sample rows with negative values and zeros of both signs."""
    x = rng.normal(size=(n, K))
    x[rng.random((n, K)) < 0.1] = 0.0
    x[rng.random((n, K)) < 0.1] = -0.0
    return x


def _assemble(rng, split, data, sel, K):
    """Each rank's -0.0-prefilled buffer with the rows it owns, summed in a random rank order."""
    rank_counts = [sum(u) for u in split]
    bufs = []
    for r, units in enumerate(split):
        buf = np.full((len(sel), K), -0.0)
        for (rows, local), unit_data in zip(ot_owned_rows(sel, rank_counts, r, units), data[r]):
            assert np.all((local >= 0) & (local < len(unit_data)))
            buf[rows] = unit_data[local]
        bufs.append(buf)
    total = np.full((len(sel), K), -0.0)
    for r in rng.permutation(len(bufs)):
        total = total + bufs[r]
    return total


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("seed", range(6))
def test_union_assembly_reproduces_concatenation(world, seed):
    rng = np.random.default_rng(100 * world + seed)
    K = int(rng.choice([1, 3, 12]))
    split = _split(rng, world)
    data = [[_rows(rng, n, K) for n in units] for units in split]
    pieces = [d for rank in data for d in rank]
    X_all = np.concatenate(pieces) if pieces else np.zeros((0, K))
    N = len(X_all)
    if N == 0:
        return
    n_samples = int(rng.integers(1, N + 5))
    sel = np.random.default_rng(seed).choice(N, size=min(n_samples, N), replace=False)
    got = _assemble(rng, split, data, sel, K)
    want = X_all[sel]
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
    # every sample is owned by exactly one unit of one rank
    rank_counts = [sum(u) for u in split]
    owners = np.zeros(len(sel), int)
    for r, units in enumerate(split):
        for rows, _ in ot_owned_rows(sel, rank_counts, r, units):
            owners[rows] += 1
    assert np.all(owners == 1)


def test_global_to_rank_unit_local_mapping():
    split = [[3, 0, 2], [], [4], [0, 1]]
    rank_counts = [sum(u) for u in split]
    sel = np.arange(sum(rank_counts))
    where = {}
    for r, units in enumerate(split):
        for u, (rows, local) in enumerate(ot_owned_rows(sel, rank_counts, r, units)):
            for g, i in zip(sel[rows], local):
                where[int(g)] = (r, u, int(i))
    assert where == {0: (0, 0, 0), 1: (0, 0, 1), 2: (0, 0, 2), 3: (0, 2, 0), 4: (0, 2, 1),
                     5: (2, 0, 0), 6: (2, 0, 1), 7: (2, 0, 2), 8: (2, 0, 3), 9: (3, 1, 0)}


def test_minus_zero_is_the_identity_of_the_sum():
    v = np.array([0.0, -0.0, 1.5, -2.25, 5e-324, -5e-324, np.finfo(np.float64).max])
    for order in range(4):
        acc = v.copy()
        for _ in range(order + 1):
            acc = np.full_like(v, -0.0) + acc
            acc = acc + np.full_like(v, -0.0)
        assert np.array_equal(acc.view(np.int64), v.view(np.int64))
    assert np.signbit(np.float64(0.0) + np.float64(-0.0)) == np.False_      # +0.0 would turn a -0.0 sample into +0.0
