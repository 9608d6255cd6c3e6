"""CPU: the host reference of K16 (oracle/cooccurrence.py) pinned on scipy's cKDTree.count_neighbors, its two
enumerations against each other (strips included), co_occurrence's occ against a literal per-interval restatement,
Ripley's K of a Poisson pattern against pi r^2, and the input checks of co_occurrence / ripley (raised before any
device is touched, so they hold on a machine without a GPU)."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import cooccurrence as oc
from path_gene_multimodal_b200 import co_occurrence, ripley
from path_gene_multimodal_b200.cell_graph import occurrence_ratio


def kdtree_hist(xy, types, thresholds, n_types):
    """hist [B,T,T] from cKDTree.count_neighbors(cumulative=False) per type pair. Its first bin is d <= t_0 as K16's;
    on one tree it also counts the n_a pairs (i, i), taken out of diagonal bin 0."""
    r = np.asarray(thresholds, dtype=np.float64)
    out = np.zeros((len(r), n_types, n_types), dtype=np.int64)
    trees = {a: cKDTree(xy[types == a]) for a in range(1, n_types + 1)}
    for a in range(1, n_types + 1):
        for c in range(1, n_types + 1):
            if trees[a].n == 0 or trees[c].n == 0:
                continue
            cnt = trees[a].count_neighbors(trees[c], r, cumulative=False).astype(np.int64)
            if a == c:
                cnt[0] -= trees[a].n
            out[:, a - 1, c - 1] = cnt
    return out


def random_case(n=1500, seed=0, n_types=4):
    rng = np.random.default_rng(seed)
    xy = rng.random((n, 2)) * 300.0
    types = rng.integers(-1, n_types + 2, size=n).astype(np.int32)
    return xy, types


def lattice_case(shift, n=900, seed=1):
    """Points on the half-pixel lattice shifted by `shift`: many pairs exactly at 0.5, 1, 1.5, 2, 2.5 (d^2 exact)."""
    rng = np.random.default_rng(seed)
    q = rng.integers(0, 60, size=(n, 2))
    xy = shift + q * 0.5
    return xy, rng.integers(1, 4, size=n).astype(np.int32), np.array([0.5, 1.0, 1.5, 2.0, 2.5])


@pytest.mark.parametrize("case", ["random", "lattice_1e5", "lattice_1e7", "duplicates"])
def test_oracle_matches_count_neighbors(case):
    if case == "random":
        xy, types = random_case()
        thr, t = np.sort(np.random.default_rng(3).random(12)) * 60.0, 4
    elif case == "duplicates":
        xy, types = random_case(600, seed=5, n_types=3)
        xy = np.concatenate([xy, xy[:200], xy[:50]])            # points repeated twice and three times
        types = np.concatenate([types, types[:200], types[:50]])
        thr, t = np.array([0.0, 5.0, 20.0, 40.0]), 3
    else:
        xy, types, thr = lattice_case(1e5 if case == "lattice_1e5" else 1e7)
        t = 3
    ref = kdtree_hist(xy, types, thr, t)
    assert ref.sum() > 0
    np.testing.assert_array_equal(oc.pair_hist_brute(xy, types, thr, t), ref)
    np.testing.assert_array_equal(oc.pair_hist(xy, types, thr, t), ref)
    if case.startswith("lattice"):
        assert ref[-1].sum() > 0 and ref[0].sum() > 0          # pairs exactly on the first and last threshold


def test_oracle_enumerations_agree_on_strips():
    """n_query + ids (a strip with its halo): the two enumerations agree, and the strips' histograms sum to the whole."""
    xy, types = random_case(2000, seed=9, n_types=5)
    thr = np.array([3.0, 10.0, 25.0])
    whole = oc.pair_hist_brute(xy, types, thr, 5)
    edges = [0.0, 100.0, 170.0, 300.0001]
    total = np.zeros_like(whole)
    for lo, hi in zip(edges[:-1], edges[1:]):
        own = (xy[:, 0] >= lo) & (xy[:, 0] < hi)
        halo = ~own & (xy[:, 0] >= lo - thr[-1]) & (xy[:, 0] < hi + thr[-1])
        sel = np.concatenate([np.nonzero(own)[0], np.nonzero(halo)[0]])
        h = oc.pair_hist_brute(xy[sel], types[sel], thr, 5, n_query=int(own.sum()), ids=sel)
        np.testing.assert_array_equal(oc.pair_hist(xy[sel], types[sel], thr, 5, n_query=int(own.sum()), ids=sel), h)
        total += h
    np.testing.assert_array_equal(total, whole)
    np.testing.assert_array_equal(oc.type_count(types, 5), np.bincount(types[(types >= 1) & (types <= 5)] - 1, minlength=5))


def test_occurrence_ratio_literal():
    rng = np.random.default_rng(4)
    count = rng.integers(0, 50, size=(4, 4, 6)).astype(np.int64)
    count += count.transpose(1, 0, 2)                           # ordered pairs of a whole slide: symmetric
    count[2, :, 1] = 0                                           # an empty row in one interval: NaN row and column
    count[:, :, 3] = 0                                           # an empty interval: all NaN
    got, ref = occurrence_ratio(count), oc.occurrence(count)
    np.testing.assert_array_equal(got, ref)
    assert np.isnan(got[2, :, 1]).all() and np.isnan(got[:, 2, 1]).all() and np.isnan(got[:, :, 3]).all()
    # p(c | a) / p(c), restated per interval from the counts (row sums = column sums)
    b = 0
    c = count[:, :, b].astype(np.float64)
    p_c_given_a = c / c.sum(axis=1, keepdims=True)
    p_c = c.sum(axis=0) / c.sum()
    np.testing.assert_allclose(got[:, :, b], p_c_given_a / p_c[None, :], rtol=1e-13)


def test_ripley_k_of_a_poisson_pattern():
    """Without edge correction K underestimates pi r^2 by about perimeter * 2r / (3 pi area) (1.7 % at r = 2 % of a
    unit square); with 20 000 points the counting noise at r = 0.005 is under 1 %: 5 % holds both."""
    rng = np.random.default_rng(12)
    n = 20_000
    xy = rng.random((n, 2))
    radii = np.array([0.005, 0.01, 0.02])
    hist = oc.pair_hist(xy, np.ones(n, dtype=np.int32), radii, 1)
    k = oc.ripley_k(np.moveaxis(np.cumsum(hist, axis=0), 0, -1), [n], 1.0)[0, 0]
    np.testing.assert_allclose(k, np.pi * radii ** 2, rtol=0.05)
    assert (k < np.pi * radii ** 2).all()                        # the missing edge correction only ever loses pairs


@pytest.mark.parametrize("fn", ["co_occurrence", "ripley"])
def test_value_errors_before_any_launch(fn):
    xy, types = random_case(50)

    def call(coords=xy, t=types, thr=(0.0, 5.0, 10.0), n_types=4, **kw):
        if fn == "co_occurrence":
            return co_occurrence(coords, t, thr, n_types=n_types, **kw)
        return ripley(coords, thr, types=t, n_types=n_types, **kw)

    bad = [dict(coords=xy[:, :1]), dict(coords=xy.ravel()), dict(coords=np.where(np.arange(100).reshape(50, 2) == 7, np.nan, xy)),
           dict(coords=np.where(np.arange(100).reshape(50, 2) == 3, np.inf, xy)), dict(t=types[:-1]),
           dict(thr=(0.0, np.nan)), dict(thr=(-1.0, 2.0)), dict(thr=(1.0, 1.0)), dict(thr=(2.0, 1.0)),
           dict(thr=np.arange(65.0)), dict(thr=np.ones((2, 2))), dict(thr=(0.0, np.inf)), dict(n_types=0), dict(n_types=17)]
    if fn == "co_occurrence":
        bad += [dict(thr=(1.0,)), dict(thr=1), dict(thr=5), dict(thr=5, max_dist=np.nan), dict(thr=65, max_dist=10.0),
                dict(thr=(0.0, 1.0), max_dist=3.0)]
    else:
        bad += [dict(thr=()), dict(area=0.0), dict(area=np.nan), dict(area=-3.0)]
    for kw in bad:
        with pytest.raises(ValueError):
            call(**kw)
