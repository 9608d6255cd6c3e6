"""CPU: the statistics of spatial autocorrelation (K17) pinned on mathematics, independently of the CUDA code - the
oracle (oracle/autocorr.py) against a literal double loop, exact answers on lattices, the kernel's degree shortcuts for
S0 / S1 / S2 against W's general definitions, the permutation null (numpy's uniform permutations, squidpy's procedure,
and K15's Feistel family) against the closed-form expectation and the randomisation variance, and the host-side
p-values, Benjamini-Hochberg and input errors of ``spatial_autocorr``."""
import math

import numpy as np
import pandas as pd
import pytest
from scipy import stats
from scipy.spatial import cKDTree

from oracle import autocorr as oa
from oracle import enrichment as oe
from oracle import graph as ograph
from path_gene_multimodal_b200 import cell_graph, spatial_autocorr

SE_MAX = 4.5
MODES = ("moran", "geary")


def tile_csr(n, r, seed):
    """n random points in a 521 px tile, radius graph as a symmetric CSR."""
    rng = np.random.default_rng(seed)
    xy = rng.random((n, 2)) * 521.0
    edges = cKDTree(xy).query_pairs(r, output_type="ndarray").reshape(-1, 2)
    rp, col, _ = ograph.symmetric_csr(edges, np.zeros(len(edges)), n)
    return rp, col, xy


def features(xy, rng):
    """A normal column, a heavy-tailed one, and a spatial gradient."""
    n = len(xy)
    return np.stack([rng.normal(size=n), rng.lognormal(3.0, 0.8, size=n), xy[:, 0] + 0.1 * rng.normal(size=n)], axis=1)


def rook_lattice(side):
    """Rook-adjacency lattice of side x side nodes as a symmetric CSR (node = y * side + x)."""
    idx = np.arange(side * side).reshape(side, side)
    e = np.concatenate([np.stack([idx[:, :-1].ravel(), idx[:, 1:].ravel()], 1),
                        np.stack([idx[:-1, :].ravel(), idx[1:, :].ravel()], 1)])
    rp, col, _ = ograph.symmetric_csr(e, np.zeros(len(e)), side * side)
    return rp, col, idx


@pytest.mark.parametrize("transformation", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_oracle_against_literal_double_loop(mode, transformation):
    rp, col, xy = tile_csr(150, 70.0, seed=3)
    x = features(xy, np.random.default_rng(1))
    n = len(xy)
    w = oa.weight_matrix(rp, col, n, transformation).toarray()
    got = oa.statistic(mode, oa.weight_matrix(rp, col, n, transformation), oa.centred(x))
    for f in range(x.shape[1]):
        mean = math.fsum(x[:, f]) / n
        z = [v - mean for v in x[:, f]]
        m2 = math.fsum(v * v for v in z)
        s0 = math.fsum(w.ravel())
        if mode == "moran":
            num = math.fsum(w[i, j] * z[i] * z[j] for i in range(n) for j in range(n))
            ref = n * num / (s0 * m2)
        else:
            num = math.fsum(w[i, j] * (z[i] - z[j]) ** 2 for i in range(n) for j in range(n))
            ref = (n - 1) * num / (2 * s0 * m2)
        assert got[f] == pytest.approx(ref, rel=1e-12, abs=1e-14)


@pytest.mark.parametrize("transformation", [False, True])
@pytest.mark.parametrize("side", [4, 10, 32])
def test_checkerboard_and_gradient_on_rook_lattice(side, transformation):
    rp, col, idx = rook_lattice(side)
    n = side * side
    yy, xx = np.divmod(np.arange(n), side)
    board = ((xx + yy) % 2).astype(np.float64)
    w = oa.weight_matrix(rp, col, n, transformation)
    z = oa.centred(np.stack([board, xx.astype(np.float64)], 1))
    i = oa.statistic("moran", w, z)
    c = oa.statistic("geary", w, z)
    if transformation:  # weights 1/3 and 1/2 are not exact in binary; 1/4 is
        assert i[0] == pytest.approx(-1.0, rel=4e-16)
    else:
        assert i[0] == -1.0
    assert c[0] == pytest.approx(2.0 * (n - 1) / n, rel=4e-16)
    assert i[1] > 1.0 - 2.5 / side  # a linear gradient is strongly, not perfectly, autocorrelated (the edges)


@pytest.mark.parametrize("mode", MODES)
def test_constant_column_and_empty_graph_give_nan(mode):
    rp, col, xy = tile_csr(60, 80.0, seed=2)
    x = np.stack([np.full(60, 3.25), xy[:, 0]], 1)
    got = oa.statistic(mode, oa.weight_matrix(rp, col, 60, True), oa.centred(x))
    assert np.isnan(got[0]) and np.isfinite(got[1])
    empty = oa.statistic(mode, oa.weight_matrix(np.zeros(61, np.int64), np.zeros(0, np.int64), 60, False), oa.centred(x))
    assert np.isnan(empty).all()


def graphs():
    rp, col, _ = tile_csr(3000, 15.0, seed=4)
    yield "radius", rp, col, 3000
    xy = np.random.default_rng(5).random((2000, 2)) * 400
    idx, dist = ograph.knn(xy, 8)
    _, _, rpk, colk, _ = ograph.undirected_union(idx, dist)
    yield "knn_union", rpk, colk, 2000
    rp, col, _ = tile_csr(2000, 6.0, seed=6)  # many isolated nodes
    assert (np.diff(rp) == 0).sum() > 100
    yield "isolated", rp, col, 2000
    # foreign ids (skipped): appended to some rows, outside [0, n)
    rp, col, _ = tile_csr(1000, 20.0, seed=7)
    rows = np.repeat(np.arange(1000), np.diff(rp))
    extra_rows = np.arange(0, 1000, 7)
    rows = np.concatenate([rows, extra_rows, extra_rows])
    cols = np.concatenate([col, np.full(len(extra_rows), 1000 + 5), np.full(len(extra_rows), -1)])
    order = np.argsort(rows, kind="stable")
    yield "foreign", np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=1000))]), cols[order], 1000


@pytest.mark.parametrize("transformation", [False, True])
def test_degree_shortcuts_equal_general_definitions(transformation):
    for name, rp, col, n in graphs():
        general = oa.weight_sums(oa.weight_matrix(rp, col, n, transformation))
        short = oa.weight_sums_shortcut(rp, col, n, transformation)
        if transformation:
            np.testing.assert_allclose(short, general, rtol=1e-14, err_msg=name)
        else:
            assert short == general, name


@pytest.mark.parametrize("n, r, n_perms", [(20, 150.0, 6000), (101, 80.0, 6000), (5000, 12.0, 3000)])
@pytest.mark.parametrize("transformation", [False, True])
def test_permutation_null_matches_closed_forms(n, r, n_perms, transformation):
    rp, col, xy = tile_csr(n, r, seed=11)
    rng = np.random.default_rng(12)
    z = oa.centred(features(xy, rng))
    w = oa.weight_matrix(rp, col, n, transformation)
    for mode in MODES:
        expect = -1.0 / (n - 1) if mode == "moran" else 1.0
        var_r = oa.randomisation_variance(mode, w, z)
        feistel = oa.permuted(mode, w, z, seed=321, perms=range(n_perms))
        uniform = np.stack([oa.statistic(mode, w, z[rng.permutation(n)]) for _ in range(n_perms)])
        for name, sims in (("feistel", feistel), ("numpy", uniform)):
            se = np.sqrt(var_r / n_perms)
            dev = np.abs(sims.mean(0) - expect) / se
            assert dev.max() <= SE_MAX, (mode, name, dev)
            ratio = sims.var(0) / var_r
            assert 0.9 <= ratio.min() and ratio.max() <= 1.1, (mode, name, ratio)


def test_permuted_uses_k15_permutations():
    rp, col, xy = tile_csr(500, 40.0, seed=9)
    z = oa.centred(features(xy, np.random.default_rng(2)))
    w = oa.weight_matrix(rp, col, 500, True)
    pi = oe.permutations(500, 77, [3])[0]
    assert np.array_equal(oa.permuted("moran", w, z, 77, [3])[0], oa.statistic("moran", w, z[pi]))


def test_benjamini_hochberg_against_step_up():
    rng = np.random.default_rng(3)
    for m in (1, 2, 7, 50):
        p = rng.random(m) ** 3
        p[rng.integers(0, m)] = p[0]  # a tie
        got = cell_graph.fdr_bh(p)
        order = np.argsort(p, kind="stable")
        ref = np.empty(m)
        for rank in range(m):  # literal: adj_(k) = min over j >= k of p_(j) m / j, capped at 1
            ref[order[rank]] = min(1.0, min(p[order[j]] * m / (j + 1) for j in range(rank, m)))
        np.testing.assert_allclose(got, ref, rtol=1e-15)
    got = cell_graph.fdr_bh([0.01, np.nan, 0.04])
    assert np.isnan(got[1]) and got[0] == 0.02 and got[2] == 0.04


def test_host_p_values_and_moments():
    z = np.array([-3.0, -0.5, 0.0, 0.7, 2.5, np.inf, -np.inf, np.nan])
    got = cell_graph._normal_tail(z)
    np.testing.assert_allclose(got[:7], stats.norm.sf(np.abs(z[:7])), rtol=1e-14)
    assert np.isnan(got[7])
    # analytic moments from S0 / S1 / S2 against the formulas evaluated on W directly
    rp, col, _ = tile_csr(400, 40.0, seed=1)
    for transformation in (False, True):
        s0, s1, s2 = oa.weight_sums(oa.weight_matrix(rp, col, 400, transformation))
        n = 400.0
        e, v = cell_graph.autocorr_moments("moran", 400, s0, s1, s2)
        assert e == -1 / (n - 1)
        assert v == pytest.approx((n * n * s1 - n * s2 + 3 * s0 * s0) / ((n * n - 1) * s0 * s0) - e * e, rel=1e-14)
        e, v = cell_graph.autocorr_moments("geary", 400, s0, s1, s2)
        assert e == 1.0
        assert v == pytest.approx(((2 * s1 + s2) * (n - 1) - 4 * s0 * s0) / (2 * (n + 1) * s0 * s0), rel=1e-14)


def test_p_sim_and_z_sim_formulas():
    """The permutation p-values spatial_autocorr derives from the device outputs equal squidpy's expressions."""
    rng = np.random.default_rng(8)
    sims = rng.normal(size=(999, 4))
    score = np.array([0.5, -2.9, 0.0, 3.4])
    p = sims.shape[0]
    n_ge = (sims >= score).sum(0)
    large = n_ge.copy()
    flip = (p - large) < large
    large[flip] = p - large[flip]
    np.testing.assert_array_equal((np.minimum(n_ge, p - n_ge) + 1.0) / (p + 1.0), (large + 1) / (p + 1))
    zs = (score - sims.mean(0)) / sims.std(0)
    ref = np.where(zs > 0, 1 - stats.norm.cdf(zs), stats.norm.cdf(zs))
    np.testing.assert_allclose(cell_graph._normal_tail(zs), ref, rtol=1e-9)


def test_value_errors_before_any_launch():
    rp, col, xy = tile_csr(50, 80.0, seed=1)
    x = features(xy, np.random.default_rng(0))
    good = dict(row_ptr=rp, col=col, features=x)

    def bad(**kw):
        with pytest.raises(ValueError):
            spatial_autocorr(**{**good, **kw}, device=0)

    bad(row_ptr=rp[1:])                                   # does not start at 0 / wrong length
    bad(row_ptr=rp[::-1].copy())                          # decreasing
    bad(row_ptr=rp.reshape(1, -1))                        # not 1-D
    bad(row_ptr=rp.astype(np.float64))                    # not integer
    bad(col=np.where(col == col.max(), 50, col))          # id out of range
    bad(col=np.where(col == 0, -1, col))                  # negative id
    bad(col=col[:-1])                                     # row_ptr[-1] != len(col)
    bad(features=x[:-1])                                  # N mismatch
    bad(features=np.zeros((50, 0)))                       # F = 0
    bad(features=np.zeros((50, 257)))                     # F > 256
    with_nan = pd.DataFrame(x, columns=["area", "perimeter", "eccentricity"])
    with_nan.loc[7, "perimeter"] = np.nan
    with pytest.raises(ValueError, match="perimeter"):
        spatial_autocorr(rp, col, with_nan, device=0)
    bad(features=np.where(x > 1e9, 0, np.where(np.arange(50)[:, None] == 3, np.inf, x)))
    bad(mode="moranI")
    bad(corr_method="bonferroni")
    for n_perms in (0, -1, 100001, 2.5):
        bad(n_perms=n_perms)
