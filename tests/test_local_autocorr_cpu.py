"""CPU tests that pin the K18 oracle (oracle/local_autocorr.py) on mathematics, and the host side of local_autocorr:
a literal restatement of esda's conditional-randomisation loop; exhaustive enumeration of the conditional null at
n = 6..8 against the Gi / Gi* denominators and the local Moran permutation moments; the centred Gi / Gi* forms against
Ord & Getis's textbook forms; exact lattice answers; the sum of I_i against the global Moran's I; the Feistel draws
against numpy's as a null; the DataFrame (quadrants, G, p-values, clusters) on a planted hot spot and on isolated
nodes; and the input errors raised before anything launches."""
import itertools
import math

import numpy as np
import pytest

from oracle import autocorr as oa
from oracle import graph as ograph
from oracle import local_autocorr as ol
from path_gene_multimodal_b200 import local_autocorr
from path_gene_multimodal_b200.cell_graph import fdr_bh, local_frame


def random_graph(n, p, seed):
    rng = np.random.default_rng(seed)
    a = np.triu(rng.random((n, n)) < p, 1)
    e = np.argwhere(a)
    rp, col, _ = ograph.symmetric_csr(e, np.zeros(len(e)), n)
    return rp, col


def rook_lattice(h, w):
    idx = np.arange(h * w).reshape(h, w)
    e = np.concatenate([np.stack([idx[:, :-1].ravel(), idx[:, 1:].ravel()], 1),
                        np.stack([idx[:-1, :].ravel(), idx[1:, :].ravel()], 1)])
    rp, col, _ = ograph.symmetric_csr(e, np.zeros(len(e)), h * w)
    return rp, col


def esda_crand_literal(row_ptr, col, x, rids, transformation):
    """esda's _crand_plus / local_moran for one column, restated loop for loop: z_no_i is z without node i, the node
    takes permuted_ids[:, :cardinality] of it, the lag is the weighted sum, the statistic z_i lag (n - 1) / sum z^2;
    then the folded p-value."""
    z = np.asarray(x, dtype=np.float64) - np.mean(x)
    n = len(z)
    scaling = (n - 1) / (z * z).sum()
    rows = np.repeat(np.arange(n), np.diff(row_ptr))
    sims, p_sim = [], []
    for i in range(n):
        nbrs = [int(j) for r, j in zip(rows, col) if r == i and 0 <= j < n and j != i]
        card = len(nbrs)
        wi = np.full(card, 1.0 / card if transformation else 1.0)
        obs = z[i] * (wi * z[nbrs]).sum() * scaling
        mask = np.ones(n, dtype=bool)
        mask[i] = False
        z_no_i = z[mask]
        zrand = z_no_i[rids[:, :card]]
        rstats = z[i] * (zrand * wi).sum(1) * scaling
        larger = int((rstats >= obs).sum())
        if len(rids) - larger < larger:
            larger = len(rids) - larger
        sims.append(rstats)
        p_sim.append((larger + 1.0) / (len(rids) + 1.0))
    return np.array(sims).T, np.array(p_sim)


@pytest.mark.parametrize("transformation", [False, True])
def test_literal_esda_loop_matches_vectorised_oracle(transformation):
    rp, col = random_graph(60, 0.1, 1)
    x = np.random.default_rng(2).lognormal(1.0, 0.6, size=(60, 1))
    ref = ol.local_autocorr(rp, col, x, "moran", transformation, 50, 9)
    rids = ol.draws(60, 9, range(50), int(ref["d"].max()))
    sims, p_sim = esda_crand_literal(rp, col, x[:, 0], rids, transformation)
    np.testing.assert_allclose(ref["sims"][:, 0], sims, rtol=1e-13, atol=1e-13)
    n_ge = ref["n_ge"][0]
    np.testing.assert_array_equal((np.minimum(n_ge, 50 - n_ge) + 1) / 51.0, p_sim)


def conditional_sums(z, i, d):
    """Every sum of d values drawn from the nodes other than i (unordered subsets: the sum does not see the order)."""
    others = np.delete(z, i)
    return np.array([others[list(c)].sum() for c in itertools.combinations(range(len(others)), d)])


@pytest.mark.parametrize("n", [6, 7, 8])
@pytest.mark.parametrize("transformation", [False, True])
def test_exhaustive_conditional_null(n, transformation):
    rp, col = random_graph(n, 0.5, n)
    x = np.random.default_rng(n).normal(size=(n, 1)) * 3 + 1
    z = ol.centred(x)
    m2 = (z * z).sum(0)
    d = ol.degrees(rp, col, n)
    for i in np.flatnonzero(d > 0):
        s = conditional_sums(z[:, 0], i, int(d[i]))[:, None, None]       # [subsets, 1 node, 1 column]
        # Gi: mean 0 and variance 1 under the conditional null, i.e. the denominator is the null's standard deviation
        gi = ol.finish("gi", transformation, n, d[[i]], z[[i]], m2, s)[:, 0, 0]
        if np.isfinite(gi).all():
            assert abs(gi.mean()) < 1e-12 and abs(gi.var() - 1.0) < 1e-12
        # local Moran: the enumerated moments against E[S] = -d z_i / (n - 1), Var[S] = d (n-1-d) / (n-2) sigma^2
        mo = ol.finish("moran", transformation, n, d[[i]], z[[i]], m2, s)[:, 0, 0]
        others = np.delete(z[:, 0], i)
        es = d[i] * others.mean()
        vs = d[i] * (n - 1 - d[i]) / (n - 2) * others.var()
        k = (n - 1) / m2[0] * z[i, 0] * (1.0 / d[i] if transformation else 1.0)
        np.testing.assert_allclose(mo.mean(), k * es, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(mo.var(), k * k * vs, rtol=1e-12, atol=1e-12)
    # Gi*: Ord & Getis's null permutes every value, node i's too: mean 0 and variance 1 over all n! labellings
    # the oracle's Gi* denominator is the numerator's standard deviation over all n! labellings, whose mean is 0
    ob = ol.observed("gi_star", rp, col, x, transformation)
    ws = ol.weights(rp, col, n, transformation, star=True).toarray()
    den = (ws @ z[:, 0]) / ob["stat"][:, 0]
    perms = np.array(list(itertools.permutations(range(n))))
    num = z[perms, 0] @ ws.T                                            # [n!, n]
    np.testing.assert_allclose(num.mean(0), 0.0, atol=1e-12)
    np.testing.assert_allclose(num.std(0), den, rtol=1e-12)


@pytest.mark.parametrize("star", [False, True])
@pytest.mark.parametrize("transformation", [False, True])
def test_centred_forms_equal_textbook_forms(star, transformation):
    rp, col = random_graph(300, 0.03, 4)
    x = np.random.default_rng(5).lognormal(2.0, 0.5, size=300) + 50.0
    ob = ol.observed("gi_star" if star else "gi", rp, col, x[:, None], transformation)["stat"][:, 0]
    tb = ol.textbook_g(rp, col, x, transformation, star)["Z"]
    assert np.array_equal(np.isnan(ob), np.isnan(tb))
    np.testing.assert_allclose(ob, tb, rtol=1e-9, atol=1e-11)


def test_checkerboard_on_rook_lattice():
    h, w = 8, 10
    rp, col = rook_lattice(h, w)
    n = h * w
    x = ((np.arange(h)[:, None] + np.arange(w)[None, :]) % 2).ravel()[:, None].astype(float)
    interior = np.zeros((h, w), dtype=bool)
    interior[1:-1, 1:-1] = True
    interior = interior.ravel()
    binary = ol.observed("moran", rp, col, x, False)["stat"][:, 0]
    rowstd = ol.observed("moran", rp, col, x, True)["stat"][:, 0]
    np.testing.assert_allclose(binary[interior], -4 * (n - 1) / n, rtol=1e-14)
    np.testing.assert_allclose(rowstd[interior], -(n - 1) / n, rtol=1e-14)


@pytest.mark.parametrize("transformation", [False, True])
def test_sum_of_local_moran_is_scaled_global_moran(transformation):
    rp, col = random_graph(400, 0.02, 6)
    x = np.random.default_rng(7).normal(size=(400, 3))
    loc = ol.observed("moran", rp, col, x, transformation)["stat"]
    w = oa.weight_matrix(rp, col, 400, transformation)
    glob = oa.statistic("moran", w, oa.centred(x))
    np.testing.assert_allclose(loc.sum(0), (400 - 1) * w.sum() / 400 * glob, rtol=1e-12)


@pytest.mark.parametrize("n", [20, 101, 5000])
def test_feistel_draws_give_the_conditional_null(n):
    rng = np.random.default_rng(n)
    z = rng.normal(size=n)
    z -= z.mean()
    p = 4000
    k = min(12, n - 2)
    feistel = ol.draws(n, 11, range(p), k)
    numpy_draws = np.stack([rng.permutation(n - 1)[:k] for _ in range(p)])
    for i in (0, n // 2, n - 1):
        others = np.delete(z, i)
        for d in (1, k // 2, k):
            es, vs = d * others.mean(), d * (n - 1 - d) / (n - 2) * others.var()
            for r in (feistel, numpy_draws):
                s = others[r[:, :d]].sum(1)
                assert abs(s.mean() - es) <= 4.5 * math.sqrt(vs / p), (n, i, d)
                assert 0.9 <= s.var() / vs <= 1.1, (n, i, d)


def frame_from_oracle(rp, col, x, mode, transformation, p, seed, alpha=0.05, corr_method="fdr_bh"):
    ref = ol.local_autocorr(rp, col, x, mode, transformation, p, seed)
    res = {k: ref[k] for k in ("stat", "lag", "n_ge", "perm_mean", "perm_var", "mean")}
    api, star = ("moran", True) if mode == "moran" else ("getis_ord", mode == "gi_star")
    return local_frame(res, x, list(range(x.shape[1])), ref["d"], api, transformation, star, p, alpha,
                       corr_method), ref


def test_planted_hot_spot_frame():
    rng = np.random.default_rng(8)
    xy = rng.random((3000, 2)) * 1000
    g = ograph.radius_graph(xy, 60.0)
    rp, col = g["row_ptr"], g["col"]
    r = np.hypot(*(xy - 500).T)
    x = (rng.normal(size=3000) + 4.0 * (r < 200))[:, None]
    deep = (r < 150) & (np.diff(rp) >= 4)
    gi, _ = frame_from_oracle(rp, col, x, "gi_star", True, 199, 1, corr_method=None)
    mo, _ = frame_from_oracle(rp, col, x, "moran", True, 199, 1, corr_method=None)
    assert (gi[(0, "cluster")].to_numpy()[deep] == 1).mean() > 0.9
    assert (mo[(0, "cluster")].to_numpy()[deep] == 1).mean() > 0.9
    assert (mo[(0, "q")].to_numpy()[deep] == 1).all()
    assert (gi[(0, "cluster")].to_numpy()[r > 300] == 1).mean() < 0.05
    assert list(gi.columns.get_level_values(1)) == ["Z", "G", "p_norm", "EZ_sim", "VZ_sim", "z_sim", "p_z_sim", "p_sim",
                                                    "cluster"]


@pytest.mark.parametrize("star", [False, True])
@pytest.mark.parametrize("transformation", [False, True])
def test_frame_fields(star, transformation):
    rp, col = random_graph(500, 0.01, 12)
    x = np.random.default_rng(13).lognormal(1.0, 0.5, size=(500, 2))
    df, ref = frame_from_oracle(rp, col, x, "gi_star" if star else "gi", transformation, 99, 3)
    iso = ref["d"] == 0
    assert iso.sum() > 0
    for f in range(2):
        tb = ol.textbook_g(rp, col, x[:, f], transformation, star)
        g = df[(f, "G")].to_numpy()
        np.testing.assert_allclose(g[~iso], tb["G"][~iso], rtol=1e-12)
        p = df[(f, "p_sim")].to_numpy()
        assert np.isnan(p[iso]).all() and (df[(f, "cluster")].to_numpy()[iso] == 0).all()
        n_ge = ref["n_ge"][f][~iso]
        np.testing.assert_array_equal(p[~iso], (np.minimum(n_ge, 99 - n_ge) + 1) / 100.0)
        adj = df[(f, "p_sim_fdr_bh")].to_numpy()
        np.testing.assert_array_equal(adj, fdr_bh(p))
        z = df[(f, "Z")].to_numpy()
        want = np.where(adj <= 0.05, np.sign(np.nan_to_num(z)), 0)
        np.testing.assert_array_equal(df[(f, "cluster")].to_numpy(), want)
    mo, ref = frame_from_oracle(rp, col, x, "moran", transformation, 99, 3)
    for f in range(2):
        zx = x[:, f] - x[:, f].mean()
        lag = ref["lag"][f]
        want = np.select([(zx > 0) & (lag > 0), (zx <= 0) & (lag > 0), (zx <= 0) & (lag <= 0)], [1, 2, 3], 4)
        np.testing.assert_array_equal(mo[(f, "q")].to_numpy(), want)
        np.testing.assert_array_equal(mo[(f, "EI_sim")].to_numpy(), ref["perm_mean"][f])


def test_nan_rules():
    # a constant column (m2 = 0): NaN everywhere; Gi of a node without neighbours: NaN; n too small: NaN
    rp, col = random_graph(30, 0.2, 3)
    x = np.column_stack([np.ones(30), np.random.default_rng(1).normal(size=30)])
    for mode in ol.MODES:
        ref = ol.local_autocorr(rp, col, x, mode, True, 5, 0)
        assert np.isnan(ref["stat"][0]).all() and np.isnan(ref["sims"][:, 0]).all()
        assert np.isfinite(ref["stat"][1][ref["d"] > 0]).all()
    rp1, col1 = random_graph(2, 1.0, 0)
    assert np.isnan(ol.observed("gi", rp1, col1, np.array([[1.0], [2.0]]), False)["stat"]).all()
    # Gi*, binary, n = 2: n S1 - W^2 = 2 * 2 - 2^2 = 0 under the square root
    assert np.isnan(ol.observed("gi_star", rp1, col1, np.array([[1.0], [2.0]]), False)["stat"]).all()
    # isolated node: Moran keeps 0, Gi* keeps z_i / sqrt(m2 / n), Gi is NaN
    rp, col, _ = ograph.symmetric_csr(np.array([[0, 1], [1, 2]]), np.zeros(2), 4)
    x = np.array([[1.0], [3.0], [2.0], [7.0]])
    z = x[:, 0] - x.mean()
    assert ol.observed("moran", rp, col, x, True)["stat"][3, 0] == 0.0
    np.testing.assert_allclose(ol.observed("gi_star", rp, col, x, True)["stat"][3, 0], z[3] / math.sqrt((z * z).sum() / 4))
    assert np.isnan(ol.observed("gi", rp, col, x, True)["stat"][3, 0])


def test_input_errors_before_launch():
    rp, col = random_graph(20, 0.2, 0)
    x = np.random.default_rng(0).normal(size=(20, 2))
    for kw in ({"mode": "geary"}, {"corr_method": "bonferroni"}, {"n_perms": 0}, {"n_perms": 100001},
               {"n_perms": 9.5}, {"alpha": 0.0}, {"alpha": 1.0}):
        with pytest.raises(ValueError):
            local_autocorr(rp, col, x, **kw)
    with pytest.raises(ValueError, match="features"):
        local_autocorr(rp, col, x[:19])
    with pytest.raises(ValueError, match="columns"):
        local_autocorr(rp, col, np.zeros((20, 257)))
    with pytest.raises(ValueError, match="row_ptr"):
        local_autocorr(rp[::-1], col, x)
    with pytest.raises(ValueError, match="col ids"):
        local_autocorr(rp, col + 20, x)
    import pandas as pd

    bad = pd.DataFrame({"area": x[:, 0], "perimeter": x[:, 1]})
    bad.iloc[3, 1] = np.inf
    with pytest.raises(ValueError, match="perimeter"):
        local_autocorr(rp, col, bad)
