"""CPU: the permutation generator and statistics of neighbourhood enrichment (K15), pinned on the oracle
(oracle/enrichment.py) independently of the CUDA code - pi_p is a bijection, its null distribution of the type-pair
counts is the one of numpy's uniform permutations (squidpy's procedure), the permutation mean matches its closed
form, and the exact z formula equals numpy's."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import enrichment as oe
from oracle import graph as ograph
from path_gene_multimodal_b200 import synth

SE_MAX = 4.5
T = 5


def tile_graph(n, r, seed):
    """n points at the notebook tile's type mix in a 521 px tile, radius graph i<j."""
    rng = np.random.default_rng(seed)
    xy = rng.random((n, 2)) * 521.0
    types = rng.choice(np.arange(1, 6, dtype=np.int32), n, p=synth.TYPE_P)
    return cKDTree(xy).query_pairs(r, output_type="ndarray"), types


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 15, 16, 17, 255, 256, 257, 4 ** 8 - 1, 4 ** 8, 4 ** 8 + 1, 100_003])
def test_permutation_is_a_bijection(n):
    pi = oe.permutations(n, 12345, [0, 1, 999])
    for row in pi:
        assert np.array_equal(np.sort(row), np.arange(n))


def test_permutations_differ_by_index_and_seed():
    n = 1000
    a = oe.permutations(n, 0, range(8))
    assert len({tuple(r) for r in a}) == 8
    b = oe.permutations(n, 1, range(8))
    assert all(not np.array_equal(a[k], b[k]) for k in range(8))
    assert not np.array_equal(a[0], np.arange(n))


def test_splitmix64_known_values():
    # the first outputs of the reference splitmix64 stream seeded with 0 (state advanced by the golden gamma)
    assert int(oe.splitmix64(0)) == 0xE220A8397B1DCDAF
    assert int(oe.splitmix64(0x9E3779B97F4A7C15)) == 0x6E789E6AA1B965F4


@pytest.mark.parametrize("n, r, n_perms", [(20, 150.0, 6000), (101, 80.0, 6000), (5000, 12.0, 2000)])
def test_null_distribution_matches_uniform_permutations(n, r, n_perms):
    edges, types = tile_graph(n, r, seed=5)
    assert len(edges) > n // 2
    lab = oe.labels(types, T)
    ours = oe.permuted_counts(edges, types, T, seed=123, perms=range(n_perms))
    rng = np.random.default_rng(9)
    ref = np.concatenate([oe.pair_counts(np.stack([lab[rng.permutation(n)] for _ in range(500)]), edges, T)
                          for _ in range(n_perms // 500)])
    assert ref.shape == ours.shape
    sd_ref, sd_ours = ref.std(0), ours.std(0)
    ok = sd_ref > 0
    assert ok.sum() >= 10
    se = np.sqrt((sd_ref ** 2 + sd_ours ** 2) / n_perms)
    diff = np.abs(ours.mean(0) - ref.mean(0))[ok] / se[ok]
    assert diff.max() <= SE_MAX, diff.max()
    ratio = sd_ours[ok] / sd_ref[ok]
    assert 0.9 <= ratio.min() and ratio.max() <= 1.1, (ratio.min(), ratio.max())
    # nothing varies where numpy's permutations do not vary either
    assert (sd_ours[~ok] == 0).all()


@pytest.mark.parametrize("n, r", [(101, 80.0), (5000, 12.0)])
def test_permutation_mean_matches_closed_form(n, r):
    edges, types = tile_graph(n, r, seed=8)
    n_perms = 2000
    pc = oe.permuted_counts(edges, types, T, seed=77, perms=range(n_perms))
    d = 2 * len(edges)
    na = np.array([(types == t).sum() for t in range(1, T + 1)], dtype=np.float64)
    expect = d * np.outer(na, na) / (n * (n - 1.0))
    expect[np.diag_indices(T)] = d * na * (na - 1) / (n * (n - 1.0))
    sd = pc.std(0)
    ok = sd > 0
    z = np.abs(pc.mean(0) - expect)[ok] / (sd[ok] / np.sqrt(n_perms))
    assert z.max() <= SE_MAX, z.max()


def test_observed_count_is_the_type_interaction_matrix():
    edges, types = tile_graph(400, 60.0, seed=2)
    types = types.copy()
    types[::17] = 0
    types[::23] = 9
    csr = ograph.symmetric_csr(edges, np.zeros(len(edges)), len(types))
    comp = ograph.composition(csr[0], csr[1], types, T).astype(np.int64)
    inter = np.zeros((T, T), dtype=np.int64)
    for t in range(1, T + 1):
        inter[t - 1] = comp[types == t].sum(0)
    got = oe.pair_counts(oe.labels(types, T)[None, :], edges, T)[0]
    assert np.array_equal(got, inter)
    # rows with a foreign id count nowhere
    bad = np.concatenate([edges, [[0, len(types)], [-1, 3]]])
    assert np.array_equal(oe.pair_counts(oe.labels(types, T)[None, :], bad, T)[0], inter)


def test_exact_z_formula_equals_numpy():
    rng = np.random.default_rng(4)
    perms = rng.integers(0, 5000, size=(300, 4, 4))
    count = rng.integers(0, 5000, size=(4, 4))
    got = oe.statistics(count, perms)
    np.testing.assert_allclose(got["perm_mean"], perms.mean(0), rtol=1e-12)
    np.testing.assert_allclose(got["perm_std"], perms.std(0), rtol=1e-12)
    np.testing.assert_allclose(got["zscore"], (count - perms.mean(0)) / perms.std(0), rtol=1e-12)


def test_zero_variance_gives_nan_and_inf():
    perms = np.full((50, 1, 3), 7, dtype=np.int64)
    got = oe.statistics(np.array([[7, 9, 2]]), perms)
    assert np.isnan(got["zscore"][0, 0])
    assert got["zscore"][0, 1] == np.inf and got["zscore"][0, 2] == -np.inf
    assert (got["perm_std"] == 0).all() and (got["perm_mean"] == 7).all()
    with np.errstate(divide="ignore", invalid="ignore"):
        np.testing.assert_array_equal(got["zscore"], (np.array([[7, 9, 2]]) - perms.mean(0)) / perms.std(0))


def test_empty_inputs():
    for edges, types in ((np.zeros((0, 2), np.int64), np.zeros(0, np.int32)),
                         (np.zeros((0, 2), np.int64), np.array([1, 2, 3], np.int32))):
        got = oe.nhood_enrichment(edges, types, n_types=3, n_perms=4, seed=1)
        assert (got["count"] == 0).all() and (got["perm_mean"] == 0).all() and (got["perm_std"] == 0).all()
        assert np.isnan(got["zscore"]).all()
