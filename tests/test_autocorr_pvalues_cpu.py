"""CPU: spatial_autocorr's p-value columns where a statistic is undefined. A constant column (m2 = 0) or a graph
without edges (S0 = 0) gives NaN from the kernel with n_ge = 0; every p-value of that column must be NaN too - not
pval_sim = 1 / (P + 1), the smallest value a permutation test can give - and the Benjamini-Hochberg adjustment of the
other columns must be the one over those columns alone."""
import numpy as np

from path_gene_multimodal_b200.cell_graph import autocorr_frame, fdr_bh

P = 99
PVALS = ("pval_norm", "pval_z_sim", "pval_sim")


def outputs(stat, perm_mean, perm_var, n_ge, s012):
    return {"stat": np.array(stat), "perm_mean": np.array(perm_mean), "perm_var": np.array(perm_var),
            "n_ge": np.array(n_ge, dtype=np.int64), "s012": np.array(s012)}


def test_constant_column_has_nan_p_values_and_leaves_the_adjustment_alone():
    nan = np.nan
    res = outputs([0.31, nan, -0.002, 0.05], [-0.001, nan, -0.001, -0.001], [4e-4, nan, 4e-4, 4e-4], [0, 0, 41, 3],
                  (5000.0, 9100.0, 61000.0))
    for two_tailed in (False, True):
        for mode in ("moran", "geary"):
            df = autocorr_frame(res, ["a", "const", "b", "c"], mode, 5000, P, two_tailed)
            for k in PVALS + ("var_sim",):
                assert np.isnan(df[k]["const"]), k
            for k in PVALS:
                keep = ["a", "b", "c"]
                assert np.isfinite(df[k][keep]).all(), k
                np.testing.assert_array_equal(df[f"{k}_fdr_bh"][keep].to_numpy(), fdr_bh(df[k][keep].to_numpy()))
                assert np.isnan(df[f"{k}_fdr_bh"]["const"])


def test_graph_without_edges_is_never_significant():
    nan = np.nan
    res = outputs([nan, nan, nan], [nan, nan, nan], [nan, nan, nan], [0, 0, 0], (0.0, 0.0, 0.0))
    for mode in ("moran", "geary"):
        df = autocorr_frame(res, ["area", "perimeter", "eccentricity"], mode, 300, P, two_tailed=True)
        assert df.drop(columns=["I" if mode == "moran" else "C"]).isna().all().all()
    # the analytic-only frame too
    df = autocorr_frame(res, ["area", "perimeter", "eccentricity"], "moran", 300, 0)
    assert list(df.columns) == ["I", "pval_norm", "var_norm", "pval_norm_fdr_bh"]
    assert df.isna().all().all()


def test_defined_statistics_keep_their_permutation_p_values():
    res = outputs([0.2, -0.3], [0.0, 0.0], [1e-3, 1e-3], [0, P], (100.0, 200.0, 900.0))
    df = autocorr_frame(res, [0, 1], "moran", 100, P)
    np.testing.assert_array_equal(df["pval_sim"].to_numpy(), [1 / (P + 1), 1 / (P + 1)])
