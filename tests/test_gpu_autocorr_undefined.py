"""GPU: spatial_autocorr end to end where a statistic is undefined - a constant feature column, and a graph without
edges (for example a radius given in the wrong unit). Those columns come back with NaN statistics and NaN p-values,
never as significant, and the other columns' values and Benjamini-Hochberg adjustment are those of a table without
the undefined column."""
import numpy as np
import pandas as pd
import pytest

from oracle import graph as ograph
from path_gene_multimodal_b200 import spatial_autocorr, synth
from path_gene_multimodal_b200.cell_graph import fdr_bh

pytestmark = pytest.mark.gpu
PVALS = ("pval_norm", "pval_z_sim", "pval_sim")


@pytest.fixture(scope="module")
def slide():
    xy, _, _ = synth.make_points(20_000, 77)
    rng = np.random.default_rng(3)
    span = float(np.ptp(xy[:, 0]))
    df = pd.DataFrame({"gradient": xy[:, 0] / span + 0.3 * rng.normal(size=len(xy)),
                       "constant": np.full(len(xy), 42.5),
                       "noise": rng.normal(size=len(xy)),
                       "wave": np.sin(8 * np.pi * xy[:, 1] / span) + rng.normal(size=len(xy))})
    return xy, df


@pytest.mark.parametrize("mode, transformation", [("moran", True), ("geary", False)])
def test_constant_column(slide, mode, transformation):
    xy, df = slide
    g = ograph.radius_graph(xy, 50.0)
    out = spatial_autocorr(g["row_ptr"], g["col"], df, mode=mode, transformation=transformation, n_perms=99, seed=1,
                           device=0)
    score = "I" if mode == "moran" else "C"
    assert np.isnan(out[score]["constant"])
    for k in PVALS + ("var_sim",) + tuple(f"{p}_fdr_bh" for p in PVALS):
        assert np.isnan(out[k]["constant"]), k
    # the other columns are exactly what they are without the constant one
    rest = spatial_autocorr(g["row_ptr"], g["col"], df.drop(columns="constant"), mode=mode,
                            transformation=transformation, n_perms=99, seed=1, device=0)
    pd.testing.assert_frame_equal(out.drop(index="constant"), rest)
    for k in PVALS:
        np.testing.assert_array_equal(out[f"{k}_fdr_bh"].drop(index="constant").to_numpy(), fdr_bh(rest[k].to_numpy()))


@pytest.mark.parametrize("mode", ["moran", "geary"])
def test_graph_without_edges(slide, mode):
    xy, df = slide
    g = ograph.radius_graph(xy, 0.05)  # a radius in the wrong unit: no pair is that close
    assert len(g["col"]) == 0
    for n_perms in (None, 99):
        out = spatial_autocorr(g["row_ptr"], g["col"], df, mode=mode, n_perms=n_perms, seed=1, two_tailed=True,
                               device=0)
        assert out.isna().all().all(), out
