"""GPU tests of K17 (pg_spatial_autocorr) against the oracle (oracle/autocorr.py): the statistic and every permuted
statistic within the float64 bound the oracle computes per value, n_ge between the oracle's counts with that bound, the
weight sums bit for bit for binary weights, on radius, kNN-union and dense-clump graphs, isolated nodes and foreign ids,
n = 0 / 1 / 2 and no edges, 1 to 256 columns, 0, 1 and more permutations than one chunk holds, both statistics with
both weightings; determinism across calls, handles and chunks; a non-finite column that poisons only itself; the
public function end to end on the morphology table of a 250 k slide; and one C2-sized run."""
import numpy as np
import pytest
import torch

from oracle import autocorr as oa
from oracle import graph as ograph
from path_gene_multimodal_b200 import build_radius_graph, nuclei_morphology_table, spatial_autocorr, synth
from path_gene_multimodal_b200.cell_graph import autocorr_moments, fdr_bh, _normal_tail
from path_gene_multimodal_b200.engine import Engine
from path_gene_multimodal_b200.polygon_morphology import CONT_COLS
from test_gpu_enrichment import radius_clump

pytestmark = pytest.mark.gpu
MODES = [(m, t) for m in ("moran", "geary") for t in (False, True)]


def feature_columns(xy, n_feat, seed):
    """Columns of mixed character: spatial gradients and waves (strong autocorrelation), noise, heavy tails, a
    large offset with a small spread."""
    rng = np.random.default_rng(seed)
    n = len(xy)
    x, y = (xy[:, 0], xy[:, 1]) if n else (np.zeros(0), np.zeros(0))
    span = max(float(np.ptp(x)) if n else 1.0, 1.0)
    cols = []
    for f in range(n_feat):
        kind = f % 5
        if kind == 0:
            cols.append(x / span + 0.3 * rng.normal(size=n))
        elif kind == 1:
            cols.append(rng.normal(size=n))
        elif kind == 2:
            cols.append(rng.lognormal(4.0, 0.7, size=n))
        elif kind == 3:
            cols.append(np.sin(8 * np.pi * y / span) + rng.normal(size=n))
        else:
            cols.append(1e4 + rng.random(n))
    return np.stack(cols, axis=1) if n_feat else np.zeros((n, 0))


def run(eng, rp, col, x, mode, transformation, n_perms, seed, want_sims=True):
    dev = eng.device
    d_rp = torch.from_numpy(np.asarray(rp, dtype=np.int32)).to(dev)
    d_c = torch.from_numpy(np.asarray(col, dtype=np.int32)).to(dev)
    d_x = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64).T)).to(dev)
    res = eng.spatial_autocorr(d_rp, d_c, d_x, mode, transformation, n_perms, seed, want_sims=want_sims)
    return {k: v.cpu().numpy() for k, v in res.items()}


def close(got, ref, tol, what):
    both_nan = np.isnan(got) & np.isnan(ref)
    ok = both_nan | (np.abs(got - ref) <= tol)
    assert ok.all(), (what, got[~ok][:5], ref[~ok][:5], np.broadcast_to(tol, ok.shape)[~ok][:5])


def check(got, ref, transformation):
    close(got["stat"], ref["stat"], ref["bound"], "stat")
    p = ref["sims"].shape[0]
    if p:
        close(got["sims"], ref["sims"], ref["sims_bound"], "sims")
        tol = ref["bound"] + ref["sims_bound"]
        lo = (ref["sims"] > ref["stat"] + tol).sum(0)
        hi = (ref["sims"] >= ref["stat"] - tol).sum(0)
        fin = ~np.isnan(ref["stat"])
        assert ((lo <= got["n_ge"]) & (got["n_ge"] <= hi))[fin].all(), (lo, got["n_ge"], hi)
        assert (got["n_ge"][~fin] == 0).all()
        d = ref["sims_bound"].max(0)
        close(got["perm_mean"], ref["perm_mean"], d + 1e-15 * np.abs(ref["perm_mean"]), "perm_mean")
        sd = np.sqrt(ref["perm_var"])
        close(got["perm_var"], ref["perm_var"], 4 * sd * d + 4 * d * d + 1e-13 * ref["perm_var"], "perm_var")
    else:
        assert np.isnan(got["perm_mean"]).all() and np.isnan(got["perm_var"]).all() and (got["n_ge"] == 0).all()
    if transformation:
        np.testing.assert_allclose(got["s012"], ref["s012"], rtol=1e-13)
    else:
        assert np.array_equal(got["s012"], ref["s012"])


def run_and_check(eng, rp, col, x, mode, transformation, n_perms, seed):
    got = run(eng, rp, col, x, mode, transformation, n_perms, seed)
    check(got, oa.spatial_autocorr(rp, col, x, mode, transformation, n_perms, seed), transformation)
    return got


@pytest.fixture(scope="module")
def g50k():
    xy, _, _ = synth.make_points(50_000, 1002)
    g = ograph.radius_graph(xy, 50.0)
    return {"rp": g["row_ptr"], "col": g["col"], "xy": xy, "x": feature_columns(xy, 5, 1)}


@pytest.mark.parametrize("mode, transformation", MODES)
def test_radius_graph_c2_density(engine, g50k, mode, transformation):
    got = run_and_check(engine, g50k["rp"], g50k["col"], g50k["x"], mode, transformation, 100, 0)
    assert np.isfinite(got["stat"]).all()
    # the gradient column is clustered, the noise column is not
    assert got["n_ge"][0] == (0 if mode == "moran" else 100)


@pytest.mark.parametrize("mode, transformation", MODES)
def test_knn_union_graph(engine, mode, transformation):
    xy, _, _ = synth.make_points(20_000, 31)
    idx, dist = ograph.knn(xy, 8)
    _, _, rp, col, _ = ograph.undirected_union(idx, dist)
    run_and_check(engine, rp, col, feature_columns(xy, 4, 2), mode, transformation, 50, 3)


@pytest.mark.parametrize("mode, transformation", MODES)
def test_dense_clump(engine, mode, transformation):
    c = radius_clump()
    g = ograph.radius_graph(c["xy"], c["r"])
    assert np.diff(g["row_ptr"]).max() >= 4199
    run_and_check(engine, g["row_ptr"], g["col"], feature_columns(c["xy"], 5, 3), mode, transformation, 12, 5)


@pytest.mark.parametrize("mode, transformation", MODES)
def test_isolated_nodes_and_foreign_ids(engine, mode, transformation):
    xy, _, _ = synth.make_points(8000, 44)
    g = ograph.radius_graph(xy, 12.0)
    rp, col = g["row_ptr"], g["col"]
    assert (np.diff(rp) == 0).sum() > 1000
    rows = np.repeat(np.arange(8000), np.diff(rp))
    extra = np.arange(0, 8000, 5)
    rows = np.concatenate([rows, extra, extra])
    cols = np.concatenate([col, np.full(len(extra), 8000), np.full(len(extra), -7)])
    order = np.argsort(rows, kind="stable")
    rp2 = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=8000))])
    run_and_check(engine, rp2, cols[order], feature_columns(xy, 3, 4), mode, transformation, 30, 6)


@pytest.mark.parametrize("case", ["n0", "n1", "n2", "n2_edge", "no_edges"])
@pytest.mark.parametrize("mode, transformation", MODES)
def test_tiny_and_empty(engine, case, mode, transformation):
    n, edges = {"n0": (0, []), "n1": (1, []), "n2": (2, []), "n2_edge": (2, [[0, 1]]), "no_edges": (50, [])}[case]
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    rp, col, _ = ograph.symmetric_csr(e, np.zeros(len(e)), n)
    x = np.random.default_rng(n).normal(size=(n, 3))
    for p in (0, 3):
        got = run(engine, rp, col, x, mode, transformation, p, 1)
        ref = oa.spatial_autocorr(rp, col, x, mode, transformation, p, 1)
        check(got, ref, transformation)
        if case != "n2_edge":
            assert np.isnan(got["stat"]).all()


@pytest.mark.parametrize("n_feat", [1, 3, 4, 5, 64, 256])
def test_column_counts(engine, n_feat):
    xy, _, _ = synth.make_points(5000, 60 + n_feat)
    g = ograph.radius_graph(xy, 50.0)
    x = feature_columns(xy, n_feat, n_feat)
    for mode, transformation in (MODES[0], MODES[3]):
        run_and_check(engine, g["row_ptr"], g["col"], x, mode, transformation, 20, n_feat)


@pytest.mark.parametrize("n_perms", [0, 1])
def test_no_and_one_permutation(engine, g50k, n_perms):
    for mode, transformation in MODES:
        run_and_check(engine, g50k["rp"], g50k["col"], g50k["x"], mode, transformation, n_perms, 8)


def test_more_permutations_than_one_chunk_and_chunk_independence(engine, g50k):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"]
    engine.profile(True)
    try:
        got = run(engine, rp, col, x, "geary", True, 300, 21)
        recs = engine.profile_records()
    finally:
        engine.profile(False)
    assert sum(name == "ac_index_kernel" for name, _ in recs) > 2
    check(got, oa.spatial_autocorr(rp, col, x, "geary", True, 300, 21), True)
    # permutation p gives the same bits whichever chunk and slot it lands in
    small = run(engine, rp, col, x, "geary", True, 7, 21)
    assert small["sims"].tobytes() == got["sims"][:7].tobytes()
    assert small["stat"].tobytes() == got["stat"].tobytes()


def test_determinism(engine, g50k):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"]
    a = run(engine, rp, col, x, "moran", True, 150, 2 ** 64 - 1)
    b = run(engine, rp, col, x, "moran", True, 150, 2 ** 64 - 1)
    fresh = Engine(0)
    try:
        c = run(fresh, rp, col, x, "moran", True, 150, 2 ** 64 - 1)
    finally:
        fresh.close()
    d = run(engine, rp, col, x, "moran", True, 150, 2 ** 64 - 2)
    for k in a:
        assert a[k].tobytes() == b[k].tobytes() == c[k].tobytes(), k
    assert a["stat"].tobytes() == d["stat"].tobytes()
    assert not np.array_equal(a["sims"], d["sims"])


def test_non_finite_column_poisons_only_itself(engine, g50k):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"].copy()
    clean = run(engine, rp, col, x, "moran", False, 40, 4)
    x[123, 2] = np.nan
    x[77, 4] = np.inf
    got = run(engine, rp, col, x, "moran", False, 40, 4)
    for f in (2, 4):
        assert np.isnan(got["stat"][f]) and np.isnan(got["sims"][:, f]).all() and got["n_ge"][f] == 0
        assert np.isnan(got["perm_mean"][f]) and np.isnan(got["perm_var"][f])
    for f in (0, 1, 3):
        for k in ("stat", "perm_mean", "perm_var", "n_ge"):
            assert got[k][f] == clean[k][f], (k, f)
        assert got["sims"][:, f].tobytes() == clean["sims"][:, f].tobytes()


def test_engine_rejects_bad_arguments(engine):
    dev = engine.device
    rp = torch.zeros(3, dtype=torch.int32, device=dev)
    col = torch.zeros(0, dtype=torch.int32, device=dev)
    x = torch.zeros(2, 2, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError):
        engine.spatial_autocorr(rp, col, x, "moranI")
    with pytest.raises(ValueError):
        engine.spatial_autocorr(rp, col, x[:, :1], "moran")
    with pytest.raises(Exception):  # PG_ERR_INVALID from the library
        engine.spatial_autocorr(rp, col, x, "moran", n_perms=100001)
    with pytest.raises(Exception):
        engine.spatial_autocorr(rp, col, torch.zeros(257, 2, dtype=torch.float64, device=dev), "moran")


def test_public_function_on_morphology_table():
    tab = synth.make_table(250_000, seed=250)
    df = nuclei_morphology_table(tab.poly_xy, poly_off=tab.poly_off, hull=True, device=0)[CONT_COLS]
    g = build_radius_graph(tab.wsi_centroids(), r=50.0, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    for mode, transformation in (("moran", True), ("geary", False)):
        out = spatial_autocorr(rp, col, df, mode=mode, transformation=transformation, n_perms=60, seed=5,
                               two_tailed=mode == "geary", device=0)
        score = "I" if mode == "moran" else "C"
        assert list(out.index) == CONT_COLS
        assert list(out.columns) == [score, "pval_norm", "var_norm", "pval_z_sim", "pval_sim", "var_sim",
                                     "pval_norm_fdr_bh", "pval_z_sim_fdr_bh", "pval_sim_fdr_bh"]
        ref = oa.spatial_autocorr(rp, col, df.to_numpy(), mode, transformation, 60, 5)
        close(out[score].to_numpy(), ref["stat"], ref["bound"], score)
        close(out["var_sim"].to_numpy(), ref["perm_var"], 1e-9 * ref["perm_var"], "var_sim")
        k = 2.0 if mode == "geary" else 1.0
        e, v = autocorr_moments(mode, len(df), *ref["s012"])
        np.testing.assert_allclose(out["var_norm"], v, rtol=1e-12)
        np.testing.assert_allclose(out["pval_norm"], k * _normal_tail((ref["stat"] - e) / np.sqrt(v)),
                                   rtol=1e-6, atol=1e-300)
        n_ge = (ref["sims"] >= ref["stat"]).sum(0)
        np.testing.assert_allclose(out["pval_sim"], k * (np.minimum(n_ge, 60 - n_ge) + 1) / 61.0)
        np.testing.assert_allclose(out["pval_sim_fdr_bh"], fdr_bh(out["pval_sim"].to_numpy()))
    # a nucleus without a polygon has NaN morphology: rejected, naming the column
    bad = df.copy()
    bad.iloc[10, 0] = np.nan
    with pytest.raises(ValueError, match="area"):
        spatial_autocorr(rp, col, bad, device=0)


def test_full_c2_slide():
    xy, _, _ = synth.make_points(1_000_000, synth.SEEDS["C2"])
    g = build_radius_graph(xy, r=50.0, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    assert len(col) > 2_800_000
    x = feature_columns(xy, 10, 7)
    from path_gene_multimodal_b200.engine import get_engine

    got = run(get_engine(0), rp, col, x, "moran", True, 100, 0)
    w = oa.weight_matrix(rp, col, len(xy), True)
    z = oa.centred(x)
    close(got["stat"], oa.statistic("moran", w, z), oa.bound("moran", w, z), "stat")
    picks = [0, 1, 57, 99]
    sims, sb = oa.permuted("moran", w, z, 0, picks, with_bound=True)
    close(got["sims"][picks], sims, sb, "sims")
    np.testing.assert_allclose(got["s012"], oa.weight_sums(w), rtol=1e-13)
    np.testing.assert_allclose(got["perm_mean"], got["sims"].mean(0), rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(got["perm_var"], got["sims"].var(0), rtol=1e-9)
    assert np.array_equal(got["n_ge"], (got["sims"] >= got["stat"]).sum(0))
