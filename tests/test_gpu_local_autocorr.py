"""GPU tests of K18 (pg_local_autocorr) against the oracle (oracle/local_autocorr.py): stat, lag and every permuted
statistic within the float64 bound the oracle computes per value, n_ge between the oracle's counts with that bound,
perm_mean / perm_var within it, on radius, kNN-union and dense-clump graphs, isolated nodes with foreign ids and self
entries, n = 0..3 and no edges; 1 to 256 columns; 0, 1 and many permutations; local Moran, Gi and Gi* with both
weightings; determinism across calls, handles and permutation counts; a non-finite column that poisons only itself;
the sum of I_i against K17's global I; the public function end to end on a 250 k slide's morphology table; and a
C2-sized run checked on a node sample."""
import numpy as np
import pytest
import torch

from oracle import graph as ograph
from oracle import local_autocorr as ol
from path_gene_multimodal_b200 import build_radius_graph, local_autocorr, nuclei_morphology_table, synth
from path_gene_multimodal_b200.cell_graph import fdr_bh
from path_gene_multimodal_b200.engine import Engine, get_engine
from path_gene_multimodal_b200.polygon_morphology import CONT_COLS
from test_gpu_autocorr import feature_columns, run as run_global
from test_gpu_enrichment import radius_clump

pytestmark = pytest.mark.gpu
MODES = [(m, t) for m in ol.MODES for t in (False, True)]
API = {"moran": ("moran", True), "gi": ("getis_ord", False), "gi_star": ("getis_ord", True)}


def run(eng, rp, col, x, mode, transformation, n_perms, seed, want_sims=True):
    dev = eng.device
    d_rp = torch.from_numpy(np.asarray(rp, dtype=np.int32)).to(dev)
    d_c = torch.from_numpy(np.asarray(col, dtype=np.int32)).to(dev)
    d_x = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64).T)).to(dev)
    api, star = API[mode]
    res = eng.local_autocorr(d_rp, d_c, d_x, api, transformation, star, n_perms, seed, want_sims=want_sims)
    return {k: v.cpu().numpy() for k, v in res.items()}


def close(got, ref, tol, what):
    both_nan = np.isnan(got) & np.isnan(ref)
    ok = both_nan | (np.abs(got - ref) <= tol)
    assert ok.all(), (what, int((~ok).sum()), got[~ok][:5], ref[~ok][:5], np.broadcast_to(tol, ok.shape)[~ok][:5])


def check(got, ref):
    nodes = ref["nodes"]
    close(got["stat"], ref["stat"], ref["bound"], "stat")
    close(got["lag"], ref["lag"], ref["lag_bound"], "lag")
    close(got["mean"], ref["mean"], ref["mean_bound"], "mean")
    np.testing.assert_allclose(got["m2"], ref["m2"], rtol=1e-12, atol=1e-300)
    p = ref["sims"].shape[0]
    isolated = ref["d"][nodes] == 0
    if p:
        close(got["sims"][:, :, nodes], ref["sims"], ref["sims_bound"], "sims")
        stat, sb = ref["stat"][:, nodes], ref["bound"][:, nodes]
        tol = sb[None] + ref["sims_bound"]
        lo = (ref["sims"] > stat[None] + tol).sum(0)
        hi = (ref["sims"] >= stat[None] - tol).sum(0)
        fin = ~np.isnan(stat) & ~isolated[None]
        n_ge = got["n_ge"][:, nodes]
        assert ((lo <= n_ge) & (n_ge <= hi))[fin].all()
        assert (n_ge[~fin] == 0).all()
        d = ref["sims_bound"].max(0) + sb
        close(got["perm_mean"][:, nodes], ref["perm_mean"], d + 1e-13 * np.abs(ref["perm_mean"]), "perm_mean")
        sd = np.sqrt(ref["perm_var"])
        close(got["perm_var"][:, nodes], ref["perm_var"],
              4 * sd * d + 4 * d * d + 1e-10 * (ref["perm_var"] + np.abs(ref["perm_mean"] - stat) ** 2), "perm_var")
        assert np.isnan(got["perm_mean"][:, nodes][:, isolated]).all()
    else:
        assert np.isnan(got["perm_mean"]).all() and np.isnan(got["perm_var"]).all() and (got["n_ge"] == 0).all()


@pytest.fixture(scope="module")
def g50k():
    xy, _, _ = synth.make_points(50_000, 1002)
    g = ograph.radius_graph(xy, 50.0)
    return {"rp": g["row_ptr"], "col": g["col"], "xy": xy, "x": feature_columns(xy, 5, 1)}


@pytest.mark.parametrize("mode, transformation", MODES)
def test_radius_graph_c2_density(engine, g50k, mode, transformation):
    got = run(engine, g50k["rp"], g50k["col"], g50k["x"], mode, transformation, 40, 0)
    ref = ol.local_autocorr(g50k["rp"], g50k["col"], g50k["x"], mode, transformation, 40, 0)
    check(got, ref)
    assert np.isfinite(got["stat"][:, ref["d"] > 0]).all()


@pytest.mark.parametrize("mode, transformation", MODES)
def test_knn_union_graph(engine, mode, transformation):
    xy, _, _ = synth.make_points(20_000, 31)
    idx, dist = ograph.knn(xy, 8)
    _, _, rp, col, _ = ograph.undirected_union(idx, dist)
    x = feature_columns(xy, 4, 2)
    check(run(engine, rp, col, x, mode, transformation, 30, 3), ol.local_autocorr(rp, col, x, mode, transformation, 30, 3))


@pytest.mark.parametrize("mode, transformation", MODES)
def test_dense_clump(engine, mode, transformation):
    # rows of ~4 200 entries: more than one shared-memory tile of draws per permutation
    c = radius_clump()
    g = ograph.radius_graph(c["xy"], c["r"])
    assert np.diff(g["row_ptr"]).max() >= 4199
    x = feature_columns(c["xy"], 5, 3)
    got = run(engine, g["row_ptr"], g["col"], x, mode, transformation, 6, 5)
    check(got, ol.local_autocorr(g["row_ptr"], g["col"], x, mode, transformation, 6, 5))


@pytest.mark.parametrize("mode, transformation", MODES)
def test_isolated_nodes_foreign_ids_and_self_entries(engine, mode, transformation):
    xy, _, _ = synth.make_points(8000, 44)
    g = ograph.radius_graph(xy, 12.0)
    rp, col = g["row_ptr"], g["col"]
    assert (np.diff(rp) == 0).sum() > 1000
    rows = np.repeat(np.arange(8000), np.diff(rp))
    extra = np.arange(0, 8000, 5)
    rows = np.concatenate([rows, extra, extra, extra])
    cols = np.concatenate([col, np.full(len(extra), 8000), np.full(len(extra), -7), extra])
    order = np.argsort(rows, kind="stable")
    rp2 = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=8000))])
    x = feature_columns(xy, 3, 4)
    got = run(engine, rp2, cols[order], x, mode, transformation, 20, 6)
    ref = ol.local_autocorr(rp2, cols[order], x, mode, transformation, 20, 6)
    check(got, ref)
    # the self entries change nothing: the same graph without them gives the same bits
    clean = run(engine, rp, col, x, mode, transformation, 20, 6)
    for k in clean:
        assert clean[k].tobytes() == got[k].tobytes(), k


@pytest.mark.parametrize("case", ["n0", "n1", "n2", "n2_edge", "n3_path", "no_edges"])
@pytest.mark.parametrize("mode, transformation", MODES)
def test_tiny_and_empty(engine, case, mode, transformation):
    n, edges = {"n0": (0, []), "n1": (1, []), "n2": (2, []), "n2_edge": (2, [[0, 1]]), "n3_path": (3, [[0, 1], [1, 2]]),
                "no_edges": (50, [])}[case]
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    rp, col, _ = ograph.symmetric_csr(e, np.zeros(len(e)), n)
    x = np.random.default_rng(n).normal(size=(n, 3))
    for p in (0, 3):
        check(run(engine, rp, col, x, mode, transformation, p, 1), ol.local_autocorr(rp, col, x, mode, transformation, p, 1))


@pytest.mark.parametrize("n_feat", [1, 4, 5, 256])
def test_column_counts(engine, n_feat):
    xy, _, _ = synth.make_points(3000, 60 + n_feat)
    g = ograph.radius_graph(xy, 50.0)
    x = feature_columns(xy, n_feat, n_feat)
    for mode, transformation in (MODES[1], MODES[4]):
        check(run(engine, g["row_ptr"], g["col"], x, mode, transformation, 8, n_feat),
              ol.local_autocorr(g["row_ptr"], g["col"], x, mode, transformation, 8, n_feat))


@pytest.mark.parametrize("n_perms", [0, 1])
def test_no_and_one_permutation(engine, g50k, n_perms):
    for mode, transformation in MODES:
        check(run(engine, g50k["rp"], g50k["col"], g50k["x"], mode, transformation, n_perms, 8),
              ol.local_autocorr(g50k["rp"], g50k["col"], g50k["x"], mode, transformation, n_perms, 8))


def test_many_permutations_and_permutation_count_independence(engine, g50k):
    # 300 permutations span many shared-memory steps; permutation p gives the same bits whatever the step it lands in
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"][:, :2]
    got = run(engine, rp, col, x, "gi_star", True, 300, 21)
    picks = np.random.default_rng(0).choice(50_000, 400, replace=False)
    ref = ol.local_autocorr(rp, col, x, "gi_star", True, 300, 21, nodes=picks)
    close(got["sims"][:, :, picks], ref["sims"], ref["sims_bound"], "sims")
    check(got, ref)
    small = run(engine, rp, col, x, "gi_star", True, 7, 21)
    assert small["sims"].tobytes() == got["sims"][:7].tobytes()
    assert small["stat"].tobytes() == got["stat"].tobytes()


def test_determinism(engine, g50k):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"]
    a = run(engine, rp, col, x, "moran", True, 50, 2 ** 64 - 1)
    b = run(engine, rp, col, x, "moran", True, 50, 2 ** 64 - 1)
    fresh = Engine(0)
    try:
        c = run(fresh, rp, col, x, "moran", True, 50, 2 ** 64 - 1)
    finally:
        fresh.close()
    d = run(engine, rp, col, x, "moran", True, 50, 2 ** 64 - 2)
    for k in a:
        assert a[k].tobytes() == b[k].tobytes() == c[k].tobytes(), k
    assert a["stat"].tobytes() == d["stat"].tobytes()
    assert not np.array_equal(a["sims"], d["sims"])


def test_non_finite_column_poisons_only_itself(engine, g50k):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"].copy()
    clean = run(engine, rp, col, x, "gi", False, 20, 4)
    x[123, 2] = np.nan
    x[77, 4] = np.inf
    got = run(engine, rp, col, x, "gi", False, 20, 4)
    for f in (2, 4):
        assert np.isnan(got["stat"][f]).all() and np.isnan(got["sims"][:, f]).all() and (got["n_ge"][f] == 0).all()
        assert np.isnan(got["perm_mean"][f]).all() and np.isnan(got["perm_var"][f]).all()
    for k in got:
        if k in ("mean", "m2"):
            assert got[k][[0, 1, 3]].tobytes() == clean[k][[0, 1, 3]].tobytes()
        elif k == "sims":
            assert got[k][:, [0, 1, 3]].tobytes() == clean[k][:, [0, 1, 3]].tobytes()
        else:
            assert got[k][[0, 1, 3]].tobytes() == clean[k][[0, 1, 3]].tobytes(), k


@pytest.mark.parametrize("transformation", [False, True])
def test_sum_of_local_moran_is_global_moran(engine, g50k, transformation):
    rp, col, x = g50k["rp"], g50k["col"], g50k["x"]
    loc = run(engine, rp, col, x, "moran", transformation, 0, 0, want_sims=False)
    glob = run_global(engine, rp, col, x, "moran", transformation, 0, 0, want_sims=False)
    n, s0 = len(x), glob["s012"][0]
    np.testing.assert_allclose(loc["stat"].sum(1), (n - 1) * s0 / n * glob["stat"], rtol=1e-9)


def test_engine_rejects_bad_arguments(engine):
    dev = engine.device
    rp = torch.zeros(3, dtype=torch.int32, device=dev)
    col = torch.zeros(0, dtype=torch.int32, device=dev)
    x = torch.zeros(2, 2, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError):
        engine.local_autocorr(rp, col, x, "geary")
    with pytest.raises(ValueError):
        engine.local_autocorr(rp, col, x[:, :1], "moran")
    with pytest.raises(Exception):  # PG_ERR_INVALID from the library
        engine.local_autocorr(rp, col, x, "moran", n_perms=100001)
    with pytest.raises(Exception):
        engine.local_autocorr(rp, col, torch.zeros(257, 2, dtype=torch.float64, device=dev), "moran")


def test_public_function_on_morphology_table():
    tab = synth.make_table(250_000, seed=250)
    df = nuclei_morphology_table(tab.poly_xy, poly_off=tab.poly_off, hull=True, device=0)[CONT_COLS]
    g = build_radius_graph(tab.wsi_centroids(), r=50.0, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    x = df.to_numpy()
    picks = np.random.default_rng(1).choice(len(df), 300, replace=False)
    for mode, star in (("moran", True), ("getis_ord", True), ("getis_ord", False)):
        out = local_autocorr(rp, col, df, mode=mode, star=star, n_perms=49, seed=5, device=0)
        omode = "moran" if mode == "moran" else ("gi_star" if star else "gi")
        score = "I" if mode == "moran" else "Z"
        assert list(out.columns.get_level_values(0).unique()) == CONT_COLS
        assert len(out) == len(df)
        ref = ol.local_autocorr(rp, col, x, omode, True, 49, 5, nodes=picks)
        for f, name in enumerate(CONT_COLS):
            close(out[(name, score)].to_numpy(), ref["stat"][f], ref["bound"][f], score)
            stat = ref["stat"][f, picks]
            n_ge = (ref["sims"][:, f] >= stat).sum(0)
            clear = (np.abs(ref["sims"][:, f] - stat) > ref["sims_bound"][:, f] + ref["bound"][f, picks]).all(0)
            clear &= ref["d"][picks] > 0
            p_sim = out[(name, "p_sim")].to_numpy()[picks]
            np.testing.assert_array_equal(p_sim[clear], ((np.minimum(n_ge, 49 - n_ge) + 1) / 50.0)[clear])
            assert np.isnan(p_sim[ref["d"][picks] == 0]).all()
            np.testing.assert_array_equal(out[(name, "p_sim_fdr_bh")].to_numpy(), fdr_bh(out[(name, "p_sim")].to_numpy()))
    bad = df.copy()
    bad.iloc[10, 0] = np.nan
    with pytest.raises(ValueError, match="area"):
        local_autocorr(rp, col, bad, device=0)


def test_planted_hot_spot():
    xy, _, _ = synth.make_points(40_000, 9)
    g = build_radius_graph(xy, r=100.0, symmetric_csr=True, device=0)
    deg = np.diff(g["row_ptr"])
    r = np.hypot(*(xy - np.median(xy, axis=0)).T)
    val = np.random.default_rng(3).normal(size=len(xy)) + 4.0 * (r < 600)
    deep, outside = (r < 450) & (deg >= 4), r > 750
    for mode, want in (("getis_ord", 1), ("moran", 1)):
        out = local_autocorr(g["row_ptr"], g["col"], val, mode=mode, n_perms=199, seed=1, corr_method=None, device=0)
        cl = out[(0, "cluster")].to_numpy()
        assert (cl[deep] == want).mean() > 0.9, mode
        assert (cl[outside] == want).mean() < 0.05, mode


def test_full_c2_slide():
    xy, _, _ = synth.make_points(1_000_000, synth.SEEDS["C2"])
    g = build_radius_graph(xy, r=50.0, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    assert len(col) > 2_800_000
    x = feature_columns(xy, 10, 7)
    eng = get_engine(0)
    got = run(eng, rp, col, x, "moran", True, 99, 0, want_sims=False)
    picks = np.random.default_rng(2).choice(len(xy), 20_000, replace=False)
    ref = ol.local_autocorr(rp, col, x, "moran", True, 99, 0, nodes=picks)
    close(got["stat"], ref["stat"], ref["bound"], "stat")
    close(got["lag"], ref["lag"], ref["lag_bound"], "lag")
    stat, sb = ref["stat"][:, picks], ref["bound"][:, picks]
    tol = sb[None] + ref["sims_bound"]
    lo = (ref["sims"] > stat[None] + tol).sum(0)
    hi = (ref["sims"] >= stat[None] - tol).sum(0)
    n_ge = got["n_ge"][:, picks]
    assert ((lo <= n_ge) & (n_ge <= hi)).all()
    d = ref["sims_bound"].max(0) + sb
    close(got["perm_mean"][:, picks], ref["perm_mean"], d + 1e-13 * np.abs(ref["perm_mean"]), "perm_mean")
    close(got["perm_var"][:, picks], ref["perm_var"], 4 * np.sqrt(ref["perm_var"]) * d + 4 * d * d
          + 1e-10 * (ref["perm_var"] + (ref["perm_mean"] - stat) ** 2), "perm_var")
