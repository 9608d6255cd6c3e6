"""GPU tests of K15 (pg_nhood_enrichment): count, zscore, perm_mean and perm_std bit for bit against the oracle
(oracle/enrichment.py) on radius, kNN-union and dense-clump graphs, 1..16 types with labels outside the range, empty
and tiny inputs, int32 / int64 / misaligned edge arrays, more permutations than one label chunk holds, determinism,
agreement with type_interaction_matrix, input validation, and one full C2-sized slide."""
import numpy as np
import pytest
import torch

from oracle import enrichment as oe
from oracle import graph as ograph
from path_gene_multimodal_b200 import (build_knn_graph, build_radius_graph, neighbourhood_enrichment, synth,
                                       type_interaction_matrix)
from path_gene_multimodal_b200.engine import Engine

pytestmark = pytest.mark.gpu
FIELDS = ("count", "zscore", "perm_mean", "perm_std")


def mixed_types(rng, n, n_types):
    """Types drawn from -2..n_types+3, plus a few 17 and 2**31-1 (everything outside 1..n_types counts nowhere)."""
    t = rng.integers(-2, n_types + 4, size=n).astype(np.int64)
    pick = rng.choice(n, size=max(2, n // 100), replace=False)
    t[pick[0::2]] = 17
    t[pick[1::2]] = 2 ** 31 - 1
    return t.astype(np.int32)


def radius_clump(r=40.0, n_clump=4200, n_background=1000, seed=7):
    """About 4 200 points of type 3 inside a disc of radius 0.4 r (a clique), plus a sparse background of mixed types
    (the dense clump of test_gpu_graph_variants.py)."""
    rng = np.random.default_rng(seed)
    side = 2000.0
    cell = 0.9 * r
    centre = (np.floor(side / 2 / cell) + 0.5) * cell
    rho = 0.4 * r * np.sqrt(rng.random(n_clump))
    phi = rng.random(n_clump) * 2 * np.pi
    clump = np.stack([centre + rho * np.cos(phi), centre + rho * np.sin(phi)], axis=1)
    back = rng.random((n_background, 2)) * side
    xy = np.concatenate([clump, back])
    types = np.concatenate([np.full(n_clump, 3, dtype=np.int32), mixed_types(rng, n_background, 7)])
    order = rng.permutation(len(xy))
    return {"xy": np.ascontiguousarray(xy[order]), "types": types[order], "r": r}


def radius_edges(n, seed, r=50.0):
    xy, types, _ = synth.make_points(n, seed)
    return ograph.radius_graph(xy, r)["edges"], types, xy


def check(got, ref):
    for f in FIELDS:
        np.testing.assert_array_equal(got[f], ref[f], err_msg=f)


def run_and_check(edges, types, n_types, n_perms, seed):
    got = neighbourhood_enrichment(edges, types, n_types=n_types, n_perms=n_perms, seed=seed, device=0)
    check(got, oe.nhood_enrichment(edges, types, n_types, n_perms, seed))
    return got


@pytest.fixture(scope="module")
def g50k():
    edges, types, xy = radius_edges(50_000, 1002)
    return {"edges": edges, "types": types, "xy": xy}


def test_radius_graph_c2_density(g50k):
    got = run_and_check(g50k["edges"], g50k["types"], 5, 200, 0)
    assert got["count"].sum() == 2 * len(g50k["edges"])
    assert np.isfinite(got["zscore"]).all()


def test_knn_union_graph():
    xy, types, _ = synth.make_points(20_000, 31)
    idx, dist = ograph.knn(xy, 8)
    edges = ograph.undirected_union(idx, dist)[0]
    run_and_check(edges, types, 5, 100, 3)


@pytest.mark.parametrize("n_types", [5, 8])
def test_dense_clump(n_types):
    c = radius_clump()
    edges = ograph.radius_graph(c["xy"], c["r"])["edges"]
    assert len(edges) > 4200 * 4199 // 2
    run_and_check(edges, c["types"], n_types, 12, 5)


@pytest.mark.parametrize("n_types", [1, 2, 5, 8, 9, 16])
def test_type_ranges_with_foreign_labels(n_types):
    xy, _, _ = synth.make_points(20_000, 40 + n_types)
    types = mixed_types(np.random.default_rng(n_types), len(xy), n_types)
    edges = ograph.radius_graph(xy, 50.0)["edges"]
    run_and_check(edges, types, n_types, 64, 11)


@pytest.mark.parametrize("case", ["n0", "n1", "n2_one_edge", "no_edges", "p1"])
def test_tiny_and_empty(case):
    if case == "n0":
        edges, types, p = np.zeros((0, 2), np.int64), np.zeros(0, np.int32), 5
    elif case == "n1":
        edges, types, p = np.zeros((0, 2), np.int64), np.array([2], np.int32), 5
    elif case == "n2_one_edge":
        edges, types, p = np.array([[0, 1]]), np.array([1, 2], np.int32), 7
    elif case == "no_edges":
        edges, types, p = np.zeros((0, 2), np.int32), np.array([1, 2, 3, 1], np.int32), 3
    else:
        edges, types, _ = radius_edges(3000, 77)
        p = 1
    got = run_and_check(edges, types, 5, p, 9)
    if len(edges) == 0:
        assert (got["count"] == 0).all() and np.isnan(got["zscore"]).all()


def test_edge_dtypes_and_offset(g50k, engine):
    e64 = g50k["edges"].astype(np.int64)
    a = neighbourhood_enrichment(e64, g50k["types"], n_perms=50, seed=4, device=0)
    b = neighbourhood_enrichment(e64.astype(np.int32), g50k["types"], n_perms=50, seed=4, device=0)
    check(a, b)
    dev = engine.device
    e32 = torch.from_numpy(e64.astype(np.int32)).to(dev)
    t = torch.from_numpy(g50k["types"]).to(dev)
    buf = torch.zeros(e32.numel() + 1, dtype=torch.int32, device=dev)
    buf[1:] = e32.reshape(-1)
    shifted = buf[1:].view(-1, 2)
    assert shifted.data_ptr() % 16 == 4
    c = engine.nhood_enrichment(shifted, t, 5, 50, 4)
    check({k: v.cpu().numpy() for k, v in c.items()}, a)


def test_more_permutations_than_one_chunk(g50k, engine):
    n, p = len(g50k["types"]), 1400
    assert (p + 1) * n > 64 << 20  # PG_ENRICH_CHUNK_BYTES
    dev = engine.device
    e = torch.from_numpy(g50k["edges"].astype(np.int32)).to(dev)
    t = torch.from_numpy(g50k["types"]).to(dev)
    engine.profile(True)
    try:
        got = engine.nhood_enrichment(e, t, 5, p, 21)
        recs = engine.profile_records()
    finally:
        engine.profile(False)
    assert sum(name == "perm_labels_kernel" for name, _ in recs) > 1
    check({k: v.cpu().numpy() for k, v in got.items()}, oe.nhood_enrichment(g50k["edges"], g50k["types"], 5, p, 21))


def test_determinism(g50k, engine):
    dev = engine.device
    e = torch.from_numpy(g50k["edges"].astype(np.int32)).to(dev)
    t = torch.from_numpy(g50k["types"]).to(dev)
    a = {k: v.cpu().numpy() for k, v in engine.nhood_enrichment(e, t, 5, 300, 2 ** 64 - 1).items()}
    b = {k: v.cpu().numpy() for k, v in engine.nhood_enrichment(e, t, 5, 300, 2 ** 64 - 1).items()}
    fresh = Engine(0)
    try:
        c = {k: v.cpu().numpy() for k, v in fresh.nhood_enrichment(e, t, 5, 300, 2 ** 64 - 1).items()}
    finally:
        fresh.close()
    d = {k: v.cpu().numpy() for k, v in engine.nhood_enrichment(e, t, 5, 300, 2 ** 64 - 2).items()}
    for f in FIELDS:
        assert a[f].tobytes() == b[f].tobytes() == c[f].tobytes(), f
    assert np.array_equal(a["count"], d["count"])
    assert not np.array_equal(a["perm_mean"], d["perm_mean"])


def test_count_equals_type_interaction_matrix():
    xy, types, _ = synth.make_points(30_000, 55)
    g = build_radius_graph(xy, r=50.0, types=types, outputs="compact", device=0)
    got = neighbourhood_enrichment(g["edges"], types, n_perms=8, device=0)
    assert np.array_equal(got["count"], type_interaction_matrix(types, g["nbr_count"], device=0))
    k = build_knn_graph(xy, k=8, types=types, device=0)
    got = neighbourhood_enrichment(k["edges"], types, n_perms=8, device=0)
    assert np.array_equal(got["count"], type_interaction_matrix(types, k["nbr_count"], device=0))


def test_value_errors():
    types = np.array([1, 2, 3], np.int32)
    for bad in (np.array([[0, 3]]), np.array([[-1, 2]]), np.array([0, 1, 2]), np.array([[0, 1, 2]])):
        with pytest.raises(ValueError):
            neighbourhood_enrichment(bad, types, device=0)
    with pytest.raises(ValueError):
        neighbourhood_enrichment(np.array([[0, 1]]), types, n_perms=0, device=0)
    with pytest.raises(ValueError):
        neighbourhood_enrichment(np.array([[0, 1]]), types, n_types=17, device=0)


def test_full_c2_slide():
    xy, types, _ = synth.make_points(1_000_000, synth.SEEDS["C2"])
    g = build_radius_graph(xy, r=50.0, types=types, outputs="compact", device=0)
    assert len(g["edges"]) > 1_400_000
    run_and_check(g["edges"], types, 5, 20, 0)
