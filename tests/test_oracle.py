"""CPU: the oracle against the committed golden vectors (reference-generated, including the reference's own
add_wsi_coords_to_nuclei outputs and error message), the notebook's stored numbers (SURVEY Appendix D), brute force
and networkx."""
import numpy as np
import pytest

from conftest import GOLDEN, frames_from_golden
from oracle import graph as ograph
from oracle import morphology as omorph
from oracle import tile_to_wsi as omap
from path_gene_multimodal_b200 import synth


def test_tile_to_wsi_oracle_matches_reference_golden(golden_add_wsi):
    nuc, tiles, expected = frames_from_golden(golden_add_wsi)
    got = omap.add_wsi_coords_to_nuclei_oracle(nuc, tiles)
    assert list(got.columns) == golden_add_wsi["out_columns"]
    for c in golden_add_wsi["out_columns"]:
        if got[c].dtype.kind in "fi":
            assert np.array_equal(got[c].to_numpy(), expected[c].to_numpy()), c
            assert str(got[c].dtype) == golden_add_wsi["out_dtypes"][c], c
        else:
            assert got[c].tolist() == expected[c].tolist(), c
    # first occurrence of a duplicated tile stem wins (aggregated_hovernet_run.py:288-292)
    assert (got["tile_x"] < 999999).all()
    assert got["wsi_polygon"].iloc[3] is None and got["wsi_polygon"].iloc[10] is None


def test_tile_to_wsi_oracle_missing_tile_raises_like_reference(golden_add_wsi):
    # the frame the reference raised on when tests/golden/add_wsi_ref_error.txt was written (oracle/make_golden.py)
    nuc, tiles, _ = frames_from_golden(golden_add_wsi)
    nuc.loc[2, "tile_path"] = "/nowhere/patches/123_456.png"
    ref_msg = (GOLDEN / "add_wsi_ref_error.txt").read_text()
    with pytest.raises(ValueError) as ei:
        omap.add_wsi_coords_to_nuclei_oracle(nuc, tiles)
    head = "Some nuclei have tile_key with no matching tile coords:"
    assert ref_msg.startswith(head) and str(ei.value).startswith(head)
    assert "123_456" in ref_msg and "123_456" in str(ei.value)


def test_map_arrays_equals_frame_oracle():
    tab = synth.make_table(200, seed=3, dtype=np.float64)
    nuc, tiles = synth.to_frames(tab)
    df = omap.add_wsi_coords_to_nuclei_oracle(nuc, tiles)
    wsi_c, wsi_b, wsi_p = omap.map_arrays(tab.tile_x, tab.tile_y, tab.nuc_tile, tab.centroid, tab.bbox, tab.poly_off, tab.poly_xy)
    assert np.array_equal(df["wsi_centroid_x"].to_numpy(), wsi_c[:, 0])
    assert np.array_equal(df["wsi_bbox_ymax"].to_numpy(), wsi_b[:, 3])
    flat = np.array([p for poly in df["wsi_polygon"] for p in poly])
    assert np.array_equal(flat, wsi_p)


def test_radius_oracle_golden_and_bruteforce(golden_graph):
    coords = golden_graph["coords"]
    for r in (10.0, 25.0, 40.0):
        g = ograph.radius_graph(coords, r)
        assert np.array_equal(g["edges"], golden_graph[f"radius_{int(r)}_edges"])
        assert np.array_equal(g["dist"], golden_graph[f"radius_{int(r)}_dist"])
        assert np.array_equal(g["edges"], ograph.radius_graph_bruteforce(coords, r)["edges"])
        assert np.array_equal(g["edges"], ograph.radius_graph_notebook_loop(coords, r))
        assert g["edge_index"].shape == (2, 2 * len(g["edges"])) and g["edge_attr"].shape == (2 * len(g["edges"]), 1)
        assert g["edge_attr"].dtype == np.float32


def test_radius_inclusive_boundary():
    c = np.array([[0.0, 0.0], [3.0, 4.0], [5.0, 0.0], [5.0000000001, 12.0]])
    g = ograph.radius_graph(c, 5.0)
    assert g["edges"].tolist() == [[0, 1], [0, 2], [1, 2]]   # d == r is an edge (query_ball_tree is inclusive)


def test_knn_oracle_golden_bruteforce_ties(golden_graph):
    coords = golden_graph["coords"]
    for k in (5, 8, 16):
        idx, dist = ograph.knn(coords, k)
        assert np.array_equal(idx, golden_graph[f"knn_{k}_idx"]) and np.array_equal(dist, golden_graph[f"knn_{k}_dist"])
    bi, bd = ograph.knn_bruteforce(coords[:300], 7)
    idx, dist = ograph.knn(coords[:300], 7)
    assert np.array_equal(idx, bi) and np.array_equal(dist, bd)
    gx, gy = np.meshgrid(np.arange(9.0), np.arange(9.0))
    lat = np.stack([gx.ravel(), gy.ravel()], axis=1)
    lat = np.concatenate([lat, lat[:7]])
    for k in (1, 4, 5, 9):
        idx, dist = ograph.knn(lat, k)
        bi, bd = ograph.knn_bruteforce(lat, k)
        assert np.array_equal(idx, bi) and np.array_equal(dist, bd)
    with pytest.raises(ValueError):
        ograph.knn(lat[:4], 4)


def test_knn_notebook_distances(known_answers):
    c = np.array(known_answers["centroids_yx"])[:, ::-1]
    idx, dist = ograph.knn(c, 4)
    for key, val in known_answers["distances"].items():
        i, j = map(int, key.split(","))
        assert abs(dist[i][list(idx[i]).index(j)] - val) < 5e-7


def test_undirected_union_vs_networkx(golden_graph):
    coords, types = golden_graph["coords"], golden_graph["types"]
    idx, dist = ograph.knn(coords, 5)
    e, w, rp, col, ww = ograph.undirected_union(idx, dist)
    g = ograph.undirected_union_networkx(idx, dist)
    assert g.number_of_edges() == len(e) == len(golden_graph["knn_5_und_edges"])
    for (a, b), wt in zip(e, w):
        assert g.edges[int(a), int(b)]["weight"] == wt
    deg, stats = ograph.degree_stats(rp)
    assert np.array_equal(deg, [g.degree(i) for i in range(len(coords))])
    assert stats["sum"] == 2 * len(e) and stats["hist"].sum() == len(coords)
    comp = ograph.composition(rp, col, types, 5)
    assert np.array_equal(comp.sum(axis=1), deg)
    i = 17
    nb = list(g.neighbors(i))
    assert comp[i].tolist() == [sum(types[j] == t for j in nb) for t in range(1, 6)]
    nodes, sub = ograph.filter_types(e, types, (1, 2))
    h = g.subgraph([n for n in g.nodes if types[n] in (1, 2)])
    assert len(nodes) == h.number_of_nodes() and len(sub) == h.number_of_edges()   # cell 12


def test_notebook_ratio_of_union_edges(known_answers):
    # 101 nodes, k=5 -> 300 undirected of 505 directed edges in the notebook; uniform points give the same ratio
    rng = np.random.default_rng(0)
    fr = []
    for s in range(20):
        c = rng.random((101, 2)) * 521
        idx, dist = ograph.knn(c, 5)
        fr.append(len(ograph.undirected_union(idx, dist)[0]) / 505.0)
    assert abs(np.mean(fr) - known_answers["counts"]["knn_undirected_edges"] / 505.0) < 0.03


def test_derived_features_match_stored_notebook_rows(known_answers):
    rows = np.array(known_answers["morph_rows"], dtype=np.float64)
    cols = known_answers["morph_columns"]
    r = {c: rows[:, i] for i, c in enumerate(cols)}
    d = omorph.derived_features(r["area"], r["perimeter"], r["major"], r["minor"])
    for name in ("perimeter_area", "compactness", "roundness", "elongation", "eccentricity"):
        np.testing.assert_allclose(d[name], r[name], rtol=0, atol=2e-6, err_msg=name)


def test_polygon_features_analytic_shapes():
    rect = [[1.0, 2.0], [5.0, 2.0], [5.0, 5.0], [1.0, 5.0]]
    f = omorph.polygon_features_one(rect)
    assert f["area"] == 12.0 and f["perimeter"] == 14.0 and (f["centroid_x"], f["centroid_y"]) == (3.0, 3.5)
    assert abs(f["eccentricity"] - np.sqrt(1 - 9 / 16)) < 1e-12          # moments 16/12 and 9/12
    assert abs(f["major_axis_length"] - 4 * np.sqrt(16 / 12)) < 1e-12
    t = np.linspace(0, 2 * np.pi, 2001)[:-1]
    ell = np.stack([40 * np.cos(t) + 7, 25 * np.sin(t) - 3], axis=1)
    f = omorph.polygon_features_one(ell)
    assert abs(f["area"] - np.pi * 40 * 25) / (np.pi * 1000) < 1e-5
    assert abs(f["eccentricity"] - np.sqrt(1 - (25 / 40) ** 2)) < 1e-5
    assert abs(f["major_axis_length"] - 80) < 1e-3 and abs(f["minor_axis_length"] - 50) < 1e-3
    # closed ring == open ring; orientation does not matter
    g = omorph.polygon_features_one(rect + [rect[0]])
    h = omorph.polygon_features_one(rect[::-1])
    for k in ("area", "perimeter", "eccentricity", "circularity", "centroid_x"):
        assert f is not None and g[k] == omorph.polygon_features_one(rect)[k] and abs(h[k] - g[k]) < 1e-12
    a, l = omorph.geos_area_length(rect)
    assert (a, l) == (12.0, 14.0)


def test_polygon_features_csr_vs_scalar_and_degenerate():
    tab = synth.make_table(500, seed=1, v_lo=3, v_hi=40)
    f = omorph.polygon_features_csr(tab.poly_off, tab.poly_xy)
    for i in range(0, 500, 37):
        o = omorph.polygon_features_one(tab.poly_xy[tab.poly_off[i]:tab.poly_off[i + 1]])
        for k, v in o.items():
            assert np.isclose(v, f[k][i], rtol=1e-12, equal_nan=True), (i, k)
    off = np.array([0, 0, 1, 3, 6], dtype=np.int32)
    xy = np.array([[0, 0], [0, 0], [1, 1], [0, 0], [1, 1], [2, 2]], dtype=np.float64)
    f = omorph.polygon_features_csr(off, xy)
    assert np.isnan(f["area"][:3]).all() and f["area"][3] == 0.0 and np.isnan(f["eccentricity"][3])


def test_zscore_rule():
    assert omorph.zscore([2.0, 2.0, 2.0]).tolist() == [0.0, 0.0, 0.0]          # sigma == 0 -> 0.0 (ipynb:2905-2906)
    z = omorph.zscore([1.0, 2.0, 3.0])
    assert abs(z.std()) - 1 < 1e-12 and abs(z.mean()) < 1e-12


def test_feature_oracle_is_the_notebook_rule():
    # cell 21 / 23 semantics on a hand-checkable frame: NaN-skipping mean / std(ddof=0), constant -> 0.0,
    # one-hot columns only for the types present, ascending, before the z columns
    import pandas as pd
    from oracle import features as ofeat

    df = pd.DataFrame({"type": [3, 1, 3, 5], "area": [1.0, 2.0, 3.0, np.nan], "solidity": [0.5] * 4,
                       "elongation": [1.0, 1.0, 3.0, 3.0]})
    x, cols = ofeat.node_features(df)
    assert cols == ["type_1", "type_3", "type_5", "area_z", "solidity_z", "elongation_z"]
    assert x.dtype == np.float32 and x[:, :3].tolist() == [[0, 1, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]]
    s = np.sqrt(2.0 / 3.0)
    np.testing.assert_allclose(x[:3, 3], np.array([-1 / s, 0.0, 1 / s], dtype=np.float32), rtol=1e-6)
    assert np.isnan(x[3, 3]) and (x[:, 4] == 0).all() and x[:, 5].tolist() == [-1.0, -1.0, 1.0, 1.0]


def test_raster_oracle_on_analytic_shapes():
    # the restated skimage regionprops (skimage absent: parity unpinned, see oracle/raster.py) on shapes with known answers
    from oracle import raster as oraster

    m = np.zeros((40, 60), dtype=np.int32)
    m[3:8, 10:15] = 1                      # 5 x 5 square
    m[20:24, 5:17] = 2                     # 4 x 12 rectangle (rows x cols)
    rr, cc = np.mgrid[0:40, 0:60]
    m[(rr - 20) ** 2 + (cc - 40) ** 2 <= 12 ** 2] = 4   # disc r = 12 (label 3 absent)
    p = oraster.regionprops(m)
    assert p["label"].tolist() == [1, 2, 4] and p["area"][:2].tolist() == [25.0, 48.0]
    assert p["bbox"][0].tolist() == [3, 10, 8, 15] and p["bbox"][1].tolist() == [20, 5, 24, 17]
    assert p["centroid"][0].tolist() == [5.0, 12.0] and p["centroid"][1].tolist() == [21.5, 10.5]
    assert p["perimeter"][0] == 16.0 and p["perimeter"][1] == 28.0
    assert abs(p["eccentricity"][0]) < 1e-7
    assert np.isclose(p["major_axis_length"][1], 4 * np.sqrt((12 ** 2 - 1) / 12.0))     # variance of n pixels = (n^2-1)/12
    assert np.isclose(p["minor_axis_length"][1], 4 * np.sqrt((4 ** 2 - 1) / 12.0))
    assert np.isclose(p["eccentricity"][1], np.sqrt(1 - (4 ** 2 - 1) / (12 ** 2 - 1)))
    assert abs(p["orientation"][1]) == np.pi / 2                                        # long axis along the columns
    assert abs(p["perimeter"][2] / (2 * np.pi * 12) - 1) < 0.05 and p["eccentricity"][2] < 0.05
    assert abs(p["area"][2] / (np.pi * 144) - 1) < 0.03
    assert p["solidity"][0] == 1.0 and p["solidity"][1] == 1.0 and 0.93 < p["solidity"][2] <= 1.0   # convex shapes
    ell = np.zeros((9, 9), dtype=np.int32)
    ell[1:8, 1:3] = 1
    ell[6:8, 1:8] = 1                                   # an L: 7x2 + 2x5 = 24 pixels; its hull image has 2+3+4+5+6+7+7 = 34
    assert oraster.regionprops(ell)["solidity"][0] == 24 / 34


def test_contour_oracle_cycle_rule_equals_literal_assembly():
    # groundwork for SURVEY 8f-3 (second half, not built yet): the closed form the CUDA kernel will use - a contour
    # starts at the to-point of its last segment in square order, contours are numbered by their first segment -
    # reproduces skimage's dictionary bookkeeping (restated literally in oracle/contours.py) on random masks with
    # holes, several components and border contact; and the exact-arithmetic Douglas-Peucker is a valid member of
    # the family of results the float version can produce (same end points, every dropped vertex within tolerance)
    from oracle import contours as oc

    rng = np.random.default_rng(4)
    rr0, cc0 = np.mgrid[0:48, 0:48]
    for it in range(120):
        h, w = int(rng.integers(4, 40)), int(rng.integers(4, 40))
        rr, cc = rr0[:h, :w], cc0[:h, :w]
        m = np.zeros((h, w), dtype=bool)
        for _ in range(int(rng.integers(1, 5))):
            cy, cx = rng.uniform(-2, h + 2), rng.uniform(-2, w + 2)
            a, b, th = rng.uniform(2, 12), rng.uniform(1.5, 7), rng.uniform(0, np.pi)
            y, x = rr - cy, cc - cx
            u, v = x * np.cos(th) + y * np.sin(th), -x * np.sin(th) + y * np.cos(th)
            m |= (u / a) ** 2 + (v / b) ** 2 <= 1
        if rng.random() < 0.5:
            m[rng.integers(0, h), rng.integers(0, w)] ^= True
        cs = oc.find_contours(m)
        got = oc.longest_contour_by_cycles(m)
        if not cs:
            assert got is None
            continue
        want = max(cs, key=lambda c: c.shape[0])
        assert want.shape == got.shape and np.array_equal(want, got), it
        poly = np.stack([want[:, 1], want[:, 0]], axis=1)
        ex = oc.approximate_polygon_exact(poly, 0.5)
        assert np.array_equal(ex[0], poly[0]) and np.array_equal(ex[-1], poly[-1]) and len(ex) <= len(poly)
        fl = oc.approximate_polygon_float(poly, 0.5)
        assert abs(len(ex) - len(fl)) <= max(4, len(fl) // 4)          # same simplification up to tie choices
    # a 3 x 3 square: the 12-segment ring collapses to its 4 diagonal corners cut at the half-pixel + closing vertex
    sq = np.zeros((7, 7), dtype=bool)
    sq[2:5, 2:5] = True
    c = oc.find_contours(sq)[0]
    assert len(c) == 13 and np.array_equal(c[0], c[-1])
    assert oc.instance_polygons(sq.astype(np.int32))[1][0] == oc.instance_polygons(sq.astype(np.int32))[1][-1]
