"""GPU: the reference-style Python surface (DataFrame / array functions) against golden fixtures made by
the reference's own code and against the oracle."""
import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN, frames_from_golden
from oracle import graph as ograph
from oracle import morphology as omorph
from oracle import tile_to_wsi as omap
from path_gene_multimodal_b200 import synth

pytestmark = pytest.mark.gpu


def test_add_wsi_coords_matches_reference_golden(golden_add_wsi):
    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei

    nuc, tiles, expected = frames_from_golden(golden_add_wsi)
    nuc_before, tiles_before = nuc.copy(deep=True), tiles.copy(deep=True)
    got = add_wsi_coords_to_nuclei(nuc, tiles, tile_key_col_nuc="tile_path", tile_key_col_tiles="png_path")
    assert list(got.columns) == golden_add_wsi["out_columns"]
    for c in golden_add_wsi["out_columns"]:
        if c in ("polygon", "centroid", "bounding_box", "wsi_polygon"):
            assert got[c].tolist() == expected[c].tolist(), c                    # lists of exact floats / None
        elif got[c].dtype.kind in "fi":
            assert np.array_equal(got[c].to_numpy(), expected[c].to_numpy()), c  # bit-exact
            assert str(got[c].dtype) == golden_add_wsi["out_dtypes"][c], c
        else:
            assert got[c].tolist() == expected[c].tolist(), c
    pd.testing.assert_frame_equal(nuc, nuc_before)      # inputs untouched (aggregated_hovernet_run.py:281-282)
    pd.testing.assert_frame_equal(tiles, tiles_before)


def test_add_wsi_coords_missing_tile_raises(golden_add_wsi):
    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei

    nuc, tiles, _ = frames_from_golden(golden_add_wsi)
    nuc.loc[2, "tile_path"] = "/nowhere/patches/123_456.png"
    ref_msg = (GOLDEN / "add_wsi_ref_error.txt").read_text()
    with pytest.raises(ValueError) as ei:
        add_wsi_coords_to_nuclei(nuc, tiles)
    assert str(ei.value).startswith("Some nuclei have tile_key with no matching tile coords:")
    assert "123_456" in str(ei.value) and "123_456" in ref_msg


def test_add_wsi_coords_vs_oracle_2k_with_morphology():
    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei

    tab = synth.make_table(2000, seed=5, dtype=np.float64)
    nuc, tiles = synth.to_frames(tab, closed_rings=True)
    got = add_wsi_coords_to_nuclei(nuc, tiles, morphology=True)
    exp = omap.add_wsi_coords_to_nuclei_oracle(nuc, tiles)
    pd.testing.assert_frame_equal(got[exp.columns], exp)
    feat = omorph.polygon_features_csr(tab.poly_off, tab.poly_xy)
    for name in ("area", "perimeter", "circularity"):
        np.testing.assert_allclose(got[name], feat[name], rtol=1e-5)
    np.testing.assert_allclose(got["eccentricity"], feat["eccentricity"], rtol=1e-5, atol=2e-6)


def test_add_wsi_coords_empty_frame():
    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei

    tab = synth.make_table(10, seed=5, dtype=np.float64)
    nuc, tiles = synth.to_frames(tab)
    got = add_wsi_coords_to_nuclei(nuc.iloc[:0], tiles)
    assert len(got) == 0 and "wsi_polygon" in got.columns and "wsi_centroid_x" in got.columns


def test_process_nuclei_file_matches_reference_golden(tmp_path, golden_add_wsi):
    # file -> file (SURVEY 8f-1): the reference's Parquet layout in, the reference's two files out, CUDA in between
    from path_gene_multimodal_b200 import nuclei_io

    nuc, tiles, expected = frames_from_golden(golden_add_wsi)
    src, out_pq, out_csv = tmp_path / "local.parquet", tmp_path / "wsi.parquet", tmp_path / "wsi.csv"
    nuc.to_parquet(src, index=False)
    table = nuclei_io.process_nuclei_file(src, tiles, out_pq, out_csv, morphology=True)
    assert table.column_names[:len(golden_add_wsi["out_columns"])] == golden_add_wsi["out_columns"]
    ref_csv = tmp_path / "ref.csv"
    got = pd.read_parquet(out_pq)
    for c in golden_add_wsi["out_columns"]:
        if c in nuclei_io.LIST_COLUMNS:
            for a, b in zip(got[c], expected[c]):
                assert (a is None and b is None) or np.array_equal(np.array(a.tolist(), dtype=np.float64), np.array(b, dtype=np.float64)), c
        elif expected[c].dtype.kind in "fi":
            assert np.array_equal(got[c].to_numpy(), expected[c].to_numpy()), c
        else:
            assert got[c].tolist() == expected[c].tolist(), c
    expected.to_csv(ref_csv, index=False)
    twin = tmp_path / "twin.csv"
    nuclei_io.write_nuclei_table(table.select(golden_add_wsi["out_columns"]), csv_path=twin)
    assert twin.read_text() == ref_csv.read_text()           # the CSV twin, byte for byte
    assert out_csv.read_text().splitlines()[0].startswith(ref_csv.read_text().splitlines()[0])
    soa = nuclei_io.table_to_soa(table)
    feat = omorph.polygon_features_csr(soa.poly_off, soa.poly_xy)
    np.testing.assert_allclose(got["area"].to_numpy(), feat["area"], rtol=1e-5, equal_nan=True)


def test_polygon_morphology_tables(known_answers):
    from path_gene_multimodal_b200 import nuclei_morphology_table, polygon_morphology_table

    rings = [[[0, 0], [4, 0], [4, 3], [0, 3]], [[10, 10], [20, 10], [20, 20], [10, 20], [10, 10]],
             [[5 * np.cos(t) + 100, 5 * np.sin(t) - 7] for t in np.linspace(0, 2 * np.pi, 65)[:-1]]]
    tab = polygon_morphology_table(rings)
    assert list(tab.columns) == ["area_px2", "perimeter_px", "centroid_x", "centroid_y",
                                 "bbox_xmin", "bbox_ymin", "bbox_xmax", "bbox_ymax"]
    assert tab["area_px2"].tolist()[:2] == [12.0, 100.0] and tab["perimeter_px"].tolist()[:2] == [14.0, 40.0]
    np.testing.assert_allclose(tab.loc[0, ["centroid_x", "centroid_y"]].to_numpy(dtype=float), [2.0, 1.5], rtol=1e-12)
    assert tab.loc[1, ["bbox_xmin", "bbox_ymin", "bbox_xmax", "bbox_ymax"]].tolist() == [10.0, 10.0, 20.0, 20.0]
    np.testing.assert_allclose(tab.loc[2, "area_px2"], 0.5 * 64 * 25 * np.sin(2 * np.pi / 64), rtol=1e-5)
    for i, ring in enumerate(rings):
        a, l = omorph.geos_area_length(ring)
        np.testing.assert_allclose([tab.loc[i, "area_px2"], tab.loc[i, "perimeter_px"]], [a, l], rtol=1e-5)
    m = nuclei_morphology_table(rings, zscore=True)
    d = omorph.derived_features(m["area"], m["perimeter"], m["major_axis_length"], m["minor_axis_length"])
    for name in ("perimeter_area", "compactness", "roundness", "elongation"):
        np.testing.assert_allclose(m[name], d[name], rtol=1e-12)
    np.testing.assert_allclose(m["compactness"], m["circularity"], rtol=1e-5)
    np.testing.assert_allclose(m["area_z"], omorph.zscore(m["area"]), rtol=1e-12)


def test_build_radius_graph_api(golden_graph):
    from path_gene_multimodal_b200 import build_radius_graph

    coords, types = golden_graph["coords"], golden_graph["types"]
    g = build_radius_graph(coords, r=25.0, types=types, symmetric_csr=True)
    ref = ograph.radius_graph(coords, 25.0)
    assert g["edges"].dtype == np.int64 and np.array_equal(g["edges"], golden_graph["radius_25_edges"])
    assert np.array_equal(g["edge_index"], ref["edge_index"]) and g["edge_index"].shape == (2, 2 * len(ref["edges"]))
    assert g["edge_attr"].dtype == np.float32 and np.array_equal(g["edge_attr"], ref["edge_attr"])
    assert np.array_equal(g["row_ptr"], ref["row_ptr"]) and np.array_equal(g["col"], ref["col"])
    assert np.array_equal(g["nbr_count"], ograph.composition(ref["row_ptr"], ref["col"], types, 5))
    # the notebook's unit handling: r in micrometres on pixel coordinates scaled by mpp (ipynb:2046, :2966)
    g_um = build_radius_graph(coords, r=40.0, mpp=0.25)
    assert np.array_equal(g_um["edges"], ograph.radius_graph(coords * 0.25, 40.0)["edges"])


def test_build_knn_graph_api(golden_graph):
    from path_gene_multimodal_b200 import (build_knn_graph, degree_stats, filter_graph_by_type,
                                           neighbour_type_composition)

    coords, types = golden_graph["coords"], golden_graph["types"]
    g = build_knn_graph(coords, k=5, types=types)
    assert g["knn_neighbors"].dtype == np.int64 and np.array_equal(g["knn_neighbors"], golden_graph["knn_5_idx"])
    assert g["knn_neighbor_distances"].dtype == np.float64
    assert np.array_equal(g["knn_neighbor_distances"], golden_graph["knn_5_dist"])
    assert np.array_equal(g["edges"], golden_graph["knn_5_und_edges"])
    assert np.array_equal(g["weight"], golden_graph["knn_5_und_weight"])
    nx_g = ograph.undirected_union_networkx(g["knn_neighbors"], g["knn_neighbor_distances"])  # literal cell-11 loop
    assert nx_g.number_of_edges() == len(g["edges"])
    assert np.array_equal(g["degree"], np.array([nx_g.degree(i) for i in range(len(coords))]))
    comp = neighbour_type_composition(g["row_ptr"], g["col"], types)
    assert np.array_equal(comp, g["nbr_count"]) and np.array_equal(comp, ograph.composition(g["row_ptr"], g["col"], types, 5))
    st = degree_stats(g["row_ptr"])
    assert np.array_equal(st["degree"], g["degree"]) and st["max"] == g["degree"].max()
    nodes, sub = filter_graph_by_type(g["edges"], types, keep_types=(1, 2))
    on, oe = ograph.filter_types(g["edges"], types, (1, 2))
    assert np.array_equal(nodes, on) and np.array_equal(sub, oe)
    with pytest.raises(ValueError):
        build_knn_graph(coords[:5], k=5)


def test_non_finite_coordinates_raise(golden_graph):
    """cKDTree raises ValueError on NaN / inf; here the histogram kernel flags them (no host pass over the data)."""
    from path_gene_multimodal_b200 import build_knn_graph, build_radius_graph

    coords = np.array(golden_graph["coords"], dtype=np.float64, copy=True)
    for bad in (np.nan, np.inf):
        c = coords.copy()
        c[7, 1] = bad
        for bounds in (None, (0.0, 0.0, 600.0, 600.0)):
            with pytest.raises(ValueError, match="finite"):
                build_radius_graph(c, r=40.0, bounds=bounds)
            for cd in (np.int32, np.uint8, np.uint16):      # the compact path reads its flags with the output copies
                for _ in range(2):                           # (second call: with the capacity hint of the first)
                    with pytest.raises(ValueError, match="finite"):
                        build_radius_graph(c, r=40.0, bounds=bounds, outputs="compact", count_dtype=cd)
            with pytest.raises(ValueError, match="finite"):
                build_knn_graph(c, k=3, bounds=bounds)
    # and the handle is usable again afterwards
    g = build_radius_graph(coords, r=40.0)
    assert np.array_equal(g["edges"], ograph.radius_graph(coords, 40.0)["edges"])


def _feature_frame(n, seed):
    rng = np.random.default_rng(seed)
    df = pd.DataFrame({
        "type": rng.choice([1, 2, 3, 5], size=n, p=[0.5, 0.25, 0.2, 0.05]),     # type 4 absent: no type_4 column
        "area": rng.gamma(5.0, 40.0, size=n),
        "perimeter": rng.gamma(9.0, 6.0, size=n),
        "eccentricity": rng.random(n),
        "solidity": np.full(n, 0.75),                                            # constant column -> all 0.0
        "major_axis_length": rng.gamma(6.0, 3.0, size=n) + 1e6,                  # large offset: cancellation test
        "compactness": np.full(n, np.nan),                                       # empty column -> all 0.0
        "elongation": rng.random(n) + 1.0,
        "x_um": rng.random(n) * 0.25 * 508 * np.sqrt(n / 101.0),
        "y_um": rng.random(n) * 0.25 * 508 * np.sqrt(n / 101.0),
    })
    df.loc[rng.integers(0, n, size=max(1, n // 50)), "area"] = np.nan            # NaN rows are skipped by mean / std
    return df


@pytest.mark.parametrize("n", [1, 101, 50_000])
def test_node_feature_matrix_against_the_notebook_cells(n):
    from oracle import features as ofeat
    from path_gene_multimodal_b200 import node_feature_matrix

    df = _feature_frame(n, seed=40 + n)
    want, want_cols = ofeat.node_features(df)
    got = node_feature_matrix(df)
    assert got["columns"] == want_cols
    n_oh = sum(c.startswith("type_") for c in want_cols)
    assert got["x"].dtype == np.float32 and got["x"].shape == want.shape
    assert np.array_equal(got["x"][:, :n_oh], want[:, :n_oh])                    # one-hot: exact
    np.testing.assert_allclose(got["x"][:, n_oh:], want[:, n_oh:], rtol=1e-5, atol=1e-6, equal_nan=True)
    again = node_feature_matrix(df)
    assert np.array_equal(again["x"], got["x"], equal_nan=True)                  # deterministic reduction order
    for c in ("solidity_z", "compactness_z"):
        assert (got["x"][:, want_cols.index(c)] == 0.0).all()
    cols = [c[:-2] for c in want_cols[n_oh:]]
    np.testing.assert_allclose(got["mean"], [df[c].mean() for c in cols], rtol=1e-12, equal_nan=True)
    np.testing.assert_allclose(got["std"], [df[c].std(ddof=0) for c in cols], rtol=1e-9, atol=1e-12, equal_nan=True)


def test_node_feature_matrix_wide():
    # more columns than the shared-memory tile path takes: the per-element kernel
    from oracle import features as ofeat
    from path_gene_multimodal_b200 import node_feature_matrix

    rng = np.random.default_rng(3)
    n = 5000
    cols = [f"f{j}" for j in range(60)]
    df = pd.DataFrame(rng.normal(size=(n, 60)) * rng.uniform(0.1, 50, size=60) + rng.uniform(-100, 100, size=60), columns=cols)
    df["type"] = rng.integers(1, 6, size=n)
    want, want_cols = ofeat.node_features(df, cont_cols=cols)
    got = node_feature_matrix(df, cont_cols=cols)
    assert got["columns"] == want_cols and got["x"].shape == (n, 65)
    np.testing.assert_allclose(got["x"], want, rtol=1e-5, atol=1e-6)


def test_assemble_graph_data_cells_23_to_27():
    from oracle import features as ofeat
    from path_gene_multimodal_b200 import assemble_graph_data

    df = _feature_frame(3000, seed=7)
    data = assemble_graph_data(df, r=40.0)
    coords = df[["x_um", "y_um"]].to_numpy()
    ref = ograph.radius_graph(coords, 40.0)
    edges = ref["edges"]
    assert np.array_equal(data["edges"], edges)
    assert np.array_equal(data["edge_index"], np.hstack([edges.T, edges[:, ::-1].T]))          # SURVEY B-3 layout
    dists = np.linalg.norm(coords[edges[:, 0]] - coords[edges[:, 1]], axis=1)                   # cell 26
    want_attr = np.concatenate([dists[:, None], dists[:, None]], axis=0).astype(np.float32)
    assert np.array_equal(data["edge_attr"], want_attr)
    want_x, want_cols = ofeat.node_features(df)
    assert data["feat_cols"] == want_cols and data["x"].shape == want_x.shape
    np.testing.assert_allclose(data["x"], want_x, rtol=1e-5, atol=1e-6)
    assert np.array_equal(data["pos"], coords)


def test_graph_statistics_against_networkx():
    # README.md:133-136 "cell-cell interaction patterns", "degree, clustering, centrality" (SURVEY 8f-4)
    import networkx as nx
    from path_gene_multimodal_b200 import (build_knn_graph, build_radius_graph, clustering_coefficients,
                                           filter_graph_by_type, type_interaction_matrix)

    xy, types, _ = synth.make_points(4000, 21)
    for g in (build_radius_graph(xy, r=60.0, types=types, symmetric_csr=True), build_knn_graph(xy, k=6, types=types)):
        G = nx.Graph()
        G.add_nodes_from(range(len(xy)))
        G.add_edges_from(map(tuple, g["edges"]))
        st = clustering_coefficients(g["row_ptr"], g["col"])
        want = nx.clustering(G)
        # one correctly rounded division of the same exact integers on both sides: bit for bit
        assert np.array_equal(st["clustering"], [want[i] for i in range(len(xy))])
        tri = nx.triangles(G)
        assert np.array_equal(st["triangles"], [tri[i] for i in range(len(xy))])
        dc = nx.degree_centrality(G)
        np.testing.assert_allclose(st["degree_centrality"], [dc[i] for i in range(len(xy))], rtol=1e-12)
        inter = type_interaction_matrix(types, g["nbr_count"])
        e = g["edges"]
        want_i = np.zeros((5, 5), dtype=np.int64)
        np.add.at(want_i, (types[e[:, 0]] - 1, types[e[:, 1]] - 1), 1)
        np.add.at(want_i, (types[e[:, 1]] - 1, types[e[:, 0]] - 1), 1)
        assert np.array_equal(inter, want_i)
        # cell 12: the type-filtered sub-graph
        nodes, sub = filter_graph_by_type(e, types, keep_types=(1, 2))
        H = G.subgraph([i for i in range(len(xy)) if types[i] in (1, 2)])
        assert len(nodes) == H.number_of_nodes() and len(sub) == H.number_of_edges()
    empty = clustering_coefficients(np.zeros(4, dtype=np.int64), np.zeros(0, dtype=np.int64))
    assert (empty["clustering"] == 0).all() and (empty["triangles"] == 0).all()


def _blob_map(h, w, n, seed):
    rng = np.random.default_rng(seed)
    m = np.zeros((h, w), dtype=np.int32)
    rr, cc = np.mgrid[0:h, 0:w]
    for lab in range(1, n + 1):
        if lab % 17 == 0:
            continue                                            # absent labels
        cy, cx = rng.uniform(0, h), rng.uniform(0, w)           # some blobs are cut by the image border
        a, b, th = rng.uniform(3, 14), rng.uniform(2, 8), rng.uniform(0, np.pi)
        y, x = rr - cy, cc - cx
        u, v = x * np.cos(th) + y * np.sin(th), -x * np.sin(th) + y * np.cos(th)
        m[(u / a) ** 2 + (v / b) ** 2 <= 1] = lab               # later blobs overwrite earlier ones: ragged, touching regions
    m[5, 5] = n + 1                                             # a single-pixel region
    m[h - 1, 0:3] = n + 2                                       # a 1 x 3 line on the border
    return m


@pytest.mark.parametrize("shape", [(521, 521), (64, 37)])
def test_raster_regionprops_against_restated_skimage(shape):
    # SURVEY 8f-3: regionprops(inst_map) of aggregated_hovernet_run.py:172 / cell 18, one CUDA pass pair
    from oracle import raster as oraster
    from path_gene_multimodal_b200 import instance_bounding_boxes, raster_morphology_table, raster_regionprops

    m = _blob_map(*shape, n=120 if shape[0] > 100 else 9, seed=shape[1])
    want = oraster.regionprops(m)
    got = raster_regionprops(m)
    assert got["label"].tolist() == want["label"].tolist()
    assert np.array_equal(got["area"].to_numpy(), want["area"])
    assert np.array_equal(got[[f"bbox-{c}" for c in range(4)]].to_numpy(), want["bbox"])
    np.testing.assert_allclose(got[["centroid-0", "centroid-1"]].to_numpy(), want["centroid"], rtol=1e-13)
    np.testing.assert_allclose(got["perimeter"].to_numpy(), want["perimeter"], rtol=1e-13)
    for name in ("eccentricity", "major_axis_length", "minor_axis_length"):
        np.testing.assert_allclose(got[name].to_numpy(), want[name], rtol=1e-9, atol=1e-7, err_msg=name)
    assert np.array_equal(got["solidity"].to_numpy(), want["solidity"])           # integer counts: exact
    # orientation is ill-defined for (near-)isotropic regions; compare where the tensor is anisotropic
    aniso = want["eccentricity"] > 1e-3
    np.testing.assert_allclose(got["orientation"].to_numpy()[aniso], want["orientation"][aniso], rtol=1e-7, atol=1e-9)
    one = got[got["label"] == got["label"].max() - 1].iloc[0]   # the single pixel
    assert one["area"] == 1 and one["perimeter"] == 0.0 and one["eccentricity"] == 0.0 and one["major_axis_length"] == 0.0
    boxes = instance_bounding_boxes(m)
    l0 = int(want["label"][0])
    r0, c0, r1, c1 = want["bbox"][0]
    assert boxes[l0] == [c0, r0, c1, r1]                        # [x_min, y_min, x_max, y_max], aggregated_hovernet_run.py:179-180
    morph = raster_morphology_table(m, zscore=True)
    assert {"inst_id", "solidity", "perimeter_area", "compactness", "roundness", "elongation", "area_z", "solidity_z"} <= set(morph.columns)
    a, p_ = want["area"], want["perimeter"]
    np.testing.assert_allclose(morph["compactness"].to_numpy(), 4 * np.pi * a / np.clip(p_, 1, None) ** 2, rtol=1e-12)
    stacked = raster_regionprops(m[None])                        # (1, H, W) maps are squeezed like the reference does
    assert stacked["label"].tolist() == got["label"].tolist()


@pytest.mark.parametrize("shape,n", [((521, 521), 120), ((64, 37), 9), ((2, 2), 1), ((1, 9), 1)])
def test_instance_polygons_against_restated_skimage(shape, n):
    # SURVEY 8f-3, second half: find_contours + longest + approximate_polygon(0.5) per instance
    # (aggregated_hovernet_run.py:183-198), one CUDA thread per instance, exact-arithmetic tie rule (DESIGN.md)
    from oracle import contours as ocont
    from oracle import morphology as omorph2
    from path_gene_multimodal_b200 import instance_polygons, instance_polygons_csr

    if shape[0] > 2:
        m = _blob_map(*shape, n=n, seed=shape[1] + 1)
        m[30:37, 3:10] = n + 3                                             # a square ...
        m[32:35, 5:8] = 0                                                  # ... with a hole: two contours, the outer is longer
    else:
        m = np.ones(shape, dtype=np.int32)
    want = ocont.instance_polygons(m, 0.5, exact=True)
    got = instance_polygons(m)
    assert sorted(got) == sorted(want)
    for lab in want:
        assert got[lab] == want[lab], lab                                  # same vertices, same order, same start
        if len(want[lab]) > 1:
            assert got[lab][0] == got[lab][-1] or _touches_border(m, lab)  # closed unless cut by the image border
    labels, off, xy = instance_polygons_csr(m)
    assert labels.tolist() == sorted(want) and off[-1] == len(xy) == sum(len(v) for v in want.values())
    if shape[0] > 100:
        # the polygons are what the morphology kernel consumes: areas stay close to the pixel counts
        feat = omorph2.polygon_features_csr(off, xy)
        px = np.array([(m == l).sum() for l in labels], dtype=np.float64)
        big = px > 60
        assert np.all(np.abs(feat["area"][big] / px[big] - 1) < 0.25)
        # float vs exact Douglas-Peucker: same simplification up to tie choices (documented divergence)
        fl = ocont.instance_polygons(m, 0.5, exact=False)
        same = sum(fl[l] == want[l] for l in want)
        assert same >= len(want) // 2


def _touches_border(m, lab):
    rr, cc = np.nonzero(m == lab)
    return rr.min() == 0 or cc.min() == 0 or rr.max() == m.shape[0] - 1 or cc.max() == m.shape[1] - 1


def test_tile_nuclei_table_feeds_the_wsi_map():
    # run_hovernet_on_tile's table (aggregated_hovernet_run.py:135-223) from an instance map, then straight into the
    # a1-a3 drop-in: the two halves of the script path meet
    from oracle import contours as ocont
    from oracle import raster as oraster
    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei, tile_nuclei_table

    m = _blob_map(96, 80, n=14, seed=2)
    props = oraster.regionprops(m)
    labels = [int(l) for l in props["label"]]
    info = {str(l): [1 + l % 5, [0, float(c[1]), float(c[0])]] for l, c in zip(labels, props["centroid"])}
    info["9999"] = [2, [0, 1.0, 1.0]]                                       # listed by the classifier, absent from the map
    df = tile_nuclei_table(info, m, "/data/out/patches/1016_508.png")
    assert list(df.columns) == ["nuc_id", "inst_id", "type", "type_name", "bounding_box", "centroid", "polygon", "tile_name", "tile_path"]
    polys = ocont.instance_polygons(m)
    for _, row in df.iterrows():
        l = row["inst_id"]
        if l == 9999:
            assert row["bounding_box"] is None and row["polygon"] is None
            continue
        r0, c0, r1, c1 = props["bbox"][labels.index(l)]
        assert row["bounding_box"] == [c0, r0, c1, r1] and row["polygon"] == polys[l]
        assert row["type_name"] in ("neoplastic", "inflammatory", "connective", "dead", "epithelial")
    assert df["tile_name"].iloc[0] == "1016_508" and df["nuc_id"].nunique() == len(df)
    tiles = pd.DataFrame({"png_path": ["/data/out/patches/1016_508.png"], "x": [1016], "y": [508]})
    wsi = add_wsi_coords_to_nuclei(df[df["inst_id"] != 9999], tiles)
    first = wsi.iloc[0]
    assert first["wsi_polygon"][0] == [first["polygon"][0][0] + 1016.0, first["polygon"][0][1] + 508.0]
    assert first["wsi_bbox_xmin"] == first["bounding_box"][0] + 1016
