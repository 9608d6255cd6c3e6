"""GPU parity: every CUDA entry point of libpathgraph.so against the CPU oracle (oracle/).

Bars (north_star): bit-exact edge indices, degrees, type counts and (float64) distances;
float32 features within 1e-5 relative (eccentricity additionally 2e-6 absolute: for a ring whose
two principal moments coincide the value is sqrt of a rounding residue, see DESIGN.md).
"""
import numpy as np
import pytest
import torch

from oracle import graph as ograph
from oracle import morphology as omorph
from oracle import tile_to_wsi as omap
from path_gene_multimodal_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-5
ECC_ATOL = 2e-6


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


# ---------------------------------------------------------------- scan
@pytest.mark.parametrize("n", [0, 1, 31, 4095, 4096, 4097, 100_000, 1_234_567])
def test_exclusive_scan(engine, n):
    rng = np.random.default_rng(n)
    x = rng.integers(0, 50, size=n).astype(np.int32)
    out = engine.exclusive_scan(dev(x)).cpu().numpy()
    ref = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(x, out=ref[1:])
    assert np.array_equal(out, ref)


def test_exclusive_scan_repeated(engine):
    # epoch-tagged descriptors: back-to-back scans of different sizes must not see stale state
    rng = np.random.default_rng(5)
    for n in [70_000, 5_000, 300_000, 4096 * 3, 9]:
        x = rng.integers(0, 9, size=n).astype(np.int32)
        out = engine.exclusive_scan(dev(x)).cpu().numpy()
        assert out[-1] == x.sum() and np.array_equal(out[1:], np.cumsum(x))


# ---------------------------------------------------------------- K1
def _check_morph(res, off, xy, tab=None):
    feat = omorph.polygon_features_csr(off, xy)
    for name in ("area", "perimeter", "circularity"):
        np.testing.assert_allclose(res[name].cpu().numpy(), feat[name], rtol=RTOL, equal_nan=True, err_msg=name)
    np.testing.assert_allclose(res["eccentricity"].cpu().numpy(), feat["eccentricity"], rtol=RTOL, atol=ECC_ATOL,
                               equal_nan=True)
    if "major_axis" in res:
        np.testing.assert_allclose(res["major_axis"].cpu().numpy(), feat["major_axis_length"], rtol=RTOL, equal_nan=True)
        np.testing.assert_allclose(res["minor_axis"].cpu().numpy(), feat["minor_axis_length"], rtol=RTOL, atol=1e-5,
                                   equal_nan=True)
    return feat


@pytest.mark.parametrize("vt", [np.float32, np.float64])
def test_map_morph_table(engine, vt):
    tab = synth.make_table(20_000, seed=11, dtype=vt)
    res = engine.map_morph(dev(tab.poly_off), dev(tab.poly_xy), dev(tab.nuc_tile), dev(tab.tile_x), dev(tab.tile_y),
                           dev(tab.centroid), dev(tab.bbox), write_polygons=True, extra=True)
    wsi_c, wsi_b, wsi_p = omap.map_arrays(tab.tile_x, tab.tile_y, tab.nuc_tile, tab.centroid, tab.bbox, tab.poly_off,
                                          tab.poly_xy)
    assert np.array_equal(res["wsi_centroid"].cpu().numpy(), wsi_c)          # float64 add: bit-exact
    assert np.array_equal(res["wsi_bbox"].cpu().numpy().astype(np.int64), wsi_b)
    assert np.array_equal(res["wsi_poly_xy"].cpu().numpy().astype(np.float64), wsi_p)  # lattice coords: exact in f32 too
    feat = _check_morph(res, tab.poly_off, tab.poly_xy)
    tx = tab.tile_x[tab.nuc_tile].astype(np.float64)
    ty = tab.tile_y[tab.nuc_tile].astype(np.float64)
    np.testing.assert_allclose(res["centroid_x"].cpu().numpy(), feat["centroid_x"] + tx, rtol=1e-12)
    np.testing.assert_allclose(res["centroid_y"].cpu().numpy(), feat["centroid_y"] + ty, rtol=1e-12)
    bb = res["poly_bbox"].cpu().numpy()
    assert np.array_equal(bb[:, 0], feat["bbox_xmin"] + tx) and np.array_equal(bb[:, 3], feat["bbox_ymax"] + ty)


def test_map_morph_ragged_and_degenerate(engine):
    # empty rows, 1- and 2-vertex rows, a collinear ring, a long ring (> 32 vertices), closed == open ring
    rings = [
        [], [[1.0, 2.0]], [[0.0, 0.0], [3.0, 4.0]],
        [[0.0, 0.0], [1.0, 1.0], [2.0, 2.0]],                                   # zero area
        [[0.0, 0.0], [4.0, 0.0], [4.0, 3.0], [0.0, 3.0]],                       # rectangle 4x3
        [[0.0, 0.0], [4.0, 0.0], [4.0, 3.0], [0.0, 3.0], [0.0, 0.0]],           # same, explicitly closed
        [[0.0, 3.0], [4.0, 3.0], [4.0, 0.0], [0.0, 0.0]],                       # clockwise
        [[100000.5 + 10 * np.cos(t), 200000.25 + 6 * np.sin(t)] for t in np.linspace(0, 2 * np.pi, 257)[:-1]],
        [],
    ]
    off = np.zeros(len(rings) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(r) for r in rings])
    xy = np.array([p for r in rings for p in r], dtype=np.float64).reshape(-1, 2)
    res = engine.map_morph(dev(off), dev(xy), write_polygons=False, extra=True)
    feat = _check_morph(res, off, xy)
    area = res["area"].cpu().numpy()
    per = res["perimeter"].cpu().numpy()
    assert np.isnan(area[[0, 1, 2, 8]]).all() and area[3] == 0.0
    assert area[4] == 12.0 and area[5] == 12.0 and area[6] == 12.0 and per[4] == 14.0 and per[5] == 14.0
    ecc = res["eccentricity"].cpu().numpy()
    assert np.isnan(ecc[3]) and abs(ecc[4] - np.sqrt(1 - 9.0 / 16.0)) < 1e-6
    # ellipse with semi-axes 10 and 6: eccentricity -> sqrt(1 - 0.36)
    assert abs(ecc[7] - 0.8) < 1e-3
    assert np.allclose(res["centroid_x"].cpu().numpy()[7], 100000.5, atol=1e-6)
    assert feat["area"][4] == 12.0


@pytest.mark.parametrize("vt", [np.float32, np.float64])
def test_map_morph_staging_boundaries(engine, vt):
    # the warp's vertex range goes through a shared-memory slab by bulk copy (16-byte granularity) when it fits and
    # is walked straight from global memory (8-lane groups) when it does not: exercise odd range starts, vertex
    # arrays that are only 8-byte aligned, input / output with different alignment phases, rings closed explicitly
    # (33 vertices), and warps whose range is too long for the slab, all in one table
    n = 5000
    rng = np.random.default_rng(99)
    nv = rng.integers(3, 34, size=n)
    nv[32 * 7: 32 * 9] = rng.integers(40, 90, size=64)       # two warps past the slab capacity
    nv[32 * 20 + 5] = 1500                                    # one huge ring inside an otherwise ordinary warp
    nv[rng.integers(0, n, size=50)] = 0
    off = np.zeros(n + 1, dtype=np.int32)
    off[1:] = np.cumsum(nv)
    m = int(off[-1])
    owner = np.repeat(np.arange(n), nv)
    kth = np.arange(m) - off[owner]
    t = 2 * np.pi * kth / np.maximum(nv[owner], 1)
    a, b = rng.uniform(4, 12, n), rng.uniform(2, 4, n)
    cen = rng.uniform(0, 508, (n, 2))
    xy = np.stack([cen[owner, 0] + a[owner] * np.cos(t), cen[owner, 1] + b[owner] * np.sin(t)], axis=1)
    xy = (np.round(xy * 2) / 2).astype(vt)
    closed = np.flatnonzero(nv == 33)                         # make the 33-vertex rings explicitly closed
    xy[off[closed] + 32] = xy[off[closed]]
    tile_x = (np.arange(16) * 508).astype(np.int32)
    tile_y = (np.arange(16)[::-1] * 508).astype(np.int32)
    nuc_tile = rng.integers(0, 16, size=n).astype(np.int32)
    feat = omorph.polygon_features_csr(off, xy.astype(np.float64))
    want = xy.astype(np.float64) + np.stack([tile_x[nuc_tile][owner], tile_y[nuc_tile][owner]], axis=1)
    for in_shift, out_shift in ((0, 0), (1, 1), (1, 0)):
        buf = torch.zeros((m + 2, 2), dtype=dev(xy).dtype, device="cuda")
        src = buf[in_shift: in_shift + m]
        src.copy_(dev(xy))
        if vt is np.float64 and in_shift:                     # double2 rows stay 16-byte aligned under a row shift
            assert src.data_ptr() % 16 == 0
        dst_buf = torch.full((m + 2, 2), -7.0, dtype=src.dtype, device="cuda")
        dst = dst_buf[out_shift: out_shift + m]
        res = engine.map_morph(dev(off), src, dev(nuc_tile), dev(tile_x), dev(tile_y), write_polygons=True, extra=True,
                               out={"wsi_poly_xy": dst})
        assert res["wsi_poly_xy"].data_ptr() == dst.data_ptr()
        assert np.array_equal(dst.cpu().numpy().astype(np.float64), want), (in_shift, out_shift)
        guard = dst_buf.cpu().numpy()
        assert (guard[:out_shift] == -7.0).all() and (guard[out_shift + m:] == -7.0).all()   # nothing written outside
        for name in ("area", "perimeter", "circularity"):
            np.testing.assert_allclose(res[name].cpu().numpy(), feat[name], rtol=RTOL, equal_nan=True, err_msg=name)
        np.testing.assert_allclose(res["eccentricity"].cpu().numpy(), feat["eccentricity"], rtol=RTOL, atol=ECC_ATOL,
                                   equal_nan=True)
        bb = res["poly_bbox"].cpu().numpy()
        ok = nv >= 3
        assert np.array_equal(bb[ok, 0], feat["bbox_xmin"][ok] + tile_x[nuc_tile][ok])
        assert np.array_equal(bb[ok, 3], feat["bbox_ymax"][ok] + tile_y[nuc_tile][ok])


def test_map_morph_long_rings_use_bigger_slabs(engine):
    # rings of 40..90 vertices: the engine passes the mean ring length (pg_map_morph_hint) and the slabs grow, so the
    # staged path still applies; the same call after a hint for short rings takes the group path - same results
    n = 3000
    rng = np.random.default_rng(5)
    nv = rng.integers(40, 91, size=n)
    off = np.zeros(n + 1, dtype=np.int32)
    off[1:] = np.cumsum(nv)
    owner = np.repeat(np.arange(n), nv)
    t = 2 * np.pi * (np.arange(off[-1]) - off[owner]) / nv[owner]
    a, b = rng.uniform(10, 30, n), rng.uniform(5, 10, n)
    xy = np.stack([300 + a[owner] * np.cos(t), 200 + b[owner] * np.sin(t)], axis=1)
    xy = (np.round(xy * 2) / 2).astype(np.float32)
    big = engine.map_morph(dev(off), dev(xy), write_polygons=True, extra=True)
    _check_morph(big, off, xy)
    engine._check(engine.lib.pg_map_morph_hint(engine._h, n, 20 * n))      # pretend the rings are short
    fn = engine.lib.pg_map_morph_f32
    small = {k: torch.empty_like(v) for k, v in big.items()}
    from path_gene_multimodal_b200._lib import PgMorphOut
    import ctypes as C
    mo = PgMorphOut()
    for name in ("area", "perimeter", "eccentricity", "circularity", "major_axis", "minor_axis", "centroid_x", "centroid_y", "poly_bbox"):
        setattr(mo, name, small[name].data_ptr())
    engine._check(fn(engine._h, n, dev(off).data_ptr(), dev(xy).data_ptr(), None, None, None, None, None,
                     small["wsi_poly_xy"].data_ptr(), None, None, C.byref(mo), engine._stream()))
    torch.cuda.synchronize()
    assert torch.equal(small["wsi_poly_xy"], big["wsi_poly_xy"])
    for name in ("area", "perimeter", "circularity", "eccentricity"):
        np.testing.assert_allclose(small[name].cpu().numpy(), big[name].cpu().numpy(), rtol=RTOL, atol=ECC_ATOL, err_msg=name)


def test_map_morph_full_size_properties(engine):
    # C3 shape (reduced count so the oracle finishes in seconds is covered above); here: 2M x 32, invariants only
    n = 2_000_000
    off, xy = synth.make_polygons(n, seed=1003, v_fixed=32)
    rng = np.random.default_rng(3)
    side = 64
    tile_x = ((np.arange(side * side) % side) * 508).astype(np.int32)
    tile_y = ((np.arange(side * side) // side) * 508).astype(np.int32)
    nuc_tile = rng.integers(0, side * side, size=n).astype(np.int32)
    d_off, d_xy = dev(off), dev(xy)
    a = engine.map_morph(d_off, d_xy, dev(nuc_tile), dev(tile_x), dev(tile_y), write_polygons=True)
    b = engine.map_morph(d_off, d_xy, write_polygons=False)               # no shift
    c = engine.map_morph(d_off, a["wsi_poly_xy"], write_polygons=False)   # features of the shifted rings
    for name in ("area", "perimeter", "eccentricity", "circularity"):
        assert torch.equal(a[name], b[name]), name                       # translation invariance, bitwise (local frame)
        assert torch.equal(a[name], c[name]), name
    shift = torch.stack([dev(tile_x)[dev(nuc_tile).long()], dev(tile_y)[dev(nuc_tile).long()]], dim=1).float()
    owner = torch.repeat_interleave(torch.arange(n, device="cuda"), 32)
    assert torch.equal(a["wsi_poly_xy"], d_xy + shift[owner])
    assert bool((a["area"] > 0).all()) and bool((a["eccentricity"] < 1).all()) and bool((a["circularity"] <= 1.0001).all())


# ---------------------------------------------------------------- grid + radius
def _radius(engine, coords, types, r, upper, bounds=None, cell=None):
    from path_gene_multimodal_b200.engine import radius_cell

    engine.grid_build(dev(coords), dev(types), None, cell or radius_cell(r), bounds)
    return engine.radius_graph(r, upper=upper, n_types=5, want_dist32=True, want_dist64=True, want_edges=True)


def _check_radius(engine, coords, types, r, **kw):
    ref = ograph.radius_graph(coords, r)
    n = len(coords)
    g = _radius(engine, coords, types, r, upper=True, **kw)
    edges = g["edges"].cpu().numpy()
    assert np.array_equal(edges, ref["edges"])
    assert np.array_equal(g["dist64"].cpu().numpy(), ref["dist"])                    # bit-exact float64
    assert np.array_equal(g["dist32"].cpu().numpy(), ref["dist"].astype(np.float32))
    deg, stats = ograph.degree_stats(ref["row_ptr"])
    assert np.array_equal(g["degree"].cpu().numpy(), deg)
    assert np.array_equal(g["nbr_count"].cpu().numpy(), ograph.composition(ref["row_ptr"], ref["col"], types, 5))
    st = engine.decode_stats(g["stats"], g["hist"])
    assert (st["min"], st["max"], st["sum"], st["sumsq"], st["n"]) == (stats["min"], stats["max"], stats["sum"], stats["sumsq"], n)
    assert abs(st["mean"] - stats["mean"]) < 1e-12 and abs(st["std"] - stats["std"]) < 1e-9
    h = np.zeros(64, dtype=np.int64)
    np.add.at(h, np.minimum(deg, 63), 1)
    assert np.array_equal(st["hist"], h)
    s = _radius(engine, coords, types, r, upper=False, **kw)
    assert np.array_equal(s["row_ptr"].cpu().numpy(), ref["row_ptr"])
    assert np.array_equal(s["col"].cpu().numpy(), ref["col"])
    assert np.array_equal(s["dist64"].cpu().numpy(), ref["csr_dist"])
    return ref


def test_radius_golden(engine, golden_graph):
    coords, types = golden_graph["coords"], golden_graph["types"]
    for r in (10.0, 25.0, 40.0):
        ref = _check_radius(engine, coords, types, r)
        assert np.array_equal(ref["edges"], golden_graph[f"radius_{int(r)}_edges"])   # scipy's own output, committed


def test_radius_uniform_50k(engine):
    xy, types, side = synth.make_points(50_000, seed=21)
    _check_radius(engine, xy, types, 50.0)
    _check_radius(engine, xy, types, 50.0, bounds=(0.0, 0.0, float(side), float(side)))
    _check_radius(engine, xy, types, 50.0, cell=17.0)     # cell smaller than r: ring radius 3
    _check_radius(engine, xy, types, 50.0, cell=400.0)    # cell much larger than r


def test_radius_lattice_inclusive_and_duplicates(engine):
    gx, gy = np.meshgrid(np.arange(40.0) * 5.0, np.arange(40.0) * 5.0)
    c = np.stack([gx.ravel(), gy.ravel()], axis=1)
    c = np.concatenate([c, c[:100], c[:10]])  # duplicates (distance 0) are neighbours
    t = (np.arange(len(c)) % 5 + 1).astype(np.int32)
    _check_radius(engine, c, t, 5.0)      # distance exactly r is included
    _check_radius(engine, c, t, 10.0)
    _check_radius(engine, c, t, 0.0)      # only duplicates


def test_radius_heavy_rows(engine):
    # a dense clump: rows far longer than the fill kernel's chunk, plus isolated points
    rng = np.random.default_rng(8)
    c = np.concatenate([rng.normal(500.0, 3.0, size=(300, 2)), rng.random((2000, 2)) * 5000.0])
    t = rng.integers(1, 6, size=len(c)).astype(np.int32)
    _check_radius(engine, c, t, 40.0)


def test_radius_empty_and_tiny(engine):
    t1 = np.ones(1, dtype=np.int32)
    g = _radius(engine, np.zeros((1, 2)), t1, 5.0, upper=True)
    assert g["total"] == 0 and g["row_ptr"].cpu().tolist() == [0, 0] and g["degree"].cpu().tolist() == [0]
    g = _radius(engine, np.array([[0.0, 0.0], [3.0, 4.0]]), np.array([1, 2], dtype=np.int32), 5.0, upper=True)
    assert g["edges"].cpu().tolist() == [[0, 1]] and g["dist64"].cpu().tolist() == [5.0]
    assert g["nbr_count"].cpu().tolist() == [[0, 1, 0, 0, 0], [1, 0, 0, 0, 0]]
    g = _radius(engine, np.zeros((0, 2)), np.zeros(0, dtype=np.int32), 5.0, upper=True)
    assert g["total"] == 0


def test_radius_capacity_overflow(engine):
    from path_gene_multimodal_b200._lib import PathGraphError
    from path_gene_multimodal_b200.engine import radius_cell

    xy, types, _ = synth.make_points(5000, seed=2)
    engine.grid_build(dev(xy), dev(types), None, radius_cell(50.0), None)
    g = engine.radius_graph(50.0, upper=True, capacity=100_000)
    engine.check_overflow()
    total = int(g["row_ptr"][-1])
    ref = ograph.radius_graph(xy, 50.0)
    assert total == len(ref["edges"]) and np.array_equal(g["col"][:total].cpu().numpy(), ref["edges"][:, 1])
    engine.radius_graph(50.0, upper=True, capacity=10)
    with pytest.raises(PathGraphError):
        engine.check_overflow()
    engine.check_overflow()  # flag is cleared by the check


@pytest.mark.parametrize("upper", [True, False])
def test_radius_single_call_equals_count_fill(engine, upper):
    # pg_radius_graph (outputs given up front: the fill fused into the row pass) against count -> total -> fill
    from path_gene_multimodal_b200.engine import radius_cell

    for n, seed, r, with_gid in ((70_000, 31, 50.0, False), (3_000, 32, 200.0, True), (1, 33, 5.0, False), (0, 34, 5.0, False)):
        xy, types, _ = synth.make_points(max(n, 1), seed)
        xy, types = xy[:n], types[:n]
        gid = dev(np.random.default_rng(seed).permutation(n).astype(np.int32) + 7) if with_gid else None
        engine.grid_build(dev(xy) if n else torch.empty((0, 2), dtype=torch.float64, device="cuda"),
                          dev(types) if n else torch.empty((0,), dtype=torch.int32, device="cuda"), gid, radius_cell(r), None)
        a = engine.radius_graph(r, upper=upper, want_dist32=True, want_dist64=True, want_edges=True)
        e = int(a["total"])
        b = engine.radius_graph(r, upper=upper, want_dist32=True, want_dist64=True, want_edges=True, capacity=e + 100)
        engine.check_overflow()
        assert torch.equal(a["row_ptr"], b["row_ptr"]) and int(b["row_ptr"][-1]) == e
        for name in ("col", "dist32", "dist64", "edges"):
            assert torch.equal(a[name], b[name][:e]), (name, n, upper)
        for name in ("degree", "nbr_count", "stats", "hist"):
            assert torch.equal(a[name], b[name]), (name, n, upper)


# ---------------------------------------------------------------- kNN + union + composition
def _check_knn(engine, coords, types, k, cell=None, bounds=None):
    from path_gene_multimodal_b200.engine import default_knn_cell

    n = len(coords)
    ref_idx, ref_d = ograph.knn(coords, k)
    span = np.ptp(coords, axis=0)
    cell = cell or default_knn_cell(n, max(span[0], 1e-9) * max(span[1], 1e-9), k)
    engine.grid_build(dev(coords), dev(types), None, cell, bounds)
    kn = engine.knn(k, dist_dtype=torch.float64, both=True)
    assert np.array_equal(kn["knn_idx"].cpu().numpy(), ref_idx)
    assert np.array_equal(kn["dist64"].cpu().numpy(), ref_d)
    assert np.array_equal(kn["dist32"].cpu().numpy(), ref_d.astype(np.float32))
    e, w, rp, col, ww = ograph.undirected_union(ref_idx, ref_d)
    sym = engine.symmetrize(kn["knn_idx"], kn["dist64"], want_w32=True)
    assert np.array_equal(sym["row_ptr"].cpu().numpy(), rp)
    assert np.array_equal(sym["col"].cpu().numpy(), col)
    assert np.array_equal(sym["w64"].cpu().numpy(), ww)
    assert np.array_equal(sym["w32"].cpu().numpy(), ww.astype(np.float32))
    up = engine.csr_upper(sym["row_ptr"], sym["col"], sym["w64"])
    assert np.array_equal(up["edges"].cpu().numpy(), e) and np.array_equal(up["w64"].cpu().numpy(), w)
    comp = engine.compose_degree(sym["row_ptr"], sym["col"], dev(types), 5)
    deg, stats = ograph.degree_stats(rp)
    assert np.array_equal(comp["degree"].cpu().numpy(), deg)
    assert np.array_equal(comp["nbr_count"].cpu().numpy(), ograph.composition(rp, col, types, 5))
    st = engine.decode_stats(comp["stats"], comp["hist"])
    assert (st["min"], st["max"], st["sum"], st["sumsq"]) == (stats["min"], stats["max"], stats["sum"], stats["sumsq"])
    return ref_idx, ref_d, e, w


def test_knn_golden(engine, golden_graph, known_answers):
    coords, types = golden_graph["coords"], golden_graph["types"]
    for k in (5, 8, 16):
        idx, d, e, w = _check_knn(engine, coords, types, k)
        assert np.array_equal(idx, golden_graph[f"knn_{k}_idx"]) and np.array_equal(d, golden_graph[f"knn_{k}_dist"])
        assert np.array_equal(e, golden_graph[f"knn_{k}_und_edges"])
        # distances agree with scipy's own cKDTree.query(k+1) output (self at 0; tie order aside)
        full = np.sort(np.concatenate([np.zeros((len(coords), 1)), d], axis=1), axis=1)
        assert np.array_equal(full, golden_graph[f"knn_{k}_scipy_dist_sorted"])


def test_knn_notebook_distances(engine, known_answers):
    # D-1: the five centroids printed in the notebook; cell 11 swaps (y, x) -> Point(x, y)
    c = np.array(known_answers["centroids_yx"])[:, ::-1].copy()
    engine.grid_build(dev(c), None, None, 50.0, None)
    kn = engine.knn(4, dist_dtype=torch.float64)
    idx, d = kn["knn_idx"].cpu().numpy(), kn["dist"].cpu().numpy()
    for key, val in known_answers["distances"].items():
        i, j = map(int, key.split(","))
        got = d[i][list(idx[i]).index(j)]
        assert abs(got - val) < 5e-7, (key, got, val)


@pytest.mark.parametrize("k", [1, 5, 8, 16, 33])
def test_knn_uniform_30k(engine, k):
    xy, types, side = synth.make_points(30_000, seed=31)
    _check_knn(engine, xy, types, k)


def test_knn_cell_sizes_and_bounds(engine):
    xy, types, side = synth.make_points(20_000, seed=32)
    _check_knn(engine, xy, types, 8, cell=10.0)      # many rings
    _check_knn(engine, xy, types, 8, cell=1000.0)    # one big block
    _check_knn(engine, xy, types, 8, bounds=(0.0, 0.0, float(side), float(side)))
    _check_knn(engine, xy, types, 8, bounds=(1000.0, 1000.0, 3000.0, 3000.0))  # points outside the bounds are clamped


def test_knn_clustered_and_ties(engine):
    rng = np.random.default_rng(41)
    clusters = np.concatenate([rng.normal(c, 15.0, size=(800, 2)) for c in rng.random((12, 2)) * 20000.0])
    t = rng.integers(1, 6, size=len(clusters)).astype(np.int32)
    _check_knn(engine, clusters, t, 8)               # density holes: ring expansion across empty cells
    gx, gy = np.meshgrid(np.arange(30.0), np.arange(30.0))
    lat = np.stack([gx.ravel(), gy.ravel()], axis=1)
    lat = np.concatenate([lat, lat[:50]])
    tl = (np.arange(len(lat)) % 5 + 1).astype(np.int32)
    for k in (4, 5, 8):
        _check_knn(engine, lat, tl, k, cell=2.5)     # exact ties everywhere: (d^2, index) order


def test_knn_small_n(engine):
    c = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 2.0], [5.0, 5.0]])
    t = np.array([1, 2, 3, 4], dtype=np.int32)
    _check_knn(engine, c, t, 3)                      # k = N - 1
    from path_gene_multimodal_b200._lib import PathGraphError

    engine.grid_build(dev(c), dev(t), None, 1.0, None)
    with pytest.raises(PathGraphError):
        engine.knn(4)                                # k >= N is an error


def test_full_size_c2_against_scipy(engine):
    # BASELINE config 2 at full size: 1M nuclei, r = 50 px - scipy finishes in seconds, so compare outright
    xy, types, side = synth.make_points(1_000_000, seed=synth.SEEDS["C2"])
    ref = ograph.radius_graph(xy, 50.0)
    g = _radius(engine, xy, types, 50.0, upper=True, bounds=(0.0, 0.0, float(side), float(side)))
    assert np.array_equal(g["edges"].cpu().numpy(), ref["edges"])
    assert np.array_equal(g["dist32"].cpu().numpy(), ref["dist"].astype(np.float32))
    deg = np.diff(ref["row_ptr"])
    assert np.array_equal(g["degree"].cpu().numpy(), deg)
    assert np.array_equal(g["nbr_count"].cpu().numpy(), ograph.composition(ref["row_ptr"], ref["col"], types, 5))
    # size-independent properties
    assert int(g["degree"].sum()) == 2 * len(ref["edges"])
    e = g["edges"]
    assert bool((e[:, 0] < e[:, 1]).all())
    key = e[:, 0] * len(xy) + e[:, 1]
    assert bool((key[1:] > key[:-1]).all())          # strictly sorted by (i, j)
    # the single-call path the bench times (outputs given up front, fill fused into the row pass): same graph
    cap = len(ref["edges"]) + 1000
    f = engine.radius_graph(50.0, upper=True, n_types=5, want_dist32=True, want_edges=True, capacity=cap)
    engine.check_overflow()
    n_e = len(ref["edges"])
    assert int(f["row_ptr"][-1]) == n_e and torch.equal(f["edges"][:n_e], g["edges"]) and torch.equal(f["dist32"][:n_e], g["dist32"])
    assert torch.equal(f["degree"], g["degree"]) and torch.equal(f["nbr_count"], g["nbr_count"]) and torch.equal(f["row_ptr"], g["row_ptr"])


def test_full_size_c1_knn_against_scipy(engine):
    xy, types, side = synth.make_points(100_000, seed=synth.SEEDS["C1"])
    _check_knn(engine, xy, types, 8, bounds=(0.0, 0.0, float(side), float(side)))


# ---------------------------------------------------------------- fused union (K7 + edge list + K8 in one chain)
@pytest.mark.parametrize("k,dt", [(5, torch.float64), (8, torch.float32), (8, torch.float64), (16, torch.float32)])
def test_knn_union_fused_equals_separate_passes(engine, k, dt):
    from path_gene_multimodal_b200.engine import default_knn_cell

    xy, types, side = synth.make_points(30_000, 77 + k)
    xy[100:140] = xy[100]                                  # duplicates: ties by id, heavy reverse rows
    engine.grid_build(dev(xy), dev(types), None, default_knn_cell(len(xy), float(side) ** 2, k), None)
    kn = engine.knn(k, dist_dtype=dt)
    d = kn["dist"]
    sym = engine.symmetrize(kn["knn_idx"], d)
    up = engine.csr_upper(sym["row_ptr"], sym["col"], sym["w"])
    comp = engine.compose_degree(sym["row_ptr"], sym["col"], dev(types), 5)
    fu = engine.knn_union(kn["knn_idx"], d, types=dev(types), n_types=5)
    fs = engine.knn_union(kn["knn_idx"], d, types=dev(types), n_types=5, symmetric_dist=True)   # pg_knn lists: same weights
    assert torch.equal(fs["w"], fu["w"]) and torch.equal(fs["edge_w"], fu["edge_w"]) and torch.equal(fs["col"], fu["col"])
    assert torch.equal(fu["row_ptr"], sym["row_ptr"]) and torch.equal(fu["col"], sym["col"]) and torch.equal(fu["w"], sym["w"])
    assert torch.equal(fu["edges"], up["edges"])
    assert torch.equal(fu["edge_w"], up["w64"] if dt == torch.float64 else up["w32"])
    assert torch.equal(fu["nbr_count"], comp["nbr_count"]) and torch.equal(fu["degree"], comp["degree"])
    assert engine.decode_stats(fu["stats"], fu["hist"]).keys() == engine.decode_stats(comp["stats"], comp["hist"]).keys()
    a, b = engine.decode_stats(fu["stats"], fu["hist"]), engine.decode_stats(comp["stats"], comp["hist"])
    assert all(np.array_equal(a[q], b[q]) for q in a)
    # oracle: the notebook's union
    idx, dist = ograph.knn(xy, k)
    e, w, rp, col, _ = ograph.undirected_union(idx, dist)
    assert np.array_equal(fu["edges"].cpu().numpy(), e)
    # ids in another space (strips: global ids): rows permuted, lists / types by id
    n = len(xy)
    perm = torch.randperm(n, device="cuda", dtype=torch.int64)          # row r has id perm[r]
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n, device="cuda")
    idx_ids = perm[kn["knn_idx"].long()].int()                           # lists in id space, still in row order
    types_by_id = torch.empty(n, dtype=torch.int32, device="cuda")
    types_by_id[perm] = dev(types)
    fp = engine.knn_union(idx_ids.contiguous(), d, types=types_by_id, n_types=5, row_id=perm.int().contiguous(),
                          id_map=inv.int().contiguous())
    assert torch.equal(fp["row_ptr"], sym["row_ptr"]) and torch.equal(fp["degree"], comp["degree"])
    assert torch.equal(fp["nbr_count"], comp["nbr_count"])
    ee = fp["edges"]
    assert bool((ee[:, 0] < ee[:, 1]).all()) and ee.shape == up["edges"].shape
    back = torch.stack([inv[ee[:, 0]], inv[ee[:, 1]]], dim=1)
    back = torch.stack([back.min(dim=1).values, back.max(dim=1).values], dim=1)
    key = back[:, 0] * n + back[:, 1]
    assert torch.equal(back[torch.argsort(key)], up["edges"])


def test_knn_union_small_and_empty(engine):
    idx = dev(np.array([[1, 2], [0, 2], [0, 1], [0, 1]], dtype=np.int32))
    dist = dev(np.array([[1.0, 2.0], [1.0, 1.5], [2.0, 1.5], [3.0, 3.5]], dtype=np.float64))
    fu = engine.knn_union(idx, dist, types=dev(np.array([1, 2, 2, 5], dtype=np.int32)), n_types=5, hist_len=8)
    assert fu["row_ptr"].tolist() == [0, 3, 6, 8, 10] and fu["col"].tolist() == [1, 2, 3, 0, 2, 3, 0, 1, 0, 1]
    assert fu["edges"].tolist() == [[0, 1], [0, 2], [0, 3], [1, 2], [1, 3]]
    assert fu["edge_w"].tolist() == [1.0, 2.0, 3.0, 1.5, 3.5]
    assert fu["nbr_count"].tolist() == [[0, 2, 0, 0, 1], [1, 1, 0, 0, 1], [1, 1, 0, 0, 0], [1, 1, 0, 0, 0]]
    st = engine.decode_stats(fu["stats"], fu["hist"])
    assert (st["min"], st["max"], st["sum"], st["n"]) == (2, 3, 10, 4) and st["hist"][:4].tolist() == [0, 0, 2, 2]
    e0 = engine.knn_union(torch.empty((0, 3), dtype=torch.int32, device="cuda"),
                          torch.empty((0, 3), dtype=torch.float32, device="cuda"), hist_len=4)
    assert e0["row_ptr"].tolist() == [0] and e0["edges"].shape == (0, 2) and e0["hist"].tolist() == [0, 0, 0, 0]


def test_degree_statistics_of_the_empty_graph(engine, monkeypatch):
    # n = 0 through compose_degree, degree_stats and the kNN union: the statistics block (min, max, sum, sumsq, n) and
    # the histogram are all zero, with shared bins and past them. Outputs start at -1, so one left unwritten shows.
    from path_gene_multimodal_b200 import degree_stats

    monkeypatch.setattr(engine, "_empty", lambda shape, dtype: torch.full(shape, -1, dtype=dtype, device=engine.device))
    none = torch.empty(0, dtype=torch.int32, device="cuda")
    for hist_len in (4, 2049):
        cd = engine.compose_degree(torch.zeros(1, dtype=torch.int32, device="cuda"), none, none, 5, hist_len=hist_len)
        un = engine.knn_union(torch.empty((0, 3), dtype=torch.int32, device="cuda"),
                              torch.empty((0, 3), dtype=torch.float64, device="cuda"), types=none, hist_len=hist_len)
        for name, res in (("compose", cd), ("union", un)):
            assert res["stats"].tolist() == [0, 0, 0, 0], (name, hist_len)
            assert res["hist"].tolist() == [0] * hist_len, (name, hist_len)
        st = degree_stats(np.zeros(1, dtype=np.int64), hist_len=hist_len, device=0)
        assert (st["min"], st["max"], st["sum"], st["sumsq"], st["n"]) == (0, 0, 0, 0, 0), hist_len
        assert st["hist"].tolist() == [0] * hist_len and st["degree"].shape == (0,), hist_len


# ---------------------------------------------------------------- seeded fuzz against the brute-force oracles
def _fuzz_points(rng, n, kind):
    if kind == "uniform":
        xy = rng.random((n, 2)) * rng.choice([50.0, 500.0, 5000.0])
    elif kind == "clustered":                                   # tight clumps in a large empty frame (real tissue)
        c = rng.random((max(1, n // 40), 2)) * 4000.0
        xy = c[rng.integers(0, len(c), size=n)] + rng.normal(scale=rng.choice([1.0, 15.0]), size=(n, 2))
    elif kind == "lattice":                                     # exact ties everywhere
        s = int(np.ceil(np.sqrt(n)))
        g = np.stack(np.meshgrid(np.arange(s), np.arange(s)), axis=-1).reshape(-1, 2)[:n].astype(np.float64)
        xy = g * rng.choice([1.0, 7.5, 25.0])
    elif kind == "duplicates":
        base = rng.random((max(2, n // 5), 2)) * 300.0
        xy = base[rng.integers(0, len(base), size=n)]
    else:                                                       # a line: degenerate bounding box
        xy = np.stack([rng.random(n) * 1000.0, np.full(n, 3.25)], axis=1)
    return np.ascontiguousarray(xy[rng.permutation(n)], dtype=np.float64)


@pytest.mark.parametrize("seed", range(6))
def test_fuzz_radius_and_knn_against_bruteforce(engine, seed):
    rng = np.random.default_rng(1000 + seed)
    for case in range(14):
        kind = ["uniform", "clustered", "lattice", "duplicates", "line"][(seed + case) % 5]
        n = int(rng.choice([2, 3, 17, 64, 257, 900, 1500]))
        xy = _fuzz_points(rng, n, kind)
        types = rng.integers(0, 8, size=n).astype(np.int32)     # types outside 1..5 are counted in the degree only
        span = max(np.ptp(xy[:, 0]), np.ptp(xy[:, 1]), 1.0)
        r = float(rng.choice([0.0, 1.0, 7.5, 25.0, 0.05 * span, 0.3 * span]))
        cell = None if rng.random() < 0.5 else float(max(r, 1e-3) * rng.choice([0.4, 1.0, 2.7]))
        ref = ograph.radius_graph_bruteforce(xy, r)
        g = _radius(engine, xy, types, r, upper=True, cell=cell)
        tag = (seed, case, kind, n, r, cell)
        assert np.array_equal(g["edges"].cpu().numpy(), ref["edges"]), tag
        assert np.array_equal(g["dist64"].cpu().numpy(), ref["dist"]), tag
        assert np.array_equal(g["degree"].cpu().numpy(), np.diff(ref["row_ptr"])), tag
        assert np.array_equal(g["nbr_count"].cpu().numpy(), ograph.composition(ref["row_ptr"], ref["col"], types, 5)), tag
        s = _radius(engine, xy, types, r, upper=False, cell=cell)
        assert np.array_equal(s["col"].cpu().numpy(), ref["col"]) and np.array_equal(s["row_ptr"].cpu().numpy(), ref["row_ptr"]), tag
        if n >= 3:
            k = int(rng.choice([1, 2, 5, 8, 13, 16, 20, 40]))
            k = min(k, n - 1)
            from path_gene_multimodal_b200.engine import default_knn_cell

            kcell = default_knn_cell(n, span * span, k) * float(rng.choice([0.5, 1.0, 3.0]))
            engine.grid_build(dev(xy), dev(types), None, kcell, None)
            kn = engine.knn(k, dist_dtype=torch.float64)
            idx, dist = ograph.knn_bruteforce(xy, k)
            assert np.array_equal(kn["knn_idx"].cpu().numpy(), idx), tag + (k,)
            assert np.array_equal(kn["dist"].cpu().numpy(), dist), tag + (k,)
            fu = engine.knn_union(kn["knn_idx"], kn["dist"], types=dev(types), n_types=5, symmetric_dist=True)
            e, w, rp, col, _ = ograph.undirected_union(idx, dist)
            assert np.array_equal(fu["edges"].cpu().numpy(), e) and np.array_equal(fu["edge_w"].cpu().numpy(), w), tag + (k,)
            assert np.array_equal(fu["nbr_count"].cpu().numpy(), ograph.composition(rp, col, types, 5)), tag + (k,)
    engine.check_overflow()
