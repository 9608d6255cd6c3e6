"""CPU: the convex-hull oracle (oracle/hull.py) pinned on independent engines - scipy's qhull and OpenCV's
convexHull / contourArea / moments - on synthetic nuclei rings and adversarial rings, the orientation sign convention
against the raster oracle, and the host plumbing of nuclei_morphology_table(hull=True) with oracle stand-ins for the
kernels."""
import contextlib
import math
import types

import cv2
import numpy as np
import pandas as pd
import pytest
from scipy.spatial import ConvexHull

from oracle import hull as ohull
from oracle import morphology as omorph
from oracle import raster as oraster
from path_gene_multimodal_b200 import synth


def _rings(off, xy):
    return [xy[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def test_convex_area_matches_qhull_and_opencv_on_synth_rings():
    off, xy = synth.make_polygons(4000, 11)
    got = ohull.ring_hull_csr(off, xy)
    qh = np.array([ConvexHull(r.astype(np.float64)).volume for r in _rings(off, xy)])
    cvh = np.array([cv2.contourArea(cv2.convexHull(r.astype(np.float32))) for r in _rings(off, xy)])
    np.testing.assert_allclose(got["convex_area"], qh, rtol=1e-12)
    np.testing.assert_allclose(got["convex_area"], cvh, rtol=1e-12)
    area = omorph.polygon_features_csr(off, xy)["area"]      # lattice rings: the float64 shoelace is exact
    assert np.array_equal(got["solidity"], area / got["convex_area"])
    assert np.all((got["solidity"] > 0.5) & (got["solidity"] <= 1.0))


ADVERSARIAL = {
    # name: (ring, convex area, |shoelace area|)
    "triangle": ([[0, 0], [4, 0], [0, 3]], 6.0, 6.0),
    "square_with_collinear_runs": ([[0, 0], [1, 0], [2, 0], [3, 0], [3, 1.5], [3, 3], [1.5, 3], [0, 3], [0, 1]], 9.0, 9.0),
    "duplicates": ([[0, 0], [0, 0], [2, 0], [2, 0], [2, 2], [0, 2], [0, 2]], 4.0, 4.0),
    "bow_tie": ([[0, 0], [2, 2], [2, 0], [0, 2]], 4.0, 0.0),
    "star": ([[math.cos(k * 4 * math.pi / 5), math.sin(k * 4 * math.pi / 5)] for k in range(5)], None, None),
    "concave_l": ([[0, 0], [2, 0], [2, 1], [1, 1], [1, 2], [0, 2]], 3.5, 3.0),
    "all_collinear": ([[0, 0], [1, 1], [2, 2], [3, 3]], 0.0, 0.0),
}


@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
def test_adversarial_rings(name):
    ring, ca, area = ADVERSARIAL[name]
    r = np.array(ring, dtype=np.float64)
    got_ca, got_so, got_or = ohull.ring_hull_one(r)
    if ca is None:  # the pentagram: its hull is the regular pentagon through the same points
        ca = ConvexHull(r).volume
        np.testing.assert_allclose(got_ca, ca, rtol=1e-13)
        assert 0 < got_so < 1  # |shoelace| of a self-intersecting ring: the centre counts twice, the points once
    else:
        assert got_ca == ca
        if area == 0.0:
            assert np.isnan(got_so) and np.isnan(got_or)
        else:
            assert got_so == area / ca
    # closed vs open, clockwise vs counter-clockwise: identical, bit for bit
    for variant in (np.vstack([r, r[:1]]), r[::-1], np.roll(r, 2, axis=0), np.vstack([r[::-1], r[-1:]])):
        v = ohull.ring_hull_one(variant)
        np.testing.assert_array_equal(np.array(v), np.array((got_ca, got_so, got_or)))


def test_nan_rules():
    nan3 = ohull.ring_hull_one([[0, 0], [1, 1]])
    assert all(np.isnan(nan3)) and all(np.isnan(ohull.ring_hull_one([])))
    ca, so, orient = ohull.ring_hull_one([[0, 0], [1, 0], [1, 0]])     # zero area and zero convex area
    assert ca == 0.0 and np.isnan(so) and np.isnan(orient)
    out = ohull.ring_hull_csr(np.array([0, 3, 3, 5, 8], dtype=np.int32),
                              np.array([[0, 0], [1, 0], [0, 1], [0, 0], [1, 1], [0, 0], [2, 0], [0, 2]], dtype=np.float32))
    assert np.isnan(out["convex_area"][1:3]).all() and out["convex_area"][[0, 3]].tolist() == [0.5, 2.0]
    assert out["solidity"][[0, 3]].tolist() == [1.0, 1.0]


def test_non_lattice_float64_rings_are_exact():
    rng = np.random.default_rng(4)
    for _ in range(200):
        r = rng.normal(size=(int(rng.integers(3, 40)), 2)) * rng.uniform(0.1, 1e3)
        ca, so, _ = ohull.ring_hull_one(r)
        np.testing.assert_allclose(ca, ConvexHull(r).volume, rtol=1e-12)
        area = omorph.polygon_features_one(r)["area"]
        np.testing.assert_allclose(so, area / ca, rtol=1e-12)


def _cv2_orientation(ring):
    m = cv2.moments(ring.astype(np.float32).reshape(-1, 1, 2))
    # skimage's (a, b, c) = (mu_xx, -mu_xy, mu_yy) from OpenCV's contour moments
    return 0.5 * math.atan2(2.0 * m["mu11"], m["mu02"] - m["mu20"]), m


def test_orientation_matches_opencv_moments():
    off, xy = synth.make_polygons(4000, 12)
    got = ohull.ring_hull_csr(off, xy)["orientation"]
    checked = 0
    for i, r in enumerate(_rings(off, xy)):
        ref, m = _cv2_orientation(r)
        aniso = math.hypot(m["mu20"] - m["mu02"], 2 * m["mu11"]) / (m["mu20"] + m["mu02"])
        if aniso > 1e-3:
            assert abs(got[i] - ref) < 1e-9, (i, got[i], ref)
            checked += 1
    assert checked > 3900


def _ellipse_ring(a, b, theta, cx=40.0, cy=40.0, n=400):
    t = np.linspace(0, 2 * np.pi, n, endpoint=False)
    ex, ey = a * np.cos(t), b * np.sin(t)
    return np.stack([cx + ex * np.cos(theta) - ey * np.sin(theta), cy + ex * np.sin(theta) + ey * np.cos(theta)], axis=1)


def test_orientation_sign_convention_and_raster_agreement():
    along_x = ohull.ring_hull_one(_ellipse_ring(12, 4, 0.0))[2]
    along_y = ohull.ring_hull_one(_ellipse_ring(4, 12, 0.0))[2]
    assert abs(abs(along_x) - math.pi / 2) < 1e-12 and abs(along_y) < 1e-12
    rows, cols = np.mgrid[0:80, 0:80]
    for theta in np.linspace(0.05, math.pi - 0.05, 9):
        ring = _ellipse_ring(15, 6, theta)
        poly = ohull.ring_hull_one(ring)[2]
        # x = column, y = row: the same ellipse rasterised
        dx, dy = cols - 40.0, rows - 40.0
        u = dx * math.cos(theta) + dy * math.sin(theta)
        v = -dx * math.sin(theta) + dy * math.cos(theta)
        mask = ((u / 15) ** 2 + (v / 6) ** 2 <= 1).astype(np.int32)
        ras = oraster.regionprops(mask)["orientation"][0]
        diff = (poly - ras + math.pi / 2) % math.pi - math.pi / 2   # orientations are axes: equal modulo pi
        assert abs(diff) < 0.03, (theta, poly, ras)  # pixelation of a 15 x 6 ellipse: at most 0.017 rad here


def _fake_map_morph_arrays(poly_off, poly_xy, write_polygons=True, extra=False, device=None, **_):
    f = omorph.polygon_features_csr(poly_off, poly_xy)
    return {"area": f["area"].astype(np.float32), "perimeter": f["perimeter"].astype(np.float32),
            "eccentricity": f["eccentricity"].astype(np.float32), "circularity": f["circularity"].astype(np.float32),
            "major_axis": f["major_axis_length"].astype(np.float32),
            "minor_axis": f["minor_axis_length"].astype(np.float32)}


def _fake_hull_arrays(poly_off, poly_xy, device=None):
    return ohull.ring_hull_csr(poly_off, poly_xy)


class _FakeEngine:
    """node_features on numpy: one-hot of the given values, then cell-21 z-scores."""
    device = None

    def node_features(self, feat, types_, values):
        cols = [] if values is None else [(types_ == v).astype(np.float64) for v in values]
        stats = []
        for c in (feat if feat is not None else []):
            mu, sd = np.nanmean(c), np.nanstd(c)
            stats.append([mu, sd])
            cols.append(np.zeros_like(c) if sd == 0 or np.isnan(sd) else (c - mu) / sd)
        return {"x": np.stack(cols, axis=1).astype(np.float32), "stats": np.array(stats)}


def test_nuclei_morphology_table_hull_columns_and_feature_matrix(monkeypatch):
    from path_gene_multimodal_b200 import graph_features, polygon_morphology

    monkeypatch.setattr(polygon_morphology, "map_morph_arrays", _fake_map_morph_arrays)
    monkeypatch.setattr(polygon_morphology, "hull_arrays", _fake_hull_arrays)
    off, xy = synth.make_polygons(101, 13)
    plain = polygon_morphology.nuclei_morphology_table(xy, poly_off=off)
    assert "solidity" not in plain.columns and "orientation" not in plain.columns
    df = polygon_morphology.nuclei_morphology_table(xy, poly_off=off, hull=True, zscore=True)
    assert list(df.columns[:8]) == ["inst_id", "area", "perimeter", "eccentricity", "solidity", "major_axis_length",
                                    "minor_axis_length", "orientation"]
    pd.testing.assert_frame_equal(df.drop(columns=["solidity", "orientation", "solidity_z"]),
                                  polygon_morphology.nuclei_morphology_table(xy, poly_off=off, zscore=True))
    ref = ohull.ring_hull_csr(off, xy)
    assert np.array_equal(df["solidity"].to_numpy(), ref["solidity"])
    assert "solidity_z" in df.columns

    monkeypatch.setattr(graph_features, "get_engine", lambda device=None: _FakeEngine())
    monkeypatch.setattr(graph_features, "_host", types.SimpleNamespace(
        as_int32=lambda a, name: np.asarray(a, dtype=np.int32), to_device=lambda a, dt, dev: np.asarray(a, dtype=dt),
        to_host_many=lambda d: d))
    monkeypatch.setattr(graph_features, "torch", types.SimpleNamespace(
        cuda=types.SimpleNamespace(device=lambda dev: contextlib.nullcontext())))
    df["type"] = np.arange(len(df)) % 5 + 1
    nf = graph_features.node_feature_matrix(df)
    assert nf["x"].shape == (101, 15) and len(nf["columns"]) == 15
    assert nf["columns"][:5] == [f"type_{t}" for t in range(1, 6)] and "solidity_z" in nf["columns"]
