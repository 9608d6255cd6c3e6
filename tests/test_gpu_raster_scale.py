"""K12 (raster region properties) and K13 (contour polygons) on slide-scale and adversarial instance maps.

The other f3 tests use full-map generators and oracles, which stop at a few hundred pixels a side. This file brings
its own pieces, each pinned by a CPU test below:

- `exact_props`: regionprops with the central moments formed from Python-integer raw moments, each numerator
  rounded once, then skimage's eigenvalue / eccentricity / axis / orientation expressions (oracle/raster.py). Its
  error does not grow with the region's distance from the origin, so it supports bars of 1e-12 at 46340 px.
- `stamp_blobs`: ellipses drawn inside their own bounding boxes, so a 46340-row map costs what its blobs cost.
- `regionprops_by_crop` / `polygons_by_crop`: oracle.raster / oracle.contours driven label by label over the
  `scipy.ndimage.find_objects` boxes instead of one full-map scan per label. The segment generator is vectorised
  (`contour_segments_fast`) and must emit oracle.contours.contour_segments' list exactly.
"""
from fractions import Fraction

import numpy as np
import pytest
from scipy import ndimage as ndi

from oracle import contours as ocont
from oracle import raster as oraster

SQRT2 = 1.4142135623730951
HALF = (1.0 + SQRT2) / 2.0


# ------------------------------------------------------------------------------------------------ helpers
def stamp_blobs(shape, n, seed, semi=(2.0, 14.0)):
    """int32 map with labels 1..n: ellipses with sub-pixel centres anywhere on the map (some cut by the border),
    semi-axes in `semi` and random angles, each evaluated only inside its own bounding box. Later blobs overwrite
    earlier ones, so regions touch, split into several components or vanish."""
    h, w = shape
    rng = np.random.default_rng(seed)
    m = np.zeros(shape, dtype=np.int32)
    for lab in range(1, n + 1):
        cy, cx = rng.uniform(0, h), rng.uniform(0, w)
        a, b, th = rng.uniform(*semi), rng.uniform(*semi), rng.uniform(0, np.pi)
        rad = int(np.ceil(max(a, b))) + 1
        r0, r1 = max(int(cy) - rad, 0), min(int(cy) + rad + 1, h)
        c0, c1 = max(int(cx) - rad, 0), min(int(cx) + rad + 1, w)
        if r0 >= r1 or c0 >= c1:
            continue
        y, x = np.mgrid[r0:r1, c0:c1]
        y, x = y - cy, x - cx
        u, v = x * np.cos(th) + y * np.sin(th), -x * np.sin(th) + y * np.cos(th)
        m[r0:r1, c0:c1][(u / a) ** 2 + (v / b) ** 2 <= 1.0] = lab
    return m


def _fma(a, b, c):
    """a * b + c rounded once (float64)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _perimeter_classes(img):
    """The three code classes of skimage's 4-neighbourhood perimeter (oracle/raster.py:_perimeter) as counts."""
    eroded = ndi.binary_erosion(img, ndi.generate_binary_structure(2, 1), border_value=0)
    border = img.astype(np.uint8) - eroded.astype(np.uint8)
    conv = ndi.convolve(border, np.array([[10, 2, 10], [2, 1, 2], [10, 2, 10]]), mode="constant", cval=0)
    hist = np.bincount(conv.ravel(), minlength=50)
    return int(hist[[5, 7, 15, 17, 25, 27]].sum()), int(hist[[21, 33]].sum()), int(hist[[13, 23]].sum())


def _labels_and_boxes(m):
    m = np.asarray(m)
    pos = np.where(m > 0, m, 0).astype(np.int64)
    return pos, ndi.find_objects(pos)


def exact_props(m):
    """dict of arrays, one entry per label present (ascending). Integers and centroids are exact; the tensor
    entries are (n sum r^2 - (sum r)^2) / n^2, ... with the Python-integer numerator rounded once; `perimeter` is
    p1 + p2 sqrt(2) + p3 (1 + sqrt(2)) / 2 evaluated plainly and `perimeter_fma` the same with both products fused
    (the two float64 evaluations a compiler may choose)."""
    pos, boxes = _labels_and_boxes(m)
    keys = ("label", "area", "bbox", "centroid", "perimeter", "perimeter_fma", "eccentricity", "major_axis_length",
            "minor_axis_length", "orientation", "solidity", "raw")
    out = {k: [] for k in keys}
    for i, sl in enumerate(boxes):
        if sl is None:
            continue
        lab = i + 1
        r0, c0 = sl[0].start, sl[1].start
        img = pos[sl] == lab
        rr, cc = np.nonzero(img)
        R, C = rr.astype(np.int64) + r0, cc.astype(np.int64) + c0
        n = len(R)
        sr, sc = int(R.sum()), int(C.sum())
        srr, scc, src = int((R * R).sum()), int((C * C).sum()), int((R * C).sum())
        num20, num02, num11 = n * srr - sr * sr, n * scc - sc * sc, n * src - sr * sc
        n2 = float(n) * float(n)
        ta, tb, tc = float(num02) / n2, -(float(num11) / n2), float(num20) / n2
        t = np.array([[ta, tb], [tb, tc]])
        l1, l2 = np.clip(np.sort(np.linalg.eigvalsh(t))[::-1], 0, None)
        if ta - tc == 0:
            orient = np.pi / 4 if tb < 0 else -np.pi / 4
        else:
            orient = 0.5 * np.arctan2(-2 * tb, tc - ta)
        p1, p2, p3 = _perimeter_classes(img)
        out["label"].append(lab)
        out["area"].append(n)
        out["bbox"].append([r0, c0, sl[0].stop, sl[1].stop])
        out["centroid"].append([float(Fraction(sr, n)), float(Fraction(sc, n))])
        out["perimeter"].append(float(p1) + float(p2) * SQRT2 + float(p3) * HALF)
        out["perimeter_fma"].append(_fma(p3, HALF, _fma(p2, SQRT2, p1)))
        out["eccentricity"].append(0.0 if l1 == 0 else float(np.sqrt(1 - l2 / l1)))
        out["major_axis_length"].append(4 * np.sqrt(l1))
        out["minor_axis_length"].append(4 * np.sqrt(l2))
        out["orientation"].append(orient)
        out["solidity"].append(n / oraster._convex_area(img))
        out["raw"].append((n, sr, sc, srr, scc, src))
    res = {k: np.array(v) for k, v in out.items() if k != "raw"}
    res["raw"] = out["raw"]
    if not out["label"]:
        res["bbox"] = np.zeros((0, 4), dtype=np.int64)
        res["centroid"] = np.zeros((0, 2))
    return res


def regionprops_by_crop(m):
    """oracle.raster.regionprops, one label at a time on its bounding-box crop (other labels zeroed), with the
    bbox and centroid moved back to map coordinates."""
    pos, boxes = _labels_and_boxes(m)
    parts = []
    for i, sl in enumerate(boxes):
        if sl is None:
            continue
        lab = i + 1
        r = oraster.regionprops(np.where(pos[sl] == lab, lab, 0))
        r["bbox"] = r["bbox"] + np.array([sl[0].start, sl[1].start, sl[0].start, sl[1].start])
        r["centroid"] = r["centroid"] + np.array([sl[0].start, sl[1].start])
        parts.append(r)
    if not parts:
        return oraster.regionprops(np.zeros((1, 1), dtype=np.int32))
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def contour_segments_fast(mask):
    """oracle.contours.contour_segments, vectorised over the squares: the same segments in the same order."""
    b = np.asarray(mask).astype(np.uint8)
    if b.shape[0] < 2 or b.shape[1] < 2:
        return []
    case = b[:-1, :-1] + 2 * b[:-1, 1:] + 4 * b[1:, :-1] + 8 * b[1:, 1:]
    rs, cs = np.nonzero((case != 0) & (case != 15))
    table = {1: ("tl",), 2: ("rt",), 3: ("rl",), 4: ("lb",), 5: ("tb",), 6: ("rt", "lb"), 7: ("rb",), 8: ("br",),
             9: ("tl", "br"), 10: ("bt",), 11: ("bl",), 12: ("lr",), 13: ("tr",), 14: ("lt",)}
    segs = []
    for r0, c0, k in zip(rs.tolist(), cs.tolist(), case[rs, cs].tolist()):
        pt = {"t": (r0, c0 + 0.5), "b": (r0 + 1, c0 + 0.5), "l": (r0 + 0.5, c0), "r": (r0 + 0.5, c0 + 1)}
        segs.extend((pt[s[0]], pt[s[1]]) for s in table[k])
    return segs


def polygons_by_crop(m, tolerance=0.5):
    """oracle.contours.instance_polygons(exact=True) label by label: its own crop rule (bounding box + 1 pixel,
    clipped at the image border, oracle/contours.py:190-192) taken from find_objects."""
    m = np.asarray(m)
    pos, boxes = _labels_and_boxes(m)
    h, w = m.shape
    out = {}
    for i, sl in enumerate(boxes):
        if sl is None:
            continue
        lab = i + 1
        r0, c0 = max(sl[0].start - 1, 0), max(sl[1].start - 1, 0)
        r1, c1 = min(sl[0].stop + 1, h), min(sl[1].stop + 1, w)
        contours = [c + np.array([r0, c0], dtype=np.float64)
                    for c in ocont.assemble_contours(contour_segments_fast(pos[r0:r1, c0:c1] == lab))]
        if not contours:
            continue
        contour = max(contours, key=lambda c: c.shape[0])
        out[lab] = ocont.approximate_polygon_exact(np.stack([contour[:, 1], contour[:, 0]], axis=1), tolerance).tolist()
    return out


def _axis_diff(a, b):
    d = np.abs(np.asarray(a) - np.asarray(b))
    return np.minimum(d, np.pi - d)


def assert_props_exact(got, want):
    """K12 (+ solidity) output of raster_regionprops against exact_props: integers, centroids, perimeter and
    solidity exact; eccentricity and axis lengths to 1e-12; orientation as an axis to 1e-12 where it is defined."""
    assert got["label"].tolist() == want["label"].tolist()
    assert np.array_equal(got["area"].to_numpy(), want["area"].astype(np.float64))
    assert np.array_equal(got[[f"bbox-{c}" for c in range(4)]].to_numpy(), want["bbox"])
    assert np.array_equal(got["centroid-0"].to_numpy(), want["centroid"][:, 0])
    assert np.array_equal(got["centroid-1"].to_numpy(), want["centroid"][:, 1])
    per = got["perimeter"].to_numpy()
    bad = (per != want["perimeter"]) & (per != want["perimeter_fma"])
    assert not bad.any(), (got["label"].to_numpy()[bad][:5], per[bad][:5], want["perimeter"][bad][:5])
    assert np.array_equal(got["solidity"].to_numpy(), want["solidity"])
    major = want["major_axis_length"]
    for name in ("eccentricity", "major_axis_length", "minor_axis_length"):
        g, e = got[name].to_numpy(), want[name]
        err = np.abs(g - e)
        bad = err > 1e-12 * np.abs(e) + 1e-12 * major
        assert not bad.any(), (name, got["label"].to_numpy()[bad][:5], got["bbox-0"].to_numpy()[bad][:5],
                               got["bbox-1"].to_numpy()[bad][:5], err[bad][:5], err.max())
    aniso = want["eccentricity"] > 1e-3
    d = _axis_diff(got["orientation"].to_numpy(), want["orientation"])
    bad = aniso & (d > 1e-12)
    assert not bad.any(), ("orientation", got["label"].to_numpy()[bad][:5], got["bbox-0"].to_numpy()[bad][:5],
                           got["bbox-1"].to_numpy()[bad][:5], d[bad][:5], d[aniso].max())


def _blob_maps():
    from test_cv2_pins import blobs
    from test_gpu_api import _blob_map

    return [_blob_map(521, 521, 120, seed=521), _blob_map(64, 37, 9, seed=37), blobs(256, 320, 90, seed=9),
            blobs(192, 224, 60, seed=11)]


def adversarial_maps():
    """name -> small instance map that drives K12 / K13 through their special cases."""
    maps = {}
    saddle = np.zeros((6, 7), dtype=np.int32)
    saddle[1, 1] = saddle[2, 2] = 1                                   # case 6 / 9 squares: diagonal-only pixels
    saddle[1, 5] = saddle[2, 4] = 2
    saddle[4, 0] = saddle[5, 1] = 3                                   # ... on the border as well
    maps["saddle_pairs"] = saddle
    cb = np.zeros((9, 10), dtype=np.int32)
    cb[1:8, 1:9] = np.where((np.add.outer(np.arange(7), np.arange(8)) % 2) == 0, 1, 2)
    maps["checkerboard"] = cb                                         # every square a saddle, two interleaved labels
    comp = np.zeros((12, 30), dtype=np.int32)
    comp[1:4, 1:4] = 1; comp[1:4, 6:9] = 1; comp[6:11, 2:5] = 1      # equal pair first, a longer one later
    comp[1:3, 12:14] = 2; comp[5:9, 12:16] = 2; comp[5:9, 20:24] = 2  # two equal longest: the first must win
    comp[1:4, 26:29] = 3; comp[9, 27] = 3                             # a longest one, then a single pixel
    maps["components"] = comp
    hole = np.zeros((10, 10), dtype=np.int32)
    hole[1:9, 1:9] = 1
    hole[3:6, 3:7] = 0
    maps["hole"] = hole
    nest = np.zeros((12, 12), dtype=np.int32)
    nest[1:11, 1:11] = 1
    nest[3:9, 3:9] = 0
    nest[4:8, 4:7] = 2                                                # a label inside another label's hole
    nest[6, 7] = 2
    maps["nested"] = nest
    bord = np.zeros((9, 11), dtype=np.int32)
    bord[0:3, 3:6] = 1                                                # one border
    bord[6:9, 0:3] = 2                                                # two borders (a corner)
    maps["borders_1_2"] = bord
    full = np.zeros((7, 8), dtype=np.int32)
    full[:, :] = 1
    full[2:4, 3:5] = 2                                                # label 1 touches all four borders, holed
    maps["borders_4"] = full
    lines = np.zeros((16, 16), dtype=np.int32)
    lines[1, 2:12] = 1                                                # horizontal
    lines[3:13, 14] = 2                                               # vertical
    idx = np.arange(8)
    lines[4 + idx, 1 + idx] = 3                                       # main diagonal
    lines[14 - idx, 4 + idx] = 4                                      # anti-diagonal
    maps["lines"] = lines
    one = np.zeros((5, 5), dtype=np.int32)
    one[2, 3] = 1
    maps["single_pixel"] = one
    sq = np.zeros((5, 6), dtype=np.int32)
    sq[1:3, 2:4] = 1
    maps["square_2x2"] = sq
    sparse = np.full((40, 40), -1, dtype=np.int64)                    # negative background value
    sparse[2:9, 3:8] = 1
    sparse[12:20, 5:9] = 7
    sparse[25:31, 20:33] = 1000
    sparse[33:38, 2:12] = 65536
    maps["sparse_ids"] = sparse
    maps["row_1xN"] = np.array([[0, 1, 1, 2, 0, 2, 2, 2, 3]], dtype=np.int32)
    maps["col_Nx1"] = np.array([[0, 1, 1, 2, 0, 2, 2, 2, 3]], dtype=np.int32).T.copy()
    maps["tiny_2x2"] = np.array([[1, 1], [2, 1]], dtype=np.int32)
    base = stamp_blobs((48, 40), 14, seed=3, semi=(2.0, 9.0))
    maps["uint16"] = base.astype(np.uint16)
    maps["int64"] = base.astype(np.int64)
    maps["float64"] = base.astype(np.float64)
    return maps


ADVERSARIAL = adversarial_maps()


# ------------------------------------------------------------------------------------------------ CPU: the helpers
@pytest.mark.parametrize("i", range(4))
def test_exact_oracle_matches_restated_skimage(i):
    m = _blob_maps()[i]
    want = oraster.regionprops(m)
    got = exact_props(m)
    assert got["label"].tolist() == want["label"].tolist()
    assert np.array_equal(got["area"], want["area"]) and np.array_equal(got["bbox"], want["bbox"])
    np.testing.assert_allclose(got["centroid"], want["centroid"], rtol=1e-13)
    np.testing.assert_allclose(got["perimeter"], want["perimeter"], rtol=1e-13)
    np.testing.assert_allclose(got["perimeter_fma"], want["perimeter"], rtol=1e-13)
    assert np.array_equal(got["solidity"], want["solidity"])
    major = want["major_axis_length"]
    for name in ("eccentricity", "major_axis_length", "minor_axis_length"):
        np.testing.assert_allclose(got[name], want[name], rtol=1e-13, atol=1e-13 * major.max(), err_msg=name)
    aniso = want["eccentricity"] > 1e-3
    assert _axis_diff(got["orientation"], want["orientation"])[aniso].max() <= 1e-13


def test_exact_oracle_far_from_the_origin():
    # the crop-frame restatement has no cancellation either: both agree at 46000 px, where the raw-moment
    # subtraction in float64 is off by 1e-7
    m = stamp_blobs((46340, 48), 300, seed=1)
    want = regionprops_by_crop(m)
    got = exact_props(m)
    assert got["label"].tolist() == want["label"].tolist() and got["bbox"][:, 0].max() > 46000
    for name in ("eccentricity", "major_axis_length", "minor_axis_length"):
        err = np.abs(got[name] - want[name])
        assert (err <= 1e-13 * (np.abs(want[name]) + want["major_axis_length"])).all(), (name, err.max())
    aniso = want["eccentricity"] > 1e-3
    assert _axis_diff(got["orientation"], want["orientation"])[aniso].max() <= 1e-13
    # and the raw moments far out really are where float64 subtraction loses digits
    n, sr, _, srr, _, _ = got["raw"][int(np.argmax(got["bbox"][:, 0]))]
    assert float(srr) - float(sr) * float(sr) / n != float(Fraction(n * srr - sr * sr, n))


def test_exact_oracle_against_opencv():
    cv2 = pytest.importorskip("cv2")
    m = stamp_blobs((300, 260), 80, seed=4)
    got = exact_props(m)
    for k, lab in enumerate(got["label"]):
        mo = cv2.moments((m == lab).astype(np.uint8), binaryImage=True)   # x = column, y = row
        assert mo["m00"] == got["area"][k]
        np.testing.assert_allclose(got["centroid"][k], [mo["m01"] / mo["m00"], mo["m10"] / mo["m00"]], rtol=1e-12)
        mu_rr, mu_cc, mu_rc = mo["mu02"] / mo["m00"], mo["mu20"] / mo["m00"], mo["mu11"] / mo["m00"]
        mm, cc = 0.5 * (mu_rr + mu_cc), np.hypot(0.5 * (mu_rr - mu_cc), mu_rc)
        l1, l2 = mm + cc, max(mm - cc, 0.0)
        np.testing.assert_allclose(got["major_axis_length"][k], 4 * np.sqrt(l1), rtol=1e-9)
        np.testing.assert_allclose(got["minor_axis_length"][k], 4 * np.sqrt(l2), rtol=1e-9, atol=1e-9)


def test_stamp_blobs_matches_full_map_ellipses():
    shape, n, seed = (70, 90), 25, 12
    m = stamp_blobs(shape, n, seed)
    rng = np.random.default_rng(seed)
    ref = np.zeros(shape, dtype=np.int32)
    yy, xx = np.mgrid[0:shape[0], 0:shape[1]]
    for lab in range(1, n + 1):
        cy, cx = rng.uniform(0, shape[0]), rng.uniform(0, shape[1])
        a, b, th = rng.uniform(2, 14), rng.uniform(2, 14), rng.uniform(0, np.pi)
        y, x = yy - cy, xx - cx
        u, v = x * np.cos(th) + y * np.sin(th), -x * np.sin(th) + y * np.cos(th)
        ref[(u / a) ** 2 + (v / b) ** 2 <= 1.0] = lab
    assert np.array_equal(m, ref)
    assert (m[0] > 0).any() or (m[-1] > 0).any() or (m[:, 0] > 0).any() or (m[:, -1] > 0).any()


@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
def test_fast_segments_match_oracle(name):
    m = np.asarray(ADVERSARIAL[name])
    for lab in [int(v) for v in np.unique(m) if v > 0]:
        assert contour_segments_fast(m == lab) == ocont.contour_segments(m == lab)


def test_crop_drivers_match_full_map_oracles():
    maps = [_blob_maps()[1], stamp_blobs((60, 50), 30, seed=8)] + [ADVERSARIAL[k] for k in sorted(ADVERSARIAL)]
    for m in maps:
        assert polygons_by_crop(m) == ocont.instance_polygons(m, 0.5, exact=True)
        want, got = oraster.regionprops(m), regionprops_by_crop(m)
        for k in want:
            assert np.array_equal(got[k], want[k]), k
    # a label on the image border keeps its open chain (no padding beyond the border)
    edge = np.zeros((6, 6), dtype=np.int32)
    edge[0, 1:4] = 1
    assert polygons_by_crop(edge)[1][0] != polygons_by_crop(edge)[1][-1]


# ------------------------------------------------------------------------------------------------ GPU
def _scale_strip(transpose):
    m = stamp_blobs((46340, 192), 3000, seed=46340)
    return m.T.copy() if transpose else m


@pytest.mark.gpu
@pytest.mark.parametrize("transpose", [False, True], ids=["rows_46340", "cols_46340"])
def test_raster_props_at_slide_scale(transpose):
    # K12 at the largest map side it accepts: tensor entries must not lose digits with the distance from the origin
    from path_gene_multimodal_b200 import raster_regionprops

    m = _scale_strip(transpose)
    want = exact_props(m)
    assert len(want["label"]) > 2500 and want["bbox"][:, 2 if not transpose else 3].max() > 46000
    assert_props_exact(raster_regionprops(m, device=0), want)


def _contour_scale_map(transpose):
    h, w = 16384, 1024
    m = stamp_blobs((h, w), 2000, seed=16384)
    n = int(m.max())
    r = np.arange(h)
    m[r, (r * (w - 1)) // (h - 1)] = n + 1               # a one-pixel diagonal across the map: many pieces
    m[2, 2:w - 2] = m[h - 3, 2:w - 2] = n + 2            # a one-pixel rectangle outline two pixels from the border
    m[2:h - 2, 2] = m[2:h - 2, w - 3] = n + 2
    m[0, 0] = m[h - 1, w - 1] = n + 3                    # two pixels at opposite corners
    return m.T.copy() if transpose else m


@pytest.mark.gpu
@pytest.mark.parametrize("transpose", [False, True], ids=["16384x1024", "1024x16384"])
def test_contours_at_scale(transpose):
    from path_gene_multimodal_b200 import instance_polygons, raster_regionprops

    m = _contour_scale_map(transpose)
    want = polygons_by_crop(m)
    got = instance_polygons(m, device=0)
    assert sorted(got) == sorted(want)
    bad = [lab for lab in want if got[lab] != want[lab]]
    assert not bad, (len(bad), bad[:5])                 # vertex for vertex, same start
    n = int(m.max())
    assert len(want[n - 1]) == 5 and len(want[n]) == 2  # the outline: a closed rectangle; one pixel: a diamond cut to 2
    assert_props_exact(raster_regionprops(m, device=0), exact_props(m))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
def test_adversarial_maps_through_both_kernels(name):
    from path_gene_multimodal_b200 import instance_polygons, raster_regionprops

    m = ADVERSARIAL[name]
    want = exact_props(m)
    got = raster_regionprops(m, device=0)
    assert_props_exact(got, want)
    assert instance_polygons(m, device=0) == polygons_by_crop(m)
    row = {int(l): k for k, l in enumerate(got["label"])}
    if name == "lines":
        for lab in (1, 2, 3, 4):
            k = row[lab]
            assert got["minor_axis_length"].iloc[k] == 0.0 and got["eccentricity"].iloc[k] == 1.0, lab
    if name == "square_2x2":
        assert abs(got["orientation"].iloc[0]) == np.pi / 4 and got["eccentricity"].iloc[0] == 0.0
    if name == "single_pixel":
        assert got["perimeter"].iloc[0] == 0.0 and got["major_axis_length"].iloc[0] == 0.0
    if name == "sparse_ids":
        assert got["label"].tolist() == [1, 7, 1000, 65536]


@pytest.mark.gpu
def test_contour_scratch_total_past_int32_raises():
    # 70 labels whose windows each span a 16384^2 map: 70 x 6.7e7 visited bytes is past 2^31
    from path_gene_multimodal_b200 import instance_polygons_csr

    h = 16384
    m = np.zeros((h, h), dtype=np.int32)
    lab = np.arange(1, 71)
    m[0, lab] = lab
    m[h - 1, h - 1 - lab] = lab
    with pytest.raises(RuntimeError, match="int32"):
        instance_polygons_csr(m, device=0)
    small = stamp_blobs((64, 64), 10, seed=2)              # the engine stays usable
    labels, off, xy = instance_polygons_csr(small, device=0)
    want = polygons_by_crop(small)
    assert labels.tolist() == sorted(want) and off[-1] == sum(len(v) for v in want.values())


@pytest.mark.gpu
def test_solidity_scratch_total_past_int32_raises():
    # 5800 labels spanning all 46340 rows: 5800 x 4 (2 x 46340 + 1) scratch entries is past 2^31
    from path_gene_multimodal_b200 import raster_regionprops

    h, w = 46340, 5800
    m = np.zeros((h, w), dtype=np.int32)
    lab = np.arange(1, w + 1, dtype=np.int32)
    m[0, :] = lab
    m[h - 1, :] = lab
    with pytest.raises(RuntimeError, match="int32"):
        raster_regionprops(m, device=0)
