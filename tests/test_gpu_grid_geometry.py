"""GPU: the uniform grid (K2 histogram, K3 cell scan, K4 scatter) and the queries that walk it (K5 kNN, K6 radius walk and
row pass, K7 union, pg_grid_export) on adversarial geometry, bit for bit against the oracle.

The rest of the suite builds grids over points in [0, side]^2 with cells of about r. The correctness arguments of the grid
also rest on regimes those builds never reach, and each test below names the one it is aimed at:
* coordinates far from the origin, where the binning (v - x0) * (1 / cell) rounds at large magnitude;
* thin grids: nx = 1 (no left / right column in the 3x3 walk), ny = 1, and ny on both sides of a multiple of the 32-row
  strip, where the FAST walk's second pass reaches across a strip edge (rows ly == 0 / 31);
* the cell-cap doubling loop of pg_grid_build (few points spread very wide);
* caller bounds that leave most points outside the grid (clamped into border cells), a single-point box, a far box;
* cells far smaller than r (the pg_visit_block walk, R up to 200) up to a ball that covers the whole grid many times
  over (R capped at the grid's extent);
* cells a hair above r at cell coordinates above 10^6 (the slack of the host's ring radius);
* queries on a prefix of the points (ghost points behind the rows, as the strip builds append them);
* one handle rebuilt 30 times (workspace growth and shrink, stale counters / scan descriptors / parking hints);
* the cell scan across look-back groups (256 tiles x 4096 items) and pg_grid_export as the cell order;
* a coordinate span that overflows double (rejected, and the handle keeps working).

Bars: bit-exact row_ptr / col / edges / degree / type counts / statistics / float64 distances (float32 = the rounded
float64), kNN lists in (d^2, id) order. The CPU tests at the top pin this file's own references against oracle/graph.py.
"""
import math

import numpy as np
import pytest
import torch
from scipy.spatial import cKDTree

from oracle import graph as ograph
from path_gene_multimodal_b200.engine import default_knn_cell, radius_cell

STRIP = 32                   # PG_STRIP: grid rows per strip of the cell order
SCAN_GROUP = 256 * 4096      # K3: tiles of 4096 items, 256 tiles per look-back group
MIN_CAP = 1 << 20            # pg_grid_build: the cell cap is max(8 n, 2^20) (and at most 2^28)
N_TYPES = 5
HIST_LEN = 64


# ---------------------------------------------------------------------------------------------------- helpers
def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def cell_coords(xy, info):
    """The grid's own binning rule (pg_cell_coord): floor((v - v0) * (1 / cell)), clamped into the grid."""
    inv = 1.0 / info["cell"]
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    with np.errstate(invalid="ignore", over="ignore"):
        tx = np.floor((xy[:, 0] - info["x0"]) * inv)
        ty = np.floor((xy[:, 1] - info["y0"]) * inv)
    cx = np.clip(tx, 0, info["nx"] - 1).astype(np.int64)
    cy = np.clip(ty, 0, info["ny"] - 1).astype(np.int64)
    return cx, cy


def padded_cells(info):
    """Cells of the grid including the padding rows up to whole strips (the length of the scanned histogram)."""
    return info["nx"] * (-(-info["ny"] // STRIP)) * STRIP


def cell_index(info, cx, cy):
    """pg_cell_index: strip by strip, column-major inside a strip."""
    return ((cy // STRIP) * info["nx"] + cx) * STRIP + cy % STRIP


EPS = float(np.finfo(np.float64).eps)


def ring_radius(r, info):
    """The radius walk's block radius (pg_radius.cu ring_radius): cells a point within r can be away along an axis,
    with a slack that grows with the grid (the binning's rounding grows with the cell coordinate), capped at the grid's
    extent (a block that large covers the grid)."""
    big = max(info["nx"], info["ny"])
    rr = math.ceil(r * (1.0 / info["cell"]) * (1.0 + 1e-9) + 1e-9 + 4.0 * big * EPS)
    return big if rr >= big else max(rr, 1)


def ring_radius_fixed_slack(r, info):
    """The ring radius with only the fixed 1e-9 slack (what the library used before the grid-scaled term)."""
    return max(math.ceil(r * (1.0 / info["cell"]) * (1.0 + 1e-9) + 1e-9), 1)


def binade_top_pairs(r, cell, k, span=200_000):
    """Pairs (ya, ya + r) exactly r apart with ya * (1 / cell) just below 2^k, where the float64 spacing doubles: the
    second point's cell coordinate rounds up by half the wider spacing. Returns (ya, yb, row_a, row_b)."""
    b = (2.0 ** k) * cell
    ya = np.unique(b + np.arange(-span, span // 100) * (np.spacing(b) / 8))
    yb = ya + r
    ok = (yb - ya) == r
    ya, yb = ya[ok], yb[ok]
    return ya, yb, np.floor(ya * (1.0 / cell)), np.floor(yb * (1.0 / cell))


def _d2(a, b):
    dx = a[..., 0] - b[..., 0]
    dy = a[..., 1] - b[..., 1]
    return dx * dx + dy * dy


def _pairs_within(xy, r, nq):
    """(src, dst, d2): every (row i < nq, point j != i) with d2 <= r*r in float64, rows ascending."""
    n = len(xy)
    if nq == 0 or n == 0:
        z = np.zeros(0, dtype=np.int64)
        return z, z, np.zeros(0)
    r2 = np.float64(r) * np.float64(r)
    if n <= 3000:
        d2 = _d2(xy[:nq, None, :], xy[None, :, :])
        src, dst = np.nonzero(d2 <= r2)
        d2 = d2[src, dst]
    else:
        tree = cKDTree(xy)
        lists = tree.query_ball_point(xy[:nq], r * (1.0 + 1e-9) + 1e-300, workers=-1)
        cnt = np.fromiter((len(p) for p in lists), dtype=np.int64, count=nq)
        src = np.repeat(np.arange(nq, dtype=np.int64), cnt)
        dst = np.fromiter((j for p in lists for j in p), dtype=np.int64, count=int(cnt.sum()))
        d2 = _d2(xy[src], xy[dst])
        keep = d2 <= r2                                      # the exact acceptance test, not the tree's
        src, dst, d2 = src[keep], dst[keep], d2[keep]
    keep = src != dst
    return src[keep], dst[keep], d2[keep]


def radius_ref(xy, r, types, nq=None, ids=None, n_types=N_TYPES):
    """The radius graph of the rows 0..nq-1 over all points, keyed by ``ids`` (default: the point index).

    Symmetric rows hold every neighbour's id ascending; upper rows the ids above the row's own; ``edges`` are the upper
    rows' (id, id) pairs in row order. Degree and type counts are over all neighbours."""
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    n = len(xy)
    nq = n if nq is None else nq
    ids = np.arange(n, dtype=np.int64) if ids is None else np.asarray(ids, dtype=np.int64)
    src, dst, d2 = _pairs_within(xy, r, nq)
    order = np.lexsort((ids[dst], src))
    src, dst, d2 = src[order], dst[order], d2[order]
    cnt = np.bincount(src, minlength=nq)
    row_ptr = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(cnt, out=row_ptr[1:])
    up = ids[dst] > ids[src]
    up_ptr = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(np.bincount(src[up], minlength=nq), out=up_ptr[1:])
    t = np.asarray(types, dtype=np.int64)[dst]
    ok = (t >= 1) & (t <= n_types)
    comp = np.zeros((nq, n_types), dtype=np.int32)
    np.add.at(comp, (src[ok], t[ok] - 1), 1)
    return {"row_ptr": row_ptr, "col": ids[dst], "dist": np.sqrt(d2), "up_ptr": up_ptr,
            "edges": np.stack([ids[src[up]], ids[dst[up]]], axis=1), "edge_dist": np.sqrt(d2[up]),
            "degree": cnt.astype(np.int32), "comp": comp}


def knn_ref(xy, k, nq=None, ids=None):
    """kNN lists of the rows 0..nq-1 over all points in (d^2, id) order, self removed by index: (ids [nq,k], dist)."""
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    n = len(xy)
    nq = n if nq is None else nq
    ids = np.arange(n, dtype=np.int64) if ids is None else np.asarray(ids, dtype=np.int64)
    if nq == 0:
        return np.zeros((0, k), dtype=np.int64), np.zeros((0, k))
    tree = cKDTree(xy)
    kk = min(n, k + 4)
    _, nb = tree.query(xy[:nq], k=kk, workers=-1)
    nb = nb.reshape(nq, kk)
    d2 = _d2(xy[:nq, None, :], xy[nb])
    d2 = np.where(nb == np.arange(nq)[:, None], np.inf, d2)  # self sorts last and is never taken
    order = np.lexsort((ids[nb], d2), axis=-1)
    nb, d2 = np.take_along_axis(nb, order, axis=1), np.take_along_axis(d2, order, axis=1)
    out_i, out_d = ids[nb[:, :k]], d2[:, :k].copy()
    # a row is settled when its k-th candidate is strictly nearer than the farthest one fetched (every point not
    # fetched is at least that far); the others (ties across the fetched set, duplicates) are redone exactly
    far = np.where(np.isinf(d2), -1.0, d2).max(axis=1)
    redo = np.nonzero(~(out_d[:, -1] < far * (1.0 - 1e-12)) | (kk < k + 1))[0]
    for i in redo:
        cand = np.arange(n) if n <= 4096 else np.array(
            tree.query_ball_point(xy[i], math.sqrt(out_d[i, -1]) * (1.0 + 1e-9) + 1e-300), dtype=np.int64)
        cand = cand[cand != i]
        cd2 = _d2(xy[i][None, :], xy[cand])
        o = np.lexsort((ids[cand], cd2))[:k]
        out_i[i], out_d[i] = ids[cand[o]], cd2[o]
    return out_i, np.sqrt(out_d)


def assert_stats(engine, stats_t, hist_t, deg, tag):
    st = engine.decode_stats(stats_t, hist_t)
    deg = np.asarray(deg, dtype=np.int64)
    if len(deg) == 0:
        assert st["n"] == 0 and st["sum"] == 0 and (st["hist"] == 0).all(), tag
        return
    assert (st["min"], st["max"], st["sum"], st["sumsq"], st["n"]) == (
        int(deg.min()), int(deg.max()), int(deg.sum()), int((deg * deg).sum()), len(deg)), tag
    assert np.array_equal(st["hist"], np.bincount(np.minimum(deg, HIST_LEN - 1), minlength=HIST_LEN)), tag


def check_radius(engine, ref, r, tag, calls=("count", "fused")):
    """Upper and symmetric CSR through count -> total -> fill and through the fused capacity= call."""
    for upper in (True, False):
        for call in calls:
            t = tag + (("upper" if upper else "sym"), call)
            want_ptr = ref["up_ptr"] if upper else ref["row_ptr"]
            e = int(want_ptr[-1])
            kw = dict(upper=upper, n_types=N_TYPES, hist_len=HIST_LEN, want_dist32=True, want_dist64=True,
                      want_edges=upper)
            if call == "count":
                g = engine.radius_graph(r, **kw)
                assert int(g["total"]) == e, t + (int(g["total"]), e)
            else:
                g = engine.radius_graph(r, capacity=e + 64, **kw)
                engine.check_overflow()
            got_ptr = g["row_ptr"].cpu().numpy()
            assert int(got_ptr[-1]) == e, t + (int(got_ptr[-1]), e)
            assert np.array_equal(got_ptr, want_ptr), t
            col = g["col"][:e].cpu().numpy()
            d64 = g["dist64"][:e].cpu().numpy()
            if upper:
                assert np.array_equal(g["edges"][:e].cpu().numpy(), ref["edges"]), t
                assert np.array_equal(col, ref["edges"][:, 1]), t
                want_d = ref["edge_dist"]
            else:
                assert np.array_equal(col, ref["col"]), t
                want_d = ref["dist"]
            assert np.array_equal(d64, want_d), t
            assert np.array_equal(g["dist32"][:e].cpu().numpy(), want_d.astype(np.float32)), t
            assert np.array_equal(g["degree"].cpu().numpy(), ref["degree"]), t
            assert np.array_equal(g["nbr_count"].cpu().numpy(), ref["comp"]), t
            assert_stats(engine, g["stats"], g["hist"], ref["degree"], t)


def check_knn(engine, xy, k, tag, nq=None, ids=None):
    want_i, want_d = knn_ref(xy, k, nq, ids)
    kn = engine.knn(k, dist_dtype=torch.float64, both=True)
    assert np.array_equal(kn["knn_idx"].cpu().numpy(), want_i), tag + (k,)
    assert np.array_equal(kn["dist64"].cpu().numpy(), want_d), tag + (k,)
    assert np.array_equal(kn["dist32"].cpu().numpy(), want_d.astype(np.float32)), tag + (k,)
    return kn, want_i, want_d


def check_knn_union(engine, xy, types, k, tag):
    """kNN lists, then the fused union (i<j edges, symmetric CSR, composition, degree statistics) of them."""
    kn, idx, dist = check_knn(engine, xy, k, tag)
    e, w, rp, col, ww = ograph.undirected_union(idx, dist)
    u = engine.knn_union(kn["knn_idx"], kn["dist64"], types=dev(types), n_types=N_TYPES, hist_len=HIST_LEN,
                         symmetric_dist=True)
    t = tag + ("union", k)
    assert np.array_equal(u["row_ptr"].cpu().numpy(), rp) and np.array_equal(u["col"].cpu().numpy(), col), t
    assert np.array_equal(u["w"].cpu().numpy(), ww), t
    assert np.array_equal(u["edges"].cpu().numpy(), e) and np.array_equal(u["edge_w"].cpu().numpy(), w), t
    assert np.array_equal(u["nbr_count"].cpu().numpy(), ograph.composition(rp, col, types, N_TYPES)), t
    assert np.array_equal(u["degree"].cpu().numpy(), np.diff(rp)), t
    assert_stats(engine, u["stats"], u["hist"], np.diff(rp), t)


def check_export(engine, xy, types, info, ids=None):
    """pg_grid_export is the cell order: a permutation of the input whose cell index never decreases, and every cell
    holds exactly numpy's binning of the input (within a cell the order is atomic arrival order: compared as sets).
    The cell boundaries of the export are the scanned cell_start array."""
    n = len(xy)
    ids = np.arange(n, dtype=np.int64) if ids is None else np.asarray(ids, dtype=np.int64)
    ex_xy, ex_t, ex_id = (a.cpu().numpy() for a in engine.grid_export())
    ex_id = ex_id.astype(np.int64)
    by_id = np.argsort(ids)                                  # id -> input index
    src = by_id[np.searchsorted(ids[by_id], ex_id)]
    assert np.array_equal(np.sort(ex_id), np.sort(ids))      # a permutation
    assert np.array_equal(ex_xy, xy[src]) and np.array_equal(ex_t, np.asarray(types)[src])
    c_in = cell_index(info, *cell_coords(xy, info))
    c_ex = cell_index(info, *cell_coords(ex_xy, info))
    assert (np.diff(c_ex) >= 0).all()                        # cell order
    cells = padded_cells(info)
    assert c_in.max(initial=0) < cells
    start = np.zeros(cells + 1, dtype=np.int64)
    np.cumsum(np.bincount(c_in, minlength=cells), out=start[1:])
    assert np.array_equal(np.searchsorted(c_ex, np.arange(cells + 1)), start)   # cell_start
    # the same point set in every cell: sort both sides by (cell, id)
    o_in = np.lexsort((ids, c_in))
    o_ex = np.lexsort((ex_id, c_ex))
    assert np.array_equal(ids[o_in], ex_id[o_ex])


def half_pixel_points(n, side, seed):
    """Points on the half-pixel lattice (exact in float64 at any shift below 2^51), with duplicates."""
    rng = np.random.default_rng(seed)
    q = rng.integers(0, int(2 * side) + 1, size=(n, 2)).astype(np.float64) * 0.5
    q[: n // 50] = q[n // 2: n // 2 + n // 50]
    return q, rng.integers(-1, 8, size=n).astype(np.int32)


# ---------------------------------------------------------------------------------------------------- CPU tests
def test_references_against_the_oracle():
    rng = np.random.default_rng(0)
    xy = np.round(rng.random((700, 2)) * 60.0 * 2) / 2        # half-pixel lattice: ties at d == r
    types = rng.integers(0, 7, size=700).astype(np.int32)
    for r in (3.0, 5.0):
        o = ograph.radius_graph_bruteforce(xy, r)
        ref = radius_ref(xy, r, types)
        assert np.array_equal(ref["row_ptr"], o["row_ptr"]) and np.array_equal(ref["col"], o["col"])
        assert np.array_equal(ref["dist"], o["csr_dist"]) and np.array_equal(ref["edges"], o["edges"])
        assert np.array_equal(ref["edge_dist"], o["dist"])
        assert np.array_equal(ref["comp"], ograph.composition(o["row_ptr"], o["col"], types, N_TYPES))
    # the tree path (n > 3000) equals the dense path
    big = np.round(rng.random((3500, 2)) * 200.0 * 2) / 2
    tb = rng.integers(0, 7, size=3500).astype(np.int32)
    a = radius_ref(big, 4.0, tb)
    o = ograph.radius_graph_bruteforce(big, 4.0)
    assert np.array_equal(a["edges"], o["edges"]) and np.array_equal(a["col"], o["col"])
    for k in (1, 8, 17):
        i, d = knn_ref(xy, k)
        bi, bd = ograph.knn_bruteforce(xy, k)
        assert np.array_equal(i, bi) and np.array_equal(d, bd)
        i, d = knn_ref(big, k)
        bi, bd = ograph.knn(big, k)
        assert np.array_equal(i, bi) and np.array_equal(d, bd)


def test_references_on_a_prefix_with_ids():
    rng = np.random.default_rng(1)
    xy = np.round(rng.random((500, 2)) * 40.0)
    types = rng.integers(1, 6, size=500).astype(np.int32)
    ids = rng.permutation(500) + 1000
    nq = 123
    ref = radius_ref(xy, 4.0, types, nq=nq, ids=ids)
    full = ograph.radius_graph_bruteforce(xy, 4.0)
    for i in (0, 7, nq - 1):
        js = np.concatenate([full["col"][full["row_ptr"][i]:full["row_ptr"][i + 1]]])
        assert np.array_equal(ref["col"][ref["row_ptr"][i]:ref["row_ptr"][i + 1]], np.sort(ids[js]))
        up = np.sort(ids[js][ids[js] > ids[i]])
        assert np.array_equal(ref["edges"][ref["up_ptr"][i]:ref["up_ptr"][i + 1]], np.stack([np.full(len(up), ids[i]), up], 1))
    ki, kd = knn_ref(xy, 6, nq=nq, ids=ids)
    for i in (0, 50, nq - 1):
        d2 = _d2(xy[i][None, :], xy)
        j = np.array([x for x in np.lexsort((ids, d2)) if x != i][:6])
        assert np.array_equal(ki[i], ids[j]) and np.array_equal(kd[i], np.sqrt(d2[j]))


def test_binning_restatement():
    info = {"x0": -3.0, "y0": 10.0, "cell": 2.5, "nx": 4, "ny": 70}
    xy = np.array([[-3.0, 10.0], [-0.5, 12.5], [-1e9, 1e9], [7.0, 10.0 + 2.5 * 31], [7.0, 10.0 + 2.5 * 32]])
    cx, cy = cell_coords(xy, info)
    assert cx.tolist() == [0, 1, 0, 3, 3] and cy.tolist() == [0, 1, 69, 31, 32]
    assert cell_index(info, cx, cy).tolist() == [0, 33, 2 * 4 * 32 + 5, 3 * 32 + 31, 4 * 32 + 3 * 32]
    assert padded_cells(info) == 4 * 96
    assert ring_radius(1.0, {"cell": radius_cell(1.0), "nx": 9, "ny": 9}) == 1
    assert ring_radius(1e10, {"cell": 1.0, "nx": 1001, "ny": 30}) == 1001
    assert ring_radius(10.0, {"cell": 10.0 / 200, "nx": 1001, "ny": 1001}) >= 200


def test_hair_above_r_binning_stays_within_the_ring():
    # the host-side claim behind the ring radius: with the library's cell size, ring radius and binning, two points
    # exactly r apart never bin more than R cells apart - checked here on the exact expressions, at cell coordinates up
    # to 2^27, right below and above cell boundaries (see the next test for the tops of binades)
    rng = np.random.default_rng(5)
    for delta in (2.0 ** -20, 1e-9, 2e-9, 3e-9, 1e-12):
        for r in (1.0, 0.75, 3.0):
            cell = r * (1.0 + delta)
            info = {"cell": cell, "nx": 1, "ny": 1 << 28}
            R = ring_radius(r, info)
            for lo in (1 << 20, 1 << 24, 1 << 27):
                k = rng.integers(lo, 2 * lo, size=200).astype(np.float64)
                b = (k * cell)[:, None]
                ya = (b + np.spacing(b) * np.arange(-60, 20)[None, :]).ravel()
                yb = ya + r
                ok = (yb - ya) == r
                ta, tb = np.floor(ya * (1.0 / cell)), np.floor(yb * (1.0 / cell))
                assert ok.sum() > len(ok) // 2
                assert ((tb - ta)[ok] <= R).all(), (delta, r, lo)


def test_ring_radius_covers_the_top_of_a_binade():
    # just below t = 2^k the float64 spacing of the cell coordinate doubles: a point r past one that bins to 2^k - 1 can
    # round up into row 2^k + 1, two rows away, for a cell a few 1e-9 above r. A fixed slack misses that (R = 1 and the
    # FAST walk drops the edge); the slack that grows with max(nx, ny) covers it on every grid that reaches such a t.
    ya, yb, ta, tb = binade_top_pairs(13 / 64, 13 / 64 * (1.0 + 3e-9), 26)
    hit = np.flatnonzero(tb - ta >= 2)
    assert 13631488.040894464 in ya[hit].tolist()              # two rows apart: 2^26 - 1 and 2^26 + 1
    missed = 0
    for r in (13 / 64, 3 / 16, 5 / 8, 0.75, 1.0):
        for delta in (2.1e-9, 3e-9, 4e-9, 5e-9, 2.0 ** -20):
            cell = r * (1.0 + delta)
            for k in (24, 25, 26, 27, 28):
                ya, yb, ta, tb = binade_top_pairs(r, cell, k, span=40_000)
                gap = int((tb - ta).max())
                # the smallest grid that holds row 2^k + 1 on one axis: its slack is the smallest
                info = {"cell": cell, "nx": 1, "ny": (1 << k) + 2}
                assert gap <= ring_radius(r, info), (r, delta, k, gap)
                missed += gap > ring_radius_fixed_slack(r, info)
                if delta == 2.0 ** -20:
                    assert ring_radius(r, dict(info, ny=1 << 28)) == 1  # radius_cell keeps the FAST walk
    assert missed > 0                                             # the regime is reached, not just bounded


# ---------------------------------------------------------------------------------------------------- 1. far from the origin
@pytest.mark.gpu
@pytest.mark.parametrize("shift", [0.0, 1e5, 1e7, 1e9])
def test_far_from_origin(engine, shift):
    """FAST walk, select / ring kNN: binning (v - x0) * inv_cell at magnitudes up to 1e9, with exact ties at d == r."""
    xy0, types = half_pixel_points(2500, 300.0, 11)
    xy = xy0 + shift
    assert np.array_equal(xy - shift, xy0)                    # the shift is exact
    r = 5.0
    ref = radius_ref(xy, r, types)
    ref0 = radius_ref(xy0, r, types)
    assert np.array_equal(ref["edges"], ref0["edges"]) and np.array_equal(ref["dist"], ref0["dist"])
    assert (ref["dist"] == r).sum() > 100                     # (3, 4) pairs: d == r exactly
    engine.grid_build(dev(xy), dev(types), None, radius_cell(r), None)
    info = engine.grid_info()
    assert info["x0"] == xy[:, 0].min() and info["y0"] == xy[:, 1].min()
    assert ring_radius(r, info) == 1
    check_radius(engine, ref, r, ("shift", shift))
    check_export(engine, xy, types, info)
    engine.grid_build(dev(xy), dev(types), None, default_knn_cell(len(xy), 300.0 ** 2, 8), None)
    check_knn_union(engine, xy, types, 8, ("shift", shift))
    check_knn(engine, xy, 17, ("shift", shift))


# ---------------------------------------------------------------------------------------------------- 2. thin grids
def _line_points(n, r, seed, axis):
    """A line of points along ``axis`` (the other coordinate constant): lattice steps of r / 2 and r with random gaps,
    a few duplicates - pairs at exactly r and 2r."""
    rng = np.random.default_rng(seed)
    steps = rng.choice([0.0, 0.5 * r, r, 1.5 * r, 3.25 * r], size=n, p=[0.03, 0.3, 0.4, 0.2, 0.07])
    v = np.cumsum(steps)
    xy = np.zeros((n, 2))
    xy[:, axis] = v
    xy[:, 1 - axis] = 250.0
    return xy, rng.integers(0, 7, size=n).astype(np.int32)


def _thin(kind, r):
    cell = radius_cell(r)
    rng = np.random.default_rng(THIN.index(kind))
    if kind == "vertical_line":
        xy, t = _line_points(4000, r, 1, axis=1)
        return xy, t, None
    if kind == "horizontal_line":
        xy, t = _line_points(4000, r, 2, axis=0)
        return xy, t, None
    if kind == "band_2_cells":
        n = 4000
        xy = np.stack([rng.random(n) * 1.999 * cell, rng.random(n) * 3000.0], axis=1)
        return xy, rng.integers(0, 7, size=n).astype(np.int32), None
    # "rows_<m>": ny = 3 * 32 + m rows given by the bounds; points on the strip edges and on cell boundaries
    m = int(kind.split("_")[1])
    ny = 3 * STRIP + m
    height = (ny - 1) * cell + 0.5 * cell
    width = 12 * cell
    n = 3000
    xy = np.stack([rng.random(n) * width, rng.random(n) * height], axis=1)
    rows = np.array([s * STRIP + d for s in range(1, ny // STRIP + 1) for d in (-1, 0)] + [ny - 1])
    edge = np.stack([rng.random(len(rows) * 20) * width,
                     np.repeat(rows, 20) * cell + rng.choice([0.0, 0.5 * r, 0.999 * r], size=len(rows) * 20)], axis=1)
    corners = np.array([[cx * cell, cy * cell] for cx in range(0, 12, 3) for cy in rows])  # exactly on boundaries
    xy = np.concatenate([xy, edge, corners])
    xy[:, 1] = np.minimum(xy[:, 1], height)
    return xy, rng.integers(0, 7, size=len(xy)).astype(np.int32), (0.0, 0.0, width, height)


THIN = ["vertical_line", "horizontal_line", "band_2_cells", "rows_1", "rows_31", "rows_32", "rows_33"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", THIN)
def test_thin_grids(engine, kind):
    """FAST walk at the grid's edges: nx = 1 (has_l = has_r = false), ny = 1, nx = 2, and ny = 1, 31, 0, 1 (mod 32),
    where points on rows ly == 0 / 31 take the strip-edge pass into the padded strip layout."""
    r = 6.0
    xy, types, bounds = _thin(kind, r)
    ref = radius_ref(xy, r, types)
    engine.grid_build(dev(xy), dev(types), None, radius_cell(r), bounds)
    info = engine.grid_info()
    assert info["cell"] == radius_cell(r) and ring_radius(r, info) == 1
    if kind == "vertical_line":
        assert info["nx"] == 1 and info["ny"] > 8 * STRIP
    elif kind == "horizontal_line":
        assert info["ny"] == 1 and info["nx"] > 1000
    elif kind == "band_2_cells":
        assert info["nx"] == 2 and info["ny"] > 8 * STRIP
    else:
        m = int(kind.split("_")[1])
        assert info["ny"] == 3 * STRIP + m and info["ny"] % STRIP == m % STRIP
    cx, cy = cell_coords(xy, info)
    src = np.repeat(np.arange(len(xy)), np.diff(ref["row_ptr"]))
    cross = (cy[src] // STRIP) != (cy[ref["col"]] // STRIP)
    if info["ny"] > STRIP:
        assert cross.sum() > 20                              # edges across strip edges: the edge pass finds them
    check_radius(engine, ref, r, (kind,))
    check_export(engine, xy, types, info)
    k = 8 if kind != "rows_33" else 17
    engine.grid_build(dev(xy), dev(types), None, radius_cell(r), bounds)
    check_knn_union(engine, xy, types, k, (kind,))
    check_knn(engine, xy, 1, (kind,))


# ---------------------------------------------------------------------------------------------------- 3. cap doubling
@pytest.mark.gpu
def test_cell_cap_doubling(engine):
    """pg_grid_build's doubling loop: 300 points in 20 clumps 1e6 px apart ask for ~10^11 cells of radius_cell(r); the
    cap (2^20 for 8 n < 2^20) forces the cell up. The radius walk then runs with R = 1 on fat cells, and kNN with
    k = 17 (more than a clump holds) expands its rings across empty cells to the next clump."""
    rng = np.random.default_rng(3)
    centres = np.stack(np.meshgrid(np.arange(5.0), np.arange(4.0)), axis=-1).reshape(-1, 2) * 1e6
    xy = np.concatenate([c + rng.random((15, 2)) * 40.0 for c in centres])
    types = rng.integers(1, 6, size=len(xy)).astype(np.int32)
    r = 10.0
    engine.grid_build(dev(xy), dev(types), None, radius_cell(r), None)
    info = engine.grid_info()
    assert info["cell"] >= radius_cell(r) * 256             # doubled at least 8 times
    assert info["nx"] * info["ny"] <= MIN_CAP
    assert ring_radius(r, info) == 1
    ref = radius_ref(xy, r, types)
    check_radius(engine, ref, r, ("cap",))
    check_export(engine, xy, types, info)
    for k in (1, 8, 17):
        check_knn_union(engine, xy, types, k, ("cap",))


# ---------------------------------------------------------------------------------------------------- 4. clamping
BOUNDS = {
    "tenth": (450.0, 450.0, 766.0, 766.0),                   # ~10 % of the points inside
    "one_point": (500.0, 500.0, 500.0, 500.0),               # x0 == x1, y0 == y1: a 1 x 1 grid
    "far_away": (1e6, 1e6, 1e6 + 100.0, 1e6 + 100.0),        # every point clamped into one corner cell
    "thin_slice": (0.0, 400.0, 1000.0, 400.0),               # ny == 1
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BOUNDS))
def test_caller_bounds_clamp(engine, name):
    """pg_cell_coord's clamp: bounds that leave most points outside the grid put them into border cells; the radius
    walk (R = 1 and the block walk), kNN and the union must still find every neighbour."""
    rng = np.random.default_rng(4)
    xy = rng.random((3000, 2)) * 1000.0
    types = rng.integers(0, 7, size=3000).astype(np.int32)
    b = BOUNDS[name]
    inside = (xy[:, 0] >= b[0]) & (xy[:, 0] <= b[2]) & (xy[:, 1] >= b[1]) & (xy[:, 1] <= b[3])
    assert inside.mean() < 0.12
    for r in (8.0, 25.0):
        ref = radius_ref(xy, r, types)
        for cell in (radius_cell(r), r / 2.5):
            engine.grid_build(dev(xy), dev(types), None, cell, b)
            info = engine.grid_info()
            assert (info["x0"], info["y0"]) == (b[0], b[1])
            check_radius(engine, ref, r, (name, r, cell))
    check_export(engine, xy, types, info)
    for k in (1, 8, 17):
        engine.grid_build(dev(xy), dev(types), None, default_knn_cell(3000, 1000.0 ** 2, k), b)
        check_knn_union(engine, xy, types, k, (name,))


# ---------------------------------------------------------------------------------------------------- 5. cells << r
@pytest.mark.gpu
@pytest.mark.parametrize("div", [3, 17, 200])
def test_cells_much_smaller_than_r(engine, div):
    """The non-FAST walk (pg_visit_block) with R = 3..200: 1500 points in [0, 50]^2, r = 10, cell = r / div."""
    rng = np.random.default_rng(div)
    xy = rng.random((1500, 2)) * 50.0
    types = rng.integers(0, 7, size=1500).astype(np.int32)
    r = 10.0
    engine.grid_build(dev(xy), dev(types), None, r / div, None)
    info = engine.grid_info()
    assert info["cell"] == r / div                           # no doubling: the grid has at most 1001 x 1001 cells
    R = ring_radius(r, info)
    assert div <= R <= div + 1 and R < max(info["nx"], info["ny"])
    check_radius(engine, radius_ref(xy, r, types), r, ("div", div))
    check_knn_union(engine, xy, types, 17, ("div", div))


@pytest.mark.gpu
def test_ball_covers_the_grid(engine):
    """r far beyond the grid on one built grid (cell = r0 / 200): r = 2 span, 1e6 span (R ~ 1e9 cells, near INT_MAX
    for the block walk's cx + R) and 1e10 span (r / cell past 2^31: the ring radius must not wrap to the 3x3 walk).
    Every one is the complete graph: 1500 points, 1 124 250 edges."""
    rng = np.random.default_rng(77)
    xy = rng.random((1500, 2)) * 50.0
    types = rng.integers(0, 7, size=1500).astype(np.int32)
    span = float(np.ptp(xy, axis=0).max())
    engine.grid_build(dev(xy), dev(types), None, 10.0 / 200, None)
    info = engine.grid_info()
    assert info["cell"] == 10.0 / 200 and max(info["nx"], info["ny"]) > 900
    ref = radius_ref(xy, 2.0 * span, types)
    n = len(xy)
    assert int(ref["up_ptr"][-1]) == n * (n - 1) // 2 and (ref["degree"] == n - 1).all()
    for mult in (2.0, 1e6, 1e10):
        r = mult * span
        assert ring_radius(r, info) == max(info["nx"], info["ny"])
        check_radius(engine, ref, r, ("covers", mult))
    check_knn_union(engine, xy, types, 17, ("covers",))


# ---------------------------------------------------------------------------------------------------- 6. a hair above r
@pytest.mark.gpu
@pytest.mark.parametrize("delta", [2.0 ** -20, 1e-9, 2e-9, 3e-9, 1e-12])
def test_cell_a_hair_above_r(engine, delta):
    """ring_radius's slack: cell = r (1 + delta), two lattice lines with pairs at exactly d == r (along and across the
    lines), at cell coordinates above 10^6 by the grid's own binning. delta = 2^-20 gives R = 1 (the FAST walk trusts
    that a point r away is at most one cell away); the smaller margins give R = 2 on this 1.15 M-row grid."""
    r = 1.0
    m = 150_000
    y = (1_000_000.0 + np.arange(m)) * r
    xy = np.concatenate([np.stack([np.zeros(m), y], 1), np.stack([np.full(m, r), y], 1)])
    types = (np.arange(2 * m) % 6).astype(np.int32)
    cell = r * (1.0 + delta)
    engine.grid_build(dev(xy), dev(types), None, cell, (0.0, 0.0, r, y[-1]))
    info = engine.grid_info()
    assert info["cell"] == cell and info["nx"] == 1 and info["ny"] > 1_100_000
    R = ring_radius(r, info)
    assert R == (1 if delta == 2.0 ** -20 else 2)
    cx, cy = cell_coords(xy, info)
    assert cy.min() >= 999_999
    ref = radius_ref(xy, r, types)
    assert (ref["dist"] == r).all() and (ref["degree"][[0, m - 1, m, 2 * m - 1]] == 2).all()
    src = np.repeat(np.arange(len(xy)), np.diff(ref["row_ptr"]))
    assert (np.abs(cy[src] - cy[ref["col"]]) <= R).all()
    check_radius(engine, ref, r, ("hair", delta), calls=("fused",))
    check_knn(engine, xy, 1, ("hair", delta))


@pytest.mark.gpu
def test_cell_a_hair_above_r_at_the_top_of_a_binade(engine):
    """The ring radius's grid-scaled slack on the device: a pair exactly r = 13/64 apart whose first point bins to row
    2^26 - 1 and whose second rounds up into row 2^26 + 1, on a one-column grid of 2^26 + 3 rows (2^23 + 1 points:
    the cell cap allows 8 n cells). cell = r (1 + 3e-9): a fixed 1e-9 slack gives R = 1 and the FAST walk would drop the
    edge; the library must take R = 2 here. The other points sit 2 r apart, far below the pair: no other edge."""
    r = 13 / 64
    cell = r * (1.0 + 3e-9)
    ya = 13631488.040894464
    n = (1 << 23) + 1
    m = n - 2
    y = np.concatenate([np.arange(m) * (2 * r), [ya, ya + r]])
    xy = np.stack([np.zeros(n), y], axis=1)
    assert y[-1] - y[-2] == r and np.diff(y[:m]).min() > r and y[m - 1] + r < ya
    types = np.ones(n, dtype=np.int32)
    engine.grid_build(dev(xy), dev(types), None, cell, (0.0, 0.0, 0.0, ((1 << 26) + 2.5) * cell))
    info = engine.grid_info()
    assert info["cell"] == cell and info["nx"] == 1 and info["ny"] >= (1 << 26) + 2
    _, cy = cell_coords(xy[-2:], info)
    assert cy.tolist() == [(1 << 26) - 1, (1 << 26) + 1]
    assert ring_radius_fixed_slack(r, info) == 1 and ring_radius(r, info) == 2
    deg = np.zeros(n, dtype=np.int32)
    deg[-2:] = 1
    comp = np.zeros((n, N_TYPES), dtype=np.int32)
    comp[-2:, 0] = 1
    row_ptr = np.concatenate([[0], np.cumsum(deg)])
    up_ptr = np.zeros(n + 1, dtype=np.int64)
    up_ptr[n - 1:] = 1
    ref = {"row_ptr": row_ptr, "col": np.array([n - 1, n - 2]), "dist": np.array([r, r]), "up_ptr": up_ptr,
           "edges": np.array([[n - 2, n - 1]]), "edge_dist": np.array([r]), "degree": deg, "comp": comp}
    check_radius(engine, ref, r, ("binade top",))


# ---------------------------------------------------------------------------------------------------- 7. query prefix
@pytest.mark.gpu
@pytest.mark.parametrize("nq", [0, 1, 37, 1999])
@pytest.mark.parametrize("with_gid", [False, True])
def test_queries_on_a_prefix(engine, nq, with_gid):
    """n_query < n: the rows are the first nq points, the points behind them are ghosts (no row, still neighbours), as
    the strip builds append their halo. Against brute force restricted to the query rows, with and without gids."""
    rng = np.random.default_rng(nq + 7 * with_gid)
    n = 2000
    xy = np.round(rng.random((n, 2)) * 200.0 * 2) / 2
    types = rng.integers(0, 7, size=n).astype(np.int32)
    ids = (rng.permutation(n) * 3 + 5).astype(np.int32) if with_gid else None
    r = 9.0
    engine.grid_build(dev(xy), dev(types), dev(ids) if with_gid else None, radius_cell(r), None, n_query=nq)
    ref = radius_ref(xy, r, types, nq=nq, ids=ids)
    check_radius(engine, ref, r, ("prefix", nq, with_gid))
    for k in (1, 8, 17):
        check_knn(engine, xy, k, ("prefix", nq, with_gid), nq=nq, ids=ids)


# ---------------------------------------------------------------------------------------------------- 8. one handle
@pytest.mark.gpu
def test_one_handle_many_builds(engine):
    """30 seeded builds on one handle: cell counts that outgrow the last allocation then shrink, n from 0 to 300 k,
    with and without gids, radius (count -> fill and fused) and kNN in between. A stale histogram counter, scan
    descriptor, parking hint or retry count shows up as a wrong graph."""
    rng = np.random.default_rng(2024)
    sizes = [0, 1, 2, 17, 300_000, 500, 3, 40_000, 0, 2500, 120_000, 9, 300_000, 64, 5000,
             33, 1, 75_000, 1000, 0, 200, 260_000, 7, 4096, 4097, 15, 31_000, 2, 800, 12_000]
    for step, n in enumerate(sizes):
        r = float(rng.choice([4.0, 12.0, 40.0]))
        side = max(math.sqrt(n), 1.0) * r * float(rng.uniform(0.5, 3.0))   # mean degree pi / u^2: 0.35 .. 12.6
        xy = rng.random((n, 2)) * side
        if n > 4:
            xy[: n // 40] = xy[n // 2: n // 2 + n // 40]         # duplicates
        types = rng.integers(0, 7, size=n).astype(np.int32)
        with_gid = step % 3 == 1
        ids = (rng.permutation(n) + 11).astype(np.int32) if with_gid else None
        cell = radius_cell(r) * float(rng.choice([1.0, 0.4]))
        engine.grid_build(dev(xy.reshape(n, 2)), dev(types), dev(ids) if with_gid else None, cell, None)
        info = engine.grid_info()
        tag = ("build", step, n)
        ref = radius_ref(xy.reshape(n, 2), r, types, ids=ids)
        call = ("count",) if step % 2 == 0 else ("fused",)
        check_radius(engine, ref, r, tag, calls=call)
        k = int(rng.choice([1, 8, 17]))
        if n > k:
            check_knn(engine, xy, k, tag, ids=ids)
        if 0 < n <= 300_000 and step % 5 == 0:
            check_export(engine, xy, types, info, ids=ids)


# ---------------------------------------------------------------------------------------------------- 9. scan groups
@pytest.mark.gpu
@pytest.mark.parametrize("n", [SCAN_GROUP - 1, SCAN_GROUP, SCAN_GROUP + 1, 3 * SCAN_GROUP + 17, (1 << 26) + 5])
def test_exclusive_scan_across_lookback_groups(engine, n):
    """K3's look-back chain across groups of 256 tiles x 4096 items, totals below 2^31."""
    rng = np.random.default_rng(n % 1000)
    hi = max(2, min(1000, (2 ** 31 - 1) // n))
    x = rng.integers(0, hi, size=n, dtype=np.int32)
    x[-1] = hi - 1
    out = engine.exclusive_scan(dev(x)).cpu().numpy()
    ref = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(x, out=ref[1:])
    assert ref[-1] < 2 ** 31
    assert np.array_equal(out, ref)


@pytest.mark.gpu
def test_grid_cell_scan_spans_several_groups(engine):
    """A grid whose padded cell count spans three scan groups (the cell scan's look-back crosses group boundaries):
    cell_start, as the cell boundaries of pg_grid_export, against numpy's binning; and the radius graph over it."""
    rng = np.random.default_rng(9)
    n = 300_000
    xy = rng.random((n, 2)) * 4000.0
    types = rng.integers(0, 7, size=n).astype(np.int32)
    cell = 4000.0 / 1500
    engine.grid_build(dev(xy), dev(types), None, cell, None)
    info = engine.grid_info()
    assert info["cell"] == cell and padded_cells(info) > 2 * SCAN_GROUP
    check_export(engine, xy, types, info)
    r = 3.0
    check_radius(engine, radius_ref(xy, r, types), r, ("groups",), calls=("fused",))


# ---------------------------------------------------------------------------------------------------- 10. export
EXPORT = ["uniform", "vertical_line", "clamped", "gid"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", EXPORT)
def test_grid_export_is_the_cell_order(engine, kind):
    """pg_grid_export (sharding.spatial_sort): a permutation of the input in cell order, each cell = numpy's binning."""
    rng = np.random.default_rng(len(kind))
    n = 50_000
    xy = rng.random((n, 2)) * 3000.0
    types = rng.integers(0, 7, size=n).astype(np.int32)
    ids, bounds = None, None
    if kind == "vertical_line":
        xy[:, 0] = 17.0
    elif kind == "clamped":
        bounds = (1000.0, 1000.0, 1900.0, 1900.0)
    elif kind == "gid":
        ids = (rng.permutation(n) * 2 + 1).astype(np.int32)
    engine.grid_build(dev(xy), dev(types), dev(ids) if ids is not None else None, 20.0, bounds)
    check_export(engine, xy, types, engine.grid_info(), ids=ids)


# ---------------------------------------------------------------------------------------------------- 11. span overflow
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["both_axes_1e308", "x_dbl_max", "bounds"])
def test_span_overflow_is_rejected(engine, case):
    """Finite coordinates whose span overflows double (b[2] - b[0] = inf): pg_grid_build rejects them with
    PG_ERR_INVALID instead of doubling the cell forever, and the handle builds a normal grid afterwards."""
    from path_gene_multimodal_b200._lib import PG_ERR_INVALID, PathGraphError

    big = np.finfo(np.float64).max
    xy = np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 0.5]])
    bounds = None
    if case == "both_axes_1e308":
        xy = np.concatenate([xy, [[-1e308, -1e308], [1e308, 1e308]]])
    elif case == "x_dbl_max":
        xy = np.concatenate([xy, [[-big, 0.0], [big, 1.0]]])
    else:
        bounds = (-1e308, 0.0, 1e308, 1.0)
    types = np.ones(len(xy), dtype=np.int32)
    with pytest.raises(PathGraphError, match="overflows double") as err:
        engine.grid_build(dev(xy), dev(types), None, 1.0, bounds)
    assert err.value.code == PG_ERR_INVALID
    with pytest.raises(PathGraphError):
        engine.grid_info()                                    # no grid is left behind
    rng = np.random.default_rng(0)
    ok = rng.random((2000, 2)) * 300.0
    t = rng.integers(0, 7, size=2000).astype(np.int32)
    engine.grid_build(dev(ok), dev(t), None, radius_cell(10.0), None)
    check_radius(engine, radius_ref(ok, 10.0, t), 10.0, ("after", case), calls=("fused",))
