"""Oracle (test infrastructure): connected components, DBSCAN and per-cluster properties - the reference for K19
(pg_connected_components, pg_dbscan, pg_cluster_props) and cell_graph.cell_clusters.

* ``dbscan_loop``: a literal restatement of sklearn.cluster.DBSCAN - ``radius_neighbors`` as
  ``cKDTree.query_ball_point`` (the point itself included), ``core = n_neighbors >= min_samples``, then the loop of
  sklearn's ``_dbscan_inner.pyx``: visit the points in index order, start a cluster at each unlabelled core point and
  finish it with a stack before starting the next. For small inputs.
* ``dbscan``: the same labels for slide-scale inputs - scipy's ``connected_components`` on the core-core subgraph of
  ``oracle.graph.radius_graph`` (clusters renumbered by their smallest core index), then every non-core point takes the
  smallest label among its core neighbours, -1 without one.
* ``connected_components``: scipy's weak components of any CSR, skipping entries outside [0, n) and self entries,
  numbered by smallest member.
* ``cluster_props``: exact counts and bounding boxes, the centroid with a float64 error bound, and the convex hull area
  (``scipy.spatial.ConvexHull``; exact ``oracle.hull`` for degenerate sets).
"""
from __future__ import annotations

import math

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components as _scipy_cc
from scipy.spatial import ConvexHull, cKDTree

from . import graph as ograph
from . import hull as ohull

EPS64 = np.finfo(np.float64).eps


def _by_smallest(lab: np.ndarray, n_comp: int) -> np.ndarray:
    """Renumber component labels in the order of each component's smallest index."""
    first = np.full(n_comp, np.iinfo(np.int64).max)
    np.minimum.at(first, lab, np.arange(lab.shape[0]))
    rank = np.empty(n_comp, dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(n_comp)
    return rank[lab]


def connected_components(row_ptr, col, n=None):
    """(n_components, labels int64 [n]) of the undirected graph of a CSR's entries (i, j), j in [0, n), j != i."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    n = rp.shape[0] - 1 if n is None else n
    c = np.asarray(col, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    keep = (c >= 0) & (c < n) & (c != rows)
    a = sp.csr_matrix((np.ones(int(keep.sum()), dtype=np.int8), (rows[keep], c[keep])), shape=(n, n))
    k, lab = _scipy_cc(a, directed=False)
    return int(k), _by_smallest(lab.astype(np.int64), k)


def dbscan_loop(coords, eps, min_samples):
    """sklearn's DBSCAN, literally: (labels int64 [n], core bool [n])."""
    x = np.asarray(coords, dtype=np.float64).reshape(-1, 2)
    n = x.shape[0]
    if n == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=bool)
    neigh = cKDTree(x).query_ball_point(x, eps)
    core = np.array([len(nb) >= min_samples for nb in neigh], dtype=bool)
    labels = np.full(n, -1, dtype=np.int64)
    label_num = 0
    stack = []
    for i in range(n):
        if labels[i] != -1 or not core[i]:
            continue
        while True:
            if labels[i] == -1:
                labels[i] = label_num
                if core[i]:
                    for v in neigh[i]:
                        if labels[v] == -1:
                            stack.append(v)
            if not stack:
                break
            i = stack.pop()
        label_num += 1
    return labels, core


def dbscan_csr(row_ptr, col, min_samples):
    """DBSCAN on a symmetric radius CSR without self entries: (labels int64 [n], core bool [n])."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    n = rp.shape[0] - 1
    c = np.asarray(col, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    keep = (c >= 0) & (c < n) & (c != rows)
    rows, c = rows[keep], c[keep]
    core = np.bincount(rows, minlength=n) + 1 >= min_samples
    labels = np.full(n, -1, dtype=np.int64)
    idx = np.flatnonzero(core)
    if idx.size:
        pos = np.full(n, -1, dtype=np.int64)
        pos[idx] = np.arange(idx.size)
        cc = core[rows] & core[c]
        a = sp.csr_matrix((np.ones(int(cc.sum()), dtype=np.int8), (pos[rows[cc]], pos[c[cc]])),
                          shape=(idx.size, idx.size))
        k, lab = _scipy_cc(a, directed=False)
        labels[idx] = _by_smallest(lab.astype(np.int64), k)  # idx ascending: smallest position = smallest core index
        border = ~core[rows] & core[c]
        best = np.full(n, np.iinfo(np.int64).max)
        np.minimum.at(best, rows[border], labels[c[border]])
        hit = ~core & (best != np.iinfo(np.int64).max)
        labels[hit] = best[hit]
    return labels, core


def dbscan(coords, eps, min_samples):
    """Vectorised DBSCAN over oracle.graph.radius_graph: (labels int64 [n], core bool [n])."""
    x = np.asarray(coords, dtype=np.float64).reshape(-1, 2)
    if x.shape[0] == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=bool)
    g = ograph.radius_graph(x, eps)
    return dbscan_csr(g["row_ptr"], g["col"], min_samples)


def hull_area(points) -> float:
    """Convex hull area: NaN below 3 points (K14's rule), 0 for collinear points, else scipy's ConvexHull."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    if p.shape[0] < 3:
        return float("nan")
    if p.shape[0] > 64:
        try:
            return float(ConvexHull(p).volume)
        except Exception:  # qhull refuses flat input: the exact monotone chain below says 0
            pass
    pts, d = ohull._scaled(p.tolist())
    return ohull.hull_area2(pts) / 2.0 / float(d) ** 2


def cluster_props(labels, k, coords, types=None, n_types=5, core=None, hull=True):
    """Per-cluster table of clusters 0..k-1: n_members, n_core, type_count [k, T], centroid [k, 2] with its bound
    centroid_bound [k, 2], bbox [k, 4] (xmin, ymin, xmax, ymax), member_off [k+1] / member_xy (members grouped by
    cluster in ascending index) and hull_area."""
    lab = np.asarray(labels, dtype=np.int64)
    x = np.asarray(coords, dtype=np.float64).reshape(-1, 2)
    member = (lab >= 0) & (lab < k)
    order = np.flatnonzero(member)
    order = order[np.argsort(lab[order], kind="stable")]
    cnt = np.bincount(lab[member], minlength=k)
    off = np.zeros(k + 1, dtype=np.int64)
    np.cumsum(cnt, out=off[1:])
    out = {"n_members": cnt, "member_off": off, "member_xy": x[order]}
    if core is not None:
        out["n_core"] = np.bincount(lab[member], weights=np.asarray(core)[member].astype(np.float64),
                                    minlength=k).astype(np.int64)
    if types is not None:
        t = np.asarray(types, dtype=np.int64)
        ok = member & (t >= 1) & (t <= n_types)
        tc = np.zeros((k, n_types), dtype=np.int64)
        np.add.at(tc, (lab[ok], t[ok] - 1), 1)
        out["type_count"] = tc
    cen = np.full((k, 2), np.nan)
    bound = np.full((k, 2), np.nan)
    bbox = np.full((k, 4), np.nan)
    areas = np.full(k, np.nan)
    for c in range(k):
        p = x[order[off[c]:off[c + 1]]]
        m = p.shape[0]
        if m == 0:
            continue
        cen[c] = [math.fsum(p[:, 0]) / m, math.fsum(p[:, 1]) / m]  # the correctly rounded sums
        # a float64 sum in any order is off by at most (m - 1) eps sum |x|; each side rounds its division once
        bound[c] = (m + 1) * EPS64 * np.abs(p).sum(axis=0) / m + 2 * EPS64 * np.abs(cen[c])
        bbox[c] = [p[:, 0].min(), p[:, 1].min(), p[:, 0].max(), p[:, 1].max()]
        if hull:
            areas[c] = hull_area(p)
    out.update({"centroid": cen, "centroid_bound": bound, "bbox": bbox})
    if hull:
        out["hull_area"] = areas
    return out

