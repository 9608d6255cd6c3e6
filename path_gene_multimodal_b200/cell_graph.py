"""Spatial cell graphs over nucleus centroids, in the notebook's vocabulary.

Mirrors /root/reference/hovernet_tile_inference.ipynb:
* ``build_knn_graph``      cell 11 (ipynb:1766-1951): ``knn_neighbors``, ``knn_neighbor_distances``, and the
  undirected ``nx.Graph`` union (edges ``i<j``, ``weight = min(dist)``);
* ``build_radius_graph``   cells 23-26 (ipynb:2963-3042): ``edges`` int64 [E,2] (``i<j``), ``edge_index``,
  ``edge_attr`` float32 [2E,1];
* ``filter_graph_by_type`` cell 12 (ipynb:1989-2002);
* ``neighbour_type_composition`` / ``degree_stats``: named in README.md:127,136 only; defined in SURVEY A.5;
* ``co_occurrence`` / ``ripley``: cell-type patterns across distance (squidpy.gr.co_occurrence / ripley's statistics);
* ``spatial_autocorr``: Moran's I / Geary's C of per-nucleus features over the graph (squidpy.gr.spatial_autocorr).

Host arrays in, host arrays out; everything in between is libpathgraph (uniform-grid binning, grid
queries, two-pass CSR) on the GPU.  No CPU fallback.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _host, _lib
from .engine import default_knn_cell, get_engine, pair_hist_cell, radius_cell

TYPE_NAMES = {1: "neoplastic", 2: "inflammatory", 3: "connective", 4: "dead", 5: "epithelial"}       # ipynb:1774-1780
CLASS_COLORS = {1: "tab:red", 2: "tab:green", 3: "tab:blue", 4: "tab:gray", 5: "tab:orange"}           # ipynb:1782-1788


def _prep(coords, types, eng):
    c = np.asarray(coords, dtype=np.float64)
    if c.ndim != 2 or c.shape[1] != 2:
        raise ValueError("coords must have shape (N, 2)")
    if c.shape[0] > _host.INT32_MAX:
        raise OverflowError("more than 2^31 points")
    # NaN / inf (cKDTree raises on them) are detected on the device by the histogram kernel and reported at the
    # first synchronisation - no extra pass over the coordinates on the host
    d_xy = _host.to_device(c, np.float64, eng.device)
    d_t = None
    if types is not None:
        t = np.asarray(types)
        if t.shape[0] != c.shape[0]:
            raise ValueError("types must have one entry per point")
        d_t = _host.to_device(_host.as_int32(t, "types"), np.int32, eng.device)
    return c, d_xy, d_t


def _bounds(c):
    if c.shape[0] == 0:
        return (0.0, 0.0, 1.0, 1.0)
    return (float(c[:, 0].min()), float(c[:, 1].min()), float(c[:, 0].max()), float(c[:, 1].max()))


def build_knn_graph(coords, k: int = 5, types=None, n_types: int = 5, undirected: bool = True,
                    bounds=None, cell_size: float | None = None, device=None, neighbor_coords: bool = False) -> dict:
    """kNN graph of cell 11.

    Returns ``knn_neighbors`` int64 [N,k] (ascending ``(d^2, index)``, self excluded by index),
    ``knn_neighbor_distances`` float64 [N,k] and, with ``undirected``: ``edges`` int64 [E,2] (``i<j``,
    sorted), ``weight`` float64 [E], symmetric CSR ``row_ptr`` / ``col`` / ``csr_weight``, ``degree`` int32 [N],
    ``nbr_count`` int32 [N,n_types] (when ``types`` is given) and ``degree_stats``.
    ``neighbor_coords`` adds ``knn_neighbor_coords`` float64 [N,k,2] (the (x, y) of every list entry, ipynb:1838-1840).
    Raises ``ValueError`` when ``k >= N`` (as cKDTree-backed KNN does for k+1 > N).
    """
    eng = get_engine(device)
    c, d_xy, d_t = _prep(coords, types, eng)
    n = c.shape[0]
    if not (1 <= k):
        raise ValueError("k must be >= 1")
    if k >= n:
        raise ValueError(f"k={k} must be smaller than the number of points ({n})")
    with torch.cuda.device(eng.device):
        b = bounds if bounds is not None else _bounds(c)
        if not np.isfinite(b).all():
            raise ValueError("coords must be finite")
        if cell_size is None:
            cell_size = default_knn_cell(n, max(b[2] - b[0], 1e-9) * max(b[3] - b[1], 1e-9), k)
        eng.grid_build(d_xy, d_t, None, cell_size, b)
        kn = eng.knn(k, dist_dtype=torch.float64)
        out = {"knn_neighbors": _host.to_host(kn["knn_idx"]).astype(np.int64),
               "knn_neighbor_distances": _host.to_host(kn["dist"])}
        if neighbor_coords:
            out["knn_neighbor_coords"] = _host.to_host(eng.knn_neighbor_coords(kn["knn_idx"], d_xy))
        eng.grid_check()
        if undirected:
            # union + i<j edges + composition + degree statistics: one fused pass chain (pg_knn_union_*)
            u = eng.knn_union(kn["knn_idx"], kn["dist"], types=d_t, n_types=n_types, symmetric_dist=True)
            host = _host.to_host_many({"edges": u["edges"], "weight": u["edge_w"], "row_ptr": u["row_ptr"], "col": u["col"],
                                       "csr_weight": u["w"], "degree": u["degree"], "stats": u["stats"], "hist": u["hist"],
                                       "nbr_count": u["nbr_count"]})
            out.update({
                "edges": host["edges"], "weight": host["weight"],
                "row_ptr": host["row_ptr"].astype(np.int64), "col": host["col"].astype(np.int64),
                "csr_weight": host["csr_weight"], "degree": host["degree"],
                "degree_stats": eng.decode_stats(host["stats"], host["hist"]),
            })
            if d_t is not None:
                out["nbr_count"] = host["nbr_count"]
    return out


def build_radius_graph(coords, r: float = 40.0, types=None, n_types: int = 5, mpp: float | None = None,
                       symmetric_csr: bool = False, bounds=None, device=None, outputs: str = "notebook",
                       count_dtype=np.int32) -> dict:
    """Radius graph of cells 23-26: ``d(i, j) <= r`` (inclusive, like query_ball_tree), ``i < j``.

    ``mpp`` scales pixel coordinates to micrometres first (``x_um = x_px * mpp``, ipynb:2046).
    ``outputs="notebook"`` (default) returns ``edges`` int64 [E,2] sorted by (i, j); ``edge_index`` int64 [2,2E] =
    hstack(edges.T, edges[:, ::-1].T) (the reference's vstack yields [4,E]; see SURVEY B-3); ``edge_attr`` float32
    [2E,1]; ``dist`` float32 [E]; ``degree`` int32 [N]; ``nbr_count`` int32 [N,n_types] (with ``types``);
    ``degree_stats``; and with ``symmetric_csr`` also ``row_ptr`` / ``col`` / ``csr_dist``.
    ``outputs="compact"`` returns the same graph without the redundant int64 tensors: ``edges`` int32 [E,2],
    ``dist`` float32 [E], ``degree``, ``nbr_count``, ``degree_stats`` - a third of the bytes that cross PCIe (the
    notebook tensors are ``graph_features.edge_index_from_edges(edges, dist)`` away, on whichever device consumes
    them), and the whole call is one enqueue + two synchronising copies once the handle has seen a slide of this kind.
    ``count_dtype`` (compact only): ``np.uint8`` / ``np.uint16`` narrow ``degree`` and ``nbr_count`` on the device
    before the copy (a quarter / half of their bytes); ``OverflowError`` if a count does not fit.
    """
    if np.dtype(count_dtype) not in (np.dtype(np.int32), np.dtype(np.uint8), np.dtype(np.uint16)):
        raise ValueError("count_dtype must be int32, uint8 or uint16")
    if outputs != "compact" and np.dtype(count_dtype) != np.dtype(np.int32):
        raise ValueError("count_dtype needs outputs='compact'")
    if outputs not in ("notebook", "compact"):
        raise ValueError("outputs must be 'notebook' or 'compact'")
    eng = get_engine(device)
    c = np.asarray(coords, dtype=np.float64)
    if mpp is not None:
        c = c * float(mpp)
    c, d_xy, d_t = _prep(c, types, eng)
    if not (r >= 0 and np.isfinite(r)):
        raise ValueError("r must be finite and >= 0")
    with torch.cuda.device(eng.device):
        eng.grid_build(d_xy, d_t, None, radius_cell(r), bounds)  # bounds=None: min/max reduced on the device
        if outputs == "compact":
            out = _radius_compact(eng, c.shape[0], r, n_types, d_t is not None, np.dtype(count_dtype))
        else:
            g = eng.radius_graph(r, upper=True, n_types=n_types, compose=True, want_dist32=False, want_edge_index=True)
            e = int(g["total"])
            host = _host.to_host_many({"edge_index": g["edge_index"], "edge_attr": g["edge_attr"], "degree": g["degree"],
                                       "nbr_count": g["nbr_count"] if d_t is not None else None,
                                       "stats": g["stats"], "hist": g["hist"]})
            out = {
                "edges": host["edge_index"][:, :e].T,      # view: rows (i, j), i < j, sorted by (i, j)
                "dist": host["edge_attr"][:e, 0],
                "edge_index": host["edge_index"],
                "edge_attr": host["edge_attr"],
                "degree": host["degree"],
                "degree_stats": eng.decode_stats(host["stats"], host["hist"]),
            }
            if d_t is not None:
                out["nbr_count"] = host["nbr_count"]
        if symmetric_csr:
            s = eng.radius_graph(r, upper=False, compose=False, stats=False, want_dist32=True)
            out["row_ptr"] = _host.to_host(s["row_ptr"]).astype(np.int64)
            out["col"] = _host.to_host(s["col"]).astype(np.int64)
            out["csr_dist"] = _host.to_host(s["dist32"])
    return out


def _radius_compact(eng, n: int, r: float, n_types: int, has_types: bool, count_dtype=np.dtype(np.int32)) -> dict:
    """The compact output set. With a capacity hint from an earlier slide (edges per nucleus seen on this handle)
    the build is pg_radius_graph - outputs given up front, nothing read back in between - followed by two batches of
    device-to-host copies: the per-nucleus arrays with the edge count, then exactly E edges (the capacity's head-room
    stays on the device). Without a hint, or when the hint proves too small, the exact count -> total -> fill sequence
    runs (and leaves a hint behind)."""
    hint = getattr(eng, "_radius_edges_per_point", None)
    for attempt in range(2):
        if hint is not None and attempt == 0 and n > 0:
            cap = int(hint * 1.15 * n) + 4096
            prev = getattr(eng, "_radius_cap", 0)
            if cap <= prev < 2 * cap:
                cap = prev  # same buffers as the last slide of this kind
            eng._radius_cap = cap
            g = eng.radius_graph(r, upper=True, n_types=n_types, compose=True, want_dist32=True, want_edges32=True,
                                 capacity=cap, out=getattr(eng, "_radius_compact_out", None))
            eng._radius_compact_out = {k: v for k, v in g.items() if k in ("col", "dist32", "edges32")}  # reused scratch
        else:
            g = eng.radius_graph(r, upper=True, n_types=n_types, compose=True, want_dist32=True, want_edges32=True)
            cap = int(g["total"])
        deg, nbr = g["degree"], (g["nbr_count"] if has_types else None)
        if count_dtype != np.dtype(np.int32):
            tdt = torch.uint8 if count_dtype == np.dtype(np.uint8) else torch.int16
            deg = eng.narrow_counts(deg, tdt)
            nbr = eng.narrow_counts(nbr, tdt) if nbr is not None else None
        # two batches of copies: the per-nucleus arrays and the edge count first, then exactly E edges - the capacity's
        # 15 % head-room never crosses the link (the second synchronisation costs less than copying it)
        host = _host.to_host_many({"degree": deg, "nbr_count": nbr, "stats": g["stats"], "hist": g["hist"],
                                   "row_end": g["row_ptr"][-1:]})
        e = int(host["row_end"][0])
        if e <= cap:
            # the edge copies are waited for by the flag read that follows them on the stream (pg_check_overflow /
            # pg_grid_check synchronise): one synchronisation for the copies, the overflow flag and the input flag
            host.update(_host.to_host_many({"edges": g["edges32"][:e], "dist": g["dist32"][:e]}, sync=False))
            if count_dtype != np.dtype(np.int32):
                rc = eng.lib.pg_check_overflow(eng._h)  # (also clears the flag; a non-finite input is reported first)
                if rc == _lib.PG_ERR_CAPACITY:
                    raise OverflowError(f"a degree / neighbour-type count does not fit {count_dtype}")
                eng._check(rc)
                if count_dtype == np.dtype(np.uint16):
                    host["degree"] = host["degree"].view(np.uint16)
                    if host.get("nbr_count") is not None:
                        host["nbr_count"] = host["nbr_count"].view(np.uint16)
            break
        eng.lib.pg_check_overflow(eng._h)  # clears the overflow flag the undersized pass has raised
        hint = None
    if n > 0:
        eng._radius_edges_per_point = max(e / n, 1e-3)
    if count_dtype == np.dtype(np.int32):
        eng.grid_check()  # synchronises (the edge copies above) and reports a non-finite input
    out = {"edges": host["edges"], "dist": host["dist"], "degree": host["degree"],
           "degree_stats": eng.decode_stats(host["stats"], host["hist"])}
    if has_types:
        out["nbr_count"] = host["nbr_count"]
    return out


def neighbour_type_composition(row_ptr, col, types, n_types: int = 5, device=None) -> np.ndarray:
    """``nbr_count[i, t-1] = #{j in N(i): type[j] == t}`` for t = 1..n_types over any CSR. int32 [N,T]."""
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_rp = _host.to_device(_host.as_int32(row_ptr, "row_ptr"), np.int32, eng.device)
        d_col = _host.to_device(_host.as_int32(col, "col"), np.int32, eng.device)
        d_t = _host.to_device(_host.as_int32(types, "types"), np.int32, eng.device)
        res = eng.compose_degree(d_rp, d_col, d_t, n_types)
        return _host.to_host(res["nbr_count"])


def degree_stats(row_ptr, hist_len: int = 64, device=None) -> dict:
    """``degree`` int32 [N] and ``min, max, sum, sumsq, mean, std`` (ddof=0, ipynb:2903 convention), ``hist``."""
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_rp = _host.to_device(_host.as_int32(row_ptr, "row_ptr"), np.int32, eng.device)
        res = eng.compose_degree(d_rp, None, None, 1, hist_len=hist_len, compose=False)
        out = eng.decode_stats(res["stats"], res["hist"])
        out["degree"] = _host.to_host(res["degree"])
        return out


def filter_graph_by_type(edges, types, keep_types=(1, 2)):
    """Cell 12 (ipynb:1989-2002): nodes whose type is kept, and the edges with both ends kept.

    Index bookkeeping on the host (two boolean masks); returns (kept node ids int64, edges int64 [E',2])."""
    t = np.asarray(types)
    keep = np.isin(t, list(keep_types))
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    return np.nonzero(keep)[0], e[keep[e[:, 0]] & keep[e[:, 1]]]


def clustering_coefficients(row_ptr, col, device=None) -> dict:
    """``triangles`` int32 [N] and ``clustering`` float64 [N] (= networkx.clustering) of a symmetric CSR with
    ascending rows (README.md:136 "clustering"); ``degree_centrality`` = degree / (N - 1) (networkx's definition)."""
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_rp = _host.to_device(_host.as_int32(row_ptr, "row_ptr"), np.int32, eng.device)
        d_col = _host.to_device(_host.as_int32(col, "col"), np.int32, eng.device)
        res = eng.clustering(d_rp, d_col)
        out = _host.to_host_many(res)
    n = len(out["clustering"])
    deg = np.diff(np.asarray(row_ptr, dtype=np.int64))
    out["degree_centrality"] = deg / (n - 1.0) if n > 1 else np.ones(n)
    return out


def type_interaction_matrix(types, nbr_count, n_types: int = 5, device=None) -> np.ndarray:
    """int64 [T,T]: number of directed edges from a node of type a+1 to a neighbour of type b+1 (README.md:133
    "cell-cell interaction patterns"); symmetric for an undirected graph, diagonal counts each edge twice."""
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_t = _host.to_device(_host.as_int32(types, "types"), np.int32, eng.device)
        d_c = _host.to_device(_host.as_int32(nbr_count, "nbr_count"), np.int32, eng.device)
        return _host.to_host(eng.type_interactions(d_t, d_c, n_types))


def neighbourhood_enrichment(edges, types, n_types: int = 5, n_perms: int = 1000, seed: int = 0, device=None) -> dict:
    """Neighbourhood enrichment of an undirected graph (squidpy.gr.nhood_enrichment's statistic): how much more
    often type a+1 neighbours type b+1 than under random relabelling of the nodes.

    ``edges`` int32 / int64 [E,2] rows (i, j), as ``build_radius_graph`` / ``build_knn_graph`` return them; ``types``
    int [N] (values outside 1..n_types count nowhere).  Every edge row adds one entry (a, b) and one (b, a), so
    ``count`` equals ``type_interaction_matrix`` of the same graph.  ``n_perms`` labellings permute ``types`` by keyed
    bijections of [0, N) derived from ``seed`` (the exact construction is in include/pathgraph.h, K15); the same
    seed gives the same result bit for bit.  Returns [T,T] arrays ``count`` int64, ``perm_mean`` / ``perm_std``
    float64 (mean and ddof-0 std of the permuted counts) and ``zscore`` = (count - perm_mean) / perm_std, NaN or
    +-inf where the permuted counts never vary.  Raises ``ValueError`` on a bad edge shape or an id outside
    [0, N), before anything is launched."""
    t = _host.as_int32(types, "types").reshape(-1)
    n = t.shape[0]
    e = np.asarray(edges)
    if e.size == 0 and e.ndim < 2:
        e = e.reshape(0, 2)
    if e.ndim != 2 or e.shape[1] != 2:
        raise ValueError("edges must have shape (E, 2)")
    if e.size and e.dtype.kind not in "iu":
        raise ValueError(f"edges must be integer ids, got dtype {e.dtype}")
    if e.size and (e.min() < 0 or e.max() >= n):
        raise ValueError(f"edge ids must lie in [0, {n})")
    if not 1 <= n_types <= _lib.PG_MAX_TYPES:
        raise ValueError(f"n_types must be in 1..{_lib.PG_MAX_TYPES}")
    if not 1 <= n_perms <= _lib.PG_ENRICH_MAX_PERMS:
        raise ValueError(f"n_perms must be in 1..{_lib.PG_ENRICH_MAX_PERMS}")
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_e = _host.to_device(e, np.int32, eng.device)  # ids < N <= 2^31 - 1 fit int32
        d_t = _host.to_device(t, np.int32, eng.device)
        return _host.to_host_many(eng.nhood_enrichment(d_e, d_t, n_types, n_perms, seed))


def _distances(values, name: str, min_len: int) -> np.ndarray:
    """Host thresholds for K16: 1-D float64, finite, >= 0, strictly ascending, min_len..PG_PAIRHIST_MAX_THR entries."""
    t = np.asarray(values, dtype=np.float64)
    if t.ndim != 1 or not min_len <= t.shape[0] <= _lib.PG_PAIRHIST_MAX_THR:
        raise ValueError(f"{name} must be a 1-D array of {min_len}..{_lib.PG_PAIRHIST_MAX_THR} distances")
    if not np.isfinite(t).all() or (t < 0).any():
        raise ValueError(f"{name} must be finite and >= 0")
    if (np.diff(t) <= 0).any():
        raise ValueError(f"{name} must be strictly ascending")
    return t


def _pair_hist(coords, types, thresholds, n_types: int, device) -> tuple:
    """Validated host input -> K16 over a grid built for thresholds[-1]: (hist int64 [B,T,T], type_count int64 [T],
    coords, the engine, the device coordinates)."""
    c = np.asarray(coords, dtype=np.float64)
    if c.ndim != 2 or c.shape[1] != 2:
        raise ValueError("coords must have shape (N, 2)")
    if c.shape[0] > _host.INT32_MAX:
        raise OverflowError("more than 2^31 points")
    if not np.isfinite(c).all():
        raise ValueError("coords must be finite")
    t = _host.as_int32(types, "types").reshape(-1)
    if t.shape[0] != c.shape[0]:
        raise ValueError("types must have one entry per point")
    if not 1 <= n_types <= _lib.PG_MAX_TYPES:
        raise ValueError(f"n_types must be in 1..{_lib.PG_MAX_TYPES}")
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_xy = _host.to_device(c, np.float64, eng.device)
        d_t = _host.to_device(t, np.int32, eng.device)
        b = _bounds(c)
        area = max(b[2] - b[0], 1e-9) * max(b[3] - b[1], 1e-9)
        eng.grid_build(d_xy, d_t, None, pair_hist_cell(float(thresholds[-1]), c.shape[0], area), b)
        res = _host.to_host_many(eng.pair_dist_hist(thresholds, n_types))
    return res["hist"], res["type_count"], c, eng, d_xy


def co_occurrence(coords, types, interval, n_types: int = 5, max_dist: float | None = None, cumulative: bool = False,
                  device=None) -> dict:
    """Co-occurrence of cell types across distance (the statistic squidpy.gr.co_occurrence documents): for each
    distance interval, how much more likely a cell of type c+1 is near a cell of type a+1 than anywhere.

    ``interval``: ascending distances t_0 < ... < t_B (2..64 of them, finite, >= 0), or an int together with
    ``max_dist`` for ``np.linspace(0, max_dist, interval)``.  Interval b is the annulus t_b < d <= t_{b+1}, or the disc
    d <= t_{b+1} with ``cumulative``.  There is no whole-slide default: squidpy's (up to half the slide's extent) makes
    every pair of the slide a candidate, which is quadratic in N; pick the distances that matter (tens to hundreds of
    micrometres) and the work is N x the cells within t_B.
    ``types`` int [N]; values outside 1..n_types count nowhere.  Pairs are ordered pairs (i, j) of distinct points (a
    duplicate point is a neighbour at distance 0), with squared distances compared exactly as ``build_radius_graph``
    does.  Returns ``interval`` float64 [B+1], ``count`` int64 [T,T,B] (squidpy's layout: count[a, c, b] = pairs with
    i of type a+1, j of type c+1 in interval b), ``occ`` float64 [T,T,B] = count * S / (R_a R_c) per interval, R = the
    row sums and S = the total of that interval's counts - p(c | a) / p(c), NaN where R_a or R_c is 0 - and
    ``type_count`` int64 [T].  This follows squidpy's documented definition, not its code: its versions differ on
    whether an interval is an annulus or a disc.  Raises ``ValueError`` on bad shapes, non-finite coordinates or
    distances, distances that are negative or not strictly ascending, more than 64 of them, or ``n_types`` outside
    1..16, before anything is launched."""
    if isinstance(interval, (int, np.integer)):
        if max_dist is None or not (np.isfinite(max_dist) and max_dist > 0):
            raise ValueError("an int interval needs a finite max_dist > 0")
        thr = _distances(np.linspace(0.0, float(max_dist), int(interval)), "interval", 2)
    else:
        if max_dist is not None:
            raise ValueError("max_dist only goes with an int interval")
        thr = _distances(interval, "interval", 2)
    hist, type_count, *_ = _pair_hist(coords, types, thr, n_types, device)
    cnt = np.cumsum(hist, axis=0)[1:] if cumulative else hist[1:]
    count = np.ascontiguousarray(np.moveaxis(cnt, 0, -1))
    return {"interval": thr, "count": count, "occ": occurrence_ratio(count), "type_count": type_count}


def occurrence_ratio(count) -> np.ndarray:
    """occ[a, c, b] = count[a, c, b] * S_b / (R_ab R_cb) in float64, R = row sums, S = total of interval b; NaN where a
    row sum is 0 (co_occurrence's ``occ`` from its ``count``)."""
    cnt = np.asarray(count, dtype=np.int64)
    row = cnt.sum(axis=1).astype(np.float64)                  # [T, B]
    tot = cnt.sum(axis=(0, 1)).astype(np.float64)             # [B]
    den = row[:, None, :] * row[None, :, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        occ = cnt.astype(np.float64) * tot / den
    occ[den == 0] = np.nan
    return occ


def ripley(coords, radii, types=None, n_types: int = 5, area: float | None = None, device=None) -> dict:
    """Ripley's K and L functions at ``radii`` (ascending, 1..64 distances, finite, >= 0), without edge correction.

    K_ac(r) = A C_ac(r) / (n_a n_c) and, on the diagonal, A C_aa(r) / (n_a (n_a - 1)), where C_ac(r) counts ordered
    pairs of distinct points of types a+1 and c+1 at distance <= r (the squared-distance rule of ``build_radius_graph``)
    and n_a the points of type a+1; L = sqrt(K / pi).  ``types=None`` gives the univariate K over all points (``K`` and
    ``L`` of shape [len(radii)]); otherwise they are [T,T,len(radii)] (NaN where a count of points is too small).
    ``area`` defaults to the area of the points' convex hull, as squidpy.gr.ripley uses, computed on the GPU by the
    polygon hull kernel (K14) over one ring of all N points.  Returns ``radii``, ``K``, ``L``, ``area``, ``n`` (points
    per type) and ``count`` (C, int64, same layout as ``K``).  Raises ``ValueError`` on the inputs ``co_occurrence``
    rejects and on an ``area`` that is not finite and > 0."""
    r = _distances(radii, "radii", 1)
    univariate = types is None
    c = np.asarray(coords, dtype=np.float64)
    if univariate:
        n_types = 1
        types = np.ones(c.shape[0] if c.ndim == 2 else 0, dtype=np.int32)
    if area is not None and not (np.isfinite(area) and area > 0):
        raise ValueError("area must be finite and > 0")
    hist, n_t, c, eng, d_xy = _pair_hist(c, types, r, n_types, device)
    if area is None:
        with torch.cuda.device(eng.device):
            off = _host.to_device(np.array([0, c.shape[0]], dtype=np.int32), np.int32, eng.device)
            area = float(_host.to_host(eng.ring_hull(off, d_xy)["convex_area"])[0])
    count = np.ascontiguousarray(np.moveaxis(np.cumsum(hist, axis=0), 0, -1))   # [T, T, len(radii)]
    den = n_t[:, None] * n_t[None, :] - np.diag(n_t)                              # n_a n_c, n_a (n_a - 1)
    with np.errstate(divide="ignore", invalid="ignore"):
        k = float(area) * count.astype(np.float64) / den[:, :, None].astype(np.float64)
    k[np.broadcast_to(den[:, :, None] <= 0, k.shape)] = np.nan
    lf = np.sqrt(k / np.pi)
    if univariate:
        k, lf, count = k[0, 0], lf[0, 0], count[0, 0]
    return {"radii": r, "K": k, "L": lf, "area": float(area), "n": n_t, "count": count}


def _normal_tail(z) -> np.ndarray:
    """P(Z > |z|) of a standard normal, elementwise (NaN stays NaN)."""
    z = np.asarray(z, dtype=np.float64)
    out = np.full(z.shape, np.nan)
    ok = ~np.isnan(z)
    out[ok] = [0.5 * math.erfc(abs(v) / math.sqrt(2.0)) for v in z[ok]]
    return out


def fdr_bh(pvals) -> np.ndarray:
    """Benjamini-Hochberg adjusted p-values (statsmodels' ``multipletests(method="fdr_bh")``): p_(k) n / k with the
    running minimum taken from the largest p down, clipped at 1. NaN p-values are left out and stay NaN."""
    p = np.asarray(pvals, dtype=np.float64)
    out = np.full(p.shape, np.nan)
    ok = np.flatnonzero(~np.isnan(p))
    if ok.size:
        order = ok[np.argsort(p[ok], kind="stable")]
        adj = p[order] * ok.size / np.arange(1, ok.size + 1)
        out[order] = np.minimum(np.minimum.accumulate(adj[::-1])[::-1], 1.0)
    return out


def autocorr_moments(mode: str, n: int, s0: float, s1: float, s2: float) -> tuple[float, float]:
    """Expectation and variance of Moran's I / Geary's C under the normality assumption, from the weight sums."""
    with np.errstate(divide="ignore", invalid="ignore"):
        n, s0, s1, s2 = (np.float64(v) for v in (n, s0, s1, s2))
        if mode == "moran":
            e = -1.0 / (n - 1.0)
            v = (n * n * s1 - n * s2 + 3.0 * s0 * s0) / ((n * n - 1.0) * s0 * s0) - e * e
        else:
            e = np.float64(1.0)
            v = ((2.0 * s1 + s2) * (n - 1.0) - 4.0 * s0 * s0) / (2.0 * (n + 1.0) * s0 * s0)
    return float(e), float(v)


def _csr_host(row_ptr, col) -> tuple[np.ndarray, np.ndarray]:
    """Validated symmetric-CSR arrays as int32: row_ptr [N+1] starting at 0, non-decreasing, ending at len(col), and
    col ids in [0, N)."""
    rp, c = np.asarray(row_ptr), np.asarray(col)
    if rp.ndim != 1 or rp.shape[0] < 1 or (rp.size and rp.dtype.kind not in "iu"):
        raise ValueError("row_ptr must be a 1-D integer array of N + 1 offsets")
    if c.ndim != 1 or (c.size and c.dtype.kind not in "iu"):
        raise ValueError("col must be a 1-D integer array")
    rp, c = rp.astype(np.int64), c.astype(np.int64)
    n = rp.shape[0] - 1
    if n > _host.INT32_MAX or c.shape[0] > _host.INT32_MAX:
        raise ValueError("the graph must have fewer than 2^31 nodes and entries")
    if rp[0] != 0 or rp[-1] != c.shape[0] or (np.diff(rp) < 0).any():
        raise ValueError("row_ptr must start at 0, never decrease and end at len(col)")
    if c.size and (c.min() < 0 or c.max() >= n):
        raise ValueError(f"col ids must lie in [0, {n})")
    return rp.astype(np.int32), c.astype(np.int32)


def spatial_autocorr(row_ptr, col, features, mode: str = "moran", transformation: bool = True, n_perms=None,
                     seed: int = 0, two_tailed: bool = False, corr_method: str | None = "fdr_bh", device=None):
    """Spatial autocorrelation of per-nucleus features over a cell graph (squidpy.gr.spatial_autocorr's statistic):
    Moran's I (``mode="moran"``) or Geary's C (``"geary"``) of every column, with its analytic and permutation p-values.

    ``row_ptr`` / ``col``: a symmetric CSR without duplicate entries over N nodes (``build_radius_graph(...,
    symmetric_csr=True)`` or ``build_knn_graph``).  ``features``: [N, F] array or DataFrame (for example
    ``nuclei_morphology_table(...)[CONT_COLS]``), 1 <= F <= 256; column names become the index, rows keep the column
    order.  ``transformation``: row-standardised weights 1 / degree (squidpy's default) instead of binary ones.
    ``n_perms``: None for the analytic test only, else 1..100 000 permutations of the nodes, all columns shuffled
    together (squidpy's procedure), drawn from ``seed`` by K15's keyed bijections (include/pathgraph.h) - the same
    seed gives the same result bit for bit.

    Returns a DataFrame with squidpy's columns: ``I`` or ``C``, ``pval_norm`` (the normal tail of (stat - E) / sqrt(V)
    under the normality assumption) and ``var_norm`` (V); with permutations also ``pval_z_sim`` (the normal tail of
    (stat - perm mean) / perm std), ``pval_sim`` = (min(n_ge, P - n_ge) + 1) / (P + 1), n_ge = permutations at or above
    the observed value, and ``var_sim`` (ddof 0).  ``two_tailed`` doubles the three p-values, as squidpy does.
    ``corr_method="fdr_bh"`` adds Benjamini-Hochberg ``<pval>_fdr_bh`` columns across the features (None: no
    correction).  A constant column, or a graph without edges, gives a NaN statistic and NaN p-values (left out of the
    adjustment).  Raises ``ValueError`` before anything is launched on a malformed CSR,
    a feature table of the wrong length or width, a non-finite feature value (naming its column: a nucleus without a
    polygon has NaN morphology and must be dropped or filled first), an unknown ``mode`` or ``corr_method``, or
    ``n_perms`` out of range."""
    import pandas as pd

    if mode not in ("moran", "geary"):
        raise ValueError(f"mode must be 'moran' or 'geary', got {mode!r}")
    if corr_method not in (None, "fdr_bh"):
        raise ValueError(f"corr_method must be 'fdr_bh' or None, got {corr_method!r}")
    if n_perms is not None and not (isinstance(n_perms, (int, np.integer)) and 1 <= n_perms <= _lib.PG_ENRICH_MAX_PERMS):
        raise ValueError(f"n_perms must be None or an int in 1..{_lib.PG_ENRICH_MAX_PERMS}")
    rp, c = _csr_host(row_ptr, col)
    n = rp.shape[0] - 1
    if isinstance(features, pd.DataFrame):
        names = list(features.columns)
        x = features.to_numpy(dtype=np.float64)
    else:
        x = np.asarray(features, dtype=np.float64)
        if x.ndim == 1:
            x = x[:, None]
        names = list(range(x.shape[1])) if x.ndim == 2 else []
    if x.ndim != 2 or x.shape[0] != n:
        raise ValueError(f"features must have shape (N, F) with N = {n} graph nodes")
    if not 1 <= x.shape[1] <= _lib.PG_AUTOCORR_MAX_FEAT:
        raise ValueError(f"features must have 1..{_lib.PG_AUTOCORR_MAX_FEAT} columns, got {x.shape[1]}")
    bad = np.flatnonzero(~np.isfinite(x).all(axis=0))
    if bad.size:
        raise ValueError(f"feature column {names[bad[0]]!r} has non-finite values")
    p = int(n_perms or 0)
    eng = get_engine(device)
    with torch.cuda.device(eng.device):
        d_rp = _host.to_device(rp, np.int32, eng.device)
        d_c = _host.to_device(c, np.int32, eng.device)
        d_x = _host.to_device(np.ascontiguousarray(x.T), np.float64, eng.device)
        res = _host.to_host_many(eng.spatial_autocorr(d_rp, d_c, d_x, mode, transformation, p, seed))
    return autocorr_frame(res, names, mode, n, p, two_tailed, corr_method)


def autocorr_frame(res: dict, names, mode: str, n: int, n_perms: int, two_tailed: bool = False,
                   corr_method: str | None = "fdr_bh"):
    """spatial_autocorr's DataFrame from the host copies of pg_spatial_autocorr's outputs (``stat``, ``perm_mean``,
    ``perm_var``, ``n_ge``, ``s012``) over n nodes and ``n_perms`` permutations. Where the statistic is undefined (NaN:
    a constant column, or a graph without edges) every p-value is NaN too, so it never reads as significant and the
    Benjamini-Hochberg adjustment leaves it out."""
    import pandas as pd

    stat = np.asarray(res["stat"], dtype=np.float64)
    undefined = np.isnan(stat)
    e, v = autocorr_moments(mode, n, *res["s012"])
    with np.errstate(divide="ignore", invalid="ignore"):
        cols = {"I" if mode == "moran" else "C": stat, "pval_norm": _normal_tail((stat - e) / np.sqrt(v)),
                "var_norm": np.full(stat.shape, v)}
        if n_perms:
            cols["pval_z_sim"] = _normal_tail((stat - res["perm_mean"]) / np.sqrt(res["perm_var"]))
            n_ge = np.asarray(res["n_ge"])
            cols["pval_sim"] = np.where(undefined, np.nan, (np.minimum(n_ge, n_perms - n_ge) + 1.0) / (n_perms + 1.0))
            cols["var_sim"] = np.where(undefined, np.nan, res["perm_var"])
    if two_tailed:
        for k in ("pval_norm", "pval_z_sim", "pval_sim"):
            if k in cols:
                cols[k] = cols[k] * 2.0
    df = pd.DataFrame(cols, index=pd.Index(names))
    if corr_method is not None:
        for k in ("pval_norm", "pval_z_sim", "pval_sim"):
            if k in df.columns:
                df[f"{k}_{corr_method}"] = fdr_bh(df[k].to_numpy())
    return df


def knn_graph_frame(final_df, k: int = 5, centroid_col: str = "centroid", centroid_order: str = "yx",
                    type_col: str | None = None, device=None):
    """Cell 11 at DataFrame level (ipynb:1766-1951): returns ``(df, graph)``.

    ``df`` is a copy of ``final_df`` with the columns the notebook copies back (:1945-1951): ``type_id``, ``color``,
    ``knn_neighbors`` (list of k row positions), ``knn_neighbor_coords`` (list of (x, y) tuples),
    ``knn_neighbor_points`` (shapely Points when shapely is importable, else the same tuples) and
    ``knn_neighbor_distances`` (list of k floats).  ``centroid`` cells are [y, x] as HoverNeXt stores them (the
    notebook builds ``Point(c[1], c[0])``, :1799); pass ``centroid_order="xy"`` for already swapped data.
    ``graph`` is the dict of ``build_knn_graph`` (edges, weights, degree, composition);
    ``interop.to_networkx(graph, df)`` makes the notebook's ``G_knn``."""
    import pandas as pd

    df = final_df.copy()
    c = np.array(df[centroid_col].tolist(), dtype=np.float64).reshape(-1, 2)
    coords = np.ascontiguousarray(c[:, ::-1]) if centroid_order == "yx" else c
    if "type_id" not in df.columns:                                  # ipynb:1807-1813
        if type_col is None and "type_name" in df.columns:
            name_to_id = {v: kk for kk, v in TYPE_NAMES.items()}
            df["type_id"] = df["type_name"].map(name_to_id)
        elif (type_col or "type") in df.columns:
            df["type_id"] = df[type_col or "type"]
        else:
            raise ValueError("No type_name or type column found to map cell types.")
    tid = pd.to_numeric(df["type_id"], errors="coerce")
    types = tid.fillna(0).astype(np.int64).to_numpy()
    g = build_knn_graph(coords, k=k, types=types, device=device, neighbor_coords=True)
    df["knn_neighbors"] = pd.Series(g["knn_neighbors"].tolist(), index=df.index, dtype=object)
    nc = g["knn_neighbor_coords"]
    as_tuples = [[(float(x), float(y)) for x, y in row] for row in nc.tolist()]
    df["knn_neighbor_coords"] = pd.Series(as_tuples, index=df.index, dtype=object)
    try:
        from shapely.geometry import Point  # the notebook's type; absent here -> the coordinate tuples stand in

        df["knn_neighbor_points"] = pd.Series([[Point(x, y) for x, y in row] for row in as_tuples], index=df.index, dtype=object)
    except ImportError:
        df["knn_neighbor_points"] = df["knn_neighbor_coords"]
    df["knn_neighbor_distances"] = pd.Series(g["knn_neighbor_distances"].tolist(), index=df.index, dtype=object)
    df["color"] = [CLASS_COLORS.get(int(t), "black") if np.isfinite(t) else "black" for t in tid.to_numpy(dtype=np.float64)]
    g["pos"] = coords
    return df, g
