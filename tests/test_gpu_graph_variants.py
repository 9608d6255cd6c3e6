"""GPU: the graph kernels off their defaults - every variant a runtime argument selects, bit for bit against the oracle.

Each graph kernel picks a compile-time variant or a code path from a runtime argument, and the rest of the suite mostly
passes the defaults (5 nucleus types, k <= 16, 64 histogram bins). Covered here:
* K6 radius walk: n_types > 5 runs a second walk with per-type counters (WIDE_TYPES) that writes nbr_count itself;
  n_types < 5 takes the row pass's scalar stores; the packed 12-bit type counters are flushed every 4092 candidate
  slots, which only a row with more than 4095 neighbours of one type depends on; R = 1 and the ring walk (R > 1).
* K5 kNN: select<8> (k <= 8), select<16> (9..16), ring<32> (17..32, register list), ring<64> (33..64, list in local
  memory); the select pass hands a point to the ring pass when its 3x3 block holds 65536 candidates or more (its
  histogram counters are 16-bit).
* K7 union: mark / push / rank kernels specialised for 16-byte aligned lists (k = 4, 8, 16), generic otherwise.
* K8: compose_kernel<8> / <16>; degree histograms in shared bins up to 1024 (radius rows, union rank) or 2048
  (compose_degree) bins, global atomics above; the accumulators the last CTA publishes are re-armed for the next call.
* K11 clustering on adversarial CSRs (cliques, a 20 000-leaf hub, rows straddling the 32-row warp ranges).
* K10 node features on both sides of the tile kernel's 40-column limit, up to PG_FEAT_MAX_COLS feature columns.

The CPU tests at the top pin this file's own helpers (the triangle oracle on networkx, the graph builders, the z-score
restatement on the notebook's pandas cells); the GPU tests are marked one by one.
"""
import contextlib

import numpy as np
import pandas as pd
import pytest
import torch
from scipy import sparse

from oracle import graph as ograph
from path_gene_multimodal_b200 import sharding, synth
from path_gene_multimodal_b200.engine import default_knn_cell, radius_cell

N_TYPES = [1, 3, 5, 6, 7, 9, 16]
HIST_LENS = [1, 2, 1024, 1025, 2048, 2049]
FLUSH_SLOTS = 4095          # a 12-bit packed type counter overflows past this many hits between two flushes
SELECT_SEEN_MAX = 65536     # the kNN select pass's 16-bit histogram counters: at this many candidates it gives up
TILE_WIDTH_MAX = 40         # K10: widest output the shared-memory tile kernel assembles
FEAT_MAX_COLS = 256         # PG_FEAT_MAX_COLS


# ---------------------------------------------------------------------------------------------------- helpers
def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def mixed_types(rng, n, n_types):
    """Types drawn from -2..n_types+3, plus a few 17 and 2**31-1: everything outside 1..n_types counts in the degree
    only."""
    t = rng.integers(-2, n_types + 4, size=n).astype(np.int64)
    pick = rng.choice(n, size=max(2, n // 100), replace=False)
    t[pick[0::2]] = 17
    t[pick[1::2]] = 2 ** 31 - 1
    return t.astype(np.int32)


def typed_points(n, n_types, seed):
    xy, _, side = synth.make_points(n, seed)
    return xy, mixed_types(np.random.default_rng(seed), n, n_types), side


def hist_oracle(deg, hist_len):
    return np.bincount(np.minimum(np.asarray(deg, dtype=np.int64), hist_len - 1), minlength=hist_len)


def interactions_oracle(row_ptr, col, types, n_types):
    """inter[a, b] = directed CSR entries from a node of type a+1 to a node of type b+1 (np.add.at)."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    t = np.asarray(types, dtype=np.int64)
    src = t[np.repeat(np.arange(len(rp) - 1), np.diff(rp))]
    dst = t[np.asarray(col, dtype=np.int64)]
    ok = (src >= 1) & (src <= n_types) & (dst >= 1) & (dst <= n_types)
    out = np.zeros((n_types, n_types), dtype=np.int64)
    np.add.at(out, (src[ok] - 1, dst[ok] - 1), 1)
    return out


def csr_from_edges(n, edges):
    """Undirected edge list (any order, duplicates and self loops dropped) -> symmetric CSR with ascending rows."""
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    e = e[e[:, 0] != e[:, 1]]
    key = np.unique(np.minimum(e[:, 0], e[:, 1]) * n + np.maximum(e[:, 0], e[:, 1]))
    und = np.stack([key // n, key % n], axis=1)
    row_ptr, col, _ = ograph.symmetric_csr(und, np.zeros(len(und)), n)
    return row_ptr, col


def triangles_oracle(row_ptr, col, method=None):
    """Triangles through each node of a symmetric CSR (no self loops, no duplicates), int64.

    ``dense``: (A @ A) * A row sums, halved, with A dense float32 (every entry of A @ A is an integer <= n < 2**24, so
    the product is exact whatever the summation order). ``oriented``: edges pointed from lower to higher (degree, id)
    rank, then per triangle a < b < c: (U @ U) * U counts it at its lowest and highest node, (U^T @ U) * U at its middle
    one - in scipy.sparse int64, with work bounded by the out-degrees, so a 20 000-leaf hub costs O(n) where the
    plain (A @ A) * A would hold a 20 000^2 leaf block."""
    rp = np.asarray(row_ptr, dtype=np.int64)
    c = np.asarray(col, dtype=np.int64)
    n = len(rp) - 1
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    if method is None:
        method = "dense" if n <= 6000 else "oriented"
    if method == "dense":
        a = np.zeros((n, n), dtype=np.float32)
        a[np.repeat(np.arange(n), np.diff(rp)), c] = 1.0
        p = a @ a
        p *= a
        return p.astype(np.int64).sum(axis=1) // 2
    deg = np.diff(rp)
    rank = np.empty(n, dtype=np.int64)
    rank[np.lexsort((np.arange(n), deg))] = np.arange(n)
    src = np.repeat(np.arange(n), deg)
    keep = rank[src] < rank[c]
    u = sparse.csr_matrix((np.ones(int(keep.sum()), dtype=np.int64), (src[keep], c[keep])), shape=(n, n))
    t = (u @ u).multiply(u)
    mid = (u.T @ u).multiply(u)
    return (np.asarray(t.sum(axis=1)).ravel() + np.asarray(t.sum(axis=0)).ravel()
            + np.asarray(mid.sum(axis=1)).ravel()).astype(np.int64)


def clustering_oracle(row_ptr, col, method=None):
    """(triangles, coefficient): coefficient = 2 t / (d (d - 1)), 0 for d < 2 - networkx.clustering's definition. Both
    operands are exact integers in float64, so the value is one correctly rounded division, as in networkx's Python
    int / int."""
    tri = triangles_oracle(row_ptr, col, method)
    d = np.diff(np.asarray(row_ptr, dtype=np.int64))
    den = np.where(d < 2, 1, d * (d - 1)).astype(np.float64)
    return tri, np.where(d < 2, 0.0, (2 * tri).astype(np.float64) / den)


def clique_graph(m):
    i, j = np.triu_indices(m, 1)
    return m, np.stack([i, j], axis=1)


def star_graph(leaves):
    return leaves + 1, np.stack([np.zeros(leaves, dtype=np.int64), np.arange(1, leaves + 1)], axis=1)


def hub_path_graph(leaves):
    n, e = star_graph(leaves)
    path = np.stack([np.arange(1, leaves), np.arange(2, leaves + 1)], axis=1)
    return n, np.concatenate([e, path])


def straddling_graph(seed):
    """Long rows (40..150 entries) separated by runs of 1..40 isolated nodes, so rows start and end anywhere in a
    warp's 32-row range and in its 32-entry chunks."""
    rng = np.random.default_rng(seed)
    active, pos = [], 0
    while pos < 3000:
        run = int(rng.integers(1, 41))
        active.extend(range(pos, min(pos + run, 3000)))
        pos += run + int(rng.integers(1, 41))
    active = np.array(active)
    deg = rng.integers(20, 75, size=len(active))
    src = np.repeat(active, deg)
    dst = active[rng.integers(0, len(active), size=len(src))]
    # a little local structure, so there are triangles to find
    near = active[np.clip(np.searchsorted(active, src) + rng.integers(-3, 4, size=len(src)), 0, len(active) - 1)]
    dst = np.where(rng.random(len(src)) < 0.5, near, dst)
    return 3000, np.stack([src, dst], axis=1)


def random_graph(n, p, seed):
    rng = np.random.default_rng(seed)
    i, j = np.triu_indices(n, 1)
    keep = rng.random(len(i)) < p
    return n, np.stack([i[keep], j[keep]], axis=1)


ADVERSARIAL = {
    "clique300": lambda: clique_graph(300),
    "star20000": lambda: star_graph(20_000),
    "hub_path20000": lambda: hub_path_graph(20_000),
    "straddling": lambda: straddling_graph(5),
    "n1": lambda: (1, np.zeros((0, 2), dtype=np.int64)),
    "n31": lambda: random_graph(31, 0.3, 31),
    "n33": lambda: random_graph(33, 0.3, 33),
}


def radius_clump(r=40.0, n_clump=4200, n_background=1000, seed=7):
    """About 4 200 points of type 3 inside a disc of radius 0.4 r (every pair within 0.8 r: a clique, every clump row
    has n_clump - 1 > 4095 same-type neighbours), plus a sparse background of mixed types. The disc is centred in one
    cell of a 0.9 r grid over ``bounds``, so with that grid a single column run holds the whole clump."""
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
    order = rng.permutation(len(xy))                        # clump ids interleaved with background ids
    is_clump = np.concatenate([np.ones(n_clump, bool), np.zeros(n_background, bool)])[order]
    return {"xy": np.ascontiguousarray(xy[order]), "types": types[order], "is_clump": is_clump, "r": r,
            "ring_cell": cell, "bounds": (0.0, 0.0, side, side), "centre": centre}


def knn_clump(n_clump=65_540, n_uniform=30_000, seed=11):
    """65 540 points jittered by sigma = 2 px around one centre plus 30 000 uniform points: every clump point's 3x3
    block of a default kNN grid holds more candidates than the select pass's 16-bit counters take. Just past 2**16, so
    a wrapped counter would read a handful of candidates where there are 65 536 more, instead of more than the pass
    parks (which would send the point to the ring pass anyway)."""
    rng = np.random.default_rng(seed)
    side = 5000.0
    clump = rng.normal(side / 2, 2.0, size=(n_clump, 2))
    xy = np.concatenate([clump, rng.random((n_uniform, 2)) * side])
    types = rng.integers(1, 6, size=len(xy)).astype(np.int32)
    return xy, types, np.arange(len(xy)) < n_clump


def cell_coords(xy, info):
    """The grid's own binning rule (pg_cell_coord): floor((v - v0) * (1 / cell)), clamped."""
    inv = 1.0 / info["cell"]
    cx = np.clip(np.floor((xy[:, 0] - info["x0"]) * inv), 0, info["nx"] - 1).astype(np.int64)
    cy = np.clip(np.floor((xy[:, 1] - info["y0"]) * inv), 0, info["ny"] - 1).astype(np.int64)
    return cx, cy


def block_candidates(xy, info):
    """Points in the 3x3 block of cells around each point's cell (the point itself included)."""
    cx, cy = cell_coords(xy, info)
    nx, ny = info["nx"], info["ny"]
    h = np.zeros((nx + 2, ny + 2), dtype=np.int64)
    np.add.at(h, (cx + 1, cy + 1), 1)
    s = sum(h[1 + dx: 1 + dx + nx, 1 + dy: 1 + dy + ny] for dx in (-1, 0, 1) for dy in (-1, 0, 1))
    return s[cx, cy]


def hub_lists(n, k, seed):
    """kNN-shaped lists whose union has hubs: row i lists the k smallest ids of 0..k other than i, so ids
    0..k-1 end with degree n - 1 and every other row with degree k. Distances are random (not symmetric)."""
    rng = np.random.default_rng(seed)
    base = np.arange(k + 1)
    idx = np.array([base[base != i][:k] if i <= k else base[:k] for i in range(n)], dtype=np.int32)
    return idx, rng.random((n, k)) * 50.0


def zscore_reference(feat, types, onehot_values, mean, std):
    """x of K10 from the kernel's own mean / std: one-hot columns, then float32((v - mean) / std) per feature column
    (one float64 subtract, one divide, one rounding); a column whose std is 0 or NaN is all 0.0 (cell 21)."""
    n = feat.shape[1] if feat is not None else len(types)
    parts = []
    if onehot_values is not None and len(onehot_values):
        parts.append((np.asarray(types)[:, None] == np.asarray(onehot_values)[None, :]).astype(np.float32))
    if feat is not None and len(feat):
        with np.errstate(invalid="ignore", divide="ignore"):
            z = ((feat - mean[:, None]) / std[:, None]).T.astype(np.float32)
        z[:, (std == 0) | np.isnan(std)] = 0.0
        parts.append(z)
    return np.concatenate(parts, axis=1) if parts else np.zeros((n, 0), dtype=np.float32)


@contextlib.contextmanager
def profiled(engine):
    """Names of the kernels launched inside the block (the library's own launch records)."""
    names = []
    engine.profile(True)
    try:
        yield names
        names.extend(name for name, _ in engine.profile_records())
    finally:
        engine.profile(False)


def assert_stats(engine, stats_t, hist_t, deg, hist_len, tag):
    st = engine.decode_stats(stats_t, hist_t)
    deg = np.asarray(deg, dtype=np.int64)
    assert (st["min"], st["max"], st["sum"], st["sumsq"], st["n"]) == (
        int(deg.min()), int(deg.max()), int(deg.sum()), int((deg * deg).sum()), len(deg)), tag
    assert np.array_equal(st["hist"], hist_oracle(deg, hist_len)), tag


# ---------------------------------------------------------------------------------------------------- CPU tests
def test_mixed_types_cover_every_kind_of_type():
    t = mixed_types(np.random.default_rng(0), 5000, 7)
    assert t.dtype == np.int32
    vals = set(np.unique(t).tolist())
    assert set(range(-2, 11)) <= vals and {17, 2 ** 31 - 1} <= vals


def test_triangle_oracle_pinned_on_networkx():
    import networkx as nx

    graphs = [clique_graph(12), star_graph(30), hub_path_graph(30), random_graph(31, 0.3, 31),
              random_graph(33, 0.3, 33), random_graph(200, 0.05, 2), (1, np.zeros((0, 2), dtype=np.int64)),
              (5, np.zeros((0, 2), dtype=np.int64))]
    for n, e in graphs:
        rp, col = csr_from_edges(n, e)
        g = nx.Graph()
        g.add_nodes_from(range(n))
        g.add_edges_from(map(tuple, e.tolist()))
        tri = nx.triangles(g)
        cl = nx.clustering(g)
        for method in ("dense", "oriented"):
            t, c = clustering_oracle(rp, col, method)
            assert np.array_equal(t, [tri[i] for i in range(n)]), (n, method)
            assert np.array_equal(c, [cl[i] for i in range(n)]), (n, method)      # bit for bit
        # the plain sparse product the two methods replace
        a = sparse.csr_matrix((np.ones(len(col), dtype=np.int64), col, rp), shape=(n, n))
        assert np.array_equal(np.asarray((a @ a).multiply(a).sum(axis=1)).ravel() // 2, [tri[i] for i in range(n)])


def test_triangle_oracle_methods_agree_on_the_adversarial_shapes():
    for n, e in (straddling_graph(5), hub_path_graph(2000), clique_graph(150)):
        rp, col = csr_from_edges(n, e)
        assert np.array_equal(triangles_oracle(rp, col, "dense"), triangles_oracle(rp, col, "oriented"))
    n, e = hub_path_graph(20_000)
    t, c = clustering_oracle(*csr_from_edges(n, e))
    assert t[0] == 19_999 and (t[1] == 1) and (t[2:-1] == 2).all() and t[-1] == 1      # hub, path ends, path middle


def test_graph_builders():
    n, e = straddling_graph(5)
    rp, col = csr_from_edges(n, e)
    deg = np.diff(rp)
    assert (deg == 0).sum() > 500 and deg.max() > 64
    iso = np.flatnonzero(deg == 0)
    assert (iso % 32 != 0).any() and len(set((np.flatnonzero(deg) % 32).tolist())) == 32   # rows land everywhere
    for r in range(n):
        row = col[rp[r]:rp[r + 1]]
        assert (np.diff(row) > 0).all() and (row != r).all()                   # ascending, no duplicates / loops
    n, e = star_graph(20_000)
    rp, col = csr_from_edges(n, e)
    assert rp[1] == 20_000 and (np.diff(rp)[1:] == 1).all()


def test_clump_generators_cross_their_thresholds():
    c = radius_clump()
    cl = c["xy"][c["is_clump"]]
    assert len(cl) > FLUSH_SLOTS + 1 and (c["types"][c["is_clump"]] == 3).all()
    assert (np.hypot(*(cl - c["centre"]).T) <= 0.4 * c["r"]).all()
    info = {"x0": 0.0, "y0": 0.0, "cell": c["ring_cell"], "nx": 56, "ny": 56}
    cx, cy = cell_coords(cl, info)
    assert (cx == cx[0]).all() and (cy == cy[0]).all()                        # one cell of the 0.9 r grid
    xy, _, is_clump = knn_clump(n_clump=2000, n_uniform=500)
    assert is_clump.sum() == 2000 and np.ptp(xy[is_clump], axis=0).max() < 40.0


def test_block_candidates_against_brute_force():
    rng = np.random.default_rng(3)
    xy = rng.random((3000, 2)) * 100.0
    info = {"x0": 0.0, "y0": 0.0, "cell": 7.0, "nx": 15, "ny": 15}
    cx, cy = cell_coords(xy, info)
    got = block_candidates(xy, info)
    want = [(np.abs(cx - cx[i]) <= 1) & (np.abs(cy - cy[i]) <= 1) for i in range(0, 3000, 97)]
    assert np.array_equal(got[::97], [w.sum() for w in want])


def test_hub_lists_union_degrees():
    idx, d = hub_lists(3000, 4, 1)
    assert (idx != np.arange(3000)[:, None]).all()
    _, _, rp, _, _ = ograph.undirected_union(idx, d)
    deg = np.diff(rp)
    assert (deg[:4] == 2999).all() and (deg[4:] == 4).all()


def test_zscore_reference_is_the_notebook_cells():
    # with pandas' own mean / std the restatement is oracle/features.node_features bit for bit
    from oracle import features as ofeat

    rng = np.random.default_rng(8)
    n = 700
    cols = ["a", "b", "c", "d"]
    df = pd.DataFrame({"a": rng.normal(size=n) * 30 + 1e6, "b": np.full(n, 0.75), "c": np.full(n, np.nan),
                       "d": rng.gamma(3.0, 2.0, size=n), "type": rng.choice([1, 2, 4], size=n)})
    df.loc[rng.integers(0, n, size=20), "a"] = np.nan
    want, want_cols = ofeat.node_features(df, cont_cols=cols)
    feat = df[cols].to_numpy().T.copy()
    mean = np.array([df[c].mean() for c in cols])
    std = np.array([df[c].std(ddof=0) for c in cols])
    got = zscore_reference(feat, df["type"].to_numpy(), np.array([1, 2, 4]), mean, std)
    assert want_cols[:3] == ["type_1", "type_2", "type_4"]
    assert np.array_equal(got, want, equal_nan=True)


# ---------------------------------------------------------------------------------------------------- 1. type counts
def _check_radius_graph(g, ref, comp, upper, e, tag):
    n = len(ref["row_ptr"]) - 1
    if upper:
        assert np.array_equal(np.diff(g["row_ptr"].cpu().numpy()), np.bincount(ref["edges"][:, 0], minlength=n)), tag
        assert np.array_equal(g["edges"][:e].cpu().numpy(), ref["edges"]), tag
        assert np.array_equal(g["dist64"][:e].cpu().numpy(), ref["dist"]), tag
        assert np.array_equal(g["dist32"][:e].cpu().numpy(), ref["dist"].astype(np.float32)), tag
    else:
        assert np.array_equal(g["row_ptr"].cpu().numpy(), ref["row_ptr"]), tag
        assert np.array_equal(g["col"][:e].cpu().numpy(), ref["col"]), tag
        assert np.array_equal(g["dist64"][:e].cpu().numpy(), ref["csr_dist"]), tag
        assert np.array_equal(g["dist32"][:e].cpu().numpy(), ref["csr_dist"].astype(np.float32)), tag
    assert np.array_equal(g["degree"].cpu().numpy(), np.diff(ref["row_ptr"])), tag
    assert np.array_equal(g["nbr_count"].cpu().numpy(), comp), tag


def _radius_both_calls(engine, ref, comp, r, n_types, tag, hist_len=64):
    """count -> total -> fill, then the fused capacity= call, for upper and symmetric; returns the kernels launched."""
    deg = np.diff(ref["row_ptr"])
    names = set()
    for upper in (True, False):
        with profiled(engine) as launched:
            g = engine.radius_graph(r, upper=upper, n_types=n_types, want_dist32=True, want_dist64=True,
                                    want_edges=upper, hist_len=hist_len)
        e = int(g["total"])
        _check_radius_graph(g, ref, comp, upper, e, tag + ("count+fill", upper))
        assert_stats(engine, g["stats"], g["hist"], deg, hist_len, tag + ("count+fill", upper))
        assert "radius_gather_kernel" in launched and "radius_rows_kernel" in launched
        names.update(launched)
        with profiled(engine) as launched:
            f = engine.radius_graph(r, upper=upper, n_types=n_types, want_dist32=True, want_dist64=True,
                                    want_edges=upper, hist_len=hist_len, capacity=e + 64)
            engine.check_overflow()
        assert int(f["row_ptr"][-1]) == e
        _check_radius_graph(f, ref, comp, upper, e, tag + ("fused", upper))
        assert_stats(engine, f["stats"], f["hist"], deg, hist_len, tag + ("fused", upper))
        assert "radius_rows_gather_kernel" in launched and "radius_gather_kernel" not in launched
        names.update(launched)
    return names


@pytest.mark.gpu
@pytest.mark.parametrize("n_types", N_TYPES)
def test_radius_type_counts(engine, n_types):
    # n_types > 5 dispatches the WIDE_TYPES walk (the row pass then gets no nbr_count); n_types < 5 the scalar stores
    r = 90.0
    xy, types, _ = typed_points(20_000, n_types, 600 + n_types)
    ref = ograph.radius_graph(xy, r)
    comp = ograph.composition(ref["row_ptr"], ref["col"], types, n_types)
    assert (comp.sum(axis=0) > 0).all()                                        # every column is exercised
    deg = np.diff(ref["row_ptr"])
    assert (deg > comp.sum(axis=1)).sum() > len(xy) // 4                       # out-of-range types count in the degree
    for cell in (radius_cell(r), r / 3.0):                                     # R = 1 walk, ring walk
        engine.grid_build(dev(xy), dev(types), None, cell, None)
        R = int(np.ceil(r * (1.0 / engine.grid_info()["cell"]) * (1 + 1e-9) + 1e-9))   # the library's ring_radius
        assert (R == 1) == (cell > r) and R <= 4
        _radius_both_calls(engine, ref, comp, r, n_types, (n_types, cell))


@pytest.mark.gpu
@pytest.mark.parametrize("n_types", N_TYPES)
def test_union_compose_and_interactions_type_counts(engine, n_types):
    k = 8
    xy, types, side = typed_points(20_000, n_types, 700 + n_types)
    n = len(xy)
    d_t = dev(types)
    idx, dist = ograph.knn(xy, k)
    e, w, rp, col, _ = ograph.undirected_union(idx, dist)
    comp = ograph.composition(rp, col, types, n_types)
    assert (comp.sum(axis=0) > 0).all()
    engine.grid_build(dev(xy), d_t, None, default_knn_cell(n, float(side) ** 2, k), None)
    kn = engine.knn(k, dist_dtype=torch.float64)
    assert np.array_equal(kn["knn_idx"].cpu().numpy(), idx) and np.array_equal(kn["dist"].cpu().numpy(), dist)
    u = engine.knn_union(kn["knn_idx"], kn["dist"], types=d_t, n_types=n_types)
    assert np.array_equal(u["row_ptr"].cpu().numpy(), rp) and np.array_equal(u["col"].cpu().numpy(), col)
    assert np.array_equal(u["edges"].cpu().numpy(), e) and np.array_equal(u["edge_w"].cpu().numpy(), w)
    assert np.array_equal(u["nbr_count"].cpu().numpy(), comp)
    assert np.array_equal(u["degree"].cpu().numpy(), np.diff(rp))
    # K8 over both CSRs: the union's and a radius graph's
    r = 90.0
    ref = ograph.radius_graph(xy, r)
    comp_r = ograph.composition(ref["row_ptr"], ref["col"], types, n_types)
    variant = "compose_kernel<8>" if n_types <= 8 else "compose_kernel<16>"
    for row_ptr, c, want in ((u["row_ptr"], u["col"], comp), (dev(ref["row_ptr"], torch.int32), dev(ref["col"], torch.int32), comp_r)):
        with profiled(engine) as launched:
            cd = engine.compose_degree(row_ptr, c, d_t, n_types)
        assert variant in launched, launched
        assert np.array_equal(cd["nbr_count"].cpu().numpy(), want)
        rp_h = row_ptr.cpu().numpy()
        assert np.array_equal(cd["degree"].cpu().numpy(), np.diff(rp_h))
        assert_stats(engine, cd["stats"], cd["hist"], np.diff(rp_h), 64, (n_types, "compose"))
        # K11's neighbour: the type-type interaction matrix over the same counts
        inter = engine.type_interactions(d_t, cd["nbr_count"], n_types).cpu().numpy()
        assert np.array_equal(inter, interactions_oracle(rp_h, c.cpu().numpy(), types, n_types))
    from path_gene_multimodal_b200 import type_interaction_matrix

    assert np.array_equal(type_interaction_matrix(types, comp, n_types=n_types), interactions_oracle(rp, col, types, n_types))


@pytest.mark.gpu
def test_public_api_with_seven_types(engine):
    from path_gene_multimodal_b200 import build_knn_graph, build_radius_graph

    xy, types, _ = typed_points(8000, 7, 77)
    r = 60.0
    ref = ograph.radius_graph(xy, r)
    comp = ograph.composition(ref["row_ptr"], ref["col"], types, 7)
    deg = np.diff(ref["row_ptr"])
    assert deg.max() < 256 and (comp[:, 5:].sum(axis=0) > 0).all()
    g = build_radius_graph(xy, r=r, types=types, n_types=7)
    assert np.array_equal(g["edges"], ref["edges"]) and np.array_equal(g["edge_attr"], ref["edge_attr"])
    assert np.array_equal(g["nbr_count"], comp) and np.array_equal(g["degree"], deg)
    for cd in (np.int32, np.uint8):
        for attempt in range(2):                                # exact sequence, then the capacity path with the hint
            c = build_radius_graph(xy, r=r, types=types, n_types=7, outputs="compact", count_dtype=cd)
            assert np.array_equal(c["edges"].astype(np.int64), ref["edges"]), (cd, attempt)
            assert np.array_equal(c["dist"], ref["dist"].astype(np.float32)), (cd, attempt)
            assert c["nbr_count"].dtype == cd and c["nbr_count"].shape == (len(xy), 7)
            assert np.array_equal(c["nbr_count"].astype(np.int64), comp), (cd, attempt)
            assert np.array_equal(c["degree"].astype(np.int64), deg), (cd, attempt)
    k = build_knn_graph(xy, k=6, types=types, n_types=7)
    idx, dist = ograph.knn(xy, 6)
    e, w, rp, col, _ = ograph.undirected_union(idx, dist)
    assert np.array_equal(k["knn_neighbors"], idx) and np.array_equal(k["edges"], e) and np.array_equal(k["weight"], w)
    assert np.array_equal(k["nbr_count"], ograph.composition(rp, col, types, 7))


def _strips(xy, ty, world):
    d_xy, d_ty = dev(xy), dev(ty)
    gid = torch.arange(len(xy), dtype=torch.int32, device="cuda")
    edges = [float(xy[:, 0].min()), *np.quantile(xy[:, 0], np.arange(1, world) / world).tolist(), float(xy[:, 0].max())]
    parts = []
    for s in sharding.strips_from_edges(edges):
        m = (d_xy[:, 0] >= s.x_lo) & (d_xy[:, 0] < s.x_hi)
        parts.append((s, d_xy[m].contiguous(), d_ty[m].contiguous(), gid[m].contiguous()))
    return d_xy, d_ty, parts


@pytest.mark.gpu
def test_sharded_graphs_with_seven_types(engine):
    world, n_types, r, k = 3, 7, 60.0, 8
    xy, types, side = typed_points(30_000, n_types, 88)
    n = len(xy)
    d_xy, d_ty, parts = _strips(xy, types, world)
    # radius: single GPU, oracle, three emulated ranks
    ref = ograph.radius_graph(xy, r)
    comp = ograph.composition(ref["row_ptr"], ref["col"], types, n_types)
    engine.grid_build(d_xy, d_ty, None, radius_cell(r), None)
    single = engine.radius_graph(r, upper=True, n_types=n_types, want_edges=True)["nbr_count"].cpu().numpy()
    assert np.array_equal(single, comp)
    res = sharding.run_emulated([sharding.sharded_radius_graph(engine, x, t, g, r, s, q, world, n_types=n_types)
                                 for q, (s, x, t, g) in enumerate(parts)])
    nbr = np.full((n, n_types), -1, dtype=np.int32)
    for out, (_, _, _, g) in zip(res, parts):
        assert out["n_ghost"] > 0
        nbr[g.cpu().numpy()] = out["nbr_count"].cpu().numpy()
    assert np.array_equal(nbr, single) and np.array_equal(nbr, comp)
    # kNN + union
    idx, dist = ograph.knn(xy, k)
    _, _, rp, col, _ = ograph.undirected_union(idx, dist)
    comp_k = ograph.composition(rp, col, types, n_types)
    engine.grid_build(d_xy, d_ty, None, default_knn_cell(n, float(side) ** 2, k), None)
    kn = engine.knn(k, dist_dtype=torch.float64)
    single_k = engine.knn_union(kn["knn_idx"], kn["dist"], types=d_ty, n_types=n_types)["nbr_count"].cpu().numpy()
    assert np.array_equal(single_k, comp_k)
    res = sharding.run_emulated([sharding.sharded_knn_graph(engine, x, t, g, k, s, q, world, n_global=n, n_types=n_types)
                                 for q, (s, x, t, g) in enumerate(parts)])
    nbr = np.full((n, n_types), -1, dtype=np.int32)
    for out, (_, _, _, g) in zip(res, parts):
        nbr[g.cpu().numpy()] = out["nbr_count"].cpu().numpy()
    assert np.array_equal(nbr, single_k) and np.array_equal(nbr, comp_k)


# ---------------------------------------------------------------------------------------------------- 2. dense clumps
@pytest.fixture(scope="module")
def clump():
    c = radius_clump()
    ref = ograph.radius_graph_bruteforce(c["xy"], c["r"])
    c["ref"] = ref
    c["deg"] = np.diff(ref["row_ptr"])
    c["comp"] = {t: ograph.composition(ref["row_ptr"], ref["col"], c["types"], t) for t in (5, 7)}
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("n_types", [5, 7])
def test_radius_dense_clump_crosses_the_counter_flush(engine, clump, n_types):
    r, xy, types = clump["r"], clump["xy"], clump["types"]
    comp = clump["comp"][n_types]
    assert comp[clump["is_clump"], 2].min() > FLUSH_SLOTS                      # every clump row crosses the flush
    for cell, bounds in ((radius_cell(r), None), (clump["ring_cell"], clump["bounds"])):
        engine.grid_build(dev(xy), dev(types), None, cell, bounds)
        info = engine.grid_info()
        R = int(np.ceil(r * (1.0 / info["cell"]) * (1 + 1e-9) + 1e-9))
        if cell < r:
            # ring walk (R = 2): the whole clump sits in one cell, i.e. in one contiguous run of one column
            cx, cy = cell_coords(xy[clump["is_clump"]], info)
            assert R == 2 and (cx == cx[0]).all() and (cy == cy[0]).all()
        else:
            assert R == 1
        _radius_both_calls(engine, clump["ref"], comp, r, n_types, ("clump", n_types, cell))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 16])
def test_knn_dense_clump_gives_up_the_select_pass(engine, k):
    xy, types, is_clump = knn_clump()
    n = len(xy)
    span = np.ptp(xy, axis=0)
    engine.grid_build(dev(xy), dev(types), None, default_knn_cell(n, span[0] * span[1], k), None)
    cand = block_candidates(xy, engine.grid_info())
    assert cand[is_clump].min() >= SELECT_SEEN_MAX                             # every clump point is handed on
    with profiled(engine) as launched:
        kn = engine.knn(k, dist_dtype=torch.float64, both=True)
    assert f"knn_select_kernel<{max(k, 8)}>" in launched and f"knn_ring_kernel<{max(k, 8)}>" in launched
    idx, dist = ograph.knn(xy, k)
    assert np.array_equal(kn["knn_idx"].cpu().numpy(), idx)
    assert np.array_equal(kn["dist64"].cpu().numpy(), dist)
    assert np.array_equal(kn["dist32"].cpu().numpy(), dist.astype(np.float32))


# ---------------------------------------------------------------------------------------------------- 3. k boundaries
def _knn_variant(k):
    if k <= 8:
        return {"knn_select_kernel<8>", "knn_ring_kernel<8>"}
    if k <= 16:
        return {"knn_select_kernel<16>", "knn_ring_kernel<16>"}
    return {"knn_ring_kernel<32>"} if k <= 32 else {"knn_ring_kernel<64>"}


def _check_knn_and_union(engine, xy, types, k, idx, dist, cell):
    engine.grid_build(dev(xy), dev(types), None, cell, None)
    with profiled(engine) as launched:
        kn = engine.knn(k, dist_dtype=torch.float64, both=True)
    assert {x for x in launched if x.startswith("knn_") and x != "knn_prepare_kernel"} == _knn_variant(k), launched
    assert np.array_equal(kn["knn_idx"].cpu().numpy(), idx), k
    assert np.array_equal(kn["dist64"].cpu().numpy(), dist), k
    assert np.array_equal(kn["dist32"].cpu().numpy(), dist.astype(np.float32)), k
    # the union's generic kernels at large k (rows of up to 2k entries and more)
    e, w, rp, col, _ = ograph.undirected_union(idx, dist)
    u = engine.knn_union(kn["knn_idx"], kn["dist64"], types=dev(types), n_types=5)
    assert np.array_equal(u["row_ptr"].cpu().numpy(), rp) and np.array_equal(u["col"].cpu().numpy(), col), k
    assert np.array_equal(u["edges"].cpu().numpy(), e) and np.array_equal(u["edge_w"].cpu().numpy(), w), k
    assert np.array_equal(u["nbr_count"].cpu().numpy(), ograph.composition(rp, col, types, 5)), k


@pytest.mark.gpu
@pytest.mark.parametrize("k", [9, 16, 17, 32, 33, 64])
def test_knn_k_boundaries(engine, k):
    xy, types, side = synth.make_points(30_000, seed=31)
    idx, dist = ograph.knn(xy, k)
    _check_knn_and_union(engine, xy, types, k, idx, dist, default_knn_cell(len(xy), float(side) ** 2, k))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [17, 32, 33, 64])
def test_knn_k_boundaries_with_ties(engine, k):
    # integer lattice + duplicates: exact (d^2, id) ties all along the list, at the k-th place too
    gx, gy = np.meshgrid(np.arange(40.0), np.arange(40.0))
    lat = np.stack([gx.ravel(), gy.ravel()], axis=1)
    lat = np.concatenate([lat, lat[::37]])
    t = (np.arange(len(lat)) % 7 + 1).astype(np.int32)
    idx, dist = ograph.knn_bruteforce(lat, k)
    assert (dist[:, -1][:, None] == dist[:, :-1]).any()
    _check_knn_and_union(engine, lat, t, k, idx, dist, 2.5)


@pytest.mark.gpu
def test_knn_k64_on_65_points(engine):
    rng = np.random.default_rng(65)
    xy = rng.random((65, 2)) * 300.0
    t = rng.integers(1, 6, size=65).astype(np.int32)
    idx, dist = ograph.knn_bruteforce(xy, 64)
    assert all(set(idx[i].tolist()) == set(range(65)) - {i} for i in range(65))   # each list is every other point
    _check_knn_and_union(engine, xy, t, 64, idx, dist, default_knn_cell(65, 300.0 ** 2, 64))


# ---------------------------------------------------------------------------------------------------- 4. union alignment
@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("k", [4, 8, 16])
def test_union_on_misaligned_lists(engine, k, dt):
    # the mark / push / rank kernels take their K-specialised, vector-load variants only for 16-byte aligned lists;
    # the same lists at a 4-byte offset (8 bytes for float64 distances) take the generic ones
    xy, types, side = synth.make_points(20_000, seed=90 + k)
    n = len(xy)
    d_t = dev(types)
    engine.grid_build(dev(xy), d_t, None, default_knn_cell(n, float(side) ** 2, k), None)
    kn = engine.knn(k, dist_dtype=dt)
    idx_m = torch.empty(n * k + 1, dtype=torch.int32, device="cuda")[1:].view(n, k)
    idx_m.copy_(kn["knn_idx"])
    d_m = torch.empty(n * k + 1, dtype=dt, device="cuda")[1:].view(n, k)
    d_m.copy_(kn["dist"])
    assert idx_m.data_ptr() % 16 != 0 and d_m.data_ptr() % 16 != 0 and kn["knn_idx"].data_ptr() % 16 == 0
    a = engine.knn_union(kn["knn_idx"], kn["dist"], types=d_t, n_types=5)
    m = engine.knn_union(idx_m, d_m, types=d_t, n_types=5)
    for name in ("row_ptr", "col", "w", "edges", "edge_w", "up_ptr", "nbr_count", "degree", "stats", "hist"):
        assert torch.equal(a[name], m[name]), name
    idx, dist = ograph.knn(xy, k)
    e, w, rp, col, ww = ograph.undirected_union(idx, dist)
    cast = (lambda v: v) if dt == torch.float64 else (lambda v: v.astype(np.float32))
    assert np.array_equal(m["row_ptr"].cpu().numpy(), rp) and np.array_equal(m["col"].cpu().numpy(), col)
    assert np.array_equal(m["w"].cpu().numpy(), cast(ww))
    assert np.array_equal(m["edges"].cpu().numpy(), e) and np.array_equal(m["edge_w"].cpu().numpy(), cast(w))
    assert np.array_equal(m["nbr_count"].cpu().numpy(), ograph.composition(rp, col, types, 5))


# ---------------------------------------------------------------------------------------------------- 5. histogram lengths
@pytest.mark.gpu
@pytest.mark.parametrize("hist_len", HIST_LENS)
def test_degree_histogram_lengths(engine, clump, hist_len):
    # shared bins up to 1024 (radius rows, union rank) / 2048 (compose_degree), global atomics above; each call twice on
    # one handle, since the accumulators the last CTA publishes must be re-armed for the next call
    xy, types, r, ref = clump["xy"], clump["types"], clump["r"], clump["ref"]
    deg = clump["deg"]
    assert deg.max() > max(HIST_LENS)
    engine.grid_build(dev(xy), dev(types), None, radius_cell(r), None)
    for rep in range(2):
        g = engine.radius_graph(r, upper=True, n_types=5, want_dist32=False, hist_len=hist_len)
        assert_stats(engine, g["stats"], g["hist"], deg, hist_len, ("radius count", rep))
        f = engine.radius_graph(r, upper=True, n_types=5, want_dist32=False, hist_len=hist_len, capacity=int(g["total"]))
        engine.check_overflow()
        assert_stats(engine, f["stats"], f["hist"], deg, hist_len, ("radius fused", rep))
    d_rp, d_col = dev(ref["row_ptr"], torch.int32), dev(ref["col"], torch.int32)
    for rep in range(2):
        cd = engine.compose_degree(d_rp, d_col, dev(types), 5, hist_len=hist_len)
        assert_stats(engine, cd["stats"], cd["hist"], deg, hist_len, ("compose", rep))
    idx, dist = hub_lists(3000, 4, 2)
    _, _, rp, col, _ = ograph.undirected_union(idx, dist)
    udeg = np.diff(rp)
    assert udeg.max() > max(HIST_LENS)
    ut = np.random.default_rng(4).integers(0, 8, size=3000).astype(np.int32)
    for rep in range(2):
        u = engine.knn_union(dev(idx), dev(dist), types=dev(ut), n_types=5, hist_len=hist_len)
        assert np.array_equal(u["col"].cpu().numpy(), col)
        assert np.array_equal(u["nbr_count"].cpu().numpy(), ograph.composition(rp, col, ut, 5))
        assert_stats(engine, u["stats"], u["hist"], udeg, hist_len, ("union", rep))
    for rep in range(2):
        cd = engine.compose_degree(u["row_ptr"], u["col"], dev(ut), 5, hist_len=hist_len)
        assert_stats(engine, cd["stats"], cd["hist"], udeg, hist_len, ("compose union", rep))


# ---------------------------------------------------------------------------------------------------- 6. K11
def _check_clustering(engine, rp, col, tag):
    tri, coeff = clustering_oracle(rp, col)
    res = engine.clustering(dev(rp, torch.int32), dev(col, torch.int32))
    assert np.array_equal(res["triangles"].cpu().numpy(), tri), tag
    assert np.array_equal(res["clustering"].cpu().numpy(), coeff), tag              # bit for bit


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ADVERSARIAL))
def test_clustering_adversarial_graphs(engine, name):
    n, e = ADVERSARIAL[name]()
    rp, col = csr_from_edges(n, e)
    _check_clustering(engine, rp, col, name)


@pytest.mark.gpu
def test_clustering_dense_clump(engine, clump):
    ref = clump["ref"]
    assert clump["deg"].max() >= 4000
    _check_clustering(engine, ref["row_ptr"], ref["col"], "clump")


# ---------------------------------------------------------------------------------------------------- 7. K10 width switch
@pytest.mark.gpu
@pytest.mark.parametrize("n_onehot,n_feat", [(5, 34), (5, 35), (5, 36), (0, 40), (0, 41), (0, FEAT_MAX_COLS),
                                             (4, FEAT_MAX_COLS), (6, 0)])
def test_node_features_width_switch(engine, n_onehot, n_feat):
    n = 5000
    rng = np.random.default_rng(n_onehot * 1000 + n_feat)
    feat = None
    if n_feat:
        feat = rng.normal(size=(n_feat, n)) * rng.uniform(0.01, 80.0, size=(n_feat, 1)) + rng.uniform(-100, 100, (n_feat, 1))
        feat[0] += 1e6                                                          # cancellation
        feat[1] = 0.75                                                          # std 0 -> all 0.0
        feat[2] = np.nan                                                        # std NaN -> all 0.0
        feat[3, rng.integers(0, n, size=60)] = np.nan                           # NaN rows skipped by mean / std
    types = rng.integers(-1, 9, size=n).astype(np.int32)
    values = np.array([0, 1, 2, 5, 7, 11][:n_onehot], dtype=np.int32)           # 11: a class no node has
    with profiled(engine) as launched:
        res = engine.node_features(dev(feat) if n_feat else None, dev(types) if n_onehot or not n_feat else None,
                                   dev(values) if n_onehot else None)
    x = res["x"].cpu().numpy()
    width = n_onehot + n_feat
    assert x.shape == (n, width)
    want_kernel = "feature_assemble_tile_kernel" if width <= TILE_WIDTH_MAX else "feature_assemble_kernel"
    assert want_kernel in launched and len([s for s in launched if s.startswith("feature_assemble")]) == 1, launched
    st = res["stats"].cpu().numpy()
    mean, std = (st[:, 0], st[:, 1]) if n_feat else (np.zeros(0), np.zeros(0))
    assert np.array_equal(x, zscore_reference(feat, types, values, mean, std), equal_nan=True)
    if n_feat:
        cols = [pd.Series(v) for v in feat]
        np.testing.assert_allclose(mean, [c.mean() for c in cols], rtol=1e-12, equal_nan=True)
        np.testing.assert_allclose(std, [c.std(ddof=0) for c in cols], rtol=1e-9, atol=1e-12, equal_nan=True)
        assert (x[:, n_onehot + 1] == 0).all() and (x[:, n_onehot + 2] == 0).all()


@pytest.mark.gpu
def test_node_features_column_limit(engine):
    from path_gene_multimodal_b200._lib import PathGraphError

    feat = dev(np.random.default_rng(1).normal(size=(FEAT_MAX_COLS + 1, 100)))
    with pytest.raises(PathGraphError, match="feature columns"):
        engine.node_features(feat)
    ok = engine.node_features(feat[:FEAT_MAX_COLS].contiguous())              # the handle is usable afterwards
    assert ok["x"].shape == (100, FEAT_MAX_COLS)
