"""Device-level driver of libpathgraph.so: torch tensors in, torch tensors out.

torch is used for device memory, streams and (elsewhere) torch.distributed only; every
computation below is one or more hand-written sm_100a kernels behind the C ABI
(include/pathgraph.h).  All tensors must live on the engine's CUDA device.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import PathGraphError, PgHullOut, PgMorphOut, PgRasterOut, PgUnionOut

_INF = float("inf")


def default_knn_cell(n: int, area: float, k: int) -> float:
    """Cell size for kNN grids: about the expected k-th neighbour distance sqrt(k / (pi rho))."""
    if n <= 0 or area <= 0:
        return 1.0
    rho = n / area
    return max(1.15 * math.sqrt(k / (math.pi * rho)), 1e-12)


def radius_cell(r: float) -> float:
    """Cell size for radius grids: just above r, so the 3x3 block around a point covers its ball."""
    return r * (1.0 + 2.0 ** -20) if r > 0 else 1.0


def pair_hist_cell(t_max: float, n: int, area: float) -> float:
    """Cell size for the pair histogram (K16): t_max / 4, so the 9x9 block is 1.6x the ball's area instead of the 3x3
    block's 2.9x, but no smaller than one point per cell on average (smaller cells only add runs to the walk)."""
    floor = math.sqrt(area / n) if n > 0 and area > 0 else 0.0
    return max(t_max / 4.0, floor, 1e-12)


class Engine:
    """One libpathgraph handle (= one workspace) on one CUDA device. Not thread-safe."""

    def __init__(self, device: int | torch.device | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("path_gene_multimodal_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"Engine needs a cuda device, got {dev}")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.lib = _lib.load_library()
        h = C.c_void_p()
        rc = self.lib.pg_create(self.device.index, C.byref(h))
        if rc != 0:
            raise PathGraphError(rc, (self.lib.pg_last_error(None) or b"").decode())
        self._h = h

    # ---- plumbing ----------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.pg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            msg = (self.lib.pg_last_error(self._h) or b"").decode()
            if rc == _lib.PG_ERR_INVALID and "must be finite" in msg:
                raise ValueError("coords must be finite")  # cKDTree raises ValueError on NaN / inf as well
            raise PathGraphError(rc, msg)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _p(self, t: torch.Tensor | None, dtype: torch.dtype, name: str):
        if t is None:
            return None
        if not isinstance(t, torch.Tensor) or t.device != self.device:
            raise ValueError(f"{name}: expected a tensor on {self.device}")
        if t.dtype != dtype:
            raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError(f"{name}: tensor must be contiguous")
        return C.c_void_p(t.data_ptr())

    def _empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    @property
    def launches(self) -> int:
        """Kernels launched through this handle so far (counted inside the library)."""
        return int(self.lib.pg_launch_count(self._h))

    def profile(self, on: bool = True):
        """Start / stop per-kernel CUDA-event timing inside the library (clears earlier records)."""
        self._check(self.lib.pg_profile_enable(self._h, 1 if on else 0))

    def profile_records(self) -> list[tuple[str, float]]:
        """[(kernel name, milliseconds)] for every launch since profile(True); synchronises."""
        n = self.lib.pg_profile_count(self._h)
        out = []
        name, ms = C.c_char_p(), C.c_float()
        for i in range(n):
            self._check(self.lib.pg_profile_get(self._h, i, C.byref(name), C.byref(ms)))
            out.append((name.value.decode(), float(ms.value)))
        return out

    def capture(self, fn, warmup: int = 2):
        """Capture ``fn()`` - a sequence of calls on this engine that never reads anything back (bounds given to
        grid_build, ``capacity`` / ``presized`` outputs) - into a CUDA graph and return it (``graph.replay()``).

        The hot path of a small slide is a dozen short kernels; replaying them as one graph removes the per-launch
        host cost that bounds such a pass. ``fn`` is run ``warmup`` times first (workspace growth and output
        allocation must not happen during capture) and its tensors must be kept alive by the caller."""
        stream = torch.cuda.Stream(self.device)
        stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(stream):
            for _ in range(max(warmup, 1)):
                fn()
        torch.cuda.current_stream(self.device).wait_stream(stream)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            fn()
        return graph

    def workspace_bytes(self) -> int:
        return int(self.lib.pg_workspace_bytes(self._h))

    def check_overflow(self):
        self._check(self.lib.pg_check_overflow(self._h))

    def grid_check(self):
        """Synchronise and raise if the last grid_build met a non-finite coordinate."""
        self._check(self.lib.pg_grid_check(self._h))

    @staticmethod
    def decode_stats(stats_t: torch.Tensor, hist: torch.Tensor | None = None) -> dict:
        """pg_degree_stats block (4 x int64 on the device) -> python dict (one D2H copy)."""
        s = stats_t.cpu().numpy() if isinstance(stats_t, torch.Tensor) else np.asarray(stats_t)
        raw = s.view(np.int32)
        n = int(s[3])
        tot, sq = int(s[1]), int(s[2])
        mean = tot / n if n else float("nan")
        var = max(sq / n - mean * mean, 0.0) if n else float("nan")
        out = {"min": int(raw[0]), "max": int(raw[1]), "sum": tot, "sumsq": sq, "n": n,
               "mean": mean, "std": math.sqrt(var) if n else float("nan")}
        if hist is not None:
            out["hist"] = (hist.cpu().numpy() if isinstance(hist, torch.Tensor) else np.asarray(hist)).astype(np.int64)
        return out

    # ---- K1 ------------------------------------------------------------------------------------
    def map_morph(self, poly_off, poly_xy, nuc_tile=None, tile_x=None, tile_y=None, centroid=None, bbox=None,
                  write_polygons=True, extra=False, out=None):
        """Fused tile->WSI shift + polygon morphology (pg_map_morph_f32 / _f64).

        poly_off int32 [N+1]; poly_xy float32|float64 [M,2]; nuc_tile int32 [N]; tile_x/y int32 [n_tiles];
        centroid float64 [N,2]; bbox int32 [N,4].  Returns a dict of device tensors:
        wsi_poly_xy, wsi_centroid, wsi_bbox, area, perimeter, eccentricity, circularity and, with
        ``extra``, major_axis, minor_axis, centroid_x, centroid_y, poly_bbox.  ``out`` may carry
        preallocated tensors of the same names (reused, not reallocated).
        """
        n = int(poly_off.numel()) - 1
        vt = poly_xy.dtype
        if vt not in (torch.float32, torch.float64):
            raise ValueError("poly_xy must be float32 or float64")
        m = int(poly_xy.shape[0]) if poly_xy.dim() == 2 else int(poly_xy.numel() // 2)
        res = dict(out) if out else {}

        def get(name, shape, dtype):
            t = res.get(name)
            if t is None:
                t = self._empty(shape, dtype)
                res[name] = t
            return t

        wsi_poly = get("wsi_poly_xy", (m, 2), vt) if write_polygons else None
        wsi_c = get("wsi_centroid", (n, 2), torch.float64) if centroid is not None else None
        wsi_b = get("wsi_bbox", (n, 4), torch.int32) if bbox is not None else None
        mo = PgMorphOut()
        for name in ("area", "perimeter", "eccentricity", "circularity"):
            setattr(mo, name, self._p(get(name, (n,), torch.float32), torch.float32, name))
        if extra:
            for name in ("major_axis", "minor_axis"):
                setattr(mo, name, self._p(get(name, (n,), torch.float32), torch.float32, name))
            for name in ("centroid_x", "centroid_y"):
                setattr(mo, name, self._p(get(name, (n,), torch.float64), torch.float64, name))
            mo.poly_bbox = self._p(get("poly_bbox", (n, 4), torch.float64), torch.float64, "poly_bbox")
        self._check(self.lib.pg_map_morph_hint(self._h, n, m))
        fn = self.lib.pg_map_morph_f32 if vt == torch.float32 else self.lib.pg_map_morph_f64
        self._check(fn(self._h, n, self._p(poly_off, torch.int32, "poly_off"), self._p(poly_xy, vt, "poly_xy"),
                       self._p(nuc_tile, torch.int32, "nuc_tile"), self._p(tile_x, torch.int32, "tile_x"),
                       self._p(tile_y, torch.int32, "tile_y"), self._p(centroid, torch.float64, "centroid"),
                       self._p(bbox, torch.int32, "bbox"), self._p(wsi_poly, vt, "wsi_poly_xy"),
                       self._p(wsi_c, torch.float64, "wsi_centroid"), self._p(wsi_b, torch.int32, "wsi_bbox"),
                       C.byref(mo), self._stream()))
        return res

    # ---- K14 -----------------------------------------------------------------------------------
    def ring_hull(self, poly_off, poly_xy, out=None):
        """Convex area, solidity and orientation of every ring (pg_ring_hull_f32 / _f64).

        poly_off int32 [N+1]; poly_xy float32|float64 [M,2].  Returns a dict of float64 device tensors [N]:
        convex_area, solidity, orientation.  ``out`` may carry preallocated tensors of the same names.  Asynchronous
        and free of host synchronisation once the workspace has grown, so it can be captured (``capture``)."""
        n = int(poly_off.numel()) - 1
        vt = poly_xy.dtype
        if vt not in (torch.float32, torch.float64):
            raise ValueError("poly_xy must be float32 or float64")
        m = int(poly_xy.shape[0]) if poly_xy.dim() == 2 else int(poly_xy.numel() // 2)
        res = dict(out) if out else {}
        ho = PgHullOut()
        for name in ("convex_area", "solidity", "orientation"):
            if res.get(name) is None:
                res[name] = self._empty((n,), torch.float64)
            setattr(ho, name, self._p(res[name], torch.float64, name))
        fn = self.lib.pg_ring_hull_f32 if vt == torch.float32 else self.lib.pg_ring_hull_f64
        self._check(fn(self._h, n, m, self._p(poly_off, torch.int32, "poly_off"), self._p(poly_xy, vt, "poly_xy"),
                       C.byref(ho), self._stream()))
        return res

    # ---- K2-K4 ---------------------------------------------------------------------------------
    def grid_build(self, xy, types=None, gid=None, cell_size=1.0, bounds=None, n_query=None):
        """Bin points into the uniform grid kept inside the handle (pg_grid_build)."""
        n = int(xy.shape[0])
        nq = n if n_query is None else int(n_query)
        b = None
        if bounds is not None:
            b = (C.c_double * 4)(*[float(v) for v in bounds])
        self._check(self.lib.pg_grid_build(self._h, n, nq, self._p(xy, torch.float64, "xy"),
                                           self._p(types, torch.int32, "types"), self._p(gid, torch.int32, "gid"),
                                           float(cell_size), b, self._stream()))
        self._n, self._nq = n, nq

    def grid_export(self):
        """(xy, types, ids) of the built grid's points in cell order (pg_grid_export): a spatial sort of the input."""
        n = self._n
        xy = self._empty((n, 2), torch.float64)
        ty = self._empty((n,), torch.int32)
        gid = self._empty((n,), torch.int32)
        self._check(self.lib.pg_grid_export(self._h, self._p(xy, torch.float64, "xy"), self._p(ty, torch.int32, "types"),
                                            self._p(gid, torch.int32, "gid"), self._stream()))
        return xy, ty, gid

    def grid_info(self) -> dict:
        nx, ny = C.c_int32(), C.c_int32()
        x0, y0, cell = C.c_double(), C.c_double(), C.c_double()
        self._check(self.lib.pg_grid_info(self._h, C.byref(nx), C.byref(ny), C.byref(x0), C.byref(y0), C.byref(cell)))
        return {"nx": nx.value, "ny": ny.value, "x0": x0.value, "y0": y0.value, "cell": cell.value}

    # ---- K5 ------------------------------------------------------------------------------------
    def knn(self, k, dist_dtype=torch.float64, both=False, x_lo=-_INF, x_hi=_INF, check_halo=False, out=None):
        """kNN over the built grid. Returns dict(knn_idx int32 [nq,k], dist (f64 or f32)[, dist32][, halo_ok])."""
        nq = self._nq
        res = dict(out) if out else {}
        idx = res.get("knn_idx")
        if idx is None:
            idx = res["knn_idx"] = self._empty((nq, k), torch.int32)
        d64 = d32 = None
        if dist_dtype == torch.float64 or both:
            d64 = res.get("dist64")
            if d64 is None:
                d64 = res["dist64"] = self._empty((nq, k), torch.float64)
        if dist_dtype == torch.float32 or both:
            d32 = res.get("dist32")
            if d32 is None:
                d32 = res["dist32"] = self._empty((nq, k), torch.float32)
        ok = None
        if check_halo:
            ok = res.get("halo_ok")
            if ok is None:
                ok = res["halo_ok"] = self._empty((1,), torch.int32)
        self._check(self.lib.pg_knn(self._h, int(k), self._p(idx, torch.int32, "knn_idx"),
                                    self._p(d64, torch.float64, "dist64"), self._p(d32, torch.float32, "dist32"),
                                    float(x_lo), float(x_hi), self._p(ok, torch.int32, "halo_ok"), self._stream()))
        res["dist"] = d64 if dist_dtype == torch.float64 else d32
        return res

    def knn_neighbor_coords(self, knn_idx, xy):
        """float64 [n,k,2]: coordinates of every kNN list entry (pg_knn_neighbor_coords)."""
        n, k = int(knn_idx.shape[0]), int(knn_idx.shape[1])
        out = self._empty((n, k, 2), torch.float64)
        self._check(self.lib.pg_knn_neighbor_coords(self._h, n, k, self._p(knn_idx, torch.int32, "knn_idx"),
                                                    self._p(xy, torch.float64, "xy"), int(xy.shape[0]),
                                                    self._p(out, torch.float64, "out"), self._stream()))
        return out

    # ---- K6 + fused K8 ---------------------------------------------------------------------------
    def radius_graph(self, r, upper=False, n_types=5, compose=True, stats=True, hist_len=64, want_dist32=True,
                     want_dist64=False, want_edges=False, want_edge_index=False, capacity=None, out=None,
                     want_edges32=False):
        """Radius graph over the built grid: count (+composition / degree) -> scan -> fill.

        With ``capacity`` (entries) the whole sequence is enqueued without a host sync and the
        returned col / dist tensors have ``capacity`` rows (valid prefix = row_ptr[-1]); call
        ``check_overflow()`` later.  Without it the total is read back and outputs are exact-size.
        ``want_edge_index`` (needs ``upper`` and the exact total) adds the notebook's packed tensors
        ``edge_index`` int64 [2,2E] and ``edge_attr`` float32 [2E,1], written by the fill kernel.
        ``want_edges32``: the edge list as int32 [E,2] (``edges32``) - half the bytes of ``edges`` on the way to the host.
        """
        nq = self._nq
        res = dict(out) if out else {}

        def get(name, shape, dtype):
            t = res.get(name)
            if t is None or tuple(t.shape) != tuple(shape):
                t = res[name] = self._empty(shape, dtype)
            return t

        row_ptr = get("row_ptr", (nq + 1,), torch.int32)
        degree = get("degree", (nq,), torch.int32) if compose else None
        nbr = get("nbr_count", (nq, n_types), torch.int32) if compose else None
        st = get("stats", (4,), torch.int64) if stats else None
        hist = get("hist", (hist_len,), torch.int32) if (stats and hist_len) else None
        if capacity is not None and not want_edge_index:
            # outputs known up front: one call, the fill pass fused into the row pass (pg_radius_graph)
            cap = int(capacity)
            col = get("col", (cap,), torch.int32)
            d32 = get("dist32", (cap,), torch.float32) if want_dist32 else None
            d64 = get("dist64", (cap,), torch.float64) if want_dist64 else None
            edges = get("edges", (cap, 2), torch.int64) if want_edges else None
            edges32 = get("edges32", (cap, 2), torch.int32) if want_edges32 else None
            self._check(self.lib.pg_radius_graph(
                self._h, float(r), 1 if upper else 0, self._p(row_ptr, torch.int32, "row_ptr"),
                self._p(degree, torch.int32, "degree"), self._p(nbr, torch.int32, "nbr_count"), int(n_types),
                self._p(st, torch.int64, "stats"), self._p(hist, torch.int32, "hist"),
                int(hist_len) if hist is not None else 0, self._p(col, torch.int32, "col"),
                self._p(d32, torch.float32, "dist32"), self._p(d64, torch.float64, "dist64"),
                self._p(edges, torch.int64, "edges"), self._p(edges32, torch.int32, "edges32"), cap, self._stream()))
            return res
        if capacity is not None:
            self._check(self.lib.pg_radius_reserve(self._h, int(capacity)))
        self._check(self.lib.pg_radius_count(self._h, float(r), 1 if upper else 0,
                                             self._p(row_ptr, torch.int32, "row_ptr"), self._p(degree, torch.int32, "degree"),
                                             self._p(nbr, torch.int32, "nbr_count"), int(n_types),
                                             self._p(st, torch.int64, "stats"), self._p(hist, torch.int32, "hist"),
                                             int(hist_len) if hist is not None else 0, self._stream()))
        if capacity is None:
            total = C.c_int64()
            self._check(self.lib.pg_radius_total(self._h, C.byref(total)))
            cap = int(total.value)
            res["total"] = cap
        else:
            cap = int(capacity)
        col = get("col", (cap,), torch.int32)
        d32 = get("dist32", (cap,), torch.float32) if want_dist32 else None
        d64 = get("dist64", (cap,), torch.float64) if want_dist64 else None
        edges = get("edges", (cap, 2), torch.int64) if want_edges else None
        edges32 = get("edges32", (cap, 2), torch.int32) if want_edges32 else None
        ei = ea = None
        if want_edge_index:
            if capacity is not None or not upper:
                raise ValueError("want_edge_index needs upper=True and no capacity (exact total)")
            ei = get("edge_index", (2, 2 * cap), torch.int64)
            ea = get("edge_attr", (2 * cap, 1), torch.float32)
        self._check(self.lib.pg_radius_fill(self._h, self._p(row_ptr, torch.int32, "row_ptr"),
                                            self._p(col, torch.int32, "col"), self._p(d32, torch.float32, "dist32"),
                                            self._p(d64, torch.float64, "dist64"), self._p(edges, torch.int64, "edges"),
                                            self._p(edges32, torch.int32, "edges32"), self._p(ei, torch.int64, "edge_index"), self._p(ea, torch.float32, "edge_attr"),
                                            cap if want_edge_index else 0, cap, self._stream()))
        return res

    # ---- K7 ------------------------------------------------------------------------------------
    def symmetrize(self, knn_idx, knn_dist, want_w32=False, row_id=None, id_map=None):
        """Undirected union of directed kNN lists -> symmetric CSR (row_ptr, col ascending, weight=min).

        ``row_id`` / ``id_map`` (both or neither): the lists hold global ids, row i has id row_id[i] and
        id_map[id] is the row of an id (-1 when it has no row here) - used for strips + halo."""
        n, k = int(knn_idx.shape[0]), int(knn_idx.shape[1])
        row_ptr = self._empty((n + 1,), torch.int32)
        n_ids = int(id_map.numel()) if id_map is not None else 0
        self._check(self.lib.pg_knn_symmetrize_count(self._h, n, k, self._p(knn_idx, torch.int32, "knn_idx"),
                                                     self._p(row_id, torch.int32, "row_id"),
                                                     self._p(id_map, torch.int32, "id_map"), n_ids,
                                                     self._p(row_ptr, torch.int32, "row_ptr"), self._stream()))
        total = C.c_int64()
        self._check(self.lib.pg_knn_symmetrize_total(self._h, C.byref(total)))
        e = int(total.value)
        col = self._empty((e,), torch.int32)
        is64 = knn_dist.dtype == torch.float64
        w64 = self._empty((e,), torch.float64) if is64 else None
        w32 = self._empty((e,), torch.float32) if (want_w32 or not is64) else None
        self._check(self.lib.pg_knn_symmetrize_fill(
            self._h, n, k, self._p(knn_idx, torch.int32, "knn_idx"),
            self._p(knn_dist, torch.float64, "dist64") if is64 else None,
            None if is64 else self._p(knn_dist, torch.float32, "dist32"),
            self._p(row_id, torch.int32, "row_id"), self._p(id_map, torch.int32, "id_map"),
            self._p(row_ptr, torch.int32, "row_ptr"), self._p(col, torch.int32, "col"),
            self._p(w64, torch.float64, "w64"), self._p(w32, torch.float32, "w32"), self._stream()))
        return {"row_ptr": row_ptr, "col": col, "w64": w64, "w32": w32, "w": w64 if is64 else w32}

    def knn_union(self, knn_idx, knn_dist, types=None, n_types=5, hist_len=64, row_id=None, id_map=None,
                  want_edges=True, compose=True, symmetric_dist=False, presized=False):
        """Undirected union + i<j edge list + composition + degree statistics in one pass chain (pg_knn_union_*).

        Returns row_ptr, col, w (dtype of ``knn_dist``), edges int64 [E,2], edge_w, degree, stats, hist and, with
        ``types`` (indexed by column id), nbr_count.  One host synchronisation (the two totals).  ``symmetric_dist``:
        the lists come from ``knn()`` on one coordinate set (d(i,j) == d(j,i) bit for bit), so weight = min needs no
        reverse lookup.  ``presized``: size col / w / edges by their bounds (2 k n symmetric entries, k n edges) instead
        of reading the totals back - no host synchronisation at all; the valid prefixes are ``row_ptr[-1]`` and
        ``up_ptr[-1]`` (device values), so a whole table pass can be enqueued (or graph-captured) in one go."""
        n, k = int(knn_idx.shape[0]), int(knn_idx.shape[1])
        row_ptr = self._empty((n + 1,), torch.int32)
        up_ptr = self._empty((n + 1,), torch.int32) if want_edges else None
        n_ids = int(id_map.numel()) if id_map is not None else 0
        self._check(self.lib.pg_knn_union_count(self._h, n, k, self._p(knn_idx, torch.int32, "knn_idx"),
                                                self._p(row_id, torch.int32, "row_id"),
                                                self._p(id_map, torch.int32, "id_map"), n_ids,
                                                self._p(row_ptr, torch.int32, "row_ptr"),
                                                self._p(up_ptr, torch.int32, "up_ptr"), self._stream()))
        if presized:
            e, eu = 2 * n * k, (n * k if want_edges else 0)
        else:
            total, upper = C.c_int64(), C.c_int64()
            self._check(self.lib.pg_knn_union_total(self._h, C.byref(total), C.byref(upper)))
            e, eu = int(total.value), int(upper.value) if want_edges else 0
        is64 = knn_dist.dtype == torch.float64
        wt = torch.float64 if is64 else torch.float32
        col, w = self._empty((e,), torch.int32), self._empty((e,), wt)
        edges = self._empty((eu, 2), torch.int64) if want_edges else None
        edge_w = self._empty((eu,), wt) if want_edges else None
        do_comp = compose and types is not None
        nbr = self._empty((n, n_types), torch.int32) if do_comp else None
        degree = self._empty((n,), torch.int32)
        st = self._empty((4,), torch.int64)
        hist = self._empty((hist_len,), torch.int32) if hist_len else None
        x = PgUnionOut()
        x.edges = self._p(edges, torch.int64, "edges")
        x.edge_w64 = self._p(edge_w, torch.float64, "edge_w") if is64 else None
        x.edge_w32 = None if is64 else self._p(edge_w, torch.float32, "edge_w")
        x.type = self._p(types, torch.int32, "types") if do_comp else None
        x.n_types = int(n_types)
        x.nbr_count = self._p(nbr, torch.int32, "nbr_count")
        x.degree = self._p(degree, torch.int32, "degree")
        x.stats = self._p(st, torch.int64, "stats")
        x.hist = self._p(hist, torch.int32, "hist")
        x.hist_len = int(hist_len) if hist is not None else 0
        x.symmetric_dist = 1 if symmetric_dist else 0
        x.presized = 1 if presized else 0
        self._check(self.lib.pg_knn_union_fill(
            self._h, n, k, self._p(knn_idx, torch.int32, "knn_idx"),
            self._p(knn_dist, torch.float64, "dist64") if is64 else None,
            None if is64 else self._p(knn_dist, torch.float32, "dist32"),
            self._p(row_id, torch.int32, "row_id"), self._p(id_map, torch.int32, "id_map"),
            self._p(row_ptr, torch.int32, "row_ptr"), self._p(up_ptr, torch.int32, "up_ptr"),
            self._p(col, torch.int32, "col"), self._p(w, torch.float64, "w") if is64 else None,
            None if is64 else self._p(w, torch.float32, "w"), C.byref(x), self._stream()))
        return {"row_ptr": row_ptr, "col": col, "w": w, "edges": edges, "edge_w": edge_w, "up_ptr": up_ptr,
                "nbr_count": nbr, "degree": degree, "stats": st, "hist": hist}

    def csr_upper(self, row_ptr, col, w=None, row_id=None, want_w32=False):
        """Symmetric CSR (rows ascending) -> edges int64 [E,2] with i<j, sorted by (i,j), + weights."""
        n = int(row_ptr.numel()) - 1
        up_ptr = self._empty((n + 1,), torch.int32)
        self._check(self.lib.pg_csr_upper_count(self._h, n, self._p(row_ptr, torch.int32, "row_ptr"),
                                                self._p(col, torch.int32, "col"), self._p(row_id, torch.int32, "row_id"),
                                                self._p(up_ptr, torch.int32, "up_ptr"), self._stream()))
        total = C.c_int64()
        self._check(self.lib.pg_csr_upper_total(self._h, C.byref(total)))
        e = int(total.value)
        edges = self._empty((e, 2), torch.int64)
        w64 = w32 = ew64 = ew32 = None
        if w is not None:
            if w.dtype == torch.float64:
                w64, ew64 = w, self._empty((e,), torch.float64)
                if want_w32:
                    ew32 = self._empty((e,), torch.float32)
            else:
                w32, ew32 = w, self._empty((e,), torch.float32)
        self._check(self.lib.pg_csr_upper_fill(
            self._h, n, self._p(row_ptr, torch.int32, "row_ptr"), self._p(col, torch.int32, "col"),
            self._p(w64, torch.float64, "w64"), self._p(w32, torch.float32, "w32"),
            self._p(row_id, torch.int32, "row_id"), self._p(up_ptr, torch.int32, "up_ptr"),
            self._p(edges, torch.int64, "edges"), self._p(ew64, torch.float64, "ew64"),
            self._p(ew32, torch.float32, "ew32"), self._stream()))
        return {"edges": edges, "w64": ew64, "w32": ew32, "up_ptr": up_ptr}

    # ---- K8 ------------------------------------------------------------------------------------
    def compose_degree(self, row_ptr, col, types, n_types=5, hist_len=64, compose=True):
        n = int(row_ptr.numel()) - 1
        nbr = self._empty((n, n_types), torch.int32) if compose else None
        degree = self._empty((n,), torch.int32)
        st = self._empty((4,), torch.int64)
        hist = self._empty((hist_len,), torch.int32) if hist_len else None
        self._check(self.lib.pg_compose_degree(
            self._h, n, self._p(row_ptr, torch.int32, "row_ptr"), self._p(col, torch.int32, "col"),
            self._p(types, torch.int32, "types"), int(n_types), self._p(nbr, torch.int32, "nbr_count"),
            self._p(degree, torch.int32, "degree"), self._p(st, torch.int64, "stats"),
            self._p(hist, torch.int32, "hist"), int(hist_len) if hist is not None else 0, self._stream()))
        return {"nbr_count": nbr, "degree": degree, "stats": st, "hist": hist}

    # ---- K12 -----------------------------------------------------------------------------------
    def raster_props(self, inst_map, n_labels, solidity=False):
        """skimage-regionprops quantities of an int32 instance map [H,W] for labels 1..n_labels (pg_raster_props)."""
        hgt, wid = int(inst_map.shape[0]), int(inst_map.shape[1])
        n = int(n_labels)
        res = {"area": self._empty((n,), torch.int32), "bbox": self._empty((n, 4), torch.int32),
               "centroid": self._empty((n, 2), torch.float64)}
        for name in ("perimeter", "eccentricity", "major_axis", "minor_axis", "orientation"):
            res[name] = self._empty((n,), torch.float64)
        ro = PgRasterOut()
        ro.area, ro.bbox = self._p(res["area"], torch.int32, "area"), self._p(res["bbox"], torch.int32, "bbox")
        for name in ("centroid", "perimeter", "eccentricity", "major_axis", "minor_axis", "orientation"):
            setattr(ro, name, self._p(res[name], torch.float64, name))
        self._check(self.lib.pg_raster_props(self._h, hgt, wid, self._p(inst_map, torch.int32, "inst_map"), n,
                                             C.byref(ro), self._stream()))
        if solidity and n > 0:
            res["convex_area"] = self._empty((n,), torch.int32)
            res["solidity"] = self._empty((n,), torch.float64)
            self._check(self.lib.pg_raster_solidity(
                self._h, hgt, wid, self._p(inst_map, torch.int32, "inst_map"), n, self._p(res["area"], torch.int32, "area"),
                self._p(res["bbox"], torch.int32, "bbox"), self._p(res["convex_area"], torch.int32, "convex_area"),
                self._p(res["solidity"], torch.float64, "solidity"), self._stream()))
        return res

    # ---- K13 -----------------------------------------------------------------------------------
    def instance_contours(self, inst_map, n_labels, area, bbox, tolerance=0.5):
        """One simplified contour polygon per label of an int32 instance map (pg_instance_contours_*).

        ``area`` / ``bbox`` come from ``raster_props`` on the same map. Returns poly_off int32 [n_labels+1] and
        poly_xy float64 [M,2] (x, y), closed rings."""
        hgt, wid = int(inst_map.shape[0]), int(inst_map.shape[1])
        n = int(n_labels)
        off = self._empty((n + 1,), torch.int32)
        self._check(self.lib.pg_instance_contours_count(
            self._h, hgt, wid, self._p(inst_map, torch.int32, "inst_map"), n, self._p(area, torch.int32, "area"),
            self._p(bbox, torch.int32, "bbox"), float(tolerance), self._p(off, torch.int32, "poly_off"), self._stream()))
        total = C.c_int64()
        self._check(self.lib.pg_instance_contours_total(self._h, C.byref(total)))
        xy = self._empty((int(total.value), 2), torch.float64)
        self._check(self.lib.pg_instance_contours_fill(self._h, n, self._p(off, torch.int32, "poly_off"),
                                                       self._p(xy, torch.float64, "poly_xy"), self._stream()))
        return {"poly_off": off, "poly_xy": xy}

    # ---- K11 -----------------------------------------------------------------------------------
    def clustering(self, row_ptr, col):
        """Triangles through each node and the local clustering coefficient over a symmetric CSR (pg_clustering)."""
        n = int(row_ptr.numel()) - 1
        tri = self._empty((n,), torch.int32)
        coeff = self._empty((n,), torch.float64)
        if col is None or col.numel() == 0:  # no edges: no triangles (the C entry needs a col array to read)
            return {"triangles": tri.zero_(), "clustering": coeff.zero_()}
        self._check(self.lib.pg_clustering(self._h, n, self._p(row_ptr, torch.int32, "row_ptr"),
                                           self._p(col, torch.int32, "col"), self._p(tri, torch.int32, "triangles"),
                                           self._p(coeff, torch.float64, "coeff"), self._stream()))
        return {"triangles": tri, "clustering": coeff}

    def type_interactions(self, types, nbr_count, n_types=5):
        """inter int64 [T,T]: directed edges from type a+1 to type b+1 (pg_type_interactions)."""
        n = int(types.numel())
        inter = self._empty((n_types, n_types), torch.int64)
        self._check(self.lib.pg_type_interactions(self._h, n, self._p(types, torch.int32, "types"),
                                                  self._p(nbr_count, torch.int32, "nbr_count"), int(n_types),
                                                  self._p(inter, torch.int64, "inter"), self._stream()))
        return inter

    # ---- K15 -----------------------------------------------------------------------------------
    def nhood_enrichment(self, edges, types, n_types=5, n_perms=1000, seed=0):
        """Label-permutation enrichment of the type-interaction matrix (pg_nhood_enrichment).

        edges int32 [E,2] (e.g. ``radius_graph(..., want_edges32=True)["edges32"][:E]``; rows with an id outside
        [0, N) are skipped); types int32 [N].  Returns a dict of device tensors [T,T]: count int64, zscore, perm_mean,
        perm_std float64.  Asynchronous (no host synchronisation once the workspace has grown)."""
        n = int(types.numel())
        if edges.dim() != 2 or edges.shape[1] != 2:
            raise ValueError("edges must have shape (E, 2)")
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2**64)")
        t = int(n_types)
        res = {"count": self._empty((t, t), torch.int64)}
        for name in ("zscore", "perm_mean", "perm_std"):
            res[name] = self._empty((t, t), torch.float64)
        eo = _lib.PgEnrichOut()
        eo.count = self._p(res["count"], torch.int64, "count")
        for name in ("zscore", "perm_mean", "perm_std"):
            setattr(eo, name, self._p(res[name], torch.float64, name))
        self._check(self.lib.pg_nhood_enrichment(self._h, n, self._p(types, torch.int32, "types"), t, int(edges.shape[0]),
                                                 self._p(edges, torch.int32, "edges"), int(n_perms), seed,
                                                 C.byref(eo), self._stream()))
        return res

    # ---- K17 -----------------------------------------------------------------------------------
    def spatial_autocorr(self, row_ptr, col, feat, mode="moran", transformation=True, n_perms=0, seed=0,
                         want_sims=False):
        """Moran's I / Geary's C of every feature column over a symmetric CSR, with permutation statistics
        (pg_spatial_autocorr).

        row_ptr int32 [N+1], col int32 [E] (entries outside [0, N) are skipped); feat float64 [F, N] (one row per
        column); ``transformation``: row-standardised weights 1 / d_i instead of binary ones.  Returns a dict of device
        tensors: stat, perm_mean, perm_var float64 [F], n_ge int64 [F], s012 float64 [3] (S0, S1, S2) and, with
        ``want_sims``, sims float64 [n_perms, F].  Asynchronous (no host synchronisation once the workspace has grown)."""
        if mode not in ("moran", "geary"):
            raise ValueError(f"mode must be 'moran' or 'geary', got {mode!r}")
        if feat.dim() != 2:
            raise ValueError("feat must have shape (F, N)")
        n = int(row_ptr.numel()) - 1
        n_feat = int(feat.shape[0])
        if n < 0 or int(feat.shape[1]) != n:
            raise ValueError("feat must have one value per CSR row")
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2**64)")
        p = int(n_perms)
        flags = (_lib.PG_AUTOCORR_GEARY if mode == "geary" else 0) | (_lib.PG_AUTOCORR_ROW_STD if transformation else 0)
        res = {name: self._empty((n_feat,), torch.float64) for name in ("stat", "perm_mean", "perm_var")}
        res["n_ge"] = self._empty((n_feat,), torch.int64)
        res["s012"] = self._empty((3,), torch.float64)
        if want_sims:
            res["sims"] = self._empty((p, n_feat), torch.float64)
        ao = _lib.PgAutocorrOut()
        for name, t in res.items():
            setattr(ao, name, self._p(t, torch.int64 if name == "n_ge" else torch.float64, name))
        if col is None or col.numel() == 0:  # no entries: the C entry still wants a col array it will not read
            col = self._empty((1,), torch.int32)
        self._check(self.lib.pg_spatial_autocorr(self._h, n, self._p(row_ptr, torch.int32, "row_ptr"),
                                                 self._p(col, torch.int32, "col"), n_feat,
                                                 self._p(feat, torch.float64, "feat"), flags, p, seed, C.byref(ao),
                                                 self._stream()))
        return res

    # ---- K16 -----------------------------------------------------------------------------------
    def pair_dist_hist(self, thresholds, n_types=5):
        """Type-pair distance histogram over the built grid (pg_pair_dist_hist).

        ``thresholds``: ascending distances t_0 < ... < t_{B-1} (host, at most ``PG_PAIRHIST_MAX_THR``).  Returns a dict
        of int64 device tensors: ``hist`` [B,T,T], hist[b, a-1, c-1] = ordered pairs (query row i of type a, grid point j
        of type c, i != j) with t_{b-1} < d <= t_b (b = 0: d <= t_0), and ``type_count`` [T] (query rows per type).
        Asynchronous (no host synchronisation once the workspace has grown)."""
        t = np.asarray(thresholds, dtype=np.float64).reshape(-1)
        nt, k = int(n_types), int(t.shape[0])
        res = {"hist": self._empty((k, nt, nt), torch.int64), "type_count": self._empty((nt,), torch.int64)}
        thr = (C.c_double * max(k, 1))(*t.tolist())
        self._check(self.lib.pg_pair_dist_hist(self._h, nt, k, thr, self._p(res["hist"], torch.int64, "hist"),
                                               self._p(res["type_count"], torch.int64, "type_count"), self._stream()))
        return res

    # ---- K10 -----------------------------------------------------------------------------------
    def node_features(self, feat, types=None, onehot_values=None):
        """z-scored feature columns + type one-hot -> x float32 [N, n_onehot + n_feat] (pg_node_features).

        feat float64 [n_feat, N] (one row per feature column), types int32 [N], onehot_values int32 [n_onehot]."""
        n_feat, n = (int(feat.shape[0]), int(feat.shape[1])) if feat is not None else (0, int(types.numel()))
        n_oh = int(onehot_values.numel()) if onehot_values is not None else 0
        x = self._empty((n, n_oh + n_feat), torch.float32)
        stats = self._empty((n_feat, 2), torch.float64)
        self._check(self.lib.pg_node_features(
            self._h, n, n_feat, self._p(feat, torch.float64, "feat"), self._p(types, torch.int32, "types"),
            self._p(onehot_values, torch.int32, "onehot_values"), n_oh, self._p(x, torch.float32, "x"),
            self._p(stats, torch.float64, "stats"), self._stream()))
        return {"x": x, "stats": stats}

    # ---- K9 ------------------------------------------------------------------------------------
    def halo_pack(self, xy, types, gid, lo_edge, hi_edge, capacity):
        """Records (24 B: x, y, gid, type) of the points with x < lo_edge or x >= hi_edge."""
        n = int(xy.shape[0])
        recs = self._empty((max(int(capacity), 1), 3), torch.float64)  # 24-byte records
        count = self._empty((1,), torch.int32)
        self._check(self.lib.pg_halo_pack(self._h, n, self._p(xy, torch.float64, "xy"), self._p(types, torch.int32, "types"),
                                          self._p(gid, torch.int32, "gid"), float(lo_edge), float(hi_edge),
                                          C.c_void_p(recs.data_ptr()), int(capacity), self._p(count, torch.int32, "count"),
                                          self._stream()))
        return recs, count

    def strip_partition(self, xy, types, gid, inner_edges):
        """Records (24 B: x, y, gid, type) of all points grouped by owning strip + per-strip totals (pg_strip_partition)."""
        n = int(xy.shape[0])
        world = len(inner_edges) + 1
        recs = self._empty((max(n, 1), 3), torch.float64)
        totals = self._empty((world,), torch.int32)
        e = (C.c_double * max(world - 1, 1))(*[float(v) for v in inner_edges])
        self._check(self.lib.pg_strip_partition(self._h, n, self._p(xy, torch.float64, "xy"), self._p(types, torch.int32, "types"),
                                                self._p(gid, torch.int32, "gid"), world, e, C.c_void_p(recs.data_ptr()),
                                                self._p(totals, torch.int32, "totals"), self._stream()))
        return recs[:n], totals

    def halo_unpack_multi(self, recs, n_recs, skip_begin, skip_end, ranges, xy, types, gid, n_base):
        """Append the records of several x-ranges behind slot n_base; returns the device counts int32 [len(ranges)]."""
        counts = self._empty((len(ranges),), torch.int32)
        flat = (C.c_double * (2 * len(ranges)))(*[float(v) for ab in ranges for v in ab])
        self._check(self.lib.pg_halo_unpack_multi(self._h, C.c_void_p(recs.data_ptr()), int(n_recs), int(skip_begin), int(skip_end),
                                                  len(ranges), flat, self._p(xy, torch.float64, "xy"),
                                                  self._p(types, torch.int32, "types"), self._p(gid, torch.int32, "gid"),
                                                  int(n_base), int(xy.shape[0]), self._p(counts, torch.int32, "counts"), self._stream()))
        return counts

    def widen_halfpx(self, q: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """int16 half-pixel vertices (q = 2 * coordinate, any shape) -> float32 pixels, exact (pg_widen_halfpx)."""
        if q.dtype != torch.int16 or not q.is_contiguous():
            raise TypeError("widen_halfpx: a contiguous int16 tensor is required")
        out = out if out is not None else self._empty(tuple(q.shape), torch.float32)
        self._check(self.lib.pg_widen_halfpx(self._h, int(q.numel()), C.c_void_p(q.data_ptr()), self._p(out, torch.float32, "out"),
                                             self._stream()))
        return out

    def halo_push(self, xy, types, gid, lo_edge, hi_edge, peer_ptrs_dev: int, world: int, rank: int, cap: int):
        """Pack the edge points and store them straight into every peer's receive slab (pg_halo_push)."""
        self._check(self.lib.pg_halo_push(self._h, int(xy.shape[0]), self._p(xy, torch.float64, "xy"),
                                          self._p(types, torch.int32, "types"), self._p(gid, torch.int32, "gid"),
                                          float(lo_edge), float(hi_edge), C.c_void_p(int(peer_ptrs_dev)), int(world), int(rank),
                                          int(cap), self._stream()))

    def halo_unpack_slab(self, slab, world, rank, cap, ranges, xy, types, gid, n_base):
        """Append the valid records of the local receive slab that fall into the x-ranges; device counts per range."""
        counts = self._empty((len(ranges),), torch.int32)
        flat = (C.c_double * (2 * len(ranges)))(*[float(v) for ab in ranges for v in ab])
        self._check(self.lib.pg_halo_unpack_slab(self._h, C.c_void_p(slab.data_ptr()), int(world), int(rank), int(cap), len(ranges),
                                                 flat, self._p(xy, torch.float64, "xy"), self._p(types, torch.int32, "types"),
                                                 self._p(gid, torch.int32, "gid"), int(n_base), int(xy.shape[0]),
                                                 self._p(counts, torch.int32, "counts"), self._stream()))
        return counts

    def gid_maps(self, gid, types, n_rows, n_ids, want_id_map=True, want_types=True):
        """Dense id -> row (first n_rows points) and id -> type (all points) maps over n_ids global ids (pg_gid_maps)."""
        id_map = self._empty((n_ids,), torch.int32) if want_id_map else None
        tbg = self._empty((n_ids,), torch.int32) if want_types else None
        self._check(self.lib.pg_gid_maps(self._h, int(gid.numel()), int(n_rows), self._p(gid, torch.int32, "gid"),
                                         self._p(types, torch.int32, "types"), int(n_ids), self._p(id_map, torch.int32, "id_map"),
                                         self._p(tbg, torch.int32, "type_by_gid"), self._stream()))
        return id_map, tbg

    def narrow_counts(self, x, dtype):
        """int32 counts -> uint8 / int16-sized unsigned (torch.uint8 / torch.int16 storage) on the device (pg_narrow_counts);
        values that do not fit are reported by check_overflow()."""
        bits = 8 if dtype == torch.uint8 else 16
        out = self._empty(tuple(x.shape), torch.uint8 if bits == 8 else torch.int16)
        self._check(self.lib.pg_narrow_counts(self._h, self._p(x, torch.int32, "counts"), int(x.numel()),
                                              C.c_void_p(out.data_ptr()), bits, self._stream()))
        return out

    def exclusive_scan(self, x):
        n = int(x.numel())
        out = self._empty((n + 1,), torch.int32)
        self._check(self.lib.pg_exclusive_scan_i32(self._h, self._p(x, torch.int32, "in"), self._p(out, torch.int32, "out"),
                                                   n, self._stream()))
        return out


_engines: dict[int, Engine] = {}


def get_engine(device: int | torch.device | None = None) -> Engine:
    """Process-wide engine per CUDA device (created on first use)."""
    if not torch.cuda.is_available():
        raise RuntimeError("path_gene_multimodal_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    if device is None:
        idx = torch.cuda.current_device()
    elif isinstance(device, int):
        idx = device
    else:
        d = torch.device(device)
        idx = d.index if d.index is not None else torch.cuda.current_device()
    eng = _engines.get(idx)
    if eng is None:
        eng = _engines[idx] = Engine(idx)
    return eng
