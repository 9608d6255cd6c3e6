"""ctypes binding of libpathgraph.so (C ABI: include/pathgraph.h).

The library is the only implementation: when it is missing or cannot create a handle the
callers fail loudly; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libpathgraph.so"

PG_RADIUS_SYMMETRIC = 0
PG_RADIUS_UPPER = 1
PG_MAX_TYPES = 16
PG_MAX_K = 64
PG_ENRICH_MAX_PERMS = 100000
PG_PAIRHIST_MAX_THR = 64
PG_AUTOCORR_GEARY = 1
PG_AUTOCORR_ROW_STD = 2
PG_AUTOCORR_MAX_FEAT = 256
PG_LOCAL_GETIS_ORD = 4
PG_LOCAL_STAR = 8

PG_OK, PG_ERR_INVALID, PG_ERR_CUDA, PG_ERR_STATE, PG_ERR_CAPACITY, PG_ERR_NOMEM = 0, -1, -2, -3, -4, -5

vp = C.c_void_p
i32 = C.c_int32
i64 = C.c_int64
f64 = C.c_double


class PgDegreeStats(C.Structure):
    _fields_ = [("min_degree", C.c_int32), ("max_degree", C.c_int32), ("sum_degree", C.c_int64),
                ("sumsq_degree", C.c_int64), ("n_nodes", C.c_int64)]


class PgMorphOut(C.Structure):
    _fields_ = [(name, vp) for name in ("area", "perimeter", "eccentricity", "circularity", "major_axis",
                                        "minor_axis", "centroid_x", "centroid_y", "poly_bbox")]


class PgUnionOut(C.Structure):
    _fields_ = [("edges", vp), ("edge_w64", vp), ("edge_w32", vp), ("type", vp), ("n_types", C.c_int32),
                ("nbr_count", vp), ("degree", vp), ("stats", vp), ("hist", vp), ("hist_len", C.c_int32),
                ("symmetric_dist", C.c_int32), ("presized", C.c_int32)]


class PgRasterOut(C.Structure):
    _fields_ = [(name, vp) for name in ("area", "bbox", "centroid", "perimeter", "eccentricity", "major_axis",
                                        "minor_axis", "orientation")]


class PgHullOut(C.Structure):
    _fields_ = [(name, vp) for name in ("convex_area", "solidity", "orientation")]


class PgEnrichOut(C.Structure):
    _fields_ = [(name, vp) for name in ("count", "zscore", "perm_mean", "perm_std")]


class PgAutocorrOut(C.Structure):
    _fields_ = [(name, vp) for name in ("stat", "perm_mean", "perm_var", "n_ge", "sims", "s012")]


class PgLocalOut(C.Structure):
    _fields_ = [(name, vp) for name in ("stat", "lag", "n_ge", "perm_mean", "perm_var", "sims", "mean", "m2")]


class PgClusterOut(C.Structure):
    _fields_ = [(name, vp) for name in ("n_members", "n_core", "type_count", "centroid", "bbox", "member_off",
                                        "member_xy")]


class PathGraphError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libpathgraph error {code}: {msg}")
        self.code = code


# name -> (restype, argtypes); mirrors include/pathgraph.h one to one
SIGNATURES = {
    "pg_version": (C.c_int, []),
    "pg_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "pg_destroy": (C.c_int, [vp]),
    "pg_last_error": (C.c_char_p, [vp]),
    "pg_workspace_bytes": (C.c_int64, [vp]),
    "pg_map_morph_hint": (C.c_int, [vp, i32, i64]),
    "pg_map_morph_f32": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(PgMorphOut), vp]),
    "pg_map_morph_f64": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(PgMorphOut), vp]),
    "pg_grid_build": (C.c_int, [vp, i32, i32, vp, vp, vp, f64, C.POINTER(f64), vp]),
    "pg_grid_export": (C.c_int, [vp, vp, vp, vp, vp]),
    "pg_grid_info": (C.c_int, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(f64), C.POINTER(f64), C.POINTER(f64)]),
    "pg_knn": (C.c_int, [vp, i32, vp, vp, vp, f64, f64, vp, vp]),
    "pg_knn_neighbor_coords": (C.c_int, [vp, i32, i32, vp, vp, i32, vp, vp]),
    "pg_radius_count": (C.c_int, [vp, f64, i32, vp, vp, vp, i32, vp, vp, i32, vp]),
    "pg_radius_graph": (C.c_int, [vp, f64, i32, vp, vp, vp, i32, vp, vp, i32, vp, vp, vp, vp, vp, i64, vp]),
    "pg_radius_reserve": (C.c_int, [vp, i64]),
    "pg_radius_total": (C.c_int, [vp, C.POINTER(i64)]),
    "pg_radius_fill": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, vp]),
    "pg_launch_count": (C.c_int64, [vp]),
    "pg_profile_enable": (C.c_int, [vp, C.c_int]),
    "pg_profile_count": (C.c_int, [vp]),
    "pg_profile_get": (C.c_int, [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_float)]),
    "pg_check_overflow": (C.c_int, [vp]),
    "pg_grid_check": (C.c_int, [vp]),
    "pg_knn_symmetrize_count": (C.c_int, [vp, i32, i32, vp, vp, vp, i32, vp, vp]),
    "pg_knn_symmetrize_total": (C.c_int, [vp, C.POINTER(i64)]),
    "pg_knn_symmetrize_fill": (C.c_int, [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "pg_knn_union_count": (C.c_int, [vp, i32, i32, vp, vp, vp, i32, vp, vp, vp]),
    "pg_knn_union_total": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64)]),
    "pg_knn_union_fill": (C.c_int, [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(PgUnionOut), vp]),
    "pg_csr_upper_count": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
    "pg_csr_upper_total": (C.c_int, [vp, C.POINTER(i64)]),
    "pg_csr_upper_fill": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "pg_compose_degree": (C.c_int, [vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, i32, vp]),
    "pg_halo_pack": (C.c_int, [vp, i32, vp, vp, vp, f64, f64, vp, i32, vp, vp]),
    "pg_strip_partition": (C.c_int, [vp, i32, vp, vp, vp, i32, C.POINTER(f64), vp, vp, vp]),
    "pg_halo_unpack_multi": (C.c_int, [vp, vp, i32, i32, i32, i32, C.POINTER(f64), vp, vp, vp, i32, i32, vp, vp]),
    "pg_widen_halfpx": (C.c_int, [vp, i64, vp, vp, vp]),
    "pg_halo_push": (C.c_int, [vp, i32, vp, vp, vp, f64, f64, vp, i32, i32, i32, vp]),
    "pg_halo_unpack_slab": (C.c_int, [vp, vp, i32, i32, i32, i32, C.POINTER(f64), vp, vp, vp, i32, i32, vp, vp]),
    "pg_gid_maps": (C.c_int, [vp, i32, i32, vp, vp, i32, vp, vp, vp]),
    "pg_narrow_counts": (C.c_int, [vp, vp, i64, vp, i32, vp]),
    "pg_clustering": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
    "pg_type_interactions": (C.c_int, [vp, i32, vp, vp, i32, vp, vp]),
    "pg_nhood_enrichment": (C.c_int, [vp, i32, vp, i32, i64, vp, i32, C.c_uint64, C.POINTER(PgEnrichOut), vp]),
    "pg_spatial_autocorr": (C.c_int, [vp, i32, vp, vp, i32, vp, i32, i32, C.c_uint64, C.POINTER(PgAutocorrOut), vp]),
    "pg_local_autocorr": (C.c_int, [vp, i32, vp, vp, i32, vp, i32, i32, C.c_uint64, C.POINTER(PgLocalOut), vp]),
    "pg_connected_components": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
    "pg_dbscan": (C.c_int, [vp, i32, vp, vp, i32, vp, vp, vp, vp]),
    "pg_cluster_props": (C.c_int, [vp, i32, vp, i32, vp, vp, i32, vp, C.POINTER(PgClusterOut), vp]),
    "pg_pair_dist_hist": (C.c_int, [vp, i32, i32, C.POINTER(f64), vp, vp, vp]),
    "pg_raster_props": (C.c_int, [vp, i32, i32, vp, i32, C.POINTER(PgRasterOut), vp]),
    "pg_raster_solidity": (C.c_int, [vp, i32, i32, vp, i32, vp, vp, vp, vp, vp]),
    "pg_ring_hull_f32": (C.c_int, [vp, i32, i64, vp, vp, C.POINTER(PgHullOut), vp]),
    "pg_ring_hull_f64": (C.c_int, [vp, i32, i64, vp, vp, C.POINTER(PgHullOut), vp]),
    "pg_instance_contours_count": (C.c_int, [vp, i32, i32, vp, i32, vp, vp, f64, vp, vp]),
    "pg_instance_contours_total": (C.c_int, [vp, C.POINTER(i64)]),
    "pg_instance_contours_fill": (C.c_int, [vp, i32, vp, vp, vp]),
    "pg_node_features": (C.c_int, [vp, i32, i32, vp, vp, vp, i32, vp, vp, vp]),
    "pg_exclusive_scan_i32": (C.c_int, [vp, vp, vp, i32, vp]),
}

_lib = None


def load_library(path: str | Path | None = None) -> C.CDLL:
    """dlopen libpathgraph.so and attach the prototypes. Raises if the library is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    if path is None and os.environ.get("PG_LIBPATH"):  # debugging aid: an alternative build of the same library
        p = Path(os.environ["PG_LIBPATH"])
    else:
        p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise RuntimeError(
            f"{p} is missing: build the CUDA library first (python -m path_gene_multimodal_b200._build, "
            "or __graft_entry__.build()). There is no CPU fallback for this path.")
    lib = C.CDLL(str(p))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib
