"""Per-polygon morphology tables in the reference's column vocabulary.

* ``polygon_morphology_table``  - the island-table columns of
  /root/reference/polygon_morphology.py:238-257 (``area_px2, perimeter_px, centroid_x, centroid_y,
  bbox_xmin, bbox_ymin, bbox_xmax, bbox_ymax``; shapely ``p.area / p.length / p.centroid / p.bounds``)
  and ``tag_polygons`` of create_and_overlay_polygon_from_prediction.py:291-302.
* ``nuclei_morphology_table``   - the cell-18 columns of hovernet_tile_inference.ipynb:2415-2456
  (``area, perimeter, eccentricity, major_axis_length, minor_axis_length`` + derived
  ``perimeter_area, compactness, roundness, elongation``), evaluated on the ring's exact area moments
  instead of a raster, and the cell-21 z-scores (ipynb:2903) on request; with ``hull=True`` also cell 18's
  ``solidity`` and ``orientation`` from the per-ring convex hull (pg_ring_hull_*).

All other features come from one launch of the fused kernel (pg_map_morph_*); the derived columns are
the notebook's own pandas expressions on top.
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from . import _host
from .engine import get_engine
from .nuclei_wsi import map_morph_arrays, polygons_to_csr

ISLAND_COLUMNS = ["area_px2", "perimeter_px", "centroid_x", "centroid_y",
                  "bbox_xmin", "bbox_ymin", "bbox_xmax", "bbox_ymax"]
CONT_COLS = ["area", "perimeter", "eccentricity", "solidity", "major_axis_length", "minor_axis_length",
             "perimeter_area", "compactness", "roundness", "elongation"]  # ipynb:2886-2897


def _as_csr(polygons, poly_off=None, dtype=np.float64):
    if poly_off is not None:
        xy = np.asarray(polygons)
        return np.asarray(poly_off, dtype=np.int32), xy.reshape(-1, 2), None
    return polygons_to_csr(polygons, dtype=dtype)


def polygon_morphology_table(polygons, poly_off=None, device=None) -> pd.DataFrame:
    """One row per ring: the numeric island-table columns (float64, like ``float(p.area)`` etc.).

    ``polygons``: a sequence of rings (lists of [x, y]; closing vertex optional), or a flat [M,2]
    array together with ``poly_off`` (CSR).  Rings with fewer than 3 vertices give NaN.
    """
    off, xy, _ = _as_csr(polygons, poly_off)
    res = map_morph_arrays(off, xy, write_polygons=False, extra=True, device=device)
    bb = res["poly_bbox"]
    return pd.DataFrame({
        "area_px2": res["area"].astype(np.float64),
        "perimeter_px": res["perimeter"].astype(np.float64),
        "centroid_x": res["centroid_x"],
        "centroid_y": res["centroid_y"],
        "bbox_xmin": bb[:, 0], "bbox_ymin": bb[:, 1], "bbox_xmax": bb[:, 2], "bbox_ymax": bb[:, 3],
    })


def tag_polygons(polygons, class_name: str, min_area_px: float = 0, poly_off=None, device=None) -> list[dict]:
    """``tag_polygons`` (create_and_overlay_polygon_from_prediction.py:291-302) over coordinate rings:
    ``[{'class', 'area_px2', 'perimeter_px', 'index'}]`` with rings below ``min_area_px`` dropped."""
    tab = polygon_morphology_table(polygons, poly_off, device=device)
    out = []
    for i, (a, p) in enumerate(zip(tab["area_px2"], tab["perimeter_px"])):
        if min_area_px and a < min_area_px:
            continue
        out.append({"class": class_name, "area_px2": float(a), "perimeter_px": float(p), "index": i})
    return out


def derived_columns(df: pd.DataFrame) -> pd.DataFrame:
    """The cell-18 derived features, same expressions as ipynb:2431-2456 (clip guards included)."""
    df["perimeter_area"] = df["perimeter"] / df["area"].clip(lower=1)
    df["compactness"] = 4.0 * np.pi * df["area"] / df["perimeter"].clip(lower=1) ** 2
    df["roundness"] = 4.0 * df["area"] / (np.pi * df["major_axis_length"].clip(lower=1) ** 2)
    df["elongation"] = df["major_axis_length"] / df["minor_axis_length"].clip(lower=1)
    return df


def zscore_columns(df: pd.DataFrame, cols=CONT_COLS) -> pd.DataFrame:
    """Cell 21 (ipynb:2899-2909): ``<col>_z = (x - mean) / std(ddof=0)``, 0.0 when sigma is 0 / NaN."""
    for col in cols:
        if col in df.columns:
            mu = df[col].mean()
            sigma = df[col].std(ddof=0)
            if sigma == 0 or np.isnan(sigma):
                df[col + "_z"] = 0.0
            else:
                df[col + "_z"] = (df[col] - mu) / sigma
    return df


def hull_arrays(poly_off, poly_xy, device=None) -> dict:
    """Array-level entry of the per-ring convex hull: numpy (host) in, numpy out, one kernel in between.

    poly_off int32 [N+1]; poly_xy float32 or float64 [M,2] (the dtype chooses pg_ring_hull_f32 / _f64).  Returns
    float64 [N] ``convex_area``, ``solidity`` (|area| / convex area) and ``orientation`` (skimage's convention, x =
    column, y = row).  Rings with fewer than 3 vertices give NaN; see include/pathgraph.h for the other NaN rules."""
    eng = get_engine(device)
    dev = eng.device
    vt = np.float32 if np.asarray(poly_xy).dtype == np.float32 else np.float64
    d_off = _host.to_device(poly_off, np.int32, dev)
    d_xy = _host.to_device(np.asarray(poly_xy).reshape(-1, 2), vt, dev)
    with torch.cuda.device(dev):
        res = eng.ring_hull(d_off, d_xy)
        return {k: _host.to_host(v) for k, v in res.items()}


def nuclei_morphology_table(polygons, poly_off=None, inst_id=None, zscore: bool = False, device=None,
                            hull: bool = False) -> pd.DataFrame:
    """``morph_df`` of cell 18: ``inst_id, area, perimeter, eccentricity, major_axis_length,
    minor_axis_length, perimeter_area, compactness, roundness, elongation`` (+ ``*_z``).

    ``hull=True`` adds ``solidity`` after ``eccentricity`` and ``orientation`` after ``minor_axis_length`` (cell 18's
    order), from the ring's convex hull and area moments; ``zscore`` then also yields ``solidity_z``."""
    off, xy, _ = _as_csr(polygons, poly_off)
    res = map_morph_arrays(off, xy, write_polygons=False, extra=True, device=device)
    n = len(off) - 1
    cols = {
        "inst_id": np.arange(1, n + 1) if inst_id is None else np.asarray(inst_id),
        "area": res["area"].astype(np.float64),
        "perimeter": res["perimeter"].astype(np.float64),
        "eccentricity": res["eccentricity"].astype(np.float64),
    }
    hres = hull_arrays(off, xy, device=device) if hull else None
    if hull:
        cols["solidity"] = hres["solidity"]
    cols["major_axis_length"] = res["major_axis"].astype(np.float64)
    cols["minor_axis_length"] = res["minor_axis"].astype(np.float64)
    if hull:
        cols["orientation"] = hres["orientation"]
    df = pd.DataFrame(cols)
    df = derived_columns(df)
    df["circularity"] = res["circularity"].astype(np.float64)
    if zscore:
        df = zscore_columns(df)
    return df
