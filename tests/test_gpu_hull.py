"""GPU tests of K14 (pg_ring_hull_*): convex area, solidity and orientation per ring against the exact oracle
(oracle/hull.py) - bit for bit on the half-pixel lattice, both paths (rings staged in shared memory, and the chain
path of rings too long for a slab), edge cases, CUDA-graph capture, and the nuclei_morphology_table(hull=True) /
node_feature_matrix surface."""
import math

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import hull as ohull
from oracle import morphology as omorph
from path_gene_multimodal_b200 import synth

pytestmark = pytest.mark.gpu

# Polygon orientation (instance_polygons_csr, approximate_polygon tolerance 0.5) against the raster orientation of the
# same blob differs by the pixelation of the mask. The CPU oracles (oracle/contours.py + oracle/hull.py against
# oracle/raster.py) put the largest difference over blob_map(seed 0..9) at 0.0562 rad; the bound keeps some margin.
BLOB_ORIENTATION_TOL = 0.08


def blob_map(seed, side=400, pitch=40):
    """Elongated elliptical nuclei (semi-axes 6..14 by 0.35..0.6 of that, any angle) on a grid, one label each."""
    rng = np.random.default_rng(seed)
    m = np.zeros((side, side), dtype=np.int32)
    rows, cols = np.mgrid[0:pitch, 0:pitch]
    label = 0
    for gy in range(side // pitch):
        for gx in range(side // pitch):
            a = rng.uniform(6, 14)
            b = a * rng.uniform(0.35, 0.6)
            th = rng.uniform(0, np.pi)
            cy, cx = pitch / 2 + rng.uniform(-2, 2), pitch / 2 + rng.uniform(-2, 2)
            u = (cols - cx) * np.cos(th) + (rows - cy) * np.sin(th)
            v = -(cols - cx) * np.sin(th) + (rows - cy) * np.cos(th)
            blob = (u / a) ** 2 + (v / b) ** 2 <= 1
            label += 1
            m[gy * pitch:(gy + 1) * pitch, gx * pitch:(gx + 1) * pitch][blob] = label
    return m


def _hull(off, xy):
    from path_gene_multimodal_b200 import hull_arrays

    return hull_arrays(off, xy, device=0)


def _check_exact(off, xy, got, ref=None, orient_atol=1e-9):
    ref = ref if ref is not None else ohull.ring_hull_csr(off, xy)
    np.testing.assert_array_equal(got["convex_area"], ref["convex_area"])
    np.testing.assert_array_equal(got["solidity"], ref["solidity"])
    _check_orientation(off, xy, got, ref, orient_atol)


def _check_orientation(off, xy, got, ref, atol):
    f = omorph.polygon_features_csr(off, xy)
    aniso = 1.0 - f["minor_axis_length"] / f["major_axis_length"]   # 0 for isotropic moments
    sel = np.isfinite(ref["orientation"]) & (aniso > 1e-3)
    assert np.array_equal(np.isnan(got["orientation"]), np.isnan(ref["orientation"]))
    # an orientation is an axis: +pi/2 and -pi/2 are the same one, and which of them atan2 returns for a ring long
    # along x follows the sign of a mu_xy that is zero up to rounding
    diff = (got["orientation"][sel] - ref["orientation"][sel] + np.pi / 2) % np.pi - np.pi / 2
    assert np.abs(diff).max(initial=0.0) <= atol


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("v_fixed", [32, None])
def test_lattice_tables_bit_exact(dt, v_fixed):
    off, xy = synth.make_polygons(20_000, 21, v_fixed=v_fixed, dtype=dt)
    _check_exact(off, xy, _hull(off, xy))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_short_self_intersecting_and_degenerate_rings(dt):
    """Rings that are not two x-monotone chains take the in-place sort of the staged path."""
    from test_hull_cpu import ADVERSARIAL

    rng = np.random.default_rng(5)
    rings = [_ring(int(nv), i, convex=False) / 8 for i, nv in enumerate(rng.integers(3, 40, size=3000))]
    adv = [np.array(r, dtype=np.float64) for r, _, _ in ADVERSARIAL.values() if r is not ADVERSARIAL["star"][0]]
    for r in adv:
        rings += [r, np.vstack([r, r[:1]]), r[::-1]]
    off = np.zeros(len(rings) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(r) for r in rings])
    xy = (np.round(np.vstack(rings) * 2) / 2).astype(dt)
    _check_exact(off, xy, _hull(off, xy))


def test_non_lattice_float64_rings():
    off, xy = synth.make_polygons(5000, 22, dtype=np.float64)
    xy = xy + np.random.default_rng(1).normal(scale=0.3, size=xy.shape)
    got, ref = _hull(off, xy), ohull.ring_hull_csr(off, xy)
    np.testing.assert_allclose(got["convex_area"], ref["convex_area"], rtol=1e-12)
    np.testing.assert_allclose(got["solidity"], ref["solidity"], rtol=1e-12)
    _check_orientation(off, xy, got, ref, 1e-9)


def _ring(nv, seed, convex):
    """A ring of nv vertices on the half-pixel lattice: a convex polygon (every vertex on the hull: integer points
    on a parabola arc and its mirror) or a noisy star (self-intersections, duplicates, collinear runs)."""
    if convex:
        h = nv // 2
        k = np.arange(h, dtype=np.float64)
        lo = np.stack([k, k * k / 2], axis=1)
        hi = np.stack([k[::-1], 2.0 * h * h - k[::-1] ** 2 / 2], axis=1)
        r = np.vstack([lo, hi])[:nv]
        return (r - r.mean(axis=0).round()).astype(np.float64)
    rng = np.random.default_rng(seed)
    t = np.sort(rng.uniform(0, 2 * np.pi, nv))
    rad = rng.uniform(20, 200, nv)
    return np.round(np.stack([rad * np.cos(t), rad * np.sin(t)], axis=1) * 2) / 2


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_long_rings_and_mixed_warps(dt):
    rings = []
    for nv in (300, 2500, 20_000, 100_000):
        # a convex lattice ring of nv vertices spans ~nv^1.5 half-pixels: past 2500 vertices float32 cannot hold it
        convex = dt == np.float64 or nv <= 2500
        rings += [_ring(nv, nv, convex=False), _ring(nv, nv + 1, convex=convex)]
    short_off, short_xy = synth.make_polygons(70, 23, dtype=np.float64)
    # one long ring among short ones in a single warp, then empty / 1- / 2-vertex rows
    rings += [short_xy[short_off[i]:short_off[i + 1]] for i in range(40)]
    rings.insert(45, _ring(5000, 3, convex=False))
    rings += [np.zeros((0, 2)), np.array([[1.0, 1.0]]), np.array([[0.0, 0.0], [1.0, 0.5]]), np.array([[0.0, 0.0], [2.0, 0.0], [0.0, 2.0]])]
    off = np.zeros(len(rings) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(r) for r in rings])
    xy = np.vstack(rings).astype(dt)
    got, ref = _hull(off, xy), ohull.ring_hull_csr(off, xy)
    _check_exact(off, xy, got, ref)
    convex = [1, 3, 5, 7] if dt == np.float64 else [1, 3]
    assert np.all(got["solidity"][convex] == 1.0)
    assert np.isnan(got["convex_area"][-4:-1]).all() and got["convex_area"][-1] == 2.0


def test_empty_table_and_odd_vertex_offset():
    from path_gene_multimodal_b200.engine import get_engine

    eng = get_engine(0)
    dev = eng.device
    res = eng.ring_hull(torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros((0, 2), dtype=torch.float32, device=dev))
    assert all(v.numel() == 0 for v in res.values())
    off, xy = synth.make_polygons(3000, 24, v_lo=3, v_hi=33)
    for dt in (torch.float32, torch.float64):
        base = torch.zeros((len(xy) + 1, 2), dtype=dt, device=dev)
        base[1:] = torch.from_numpy(xy).to(dev, dt)
        view = base[1:]                 # starts one vertex into its allocation: 8-byte aligned for float32
        got = {k: v.cpu().numpy() for k, v in eng.ring_hull(torch.from_numpy(off).to(dev), view).items()}
        _check_exact(off, xy, got)


def test_capture_replay_equals_eager():
    from path_gene_multimodal_b200.engine import get_engine

    eng = get_engine(0)
    dev = eng.device
    off, xy = synth.make_polygons(50_000, 25)
    rings = [xy, _ring(20_000, 9, convex=False).astype(np.float32)]
    off = np.concatenate([off, [off[-1] + 20_000]]).astype(np.int32)
    d_off, d_xy = torch.from_numpy(off).to(dev), torch.from_numpy(np.vstack(rings)).to(dev)
    eager = {k: v.clone() for k, v in eng.ring_hull(d_off, d_xy).items()}
    out = {k: torch.full_like(v, -1.0) for k, v in eager.items()}
    g = eng.capture(lambda: eng.ring_hull(d_off, d_xy, out=out))
    for v in out.values():
        v.fill_(-1.0)
    g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(torch.nan_to_num(out[k], nan=7.0), torch.nan_to_num(eager[k], nan=7.0)), k


def test_nuclei_morphology_table_hull_surface():
    from path_gene_multimodal_b200 import nuclei_morphology_table
    from path_gene_multimodal_b200.graph_features import node_feature_matrix

    off, xy = synth.make_polygons(101, 26)
    plain = nuclei_morphology_table(xy, poly_off=off, zscore=True, device=0)
    # the parent's table: no hull columns, the same frame as before
    assert list(plain.columns) == ["inst_id", "area", "perimeter", "eccentricity", "major_axis_length",
                                   "minor_axis_length", "perimeter_area", "compactness", "roundness", "elongation",
                                   "circularity"] + [c + "_z" for c in ("area", "perimeter", "eccentricity",
                                   "major_axis_length", "minor_axis_length", "perimeter_area", "compactness",
                                   "roundness", "elongation")]
    df = nuclei_morphology_table(xy, poly_off=off, zscore=True, device=0, hull=True)
    pd.testing.assert_frame_equal(df.drop(columns=["solidity", "orientation", "solidity_z"]), plain)
    ref = ohull.ring_hull_csr(off, xy)
    assert np.array_equal(df["solidity"].to_numpy(), ref["solidity"])
    df["type"] = np.arange(len(df)) % 5 + 1
    nf = node_feature_matrix(df, device=0)
    assert nf["x"].shape == (101, 15) and "solidity_z" in nf["columns"]


def test_polygon_orientation_agrees_with_raster():
    from path_gene_multimodal_b200 import hull_arrays, instance_polygons_csr, raster_morphology_table

    m = blob_map(7)
    labels, off, xy = instance_polygons_csr(m, device=0)
    poly = hull_arrays(off, xy, device=0)["orientation"]
    ras = raster_morphology_table(m, device=0).set_index("inst_id").loc[labels, "orientation"].to_numpy()
    diff = (poly - ras + math.pi / 2) % math.pi - math.pi / 2
    assert len(labels) == 100 and np.abs(diff).max() < BLOB_ORIENTATION_TOL
