"""GPU: K1 (pg_map_morph_*, csrc/pg_morph.cu) in every variant its launcher picks, against the float64 oracle.

The launcher compiles one kernel body into five reachable instantiations, picked from the vertex type, from whether
any "extra" output (major / minor axis, centroid_x / y, poly_bbox) is wanted, and from the per-warp shared-memory slab
that the ring-length hint (pg_map_morph_hint) sizes. Within a launch each warp walks its 32 rings either out of the
slab ("staged": one bulk copy in, a lane per ring, float32 perimeter partials folded into float64 every 32 edges) or
8 lanes per ring straight from global memory ("group": a range longer than the slab, an empty range, or input and
output in different 16-byte phases).

This file restates both rules, asserts through the library's launch records which instantiation ran, asserts from the
restated per-warp predicate that each table puts warps on every path it claims, and compares every output with
oracle/morphology.polygon_features_csr in float64 on the same vertices (float32 widened). The last test fails unless
all five instantiations were compared on both paths somewhere in this module.

Bars (as tests/test_gpu_parity.py): area / perimeter / circularity / eccentricity / axes rtol 1e-5, eccentricity
atol 2e-6, minor axis atol 1e-5, centroids rtol 1e-9; bbox, wsi_centroid, wsi_bbox and lattice wsi_poly_xy exact;
the NaN pattern exact per row. Output buffers start as a sentinel, so a row the kernel skips fails too.
"""
import contextlib
import ctypes as C
import functools
import math

import numpy as np
import pytest
import torch

from oracle import morphology as omorph
from path_gene_multimodal_b200 import _lib, cohort, synth
from path_gene_multimodal_b200._lib import PgMorphOut

RTOL = 1e-5
ECC_ATOL = 2e-6
MINOR_ATOL = 1e-5
CENTROID_RTOL = 1e-9
SENTINEL = 1.0e30

# the launcher's constants (pg_morph.cu)
WARPS = 4                        # TPB / 32
SLAB_VERTS_MIN = 32 * 33 + 2     # default slab: 32 rings of 32 vertices, explicitly closed, + alignment slack
SLAB_BYTES_MAX = 200 * 1024      # per CTA
SMEM_PER_SM = 227 * 1024
CTA_SMEM_RESERVED = 1024 + 128   # per CTA beside the slabs
DENSE_MINB = 7

BASE = ("area", "perimeter", "eccentricity", "circularity")
EXTRA = ("major_axis", "minor_axis", "centroid_x", "centroid_y", "poly_bbox")
OUTPUTS = {"plain": BASE, "extra": BASE + EXTRA, "only_bbox": BASE + ("poly_bbox",),
           "only_cx": BASE + ("centroid_x",)}
VARIANTS = ["map_morph_kernel<f32, extra, 5>", "map_morph_kernel<f64, extra, 4>", "map_morph_kernel<f64, plain, 5>",
            "map_morph_kernel<f32, plain, 6>", "map_morph_kernel<f32, plain, 7>"]
COVERED = set()                  # (variant, path) pairs compared with the oracle in this module


# ---------------------------------------------------------------------------------------------------- the launcher
def vbytes(vt):
    return 2 * np.dtype(vt).itemsize


def slab_verts(mean, vt):
    """Vertices per warp slab for a hinted mean ring length (launch_map_morph)."""
    s = SLAB_VERTS_MIN
    if mean > 33.0:
        s = math.ceil(46.0 * mean) + 2
    elif 0.0 < mean <= 23.0:
        s = max(512, math.ceil(40.0 * mean) + 2)
    s = min(s, SLAB_BYTES_MAX // (WARPS * vbytes(vt)))
    return s & ~1


def cap_mean(vt):
    """Mean ring length above which the slab stops growing."""
    return (SLAB_BYTES_MAX // (WARPS * vbytes(vt)) - 2) / 46.0


def variant(vt, extra, hint_n, hint_m):
    """(instantiation name, slab) the launcher picks after pg_map_morph_hint(hint_n, hint_m)."""
    mean = hint_m / hint_n if hint_n > 0 else 0.0
    slab = slab_verts(mean, vt)
    f32 = np.dtype(vt) == np.float32
    if extra:
        minb = 5 if f32 else 4
    elif f32 and DENSE_MINB * (WARPS * slab * vbytes(vt) + CTA_SMEM_RESERVED) <= SMEM_PER_SM:
        minb = DENSE_MINB
    else:
        minb = 6 if f32 else 5
    return f"map_morph_kernel<{'f32' if f32 else 'f64'}, {'extra' if extra else 'plain'}, {minb}>", slab


def warp_paths(off, slab, src_ptr, dst_ptr):
    """Per warp: "staged", "group" (rings walked from global memory) or "empty" (group path, nothing to walk)."""
    off = np.asarray(off, dtype=np.int64)
    n = len(off) - 1
    first = np.arange(0, n, 32)
    total = off[np.minimum(first + 32, n)] - off[first]
    same_phase = dst_ptr is None or (src_ptr - dst_ptr) % 16 == 0
    staged = (total > 0) & (total <= slab - 2) & same_phase
    return np.where(staged, "staged", np.where(total > 0, "group", "empty"))


# ---------------------------------------------------------------------------------------------------- tables
def csr(nv):
    off = np.zeros(len(nv) + 1, dtype=np.int64)
    np.cumsum(nv, out=off[1:])
    assert off[-1] < 2 ** 31
    return off.astype(np.int32)


def ellipses(nv, rng, vt, lattice=True, centre_span=508.0):
    """Jittered, rotated ellipse rings of the given lengths, open; semi-axes grow with the ring length so that the
    vertices of long rings do not collapse onto the 0.5-px lattice."""
    nv = np.asarray(nv, dtype=np.int64)
    n = len(nv)
    off = csr(nv)
    m = int(off[-1])
    owner = np.repeat(np.arange(n), nv)
    kth = np.arange(m) - off[:-1][owner]
    a = rng.uniform(4.0, 12.0, n) * np.maximum(1.0, nv / 32.0)
    b = a * rng.uniform(0.5, 1.0, n)
    rot = rng.uniform(0.0, np.pi, n)
    t = 2.0 * np.pi * kth / np.maximum(nv[owner], 1)
    jit = 1.0 + rng.uniform(-0.05, 0.05, m)
    ex, ey = a[owner] * np.cos(t) * jit, b[owner] * np.sin(t) * jit
    c, s = np.cos(rot[owner]), np.sin(rot[owner])
    cen = rng.random((n, 2)) * centre_span
    xy = np.stack([c * ex - s * ey + cen[owner, 0], s * ex + c * ey + cen[owner, 1]], axis=1)
    if lattice:
        xy = np.round(xy * 2.0) / 2.0
    return off, xy.astype(vt)


def tiles_for(n, rng, n_tiles=64, pitch=508):
    tile_x = ((np.arange(n_tiles) % 8) * pitch).astype(np.int32)
    tile_y = ((np.arange(n_tiles) // 8) * pitch + 3 * pitch).astype(np.int32)
    return rng.integers(0, n_tiles, size=n).astype(np.int32), tile_x, tile_y


def tile_inputs(n, rng):
    cen = rng.random((n, 2)) * 508.0
    bb = rng.integers(0, 508, size=(n, 4)).astype(np.int32)
    return cen, bb


# ---------------------------------------------------------------------------------------------------- one call
def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


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


def padded(a, shift, fill):
    """A device view of `a` that starts `shift` rows into a buffer with a guard row on each side."""
    buf = torch.full((a.shape[0] + 2,) + tuple(a.shape[1:]), fill, dtype=a.dtype, device="cuda")
    view = buf[shift: shift + a.shape[0]]
    view.copy_(a)
    return buf, view


def run_abi(engine, off, xy, outputs="extra", tiles=None, centroid=None, bbox=None, write=True, hint="table",
            in_shift=0, out_shift=0):
    """One pg_map_morph_* call through the C ABI. hint: "table" = (n, M) of this table, as Engine.map_morph passes it;
    (n, m) = that hint; None = whatever the handle holds. Returns host outputs, the launch records, and the pointers
    the per-warp predicate needs."""
    vt = xy.dtype.type
    n, m = len(off) - 1, int(xy.shape[0])
    d_off = dev(off)
    src_buf, src = padded(dev(xy), in_shift, -7.0)
    dst_buf = dst = None
    if write:
        dst_buf, dst = padded(torch.full((m, 2), -5.0, dtype=src.dtype, device="cuda"), out_shift, -7.0)
    mo = PgMorphOut()
    got = {}
    for name in OUTPUTS[outputs]:
        shape = (n, 4) if name == "poly_bbox" else (n,)
        dt = torch.float64 if name in ("centroid_x", "centroid_y", "poly_bbox") else torch.float32
        got[name] = torch.full(shape, SENTINEL, dtype=dt, device="cuda")
        setattr(mo, name, got[name].data_ptr())
    t_tile = t_tx = t_ty = t_cen = t_bb = w_cen = w_bb = None
    if tiles is not None:
        t_tile, t_tx, t_ty = (dev(a) for a in tiles)
    if centroid is not None:
        t_cen, w_cen = dev(centroid), torch.full((n, 2), SENTINEL, dtype=torch.float64, device="cuda")
    if bbox is not None:
        t_bb, w_bb = dev(bbox), torch.full((n, 4), -9, dtype=torch.int32, device="cuda")
    if hint == "table":
        hint = (n, m)
    if hint is not None:
        engine._check(engine.lib.pg_map_morph_hint(engine._h, int(hint[0]), int(hint[1])))
    fn = engine.lib.pg_map_morph_f32 if vt is np.float32 else engine.lib.pg_map_morph_f64
    with profiled(engine) as names:
        engine._check(fn(engine._h, n, ptr(d_off), ptr(src), ptr(t_tile), ptr(t_tx), ptr(t_ty), ptr(t_cen), ptr(t_bb),
                         ptr(dst), ptr(w_cen), ptr(w_bb), C.byref(mo), engine._stream()))
    res = {k: v.cpu().numpy() for k, v in got.items()}
    if write:
        res["wsi_poly_xy"] = dst.cpu().numpy()
        g = dst_buf.cpu().numpy()
        assert (g[:out_shift] == -7.0).all() and (g[out_shift + m:] == -7.0).all(), "wrote outside wsi_poly_xy"
    if centroid is not None:
        res["wsi_centroid"] = w_cen.cpu().numpy()
    if bbox is not None:
        res["wsi_bbox"] = w_bb.cpu().numpy()
    assert torch.equal(src, dev(xy)), "poly_xy changed"
    return res, names, (src.data_ptr(), None if dst is None else dst.data_ptr())


# ---------------------------------------------------------------------------------------------------- the oracle
_ORACLE = {}


def oracle(off, xy, key=None):
    """polygon_features_csr in float64 on the rings of `off` (which may be a window into xy: off[0] != 0); `key`
    names a table that several cases share, so its oracle runs once."""
    if key is not None and key in _ORACLE:
        return _ORACLE[key]
    off = np.asarray(off, dtype=np.int64)
    feat = omorph.polygon_features_csr(off - off[0], np.asarray(xy, dtype=np.float64)[off[0]: off[-1]])
    if key is not None:
        _ORACLE[key] = feat
    return feat


def shifts(n, tiles):
    if tiles is None:
        return np.zeros(n), np.zeros(n)
    nuc_tile, tile_x, tile_y = tiles
    return tile_x[nuc_tile].astype(np.float64), tile_y[nuc_tile].astype(np.float64)


def compare(res, feat, sx, sy, tag):
    """Every feature output present in `res` against the oracle, at the suite's bars."""
    for name in ("area", "perimeter", "circularity"):
        if name in res:
            np.testing.assert_allclose(res[name], feat[name], rtol=RTOL, equal_nan=True, err_msg=f"{tag} {name}")
    if "eccentricity" in res:
        np.testing.assert_allclose(res["eccentricity"], feat["eccentricity"], rtol=RTOL, atol=ECC_ATOL, equal_nan=True,
                                   err_msg=f"{tag} eccentricity")
    if "major_axis" in res:
        np.testing.assert_allclose(res["major_axis"], feat["major_axis_length"], rtol=RTOL, equal_nan=True,
                                   err_msg=f"{tag} major_axis")
    if "minor_axis" in res:
        np.testing.assert_allclose(res["minor_axis"], feat["minor_axis_length"], rtol=RTOL, atol=MINOR_ATOL,
                                   equal_nan=True, err_msg=f"{tag} minor_axis")
    for name, ref, s in (("centroid_x", feat["centroid_x"], sx), ("centroid_y", feat["centroid_y"], sy)):
        if name in res:
            np.testing.assert_allclose(res[name], ref + s, rtol=CENTROID_RTOL, equal_nan=True, err_msg=f"{tag} {name}")
    if "poly_bbox" in res:
        want = np.stack([feat["bbox_xmin"] + sx, feat["bbox_ymin"] + sy, feat["bbox_xmax"] + sx, feat["bbox_ymax"] + sy],
                        axis=1)
        np.testing.assert_array_equal(res["poly_bbox"], want, err_msg=f"{tag} poly_bbox")


def shifted_vertices(off, xy, tiles):
    """wsi = T(x + t): the vertex type's rounding of the exact sum (exact on the half-pixel lattice)."""
    off = np.asarray(off, dtype=np.int64)
    sx, sy = shifts(len(off) - 1, tiles)
    owner = np.repeat(np.arange(len(off) - 1), np.diff(off))
    seg = xy[off[0]: off[-1]].astype(np.float64)
    return np.stack([seg[:, 0] + sx[owner], seg[:, 1] + sy[owner]], axis=1).astype(xy.dtype)


def check_case(engine, off, xy, outputs="extra", tiles=None, centroid=None, bbox=None, write=True, hint="table",
               in_shift=0, out_shift=0, covers=("staged",), key=None, tag=""):
    """Run, assert the instantiation and the claimed warp paths, compare with the oracle, record the coverage."""
    n, m = len(off) - 1, int(xy.shape[0])
    res, names, (src_ptr, dst_ptr) = run_abi(engine, off, xy, outputs, tiles, centroid, bbox, write, hint, in_shift,
                                             out_shift)
    hn, hm = (n, m) if hint == "table" else (hint or (0, 0))   # None: a handle that was never hinted
    want, slab = variant(xy.dtype, outputs != "plain", hn, hm)
    assert names == [want], (tag, names, want)
    paths = set(warp_paths(off, slab, src_ptr, dst_ptr).tolist())
    assert set(covers) <= paths, (tag, "the table does not reach the claimed paths", covers, paths, slab)
    sx, sy = shifts(n, tiles)
    compare(res, oracle(off, xy, key), sx, sy, tag)
    if write:
        assert np.array_equal(res["wsi_poly_xy"][off[0]: off[-1]], shifted_vertices(off, xy, tiles)), tag
    if centroid is not None:
        assert np.array_equal(res["wsi_centroid"], centroid + np.stack([sx, sy], axis=1)), tag
    if bbox is not None:
        want_b = bbox.astype(np.int64) + np.stack([sx, sy, sx, sy], axis=1).astype(np.int64)
        assert np.array_equal(res["wsi_bbox"].astype(np.int64), want_b), tag
    COVERED.update((want, p) for p in paths & {"staged", "group"})
    return res, want, paths


# ---------------------------------------------------------------------------------------------------- CPU: the restated rule
def test_restated_launcher_picks_the_documented_variants():
    # C3 (2M x 32 float32, no extra output) runs the 6-CTA build; the ragged C1 / C4 tables (8..32, mean 20) the dense
    # 7-CTA build; any extra output selects EXTRA
    assert variant(np.float32, False, 2_000_000, 64_000_000) == ("map_morph_kernel<f32, plain, 6>", SLAB_VERTS_MIN)
    assert variant(np.float32, False, 500_000, 10_000_000) == ("map_morph_kernel<f32, plain, 7>", 802)
    assert variant(np.float32, True, 500_000, 10_000_000)[0] == "map_morph_kernel<f32, extra, 5>"
    assert variant(np.float64, False, 500_000, 10_000_000)[0] == "map_morph_kernel<f64, plain, 5>"
    assert variant(np.float64, True, 10, 1000)[0] == "map_morph_kernel<f64, extra, 4>"
    # dense exactly while mean <= 23; slab 512 up to mean 12.75; an absent hint (n = 0) is the default slab
    assert variant(np.float32, False, 100, 2300)[0].endswith(", 7>")
    assert variant(np.float32, False, 100, 2301)[0].endswith(", 6>")
    assert slab_verts(12.75, np.float32) == 512 and slab_verts(12.8, np.float32) == 514
    assert variant(np.float32, False, 0, 0) == ("map_morph_kernel<f32, plain, 6>", SLAB_VERTS_MIN)
    # the cap: 6400 float32 / 3200 float64 vertices per warp
    assert slab_verts(139.0, np.float32) == 6396 and slab_verts(140.0, np.float32) == 6400
    assert slab_verts(69.0, np.float64) == 3176 and slab_verts(70.0, np.float64) == 3200
    assert 139 < cap_mean(np.float32) < 140 and 69 < cap_mean(np.float64) < 70


def test_restated_warp_predicate():
    off = csr([10] * 32 + [40] * 32 + [0] * 32 + [3])
    assert warp_paths(off, 512, 0, 16).tolist() == ["staged", "group", "empty", "staged"]
    assert warp_paths(off, 512, 0, None).tolist() == ["staged", "group", "empty", "staged"]
    assert warp_paths(off, 512, 8, 16).tolist() == ["group", "group", "empty", "group"]   # other 16-byte phase
    assert warp_paths(off, 1282, 8, 24).tolist() == ["staged", "staged", "empty", "staged"]
    assert warp_paths(off, 1281 & ~1, 8, 24).tolist() == ["staged", "group", "empty", "staged"]


# ---------------------------------------------------------------------------------------------------- the matrix
def regime_table(vt, regime, seed):
    """(off, xy, (lo, hi] mean bounds, paths the table reaches under its own hint)."""
    rng = np.random.default_rng(seed)
    n = 8192
    if regime == "skewed":
        # short mean (dense / slab 512), four warps of 30-90-vertex rings and one 50 000-vertex ring
        nv = rng.integers(3, 17, size=32768)
        nv[32 * 100: 32 * 104] = rng.integers(30, 91, size=128)
        nv[32 * 500 + 7] = 50_000
        bounds = (0.0, 12.75)
    else:
        lo, hi, bounds = {"mean<=12.75": (3, 22, (0.0, 12.75)), "13-23": (8, 32, (12.75, 23.0)),
                          "24-33": (20, 40, (23.0, 33.0)), "34-cap": (40, 90, (33.0, cap_mean(vt))),
                          "past-cap": ((150, 250) if vt is np.float32 else (80, 120)) + ((cap_mean(vt), 1e9),)}[regime]
        nv = rng.integers(lo, hi + 1, size=n)
        nv[32 * 9: 32 * 10] = 2 * hi          # one warp past its slab: the group path in every regime
    off, xy = ellipses(nv, rng, vt)
    return off, xy, bounds


REGIMES = ["mean<=12.75", "13-23", "24-33", "34-cap", "past-cap", "skewed"]


@functools.lru_cache(maxsize=None)
def cached_regime(vt, regime):
    off, xy, bounds = regime_table(vt, regime, seed=REGIMES.index(regime) * 10 + (vt is np.float64))
    n = len(off) - 1
    rng = np.random.default_rng(7)
    return off, xy, bounds, tiles_for(n, rng), *tile_inputs(n, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("outputs", ["plain", "extra", "only_bbox", "only_cx"])
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
def test_variant_matrix_vs_oracle(engine, vt, outputs, regime):
    off, xy, (lo, hi), tiles, cen, bb = cached_regime(vt, regime)
    mean = int(off[-1]) / (len(off) - 1)
    assert lo < mean <= hi, (regime, mean)
    check_case(engine, off, xy, outputs, tiles, cen, bb, covers=("staged", "group"), key=(vt, regime),
               tag=f"{np.dtype(vt).name} {outputs} {regime}")


# ---------------------------------------------------------------------------------------------------- ring and table edges
SPECIAL_NV = [0, 1, 2, 3, 31, 32, 33, 34, 63, 64, 65]


def edge_table(vt):
    """One special-length ring per warp among short filler rings (lane 0, 17 or 31), degenerate rings, a warp of
    empty rows, and warps of 32 long rings."""
    rng = np.random.default_rng(41)
    warps = 3 * len(SPECIAL_NV) + 8
    nv = rng.integers(4, 9, size=32 * warps)
    for i, k in enumerate(SPECIAL_NV * 3):
        nv[32 * i + (0, 17, 31)[i // len(SPECIAL_NV)]] = k
    w = 3 * len(SPECIAL_NV)
    nv[32 * w: 32 * (w + 1)] = 0                      # a warp whose 32 rings are all empty
    nv[32 * (w + 1): 32 * (w + 2)] = 65               # 2080 vertices: past slabs of 512 and 1058
    nv[32 * (w + 2): 32 * (w + 3)] = 120              # 3840 vertices: past every slab these hints give
    deg = 32 * (w + 3) + np.arange(12)                # degenerate rings in an ordinary warp
    nv[deg] = 6
    off, xy = ellipses(nv, rng, vt)
    xy[off[deg[0]]: off[deg[0] + 1]] = xy[off[deg[0]]]                          # all-identical vertices
    xy[off[deg[1]]: off[deg[1] + 1]] = np.array([[3.0, 4.0]]) + np.arange(6)[:, None] * [[1.5, -0.5]]  # collinear
    xy[off[deg[2]]: off[deg[2] + 1]] = np.array([[0, 0], [0, 3], [4, 3], [4, 0], [2, -1], [1, -0.5]])  # clockwise
    xy[off[deg[3] + 1] - 1] = xy[off[deg[3]]]                                   # explicitly closed
    xy[off[deg[4]]: off[deg[4] + 1]] = np.array([[0, 0], [2, 0], [4, 0], [4, 0], [2, 0], [0, 0]])       # back and forth
    return off, xy.astype(vt), deg[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("hint_mean", [10, 28, 60])
@pytest.mark.parametrize("outputs", ["plain", "extra"])
@pytest.mark.parametrize("vt,out_shift", [(np.float32, 0), (np.float32, 1), (np.float64, 0)],
                         ids=["f32", "f32-other-phase", "f64"])
def test_ring_edges_on_every_variant(engine, vt, out_shift, outputs, hint_mean):
    # the hint (not the table) picks the slab, so one table meets each instantiation: the special lengths straddle the
    # (k & 31) == 0 fold of the staged walk, or - output in the other 16-byte phase - all go the group path
    off, xy, deg = edge_table(vt)
    n = len(off) - 1
    covers = ("group",) if out_shift else ("staged", "group")
    res, want, paths = check_case(engine, off, xy, outputs, hint=(n, hint_mean * n), out_shift=out_shift,
                                  covers=covers, key=("edges", vt), tag=f"edges {outputs} hint {hint_mean}")
    if out_shift:
        assert paths <= {"group", "empty"}
    assert "empty" in paths
    area, per = res["area"], res["perimeter"]
    assert area[deg[0]] == 0.0 and per[deg[0]] == 0.0 and res["circularity"][deg[0]] == 0.0
    assert np.isnan(res["eccentricity"][deg[0]]) and area[deg[1]] == 0.0 and area[deg[4]] == 0.0 and per[deg[4]] == 8.0
    assert area[deg[2]] == 14.0           # clockwise: |signed area| of the 4 x 3 box and the triangle below it
    nv = np.diff(off)
    assert np.isnan(area[nv < 3]).all() and np.isnan(per[nv < 3]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 127, 128, 129, 4097])
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
def test_table_sizes(engine, vt, n):
    # partial warps and partial CTAs: the last warp's range ends at poly_off[n]
    rng = np.random.default_rng(n)
    off, xy = ellipses(rng.integers(3, 41, size=n), rng, vt)
    tiles = tiles_for(n, rng)
    for outputs in ("plain", "extra"):
        check_case(engine, off, xy, outputs, tiles, *tile_inputs(n, rng), tag=f"n={n} {outputs}")


# ---------------------------------------------------------------------------------------------------- alignment and views
@pytest.mark.gpu
@pytest.mark.parametrize("outputs", ["plain", "extra"])
@pytest.mark.parametrize("vt,in_shift,out_shift,write", [
    (np.float32, 1, 1, True), (np.float32, 1, 0, False), (np.float32, 0, 1, True), (np.float32, 1, 0, True),
    (np.float64, 1, 1, True), (np.float64, 1, 0, True)])
def test_alignment(engine, vt, in_shift, out_shift, write, outputs):
    # a row shift moves a float32 array by 8 bytes (the bulk copy's head vertex; input and output in different
    # 16-byte phases when only one of them moves) and a float64 array by 16 (same phase)
    off, xy, _, tiles, _, _ = cached_regime(vt, "13-23")
    other_phase = write and vt is np.float32 and in_shift != out_shift
    res, _, paths = check_case(engine, off, xy, outputs, tiles, write=write, in_shift=in_shift, out_shift=out_shift,
                               covers=("group",) if other_phase else ("staged", "group"), key=(vt, "13-23"),
                               tag=f"shift {in_shift}/{out_shift}")
    if other_phase:
        assert paths == {"group"}


@pytest.mark.gpu
@pytest.mark.parametrize("outputs", ["plain", "extra"])
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
def test_csr_window(engine, vt, outputs):
    # poly_off = off[a:b+1] (first offset not 0) into the whole vertex array, through Engine.map_morph (which hints
    # (b - a, M)): only the window's vertices are written, the rest of wsi_poly_xy keeps its guard values
    off, xy, *_ = cached_regime(vt, "13-23")
    a, b = 1000, 5003
    w_off = off[a: b + 1]
    n = b - a
    rng = np.random.default_rng(3)
    nuc_tile, tile_x, tile_y = tiles_for(n, rng)
    out = torch.full(xy.shape, -7.0, dtype=dev(xy).dtype, device="cuda")
    with profiled(engine) as names:
        res = engine.map_morph(dev(w_off), dev(xy), dev(nuc_tile), dev(tile_x), dev(tile_y), write_polygons=True,
                               extra=outputs == "extra", out={"wsi_poly_xy": out})
    want, slab = variant(vt, outputs == "extra", n, xy.shape[0])
    assert names == [want]
    paths = set(warp_paths(w_off, slab, 0, 0).tolist())
    assert "staged" in paths
    got = {k: v.cpu().numpy() for k, v in res.items()}
    sx, sy = shifts(n, (nuc_tile, tile_x, tile_y))
    compare(got, oracle(w_off, xy), sx, sy, "window")
    wsi = got["wsi_poly_xy"]
    assert np.array_equal(wsi[w_off[0]: w_off[-1]], shifted_vertices(w_off, xy, (nuc_tile, tile_x, tile_y)))
    assert (wsi[: w_off[0]] == -7.0).all() and (wsi[w_off[-1]:] == -7.0).all()
    COVERED.update((want, p) for p in paths & {"staged", "group"})


# ---------------------------------------------------------------------------------------------------- optional inputs
@pytest.mark.gpu
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("inputs", ["nuc_tile", "centroid", "bbox", "no_polygons"])
def test_optional_inputs(engine, vt, inputs):
    # each optional input alone (the others NULL); without nuc_tile the shift is 0
    off, xy, _, tiles, cen, bb = cached_regime(vt, "13-23")
    for outputs in ("plain", "extra"):
        res, _, _ = check_case(engine, off, xy, outputs, tiles=tiles if inputs == "nuc_tile" else None,
                               centroid=cen if inputs == "centroid" else None, bbox=bb if inputs == "bbox" else None,
                               write=inputs != "no_polygons", covers=("staged", "group"), key=(vt, "13-23"),
                               tag=f"{inputs} {outputs}")
        assert ("wsi_poly_xy" in res) == (inputs != "no_polygons")
        if inputs == "centroid":
            assert np.array_equal(res["wsi_centroid"], cen)


@pytest.mark.gpu
@pytest.mark.parametrize("outputs", ["plain", "extra"])
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
def test_off_lattice_vertices_under_wsi_scale_shifts(engine, vt, outputs):
    # vertices off the half-pixel lattice, tiles up to ~150 000 px: the shifted vertex is the vertex type's rounding
    # of x + t (float32: one rounding of the exact sum; the features come from the unshifted vertices)
    rng = np.random.default_rng(17)
    n = 6000
    nv = rng.integers(8, 60, size=n)
    off, xy = ellipses(nv, rng, vt, lattice=False)
    nuc_tile = rng.integers(0, 90_000, size=n).astype(np.int32)
    tile_x = ((np.arange(90_000) % 300) * 508).astype(np.int32)
    tile_y = ((np.arange(90_000) // 300) * 508).astype(np.int32)
    res, _, _ = check_case(engine, off, xy, outputs, (nuc_tile, tile_x, tile_y), covers=("staged",),
                           tag="off-lattice")
    sx, _ = shifts(n, (nuc_tile, tile_x, tile_y))
    assert sx.max() > 100_000
    if vt is np.float32:   # the rounding is real: the float64 sum is not representable for most vertices
        owner = np.repeat(np.arange(n), nv)
        assert (res["wsi_poly_xy"][:, 0].astype(np.float64) != xy[:, 0].astype(np.float64) + sx[owner]).mean() > 0.5


# ---------------------------------------------------------------------------------------------------- stale or absent hint
@pytest.mark.gpu
@pytest.mark.parametrize("outputs", ["plain", "extra"])
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("table,hint_mean,covers", [
    ("34-cap", 10, ("group",)),               # short-ring hint on a long table: small slabs, every warp walks global
    ("mean<=12.75", 100, ("staged",)),        # long-ring hint on a short table: big slabs
    ("34-cap", 0, ("group",)),                # hint of n = 0: the default slab
    ("mean<=12.75", 0, ("staged", "group"))])
def test_stale_or_absent_hint(engine, vt, outputs, table, hint_mean, covers):
    off, xy, _, tiles, cen, bb = cached_regime(vt, table)
    n = len(off) - 1
    hint = (n, hint_mean * n) if hint_mean else (0, 0)
    check_case(engine, off, xy, outputs, tiles, cen, bb, hint=hint, covers=covers, key=(vt, table),
               tag=f"{table} hint {hint}")


@pytest.mark.gpu
def test_fresh_handle_without_a_hint():
    from path_gene_multimodal_b200.engine import Engine

    eng = Engine(0)
    try:
        off, xy, _, tiles, cen, bb = cached_regime(np.float32, "34-cap")
        check_case(eng, off, xy, "plain", tiles, cen, bb, hint=None, covers=("group",), key=(np.float32, "34-cap"),
                   tag="fresh handle")
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------- product configurations
@pytest.mark.gpu
def test_c3_as_the_benchmark_calls_it(engine):
    # bench.py's C3 stage: 2M rings x 32 float32 vertices, nuc_tile / centroid / bbox, write_polygons=True, through
    # Engine.map_morph; every ring against the oracle (about 15 s of numpy)
    n3 = 2_000_000
    off, xy = synth.make_polygons(n3, synth.SEEDS["C3"], v_fixed=32)
    rng = np.random.default_rng(3)
    side = 73
    tile_x = ((np.arange(side * side) % side) * 508).astype(np.int32)
    tile_y = ((np.arange(side * side) // side) * 508).astype(np.int32)
    nuc_tile = rng.integers(0, side * side, size=n3).astype(np.int32)
    cen = rng.random((n3, 2)) * 508
    bb = rng.integers(0, 508, size=(n3, 4)).astype(np.int32)
    d_xy = dev(xy)
    with profiled(engine) as names:
        res = engine.map_morph(dev(off), d_xy, dev(nuc_tile), dev(tile_x), dev(tile_y), dev(cen), dev(bb),
                               write_polygons=True)
    want, slab = variant(np.float32, False, n3, xy.shape[0])
    assert names == [want] == ["map_morph_kernel<f32, plain, 6>"]
    paths = set(warp_paths(off, slab, d_xy.data_ptr(), res["wsi_poly_xy"].data_ptr()).tolist())
    assert paths == {"staged"}
    got = {k: v.cpu().numpy() for k, v in res.items()}
    feat = omorph.polygon_features_csr(off, xy)
    tiles = (nuc_tile, tile_x, tile_y)
    sx, sy = shifts(n3, tiles)
    compare(got, feat, sx, sy, "C3")
    assert np.array_equal(got["wsi_poly_xy"], shifted_vertices(off, xy, tiles))
    assert np.array_equal(got["wsi_centroid"], cen + np.stack([sx, sy], axis=1))
    assert np.array_equal(got["wsi_bbox"].astype(np.int64), bb + np.stack([sx, sy, sx, sy], axis=1).astype(np.int64))
    np.testing.assert_allclose(got["area"].astype(np.float64).sum(), feat["area"].sum(), rtol=1e-6)
    COVERED.add((want, "staged"))


@pytest.mark.gpu
@pytest.mark.parametrize("staging", ["float", "halfpx16"])
def test_c4_slide_through_process_slide(staging):
    # one 500 k-nucleus C4 slide through cohort.process_slide (float32 or int16 half-pixel staging, widened on the
    # device): the dense build; per-ring values from the map_morph call it makes, and its area_sum
    from path_gene_multimodal_b200.engine import Engine

    n = 500_000
    tab = synth.make_cohort_slide(0, n)
    off, xy = tab.poly_off, tab.poly_xy
    tiles = (tab.nuc_tile, tab.tile_x, tab.tile_y)
    eng = Engine(0)
    seen = []
    inner = eng.map_morph

    def recording(*args, **kw):
        seen.append(inner(*args, **kw))
        return seen[-1]

    eng.map_morph = recording
    try:
        with profiled(eng) as names:
            summary = cohort.process_slide(eng, cohort.pin_table(synth.make_cohort_slide(0, n), staging=staging))
        want, slab = variant(np.float32, False, n, xy.shape[0])
        assert want == "map_morph_kernel<f32, plain, 7>"
        assert [s for s in names if s.startswith("map_morph")] == [want]
        assert "staged" in set(warp_paths(off, slab, 0, 0).tolist())
        assert len(seen) == 1
        got = {k: v.cpu().numpy() for k, v in seen[0].items()}
    finally:
        eng.close()
    feat = oracle(off, xy, key=("C4", n))
    sx, sy = shifts(n, tiles)
    compare(got, feat, sx, sy, f"C4 {staging}")
    assert np.array_equal(got["wsi_poly_xy"], shifted_vertices(off, xy, tiles))
    assert np.array_equal(got["wsi_centroid"], tab.centroid + np.stack([sx, sy], axis=1))
    np.testing.assert_allclose(summary["area_sum"], feat["area"].sum(), rtol=1e-6)
    COVERED.add((want, "staged"))


# ---------------------------------------------------------------------------------------------------- in-place shift
@pytest.mark.gpu
@pytest.mark.parametrize("vt", [np.float32, np.float64], ids=["f32", "f64"])
def test_in_place_shift_is_refused(engine, vt):
    # the group path reads a ring's vertex 0 again for the closing edge after another lane has shifted it (and both
    # pointers are __restrict__): the C ABI refuses wsi_poly_xy == poly_xy, the engine any overlap, before any launch
    off, xy, _, tiles, *_ = cached_regime(vt, "skewed")
    n, m = len(off) - 1, xy.shape[0]
    d_off, t_tile, t_tx, t_ty = dev(off), *(dev(a) for a in tiles)
    buf = torch.zeros((2 * m + 1, 2), dtype=dev(xy).dtype, device="cuda")
    src = buf[:m]
    src.copy_(dev(xy))
    mo = PgMorphOut()
    area = torch.full((n,), SENTINEL, dtype=torch.float32, device="cuda")
    mo.area = area.data_ptr()
    fn = engine.lib.pg_map_morph_f32 if vt is np.float32 else engine.lib.pg_map_morph_f64
    l0 = engine.launches
    rc = fn(engine._h, n, ptr(d_off), ptr(src), ptr(t_tile), ptr(t_tx), ptr(t_ty), None, None, ptr(src), None, None,
            C.byref(mo), engine._stream())
    assert rc == _lib.PG_ERR_INVALID
    assert b"alias" in engine.lib.pg_last_error(engine._h)
    for overlap in (src, buf[m - 1: 2 * m - 1], buf[1: m + 1]):
        with pytest.raises(ValueError, match="overlaps poly_xy"):
            engine.map_morph(d_off, src, t_tile, t_tx, t_ty, write_polygons=True, out={"wsi_poly_xy": overlap})
    assert engine.launches == l0
    torch.cuda.synchronize()
    assert torch.equal(src, dev(xy)) and bool((area == SENTINEL).all())
    # the adjacent, disjoint range of the same buffer is a legal output
    res = engine.map_morph(d_off, src, t_tile, t_tx, t_ty, write_polygons=True, out={"wsi_poly_xy": buf[m: 2 * m]})
    assert engine.launches == l0 + 1
    assert np.array_equal(res["wsi_poly_xy"].cpu().numpy(), shifted_vertices(off, xy, tiles))
    compare({k: res[k].cpu().numpy() for k in BASE}, oracle(off, xy, key=(vt, "skewed")), *shifts(n, tiles), "adjacent")


# ---------------------------------------------------------------------------------------------------- coverage
@pytest.mark.gpu
def test_every_variant_was_compared_on_both_paths():
    # runs last: the cases above record (instantiation, path) only after their comparison passed
    missing = [(v, p) for v in VARIANTS for p in ("staged", "group") if (v, p) not in COVERED]
    assert not missing, missing
