"""GPU tests of K16 (pg_pair_dist_hist): histograms and type counts bit for bit against the host reference
(oracle/cooccurrence.py) on synthetic slides, half-pixel lattices with distances on the thresholds, dense clumps (the
hot counter; more than 2^32 pairs in one bin), t_max past the slide's diagonal and below the nearest-neighbour
distance, tiny inputs, 1 and 64 thresholds, and a grid built for a much smaller radius. Also: strips with halos whose
histograms sum to the slide's, determinism across calls and handles, and co_occurrence / ripley end to end."""
import numpy as np
import pytest
import torch

from oracle import cooccurrence as oc
from path_gene_multimodal_b200 import co_occurrence, ripley, synth
from path_gene_multimodal_b200.engine import Engine, pair_hist_cell

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    return Engine(0)


def mixed_types(rng, n, n_types):
    """Types 1..n_types plus -2, 0, n_types + 1, 17 and 2**31 - 1 (everything outside 1..n_types counts nowhere)."""
    t = rng.integers(-2, n_types + 2, size=n).astype(np.int64)
    pick = rng.choice(n, size=max(2, n // 50), replace=False)
    t[pick[0::2]] = 17
    t[pick[1::2]] = 2 ** 31 - 1
    return t.astype(np.int32)


def gpu_hist(engine, xy, types, thr, n_types, cell=None, n_query=None, gid=None):
    xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    n = xy.shape[0]
    if cell is None:
        span = np.ptp(xy, axis=0) if n else np.ones(2)
        cell = pair_hist_cell(float(thr[-1]), n, max(span[0], 1e-9) * max(span[1], 1e-9))
    d_xy = torch.from_numpy(xy).to(engine.device)
    d_t = torch.from_numpy(np.ascontiguousarray(types, dtype=np.int32)).to(engine.device)
    d_g = torch.from_numpy(np.ascontiguousarray(gid, dtype=np.int32)).to(engine.device) if gid is not None else None
    engine.grid_build(d_xy, d_t, d_g, cell, n_query=n_query)
    r = engine.pair_dist_hist(thr, n_types)
    return r["hist"].cpu().numpy(), r["type_count"].cpu().numpy()


def check(engine, xy, types, thr, n_types, ref=None, **kw):
    h, tc = gpu_hist(engine, xy, types, thr, n_types, **kw)
    if ref is None:
        ref = oc.pair_hist(xy, types, thr, n_types, n_query=kw.get("n_query"), ids=kw.get("gid"))
    np.testing.assert_array_equal(h, ref)
    np.testing.assert_array_equal(tc, oc.type_count(types, n_types, kw.get("n_query")))
    return h


@pytest.mark.parametrize("n,n_types,n_thr", [(20_000, 1, 50), (20_000, 5, 50), (20_000, 16, 64), (200_000, 5, 50),
                                             (200_000, 16, 64)])
def test_synth_slides(engine, n, n_types, n_thr):
    xy, _, _ = synth.make_points(n, synth.SEEDS["C2"])
    types = mixed_types(np.random.default_rng(n + n_types), len(xy), n_types)
    thr = np.linspace(0.0, 200.0, n_thr)
    h = check(engine, xy, types, thr, n_types)
    assert h.sum() > 0


@pytest.mark.parametrize("shift", [1e5, 1e7])
def test_half_pixel_lattice_on_the_thresholds(engine, shift):
    rng = np.random.default_rng(int(shift) % 97)
    xy = shift + rng.integers(0, 300, size=(20_000, 2)) * 0.5   # dense: many duplicates and exact ties
    types = rng.integers(1, 4, size=len(xy)).astype(np.int32)
    thr = np.arange(1, 21) * 0.5                                # t^2 = k^2 / 4: exact, pairs sit on every threshold
    h = check(engine, xy, types, thr, 3)
    assert (h.sum(axis=(1, 2)) > 0).all()


def test_dense_clump_hot_counter(engine):
    """4 200 type-3 points inside a disc of radius 16 (the clump of test_gpu_graph_variants.py) plus a background:
    every clump pair lands in bin 0, one (bin, 3, 3) counter for almost every lane of every clump warp."""
    rng = np.random.default_rng(7)
    side, n_clump = 2000.0, 4200
    rho, phi = 16.0 * np.sqrt(rng.random(n_clump)), rng.random(n_clump) * 2 * np.pi
    clump = np.stack([1000 + rho * np.cos(phi), 1000 + rho * np.sin(phi)], axis=1)
    xy = np.concatenate([clump, rng.random((1000, 2)) * side])
    types = np.concatenate([np.full(n_clump, 3, dtype=np.int32), mixed_types(rng, 1000, 7)])
    order = rng.permutation(len(xy))
    xy, types = xy[order], types[order]
    h = check(engine, xy, types, np.array([33.0, 80.0, 200.0]), 7)
    assert h[0, 2, 2] >= n_clump * (n_clump - 1)


def test_65540_point_clump_more_than_2_pow_32_pairs_in_one_bin(engine):
    """65 540 points around one centre (sigma 2 px) and 30 000 uniform points: the clump's 4.3e9 ordered pairs all land
    in bin 0, more than a 32-bit counter holds. The clump x clump part of the reference is its closed form."""
    rng = np.random.default_rng(11)
    side, n_clump = 5000.0, 65_540
    clump = rng.normal(side / 2, 2.0, size=(n_clump, 2))
    xy = np.concatenate([clump, rng.random((30_000, 2)) * side])
    types = rng.integers(1, 6, size=len(xy)).astype(np.int32)
    thr = np.array([40.0, 100.0, 300.0])
    assert np.hypot(*np.ptp(clump, axis=0)) < thr[0]
    ids = np.arange(len(xy))
    cl, un = ids < n_clump, ids >= n_clump
    ref = oc.pair_hist_sets(xy[un], types[un], ids[un], xy, types, ids, thr, 5)
    ref += oc.pair_hist_sets(xy[cl], types[cl], ids[cl], xy[un], types[un], ids[un], thr, 5)
    na = np.bincount(types[cl] - 1, minlength=5).astype(np.int64)
    ref[0] += np.outer(na, na) - np.diag(na)
    assert ref[0].sum() > 2 ** 32 and ref[0].max() < 2 ** 63
    check(engine, xy, types, thr, 5, ref=ref)


def test_t_max_past_the_diagonal_and_below_the_nearest_neighbour(engine):
    xy, _, side = synth.make_points(20_000, synth.SEEDS["C1"])
    types = mixed_types(np.random.default_rng(2), len(xy), 5)
    thr = np.array([500.0, 3000.0, 2.0 * side])                 # 2 side > the diagonal: every pair counts
    ref = oc.pair_hist_brute(xy, types, thr, 5)
    h = check(engine, xy, types, thr, 5, ref=ref)
    ok = (types >= 1) & (types <= 5)
    assert h.sum() == ok.sum() * (ok.sum() - 1)
    h = check(engine, xy, types, np.array([1e-3]), 5)           # below every nearest-neighbour distance
    assert h.sum() == 0


@pytest.mark.parametrize("n", [0, 1, 2])
@pytest.mark.parametrize("n_thr", [1, 64])
def test_tiny_inputs(engine, n, n_thr):
    xy = np.array([[3.0, 4.0], [3.0, 4.0 + 1e-3]])[:n]
    types = np.array([1, 2], dtype=np.int32)[:n]
    thr = np.linspace(0.0, 1.0, n_thr) if n_thr > 1 else np.array([0.5])
    h = check(engine, xy, types, thr, 2)
    assert h.sum() == (2 if n == 2 else 0)


def test_grid_for_a_small_radius_queried_at_a_large_one(engine):
    xy, _, _ = synth.make_points(20_000, synth.SEEDS["C3"])
    types = mixed_types(np.random.default_rng(5), len(xy), 5)
    thr = np.linspace(0.0, 300.0, 30)
    ref = oc.pair_hist(xy, types, thr, 5)
    check(engine, xy, types, thr, 5, ref=ref)
    check(engine, xy, types, thr, 5, ref=ref, cell=2.0)          # built as for a 2 px radius: R ~ 150 rings
    info = engine.grid_info()
    assert info["cell"] < 20.0


def test_strips_with_halos_sum_to_the_slide(engine):
    """Strips of a slide built with n_query (the strip's own points first), gid (global ids) and a halo of t_max: the
    sum of their histograms is the whole slide's, which is what a strip-sharded co_occurrence adds up."""
    xy, _, side = synth.make_points(200_000, synth.SEEDS["C2"])
    types = mixed_types(np.random.default_rng(8), len(xy), 5)
    thr = np.linspace(0.0, 150.0, 40)
    whole, tc_whole = gpu_hist(engine, xy, types, thr, 5)
    total, tc_total = np.zeros_like(whole), np.zeros_like(tc_whole)
    edges = np.linspace(xy[:, 0].min(), xy[:, 0].max() + 1.0, 5)
    for lo, hi in zip(edges[:-1], edges[1:]):
        own = (xy[:, 0] >= lo) & (xy[:, 0] < hi)
        halo = ~own & (xy[:, 0] >= lo - thr[-1]) & (xy[:, 0] < hi + thr[-1])
        sel = np.concatenate([np.nonzero(own)[0], np.nonzero(halo)[0]])
        h, tc = gpu_hist(engine, xy[sel], types[sel], thr, 5, n_query=int(own.sum()), gid=sel.astype(np.int32))
        total += h
        tc_total += tc
    np.testing.assert_array_equal(total, whole)
    np.testing.assert_array_equal(tc_total, tc_whole)
    np.testing.assert_array_equal(whole, oc.pair_hist(xy, types, thr, 5))


def test_determinism_across_calls_and_handles(engine):
    xy, _, _ = synth.make_points(200_000, synth.SEEDS["C2"])
    types = mixed_types(np.random.default_rng(9), len(xy), 16)
    thr = np.linspace(0.0, 200.0, 64)
    a = gpu_hist(engine, xy, types, thr, 16)
    b = gpu_hist(engine, xy, types, thr, 16)
    other = Engine(0)
    try:
        c = gpu_hist(other, xy, types, thr, 16)
    finally:
        other.close()
    for x in (b, c):
        np.testing.assert_array_equal(x[0], a[0])
        np.testing.assert_array_equal(x[1], a[1])


def test_co_occurrence_end_to_end():
    xy, types, _ = synth.make_points(100_000, synth.SEEDS["C2"])
    thr = np.linspace(0.0, 200.0, 21)
    hist = oc.pair_hist(xy, types, thr, 5)
    got = co_occurrence(xy, types, thr, n_types=5, device=0)
    annulus = np.moveaxis(hist[1:], 0, -1)
    np.testing.assert_array_equal(got["interval"], thr)
    np.testing.assert_array_equal(got["count"], annulus)
    np.testing.assert_array_equal(got["occ"], oc.occurrence(annulus))
    cum = co_occurrence(xy, types, 21, max_dist=200.0, cumulative=True, device=0)
    np.testing.assert_array_equal(cum["count"], np.moveaxis(np.cumsum(hist, axis=0)[1:], 0, -1))
    np.testing.assert_array_equal(cum["occ"], oc.occurrence(cum["count"]))
    assert got["count"].shape == (5, 5, 20) and np.isfinite(got["occ"]).all()


def test_ripley_end_to_end_with_the_hull_area():
    """K / L by type pair and univariate; the default area is K14's hull of all 1 M centroids as one ring, checked
    against scipy's ConvexHull."""
    from scipy.spatial import ConvexHull

    xy, types, _ = synth.make_points(1_000_000, synth.SEEDS["C2"])
    radii = np.array([10.0, 25.0, 50.0, 100.0])
    got = ripley(xy, radii, types=types, n_types=5, device=0)
    area = ConvexHull(xy).volume
    assert abs(got["area"] - area) <= 1e-12 * area
    count = np.moveaxis(np.cumsum(oc.pair_hist(xy, types, radii, 5), axis=0), 0, -1)
    np.testing.assert_array_equal(got["count"], count)
    n = oc.type_count(types, 5)
    np.testing.assert_array_equal(got["n"], n)
    np.testing.assert_array_equal(got["K"], oc.ripley_k(count, n, got["area"]))
    np.testing.assert_array_equal(got["L"], np.sqrt(oc.ripley_k(count, n, got["area"]) / np.pi))
    uni = ripley(xy[:50_000], radii, area=1234.5, device=0)
    c1 = np.cumsum(oc.pair_hist(xy[:50_000], np.ones(50_000, dtype=np.int32), radii, 1)[:, 0, 0])
    np.testing.assert_array_equal(uni["count"], c1)
    np.testing.assert_array_equal(uni["K"], 1234.5 * c1.astype(np.float64) / float(50_000 * 49_999))
    assert uni["K"].shape == (4,) and uni["area"] == 1234.5
