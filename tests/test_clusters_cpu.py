"""CPU tests of the cluster oracle (oracle/clusters.py) behind K19 and cell_clusters: the literal sklearn loop against
the vectorised form and against sklearn.cluster.DBSCAN itself on random slides, planted clusters and integer lattices
with d == eps exactly; the lower-label rule for a border point between two clusters; min_samples = 1 as connected
components; the components oracle against scipy on non-symmetric CSRs; the per-cluster table; and the input errors of
cell_clusters / connected_components, which are raised before anything needs a GPU."""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components as scipy_cc

from oracle import clusters as oc
from oracle import graph as ograph
from path_gene_multimodal_b200.cell_graph import cell_clusters, connected_components


def random_slide(n, seed, side=100.0):
    return np.random.default_rng(seed).random((n, 2)) * side


def planted(seed):
    """A sparse background with three tight aggregates of different sizes."""
    rng = np.random.default_rng(seed)
    bg = rng.random((400, 2)) * 200.0
    blobs = [rng.normal(c, s, size=(m, 2)) for c, s, m in (((50, 50), 2.0, 80), ((150, 60), 3.0, 150),
                                                            ((100, 160), 1.5, 40))]
    x = np.concatenate([bg, *blobs])
    return x[rng.permutation(len(x))]


def lattice_345(seed):
    """Integer points where many pairs lie exactly eps = 5 apart (3-4-5 triangles) or sqrt(2) * 5 apart."""
    rng = np.random.default_rng(seed)
    base = np.stack(np.meshgrid(np.arange(0, 40, 3), np.arange(0, 40, 4)), -1).reshape(-1, 2).astype(np.float64)
    extra = rng.integers(0, 40, size=(60, 2)).astype(np.float64)
    x = np.concatenate([base, extra])
    return x[rng.permutation(len(x))]


def sklearn_dbscan(x, eps, min_samples):
    skc = pytest.importorskip("sklearn.cluster")
    m = skc.DBSCAN(eps=eps, min_samples=min_samples, algorithm="kd_tree").fit(x)
    core = np.zeros(len(x), dtype=bool)
    core[m.core_sample_indices_] = True
    return m.labels_.astype(np.int64), core


CASES = [("random", lambda: random_slide(2000, 1), 2.0, 3), ("random", lambda: random_slide(2000, 2), 3.5, 6),
         ("random", lambda: random_slide(1500, 3), 1.2, 1), ("planted", lambda: planted(4), 4.0, 5),
         ("planted", lambda: planted(5), 6.0, 12), ("lattice", lambda: lattice_345(6), 5.0, 4),
         ("lattice", lambda: lattice_345(7), 5.0, 6), ("lattice", lambda: lattice_345(8), 4.0, 3)]


@pytest.mark.parametrize("name,make,eps,ms", CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(CASES)])
def test_loop_vectorised_and_sklearn_agree(name, make, eps, ms):
    x = make()
    lab_loop, core_loop = oc.dbscan_loop(x, eps, ms)
    lab_vec, core_vec = oc.dbscan(x, eps, ms)
    np.testing.assert_array_equal(lab_loop, lab_vec)
    np.testing.assert_array_equal(core_loop, core_vec)
    lab_sk, core_sk = sklearn_dbscan(x, eps, ms)
    np.testing.assert_array_equal(lab_loop, lab_sk)
    np.testing.assert_array_equal(core_loop, core_sk)
    assert lab_loop.max() >= 0 or ms > 1


def test_lattice_boundary_is_inclusive():
    # (0,0) - (3,4) at exactly 5: one pair, joined at eps = 5 and not at the float just below
    x = np.array([[0.0, 0.0], [3.0, 4.0], [20.0, 20.0]])
    lab, _ = oc.dbscan(x, 5.0, 2)
    np.testing.assert_array_equal(lab, [0, 0, -1])
    lab, _ = oc.dbscan(x, np.nextafter(5.0, 0.0), 2)
    np.testing.assert_array_equal(lab, [-1, -1, -1])
    np.testing.assert_array_equal(sklearn_dbscan(x, 5.0, 2)[0], [0, 0, -1])


SQUARE_A = [(0, 0), (1, 0), (0, 1), (1, 1)]
SQUARE_B = [(3, 0), (4, 0), (3, 1), (4, 1)]
BORDER = [(2, -0.6)]


@pytest.mark.parametrize("order,expect", [
    ((SQUARE_B, SQUARE_A, BORDER), [0] * 4 + [1] * 4 + [0]),   # b takes B's label, the lower one
    ((BORDER, SQUARE_A, SQUARE_B), [0] + [0] * 4 + [1] * 4),   # b takes A's label
])
def test_border_point_takes_lower_label(order, expect):
    x = np.array([p for group in order for p in group], dtype=np.float64)
    for fn in (oc.dbscan_loop, oc.dbscan):
        lab, core = fn(x, 1.5, 4)
        np.testing.assert_array_equal(lab, expect)
        assert not core[[i for i, p in enumerate(map(tuple, x)) if p == (2, -0.6)]].any()
    np.testing.assert_array_equal(sklearn_dbscan(x, 1.5, 4)[0], expect)


@pytest.mark.parametrize("seed", [0, 1])
def test_min_samples_one_is_connected_components(seed):
    x = random_slide(1500, seed)
    g = ograph.radius_graph(x, 2.0)
    k, cc = oc.connected_components(g["row_ptr"], g["col"])
    lab, core = oc.dbscan(x, 2.0, 1)
    assert core.all()
    np.testing.assert_array_equal(lab, cc)
    assert lab.max() + 1 == k


def test_components_oracle_equals_scipy_on_one_directional_csr():
    rng = np.random.default_rng(3)
    n = 3000
    src = rng.integers(0, n, 2500)
    dst = rng.integers(0, n, 2500)
    a = sp.csr_matrix((np.ones(2500), (src, dst)), shape=(n, n))
    a.sum_duplicates()
    a.sort_indices()
    k_ref, lab_ref = scipy_cc(a, directed=False)
    k, lab = oc.connected_components(a.indptr, a.indices)
    assert k == k_ref
    # same partition, numbered by smallest member
    np.testing.assert_array_equal(lab, oc._by_smallest(lab_ref.astype(np.int64), k_ref))
    first = np.array([np.flatnonzero(lab == c)[0] for c in range(k)])
    assert (np.diff(first) > 0).all()


def test_components_oracle_skips_foreign_ids_and_self_entries():
    rp = np.array([0, 3, 4, 6, 6])
    col = np.array([0, 7, -2, 2, 3, 1])  # self (0,0), foreign 7 and -2; 1 -> 2, 2 -> 3 and 2 -> 1
    k, lab = oc.connected_components(rp, col)
    assert k == 2
    np.testing.assert_array_equal(lab, [0, 1, 1, 1])


def test_cluster_props_oracle():
    x = np.array([[0, 0], [2, 0], [0, 2], [5, 5], [5, 6], [9, 9], [1, 1]], dtype=np.float64)
    lab = np.array([0, 0, 0, 1, 1, -1, 0])
    t = np.array([1, 2, 2, 5, 7, 1, 1])
    p = oc.cluster_props(lab, 2, x, t, 5, core=np.array([1, 1, 0, 1, 1, 0, 1], bool))
    np.testing.assert_array_equal(p["n_members"], [4, 2])
    np.testing.assert_array_equal(p["n_core"], [3, 2])
    np.testing.assert_array_equal(p["type_count"], [[2, 2, 0, 0, 0], [0, 0, 0, 0, 1]])
    np.testing.assert_array_equal(p["member_off"], [0, 4, 6])
    np.testing.assert_array_equal(p["member_xy"], x[[0, 1, 2, 6, 3, 4]])
    np.testing.assert_allclose(p["centroid"], [[0.75, 0.75], [5.0, 5.5]])
    np.testing.assert_array_equal(p["bbox"], [[0, 0, 2, 2], [5, 5, 5, 6]])
    assert p["hull_area"][0] == 2.0 and np.isnan(p["hull_area"][1])
    assert oc.hull_area(np.array([[0, 0], [1, 1], [2, 2], [3, 3.0]])) == 0.0
    rng = np.random.default_rng(0)
    big = rng.random((500, 2))
    from scipy.spatial import ConvexHull

    assert oc.hull_area(big) == ConvexHull(big).volume


def test_cell_clusters_input_errors():
    x = random_slide(10, 0)
    t = np.ones(10, dtype=np.int32)
    with pytest.raises(ValueError, match="shape"):
        cell_clusters(np.zeros((5, 3)), 1.0)
    for eps in (-1.0, np.nan, np.inf):
        with pytest.raises(ValueError, match="eps"):
            cell_clusters(x, eps)
    for ms in (0, -3, 2.5):
        with pytest.raises(ValueError, match="min_samples"):
            cell_clusters(x, 1.0, min_samples=ms)
    with pytest.raises(ValueError, match="keep_types"):
        cell_clusters(x, 1.0, types=t, keep_types=[])
    with pytest.raises(ValueError, match="keep_types"):
        cell_clusters(x, 1.0, keep_types=[1])
    with pytest.raises(ValueError, match="types"):
        cell_clusters(x, 1.0, types=t[:5])
    with pytest.raises(ValueError, match="n_types"):
        cell_clusters(x, 1.0, types=t, n_types=17)
    with pytest.raises(ValueError, match="mpp"):
        cell_clusters(x, 1.0, mpp=0.0)


def test_connected_components_input_errors():
    with pytest.raises(ValueError, match="row_ptr"):
        connected_components(np.array([1, 2]), np.array([0]))
    with pytest.raises(ValueError, match="row_ptr"):
        connected_components(np.array([0, 2, 1]), np.array([0]))
    with pytest.raises(ValueError, match="col ids"):
        connected_components(np.array([0, 1, 2]), np.array([1, 5]))
    with pytest.raises(ValueError, match="col"):
        connected_components(np.array([0, 1]), np.array([0.5]))
