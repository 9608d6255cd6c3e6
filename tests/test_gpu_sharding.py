"""GPU: strip-sharded graphs equal the single-GPU graphs bit for bit (ranks emulated in lockstep on one GPU;
the same generators run over NCCL in tests/multi_gpu_check.py and in the c5_strip_sharded stage of bench.py --gpus N)."""
import numpy as np
import pytest
import torch

from path_gene_multimodal_b200 import sharding, synth
from path_gene_multimodal_b200.engine import default_knn_cell, radius_cell

pytestmark = pytest.mark.gpu


def _split(xy, ty, world, edges=None):
    dev = torch.device("cuda", 0)
    n = len(xy)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    gid = torch.arange(n, dtype=torch.int32, device=dev)
    if edges is None:
        chunks = [slice(q * n // world, (q + 1) * n // world) for q in range(world)]
        edges = sharding.run_emulated([sharding.equal_count_edges(d_xy[c][:, 0].contiguous(), world, float(xy[:, 0].min()),
                                                                  float(xy[:, 0].max())) for c in chunks])[0]
    strips = sharding.strips_from_edges(edges)
    parts = []
    for s in strips:
        m = (d_xy[:, 0] >= s.x_lo) & (d_xy[:, 0] < s.x_hi)
        parts.append((d_xy[m].contiguous(), d_ty[m].contiguous(), gid[m].contiguous()))
    return d_xy, d_ty, strips, parts


@pytest.mark.parametrize("world", [2, 4, 7])
def test_sharded_radius_equals_single(engine, world):
    xy, ty, side = synth.make_points(60_000, seed=51)
    d_xy, d_ty, strips, parts = _split(xy, ty, world)
    engine.grid_build(d_xy, d_ty, None, radius_cell(50.0), None)
    ref = engine.radius_graph(50.0, upper=True, want_dist32=True, want_dist64=True, want_edges=True)
    ref_edges = ref["edges"].cpu().numpy()
    res = sharding.run_emulated([sharding.sharded_radius_graph(engine, p[0], p[1], p[2], 50.0, s, q, world)
                                 for q, (s, p) in enumerate(zip(strips, parts))])
    edges = np.concatenate([r["edges"].cpu().numpy() for r in res])
    d64 = np.concatenate([r["dist64"].cpu().numpy() for r in res])
    order = np.lexsort((edges[:, 1], edges[:, 0]))
    assert np.array_equal(edges[order], ref_edges)                                   # every edge once, global ids
    assert np.array_equal(d64[order], ref["dist64"].cpu().numpy())
    deg = np.zeros(len(xy), dtype=np.int32)
    nbr = np.zeros((len(xy), 5), dtype=np.int32)
    for r, p in zip(res, parts):
        g = p[2].cpu().numpy()
        deg[g] = r["degree"].cpu().numpy()
        nbr[g] = r["nbr_count"].cpu().numpy()
        assert r["n_ghost"] > 0
    assert np.array_equal(deg, ref["degree"].cpu().numpy()) and np.array_equal(nbr, ref["nbr_count"].cpu().numpy())
    # per-strip statistics combine to the whole-slide statistics
    tot = sum(int(r["stats"].cpu().numpy()[1]) for r in res)
    assert tot == int(ref["stats"].cpu().numpy()[1])


@pytest.mark.parametrize("world,k", [(2, 8), (4, 16), (5, 5)])
def test_sharded_knn_equals_single(engine, world, k):
    xy, ty, side = synth.make_points(50_000, seed=52)
    n = len(xy)
    d_xy, d_ty, strips, parts = _split(xy, ty, world)
    engine.grid_build(d_xy, d_ty, None, default_knn_cell(n, float(side) ** 2, k), None)
    kn = engine.knn(k, dist_dtype=torch.float64)
    ref_idx, ref_d = kn["knn_idx"].cpu().numpy(), kn["dist"].cpu().numpy()
    sym = engine.symmetrize(kn["knn_idx"], kn["dist"])
    up = engine.csr_upper(sym["row_ptr"], sym["col"], sym["w64"])
    comp = engine.compose_degree(sym["row_ptr"], sym["col"], d_ty, 5)
    res = sharding.run_emulated([sharding.sharded_knn_graph(engine, p[0], p[1], p[2], k, s, q, world, n_global=n, h0=20.0)
                                 for q, (s, p) in enumerate(zip(strips, parts))])   # h0 too small on purpose: must retry
    idx = np.zeros_like(ref_idx)
    dist = np.zeros_like(ref_d)
    deg = np.zeros(n, dtype=np.int32)
    nbr = np.zeros((n, 5), dtype=np.int32)
    for r, p in zip(res, parts):
        g = p[2].cpu().numpy()
        idx[g] = r["knn_idx"].cpu().numpy()
        dist[g] = r["dist"].cpu().numpy()
        deg[g] = r["degree"].cpu().numpy()
        nbr[g] = r["nbr_count"].cpu().numpy()
        assert r["halo"] > 20.0
        # owned rows of the union CSR equal the single-GPU rows
        rp = sym["row_ptr"].cpu().numpy()
        col = sym["col"].cpu().numpy()
        mine_rp = r["row_ptr"].cpu().numpy()
        mine_col = r["col"].cpu().numpy()
        for t in (0, len(g) // 2, len(g) - 1):
            assert np.array_equal(mine_col[mine_rp[t]:mine_rp[t + 1]], col[rp[g[t]]:rp[g[t] + 1]])
    assert np.array_equal(idx, ref_idx) and np.array_equal(dist, ref_d)
    assert np.array_equal(deg, comp["degree"].cpu().numpy()) and np.array_equal(nbr, comp["nbr_count"].cpu().numpy())
    edges = np.concatenate([r["edges"].cpu().numpy() for r in res])
    w = np.concatenate([r["weight"].cpu().numpy() for r in res])
    order = np.lexsort((edges[:, 1], edges[:, 0]))
    assert np.array_equal(edges[order], up["edges"].cpu().numpy()) and np.array_equal(w[order], up["w64"].cpu().numpy())


def test_sharded_with_ties_on_strip_edges(engine):
    # lattice points sitting exactly on strip boundaries and exact distance ties across strips
    gx, gy = np.meshgrid(np.arange(60.0) * 4.0, np.arange(40.0) * 4.0)
    xy = np.stack([gx.ravel(), gy.ravel()], axis=1)
    ty = (np.arange(len(xy)) % 5 + 1).astype(np.int32)
    n = len(xy)
    d_xy, d_ty, strips, parts = _split(xy, ty, 3, edges=[0.0, 80.0, 160.0, 236.0])
    engine.grid_build(d_xy, d_ty, None, radius_cell(8.0), None)
    ref = engine.radius_graph(8.0, upper=True, want_edges=True)
    res = sharding.run_emulated([sharding.sharded_radius_graph(engine, p[0], p[1], p[2], 8.0, s, q, 3)
                                 for q, (s, p) in enumerate(zip(strips, parts))])
    edges = np.concatenate([r["edges"].cpu().numpy() for r in res])
    order = np.lexsort((edges[:, 1], edges[:, 0]))
    assert np.array_equal(edges[order], ref["edges"].cpu().numpy())
    engine.grid_build(d_xy, d_ty, None, 6.0, None)
    kn = engine.knn(6, dist_dtype=torch.float64)
    res = sharding.run_emulated([sharding.sharded_knn_graph(engine, p[0], p[1], p[2], 6, s, q, 3, n_global=n, h0=5.0, union=False)
                                 for q, (s, p) in enumerate(zip(strips, parts))])
    idx = np.zeros((n, 6), dtype=np.int32)
    for r, p in zip(res, parts):
        idx[p[2].cpu().numpy()] = r["knn_idx"].cpu().numpy()
    assert np.array_equal(idx, kn["knn_idx"].cpu().numpy())      # (d^2, global id) tie-break survives sharding


def test_partition_kernel_equals_bucketize(engine):
    # pg_strip_partition against the torch expression it replaces (bucketize right=True + stable argsort)
    xy, ty, side = synth.make_points(70_001, seed=53)
    dev = torch.device("cuda", 0)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    gid = torch.arange(len(xy), dtype=torch.int32, device=dev) * 3 + 1
    for inner in ([], [float(side) / 2], [100.0, 100.0, 2500.5, float(side) - 1.0, float(side) + 5.0]):
        recs, totals = engine.strip_partition(d_xy, d_ty, gid, inner)
        owner = torch.bucketize(d_xy[:, 0].contiguous(), torch.tensor(inner, dtype=torch.float64, device=dev), right=True)
        order = torch.argsort(owner, stable=True)
        assert torch.equal(totals.long(), torch.bincount(owner, minlength=len(inner) + 1))
        assert torch.equal(recs[:, :2], d_xy[order])
        meta = recs[:, 2].contiguous().view(torch.int32).reshape(-1, 2)
        assert torch.equal(meta[:, 0], gid[order]) and torch.equal(meta[:, 1], d_ty[order])
    # the whole exchange, emulated: every point lands on the rank owning its strip, intact
    world = 3
    n = len(xy)
    chunks = [slice(q * n // world, (q + 1) * n // world) for q in range(world)]
    edges = np.array([0.0, side / 3, 2 * side / 3, float(side)])
    parts = sharding.run_emulated([sharding.partition_by_strips(engine, d_xy[c].contiguous(), d_ty[c].contiguous(),
                                                                gid[c].contiguous(), edges, q, world) for q, c in enumerate(chunks)])
    seen = torch.cat([p[2] for p in parts])
    assert torch.equal(torch.sort(seen).values, gid)
    for q, (pxy, pty, pgid) in enumerate(parts):
        assert bool(((pxy[:, 0] >= edges[q]) & ((pxy[:, 0] < edges[q + 1]) | (q == world - 1))).all())
        row = ((pgid - 1) // 3).long()
        assert torch.equal(pxy, d_xy[row]) and torch.equal(pty, d_ty[row])


def test_gid_maps(engine):
    dev = torch.device("cuda", 0)
    gid = torch.tensor([7, 2, 9, 0, 5], dtype=torch.int32, device=dev)
    ty = torch.tensor([1, 2, 3, 4, 5], dtype=torch.int32, device=dev)
    id_map, tbg = engine.gid_maps(gid, ty, n_rows=3, n_ids=11)
    assert id_map.tolist() == [-1, -1, 1, -1, -1, -1, -1, 0, -1, 2, -1]
    assert tbg.tolist() == [4, 0, 2, 0, 0, 5, 0, 1, 0, 3, 0]


def test_c5_full_size_sharded_equals_single(engine):
    """BASELINE config 5 at full size (20 M nuclei, k = 16, r = 50 px): four emulated ranks (one GPU, lockstep) go
    through equal-count strips, the all-to-all partition of a row-partitioned table and the halo exchange; the
    concatenated outputs must equal the single-GPU build bit for bit (size-independent property; scipy at this size
    takes minutes)."""
    world, n, k = 4, 20_000_000, 16
    xy, ty, side = synth.make_points(n, synth.SEEDS["C5"])
    dev = torch.device("cuda", 0)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    gid = torch.arange(n, dtype=torch.int32, device=dev)
    bounds = (0.0, 0.0, float(side), float(side))
    chunks = [slice(q * n // world, (q + 1) * n // world) for q in range(world)]
    edges = sharding.run_emulated([sharding.equal_count_edges(d_xy[c][:, 0].contiguous(), world, 0.0, float(side)) for c in chunks])[0]
    parts = sharding.run_emulated([sharding.partition_by_strips(engine, d_xy[c].contiguous(), d_ty[c].contiguous(), gid[c].contiguous(),
                                                                edges, q, world) for q, c in enumerate(chunks)])
    strips = sharding.strips_from_edges(edges)
    counts = [int(p[2].numel()) for p in parts]
    assert sum(counts) == n and max(counts) - min(counts) < n // 200          # equal-count strips
    # ---- radius graph
    res = sharding.run_emulated([sharding.sharded_radius_graph(engine, p[0], p[1], p[2], 50.0, s, q, world, bounds=bounds)
                                 for q, (s, p) in enumerate(zip(strips, parts))])
    engine.grid_build(d_xy, d_ty, None, radius_cell(50.0), bounds)
    ref = engine.radius_graph(50.0, upper=True, want_edges=True)
    e = torch.cat([r["edges"] for r in res])
    assert e.shape == ref["edges"].shape
    assert torch.equal(e[torch.argsort(e[:, 0] * n + e[:, 1])], ref["edges"])
    deg = torch.empty(n, dtype=torch.int32, device=dev)
    nbr = torch.empty((n, 5), dtype=torch.int32, device=dev)
    for r, p in zip(res, parts):
        deg[p[2].long()] = r["degree"]
        nbr[p[2].long()] = r["nbr_count"]
    assert torch.equal(deg, ref["degree"]) and torch.equal(nbr, ref["nbr_count"])
    del res, ref, e, deg, nbr
    torch.cuda.empty_cache()
    # ---- kNN lists + undirected union
    res = sharding.run_emulated([sharding.sharded_knn_graph(engine, p[0], p[1], p[2], k, s, q, world, n_global=n, bounds=bounds)
                                 for q, (s, p) in enumerate(zip(strips, parts))])
    engine.grid_build(d_xy, d_ty, None, default_knn_cell(n, float(side) ** 2, k), bounds)
    kn = engine.knn(k, dist_dtype=torch.float64)
    for r, p in zip(res, parts):
        g = p[2].long()
        assert torch.equal(r["knn_idx"], kn["knn_idx"][g]) and torch.equal(r["dist"], kn["dist"][g])
    un = engine.knn_union(kn["knn_idx"], kn["dist"], types=d_ty, n_types=5, symmetric_dist=True, hist_len=0)
    e = torch.cat([r["edges"] for r in res])
    w = torch.cat([r["weight"] for r in res])
    order = torch.argsort(e[:, 0] * n + e[:, 1])
    assert torch.equal(e[order], un["edges"]) and torch.equal(w[order], un["edge_w"])
    deg = torch.empty(n, dtype=torch.int32, device=dev)
    for r, p in zip(res, parts):
        deg[p[2].long()] = r["degree"]
    assert torch.equal(deg, un["degree"])
    # size-independent properties of the single-GPU result itself
    rp, col = un["row_ptr"].long(), un["col"]
    assert int(rp[-1]) == 2 * un["edges"].shape[0]                              # symmetric: every edge twice
    assert bool((kn["dist"][:, 1:] >= kn["dist"][:, :-1]).all())                # lists ascend by distance
    assert bool((un["edges"][:, 0] < un["edges"][:, 1]).all())


def test_spatial_sort_is_a_permutation_that_changes_nothing(engine):
    xy, ty, side = synth.make_points(80_000, seed=54)
    dev = torch.device("cuda", 0)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    gid = torch.arange(len(xy), dtype=torch.int32, device=dev)
    s_xy, s_ty, s_gid = sharding.spatial_sort(engine, d_xy, d_ty, gid, radius_cell(50.0))
    assert torch.equal(torch.sort(s_gid).values, gid)
    assert torch.equal(s_xy, d_xy[s_gid.long()]) and torch.equal(s_ty, d_ty[s_gid.long()])
    # the one-rank "sharded" builds over the sorted strip give the same graph, keyed by global id
    strip = sharding.Strip(0.0, float(side), True, True)
    comm = sharding.LocalComm()
    rg = sharding.run(sharding.sharded_radius_graph(engine, s_xy, s_ty, s_gid, 50.0, strip, 0, 1), comm)
    engine.grid_build(d_xy, d_ty, None, radius_cell(50.0), None)
    ref = engine.radius_graph(50.0, upper=True, want_edges=True)
    e = rg["edges"]
    assert torch.equal(e[torch.argsort(e[:, 0] * len(xy) + e[:, 1])], ref["edges"])
    deg = torch.empty(len(xy), dtype=torch.int32, device=dev)
    deg[s_gid.long()] = rg["degree"]
    assert torch.equal(deg, ref["degree"])
    kg = sharding.run(sharding.sharded_knn_graph(engine, s_xy, s_ty, s_gid, 8, strip, 0, 1, n_global=len(xy)), comm)
    engine.grid_build(d_xy, d_ty, None, default_knn_cell(len(xy), float(side) ** 2, 8), None)
    kn = engine.knn(8, dist_dtype=torch.float64)
    assert torch.equal(kg["knn_idx"], kn["knn_idx"][s_gid.long()]) and torch.equal(kg["dist"], kn["dist"][s_gid.long()])
    un = engine.knn_union(kn["knn_idx"], kn["dist"], types=d_ty, symmetric_dist=True)
    e = kg["edges"]
    assert torch.equal(e[torch.argsort(e[:, 0] * len(xy) + e[:, 1])], un["edges"])


def test_peer_slab_halo_equals_allgather_path(engine):
    """pg_halo_push / pg_halo_unpack_slab (the halo exchange over peer memory) against pg_halo_pack + all-gather +
    pg_halo_unpack_multi. Three emulated ranks on one GPU: the "peer" slabs are three local buffers, so the very same
    kernels run, only the stores do not cross NVLink (tests/multi_gpu_check.py with PG_PEER=1 is the real thing)."""
    world, n, cap, width = 3, 60_000, 8192, 40.0
    xy, ty, side = synth.make_points(n, 4242)
    dev = torch.device("cuda", 0)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    gid = torch.arange(n, dtype=torch.int32, device=dev)
    cuts = [0.0, side * 0.3, side * 0.55, float(side)]
    strips = sharding.strips_from_edges(cuts)
    own = [torch.nonzero((d_xy[:, 0] >= cuts[q]) & (d_xy[:, 0] < cuts[q + 1])).reshape(-1) for q in range(world)]
    parts = [(d_xy[o].contiguous(), d_ty[o].contiguous(), gid[o].contiguous()) for o in own]
    slab_bytes = world * cap * 24 + 8 * ((world * 4 + 7) // 8)
    slabs = [torch.zeros(slab_bytes, dtype=torch.uint8, device=dev) for _ in range(world)]
    ptrs = torch.tensor([s.data_ptr() for s in slabs], dtype=torch.int64, device=dev)
    inf = float("inf")
    for q, (s, p) in enumerate(zip(strips, parts)):
        engine.halo_push(p[0], p[1], p[2], -inf if s.is_first else s.lo + width, inf if s.is_last else s.hi - width,
                         ptrs.data_ptr(), world, q, cap)
    # reference path: pack + gather
    packed = []
    for q, (s, p) in enumerate(zip(strips, parts)):
        recs, cnt = engine.halo_pack(p[0], p[1], p[2], -inf if s.is_first else s.lo + width, inf if s.is_last else s.hi - width,
                                     capacity=int(p[0].shape[0]))
        packed.append(recs[:int(cnt.item())])
    max_cnt = max(int(r.shape[0]) for r in packed)
    assert 0 < max_cnt <= cap
    pad = torch.full((world, max_cnt, 3), float("nan"), dtype=torch.float64, device=dev)
    for q, r in enumerate(packed):
        pad[q, :r.shape[0]] = r
    for q, (s, p) in enumerate(zip(strips, parts)):
        ranges = [(-inf if s.is_first else s.lo - width / 2, inf if s.is_last else s.hi + width / 2),
                  (-inf if s.is_first else s.lo - width, -inf if s.is_first else s.lo - width / 2)]
        m = int(p[0].shape[0])
        a = [torch.empty((m + world * cap, 2), dtype=torch.float64, device=dev), torch.empty(m + world * cap, dtype=torch.int32, device=dev),
             torch.empty(m + world * cap, dtype=torch.int32, device=dev)]
        got = engine.halo_unpack_slab(slabs[q], world, q, cap, ranges, a[0], a[1], a[2], m).tolist()
        engine.check_overflow()
        want = sharding.merge_halo(engine, p[0], p[1], p[2], pad.reshape(world * max_cnt, 3).contiguous(), max_cnt, q, ranges)
        assert got == want[3] and sum(got) > 0
        at = m
        for c in got:                                       # same SET per range (append order inside a range is free)
            ga, gb = a[2][at:at + c], want[2][at:at + c]
            ia, ib = torch.argsort(ga), torch.argsort(gb)
            assert torch.equal(ga[ia], gb[ib]) and torch.equal(a[0][at:at + c][ia], want[0][at:at + c][ib])
            assert torch.equal(a[1][at:at + c][ia], want[1][at:at + c][ib])
            at += c
    # a slab that is too small is reported, on the packing side and on the receiving side
    tiny = [torch.zeros(world * 16 * 24 + 16, dtype=torch.uint8, device=dev) for _ in range(world)]
    tptr = torch.tensor([s.data_ptr() for s in tiny], dtype=torch.int64, device=dev)
    engine.halo_push(parts[1][0], parts[1][1], parts[1][2], strips[1].lo + width, strips[1].hi - width, tptr.data_ptr(), world, 1, 16)
    with pytest.raises(RuntimeError):
        engine.check_overflow()
    buf = [torch.empty((n, 2), dtype=torch.float64, device=dev), torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev)]
    engine.halo_unpack_slab(tiny[0], world, 0, 16, [(-inf, inf)], buf[0], buf[1], buf[2], 0)
    with pytest.raises(RuntimeError):
        engine.check_overflow()


def _meta(recs):
    """(gid, type) int32 columns of 24-byte halo records held as float64 [n, 3]."""
    m = recs[:, 2].contiguous().view(torch.int32).reshape(-1, 2)
    return m[:, 0], m[:, 1]


def test_halo_pack_past_capacity(engine):
    """pg_halo_pack with fewer slots than selected points: the count still counts every selected point, the overflow
    is reported once, and the slots that were written hold distinct selected points, intact. A NaN x is never packed."""
    dev = torch.device("cuda", 0)
    xy, ty, side = synth.make_points(20_000, seed=55)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    d_xy[::97, 0] = float("nan")
    gid = torch.arange(len(xy), dtype=torch.int32, device=dev) * 3 + 1
    lo_edge, hi_edge = side * 0.1, side * 0.9
    sel = (d_xy[:, 0] < lo_edge) | (d_xy[:, 0] >= hi_edge)
    n_sel, cap = int(sel.sum()), 500
    assert n_sel > 2 * cap
    engine.check_overflow()
    recs, count = engine.halo_pack(d_xy, d_ty, gid, lo_edge, hi_edge, capacity=cap)
    assert int(count.item()) == n_sel
    with pytest.raises(RuntimeError) as exc:
        engine.check_overflow()
    assert exc.value.code == -4
    engine.check_overflow()
    g, t = _meta(recs)
    assert torch.unique(g).numel() == cap
    row = ((g - 1) // 3).long()
    assert torch.equal(g, gid[row]) and bool(sel[row].all())
    assert torch.equal(recs[:, :2], d_xy[row]) and torch.equal(t, d_ty[row])
    # without gid / type: the gid is the row index and the type 0
    recs, count = engine.halo_pack(d_xy, None, None, lo_edge, hi_edge, capacity=n_sel)
    engine.check_overflow()
    g, t = _meta(recs)
    assert torch.equal(torch.sort(g).values, torch.nonzero(sel).reshape(-1).to(torch.int32)) and not bool(t.any())


_INF = float("inf")


def _gathered(engine, n_recs, seed):
    """Records of n_recs points (gid = row) in the layout of the all-gathered payload, every 13th a NaN padding row.
    Returns (recs, xy, types, side)."""
    dev = torch.device("cuda", 0)
    xy, ty, side = synth.make_points(n_recs, seed=seed)
    d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
    recs, count = engine.halo_pack(d_xy, d_ty, None, _INF, -_INF, capacity=n_recs)
    assert int(count.item()) == n_recs
    recs[::13] = float("nan")
    return recs, d_xy, d_ty, side


def test_halo_unpack_multi_skip_window(engine):
    """The records of [skip_begin, skip_end) (this rank's own) and NaN padding never land, in any range."""
    dev = torch.device("cuda", 0)
    n_recs, n_base, skip = 30_000, 1000, (9_000, 17_000)
    recs, d_xy, d_ty, side = _gathered(engine, n_recs, 56)
    ranges = [(side * 0.2, side * 0.6), (-_INF, side * 0.2), (side * 0.6, _INF)]
    cap = n_base + n_recs
    a = [torch.full((cap, 2), -1.0, dtype=torch.float64, device=dev), torch.full((cap,), -1, dtype=torch.int32, device=dev),
         torch.full((cap,), -1, dtype=torch.int32, device=dev)]
    engine.check_overflow()
    got = engine.halo_unpack_multi(recs, n_recs, skip[0], skip[1], ranges, a[0], a[1], a[2], n_base).tolist()
    engine.check_overflow()
    g_all = _meta(recs)[0]
    keep = ~torch.isnan(recs[:, 0])
    keep[skip[0]:skip[1]] = False
    assert sum(got) == int(keep.sum())
    assert bool((a[2][:n_base] == -1).all()) and bool((a[2][n_base + sum(got):] == -1).all())
    at = n_base
    for (lo, hi), c in zip(ranges, got):
        want = keep & (recs[:, 0] >= lo) & (recs[:, 0] < hi)
        assert c == int(want.sum())
        g = a[2][at:at + c]
        assert torch.equal(torch.sort(g).values, torch.sort(g_all[want]).values)
        assert torch.equal(a[0][at:at + c], d_xy[g.long()]) and torch.equal(a[1][at:at + c], d_ty[g.long()])
        at += c


def test_halo_unpack_multi_reports_a_small_destination(engine):
    dev = torch.device("cuda", 0)
    n_recs, n_base = 30_000, 100
    recs, _, _, side = _gathered(engine, n_recs, 57)
    cap = n_base + 1000
    a = [torch.empty((cap, 2), dtype=torch.float64, device=dev), torch.empty(cap, dtype=torch.int32, device=dev),
         torch.empty(cap, dtype=torch.int32, device=dev)]
    engine.check_overflow()
    engine.halo_unpack_multi(recs, n_recs, 0, 0, [(-_INF, side * 0.5), (side * 0.5, _INF)], a[0], a[1], a[2], n_base)
    with pytest.raises(RuntimeError) as exc:
        engine.check_overflow()
    assert exc.value.code == -4
