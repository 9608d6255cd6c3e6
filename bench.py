#!/usr/bin/env python
"""bench.py - nuclei/s of the radius-graph + neighbour-type composition + degree-statistics build on
a 1M-nucleus synthetic WSI (BASELINE.json configs[1], "C2"), per GPU, weak-scaled by slide over N GPUs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one slide:
  pg_grid_build (histogram, look-back scan, counting-sort scatter) -> pg_radius_graph (one neighbourhood walk with
  fused neighbour-type counts, then the row pass: row_ptr scan + degree statistics + gather of the parked entries:
  edges i<j, float32 distances).
`value`    : inputs resident in HBM, device time from CUDA events, L2 flushed between steps. The outputs are
             pre-sized (capacity = 1.25 E from one exact pass before the timed region), so a step is one enqueue with
             no host read; a caller who does not know E takes count -> total -> fill (one host sync, `e2e` below).
`e2e`      : the public call build_radius_graph(host coords, ..., outputs="compact") -> host arrays (H2D + kernels +
             D2H); `e2e_notebook` is the same call with the notebook's int64 edge_index / edge_attr tensors.
`roofline` : SURVEY 8(d) bytes of the step (48 N + 8 E_dir) over the dominant kernel's launch time (CUDA events
             inside the library, on its own stream); `roofline_step` the same bytes over the whole step;
             `roofline_sweep` the step at 250 k / 1 M / 4 M / 16 M nuclei.
`stages`   : other hot-path stages on one GPU and, with every --gpus N, the two multi-GPU workloads under this
             process's clock: `c5_strip_sharded` (20 M nuclei, k=16 and r=50, x-strips + NCCL halo all-gather,
             strong scaling, checksums against the single-GPU build) and `c4_cohort` (64 x 500 k nuclei slides from
             page-locked host tables, slide-parallel), plus the host-link ceiling measured with all ranks copying at once.
`cpu_baseline` / `--impl reference`: the notebook's scipy path (oracle/graph.py) on the host cores, full 1 M slide.
`--dump-outputs DIR`: rank 0 writes what the last timed step computed as DIR/<name>.npy (see last_step_outputs), so
that two builds run with the same arguments - same seeded inputs - can be compared output for output.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_NUCLEI = 1_000_000
RADIUS = 50.0
N_TYPES = 5
METRIC = "nuclei/s, kNN+radius graph+morphology, 1/2/4/8 B200; % of HBM peak"
WORKLOAD = "C2: 1M-nuclei WSI, radius graph r=50px + neighbour-type composition + degree stats"
FALLBACK_HBM_GBS = 6650.0


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/ncu_traffic.json)."""
    try:
        t = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
        return int(t["kernels"][kernel]["traffic"]), t["source"]
    except Exception:
        return None, None


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons of the first `n_gpus` GPUs, sampled every 50 ms by ONE process (rank 0's)
    while the timed regions (device-resident steps, then the end-to-end steps) run. It is started before the warm-up:
    the start-up of nvidia-smi takes driver locks that can stall kernel launches for milliseconds."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, n_gpus: int):
        self.n_gpus = n_gpus
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", ",".join(str(i) for i in range(self.n_gpus))],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict | None:
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in Path(self.path).read_text().splitlines():
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            return None
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU reference
def reference_pipeline(coords, types, r, n_types=N_TYPES):
    """The notebook's radius-graph path (cells 23-26) + numpy composition / degree. Returns n_edges."""
    from oracle import graph as ograph

    edges = ograph.radius_graph_notebook_loop(coords, r)            # cKDTree, query_ball_tree, i<j Python loop
    edge_index = np.vstack([edges.T, edges[:, ::-1].T])             # ipynb:3021 (as written)
    d = np.linalg.norm(coords[edges[:, 0]] - coords[edges[:, 1]], axis=1)
    edge_attr = np.concatenate([d[:, None], d[:, None]], axis=0).astype(np.float32)
    row_ptr, col, _ = ograph.symmetric_csr(edges, d, len(coords))
    ograph.composition(row_ptr, col, types, n_types)
    ograph.degree_stats(row_ptr)
    return len(edges), edge_index.shape, edge_attr.shape


def cpu_stage_timings():
    """SURVEY 8(d) timing protocol: the reference's CPU stages on the GPU box's host, on bounded samples of the
    BASELINE workloads (a few seconds each), next to the GPU numbers of the same run. kind = "port": the oracle's
    restatements (the reference function itself cannot travel to the GPU box; scipy / networkx are its own deps)."""
    import pandas as pd  # noqa: F401
    from scipy.spatial import cKDTree

    from oracle import graph as ograph
    from oracle import morphology as omorph
    from oracle import tile_to_wsi as omap
    from path_gene_multimodal_b200 import synth

    out = {"cores_available": len(os.sched_getaffinity(0)), "os_cpu_count": os.cpu_count()}

    def clock(fn):
        t0 = time.perf_counter()
        r = fn()
        return time.perf_counter() - t0, r

    # (i) a1-a3: add_wsi_coords_to_nuclei on a C1-style table (per-row Python loops, single-threaded by nature)
    n1 = 20_000
    tab = synth.make_table(n1, synth.SEEDS["C1"], dtype=np.float64)
    nuc, tiles = synth.to_frames(tab)
    dt, _ = clock(lambda: omap.add_wsi_coords_to_nuclei_oracle(nuc, tiles))
    out["add_wsi_coords_to_nuclei"] = {"nuclei_per_s": n1 / dt, "sample": f"{n1} nuclei of C1 (DataFrame in, DataFrame out)", "cores": 1}
    # (ii) a4-a5: per-polygon morphology (numpy restatement of the GEOS / moment formulas; shapely is absent)
    n2 = 200_000
    off, xy = synth.make_polygons(n2, synth.SEEDS["C3"], v_fixed=32)
    dt, _ = clock(lambda: omorph.polygon_features_csr(off, xy))
    out["polygon_morphology_numpy"] = {"polygons_per_s": n2 / dt, "sample": f"{n2} polygons x 32 vertices of C3 (vectorised numpy, no per-polygon GEOS object)", "cores": 1}
    # (iii) a6: cKDTree build + query(k+1), one worker and all workers
    n3 = 1_000_000
    c3, t3, _ = synth.make_points(n3, synth.SEEDS["C2"])
    dt_b, tree = clock(lambda: cKDTree(c3))
    dt1, _ = clock(lambda: tree.query(c3[:200_000], 9, workers=1))
    dta, _ = clock(lambda: tree.query(c3, 9, workers=-1))
    out["ckdtree_knn_k8"] = {"build_s": dt_b, "query_nuclei_per_s_1_worker": 200_000 / dt1, "query_nuclei_per_s_all_workers": n3 / dta,
                             "sample": "tree over the 1M-nuclei slide; 200k queries with workers=1, 1M with workers=-1"}
    # (iv) a7: the notebook's undirected-union loop (networkx has_edge / add_edge per directed edge)
    n4 = 50_000
    idx, dist = ograph.knn(c3[:n4], 8)
    dt, _ = clock(lambda: ograph.undirected_union_networkx(idx, dist))
    out["knn_union_networkx_loop"] = {"nuclei_per_s": n4 / dt, "sample": f"{n4} nuclei, k=8 (cell 11 loop)", "cores": 1}
    return out


def table_api_timings(device):
    """The a1-a3 drop-in through its two public entry points, end to end from HOST tables on one GPU: the reference's
    DataFrame format (one Python list per vertex in and out - the format, not the kernel, sets the pace) and the
    Arrow table (list<list<double>> = CSR buffers, no Python object per nucleus)."""
    import pyarrow as pa

    from path_gene_multimodal_b200 import add_wsi_coords_to_nuclei, add_wsi_coords_to_table, synth

    n = 50_000
    tab = synth.make_table(n, synth.SEEDS["C1"], dtype=np.float64)
    nuc, tiles = synth.to_frames(tab)
    tb = pa.Table.from_pandas(nuc, preserve_index=False)
    out = {}
    import functools

    for name, fn, arg in (("add_wsi_coords_to_nuclei(DataFrame)", add_wsi_coords_to_nuclei, nuc),
                          ("add_wsi_coords_to_nuclei(DataFrame, wsi_polygon_as='arrow')",
                           functools.partial(add_wsi_coords_to_nuclei, wsi_polygon_as="arrow"), nuc),
                          ("add_wsi_coords_to_table(Arrow)", add_wsi_coords_to_table, tb)):
        fn(arg, tiles, device=device)
        t0 = time.perf_counter()
        reps = 2 if "DataFrame" in name else 10
        for _ in range(reps):
            fn(arg, tiles, device=device)
        dt = (time.perf_counter() - t0) / reps
        out[name] = {"nuclei_per_s": n / dt, "ms": dt * 1e3, "sample": f"{n} nuclei of C1, host table in, host table out"}
    return out


def cpu_sample(n, seed):
    from path_gene_multimodal_b200 import synth

    xy, types, side = synth.make_points(n, seed)
    return xy, types, side


def run_reference(args, rank, world):
    """The reference's own CPU path on the SAME config as the GPU arm: the full 1M-nuclei slide every step."""
    if rank != 0:
        return
    n = N_NUCLEI
    xy, types, side = cpu_sample(n, 1002)
    n_edges = None
    for _ in range(args.warmup):
        n_edges = reference_pipeline(xy, types, RADIUS)[0]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        n_edges = reference_pipeline(xy, types, RADIUS)[0]
    dt = time.perf_counter() - t0
    val = n * args.steps / dt
    sample = (f"the full {n}-nuclei slide (seed 1002, r=50px) every step; scipy cKDTree.query_ball_tree + "
              "the notebook's i<j Python loop + np.linalg.norm + numpy composition/degree")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "nuclei/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nuclei_per_gpu": n, "nuclei_per_step": n, "radius_px": RADIUS, "n_types": N_TYPES,
                   "undirected_edges": int(n_edges) if n_edges is not None else None},
        "cpu_baseline": {"value": val, "unit": "nuclei/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": len(os.sched_getaffinity(0)),
                         "note": "query_ball_tree has no workers parameter and the edge loop is GIL-bound: 1 thread is all it can use"},
        "e2e": {"value": val, "unit": "nuclei/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ ours
def algorithmic_bytes(n, e_dir):
    """SURVEY 8(d): radius + composition + degree = 48 N + 8 E_dir bytes (E_dir = 2 E_und)."""
    return 48 * n + 8 * e_dir


def kernel_bytes(name, n, e_und, cells):
    """Compulsory bytes of one launch of each kernel (its own inputs read once + outputs written once)."""
    table = {
        "histogram_kernel": 16 * n + 4 * cells,                       # xy in; cell counters
        "scan_kernel": 8 * cells,                                     # counters in, cell starts out
        "scatter_kernel": 16 * n + 4 * n + 4 * cells + 32 * n,        # xy, type, cursors in; 32-byte records out
        "radius_walk_kernel": 32 * n + 4 * cells + 32 * n + 16 * e_und,  # records, cell starts in; per-point meta + parked entries out
        "radius_rows_kernel": 32 * n + 4 * n + 4 * n + 4 * N_TYPES * n + 4 * n,  # meta in; row_ptr, degree, nbr_count, row_off out
        "radius_rows_gather_kernel": 32 * n + 4 * n + 4 * n + 4 * N_TYPES * n + 16 * e_und + 24 * e_und,  # meta, entries in; row_ptr, degree, nbr_count, col, dist32, edges out
        "radius_gather_kernel": 8 * n + 16 * e_und + 4 * e_und + 4 * e_und + 16 * e_und,  # row_ptr, row_off, entries in; col, dist32, edges out
    }
    return table.get(name)


class C2Slide:
    """One slide of the C2 workload resident on the device, with pre-sized outputs: step() = one pass of the hot path."""

    def __init__(self, eng, dev, n, seed):
        import torch

        from path_gene_multimodal_b200 import synth
        from path_gene_multimodal_b200.engine import radius_cell

        self.eng, self.n = eng, n
        self.xy_np, self.types_np, side = synth.make_points(n, seed)
        self.bounds = (0.0, 0.0, float(side), float(side))
        self.d_xy = torch.from_numpy(self.xy_np).to(dev)
        self.d_ty = torch.from_numpy(self.types_np).to(dev)
        self.cell = radius_cell(RADIUS)
        eng.grid_build(self.d_xy, self.d_ty, None, self.cell, self.bounds)
        g0 = eng.radius_graph(RADIUS, upper=True, n_types=N_TYPES, want_edges=True)   # exact pass: E for the byte counts
        self.e_und = int(g0["total"])
        info = eng.grid_info()
        self.cells = info["nx"] * info["ny"]
        self.cap = int(self.e_und * 1.25) + 1024
        self.out = {}

    def step(self):
        self.eng.grid_build(self.d_xy, self.d_ty, None, self.cell, self.bounds)
        self.out = self.eng.radius_graph(RADIUS, upper=True, n_types=N_TYPES, want_dist32=True, want_edges=True,
                                         capacity=self.cap, out=self.out)


DUMP_ROWS = 1 << 18       # rows kept of each per-nucleus / per-edge output: ~25 MB of .npy for the 1 M slide
DUMP_MAX_BYTES = 64 * 10**6


def last_step_outputs(slide):
    """Host copies of what a C2 step hands its caller: the per-nucleus outputs (degree, nbr_count, upper-CSR row_ptr),
    the valid prefix of the pre-sized per-edge outputs (edges, col, float32 dist; row_ptr[-1] entries) and the degree
    statistics. Indices and counts are stored as float64 (exact), dist as float32. Outputs longer than DUMP_ROWS rows
    keep a fixed seeded sample of rows (node_rows / edge_rows, stored too); the sample depends only on N and E."""
    import torch

    from path_gene_multimodal_b200.engine import Engine

    o = slide.out
    n_edges = int(o["row_ptr"][-1])
    rng = np.random.default_rng(0)

    def rows(count):
        return np.arange(count) if count <= DUMP_ROWS else np.sort(rng.choice(count, DUMP_ROWS, replace=False))

    node_rows, edge_rows = rows(slide.n), rows(n_edges)
    ni = torch.from_numpy(node_rows).to(o["row_ptr"].device)
    ei = torch.from_numpy(edge_rows).to(o["row_ptr"].device)

    def f64(t):
        return t.cpu().numpy().astype(np.float64)

    st = Engine.decode_stats(o["stats"], o["hist"])
    return {
        "node_rows": node_rows.astype(np.float64), "degree": f64(o["degree"][ni]), "nbr_count": f64(o["nbr_count"][ni]),
        "row_ptr": f64(o["row_ptr"][ni]),
        "edge_rows": edge_rows.astype(np.float64), "edges": f64(o["edges"][ei]), "col": f64(o["col"][ei]),
        "dist": o["dist32"][ei].cpu().numpy(),
        "n_edges": np.array([n_edges], dtype=np.float64),
        "degree_stats": np.array([st["min"], st["max"], st["sum"], st["sumsq"], st["n"]], dtype=np.float64),
        "degree_hist": st["hist"].astype(np.float64),
    }


def write_outputs(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"output dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    for name, a in arrays.items():
        np.save(Path(out_dir) / f"{name}.npy", a)


def timed_steps(fn, flush, steps, warmup):
    """CUDA-event time of each of `steps` calls of fn, the L2 flushed (512 MB written) before every one."""
    import torch

    for _ in range(warmup):
        flush.zero_()
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def link_ceiling(dev, dist, mb=64, reps=8):
    """Pinned host <-> device copies with EVERY rank copying at the same time (one cudaMemcpyAsync per buffer): what
    the host's PCIe / memory system gives each GPU when all of them are fed at once. GB/s per rank."""
    import torch

    from path_gene_multimodal_b200 import _host

    nb = mb * 1000 * 1000
    h_in = torch.from_numpy(_host.pinned_empty((nb,), np.uint8))
    h_out = torch.from_numpy(_host.pinned_empty((nb,), np.uint8))
    d_a = torch.empty(nb, dtype=torch.uint8, device=dev)
    d_b = torch.empty(nb, dtype=torch.uint8, device=dev)
    side = torch.cuda.Stream(dev)
    out = {}
    for name in ("h2d", "d2h", "both"):
        for i in range(2):  # untimed
            d_a.copy_(h_in, non_blocking=True)
            h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        side.wait_event(e0)
        for _ in range(reps):
            if name in ("h2d", "both"):
                d_a.copy_(h_in, non_blocking=True)
            if name == "d2h":
                h_out.copy_(d_b, non_blocking=True)
            if name == "both":
                with torch.cuda.stream(side):
                    h_out.copy_(d_b, non_blocking=True)
        torch.cuda.current_stream().wait_stream(side)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        out[name + "_GBs_per_rank"] = nb * reps * (2 if name == "both" else 1) / ms / 1e6
    out["buffer_MB"] = mb
    return out


def iter_value(v):
    """A generator that yields no collective and returns v (so that a plain call fits the sharding.run driver)."""
    return v
    yield  # noqa: unreachable - makes this a generator


def checksum_edges(e):
    return int((e[:, 0] * 1000003 + e[:, 1]).sum().item()) if e.numel() else 0


def c5_stage(eng, dev, dist, rank, world, n=20_000_000, k=16, reps=3):
    """BASELINE config 5: one 20M-nuclei slide, radius r=50 graph and kNN k=16 + undirected union, strip-sharded over
    the ranks (equal-count x-strips, all-to-all partition of the row-partitioned table, ONE halo all-gather per build).
    Strong scaling: the slide is fixed. Device time (CUDA events, max over ranks) of partition / radius / kNN builds;
    order-independent checksums of every output are compared with the single-GPU build of the whole slide (rank 0)."""
    import torch

    from path_gene_multimodal_b200 import sharding, synth
    from path_gene_multimodal_b200.engine import default_knn_cell, radius_cell

    xy, ty, side = synth.make_points(n, synth.SEEDS["C5"])
    bounds = (0.0, 0.0, float(side), float(side))
    comm = sharding.TorchComm() if world > 1 else sharding.LocalComm()
    rows = slice(rank * n // world, (rank + 1) * n // world)           # the table starts row-partitioned
    l_xy, l_ty = torch.from_numpy(xy[rows]).to(dev), torch.from_numpy(ty[rows]).to(dev)
    l_gid = torch.arange(rows.start, rows.stop, dtype=torch.int32, device=dev)

    def timed(make):
        best, res = None, None
        for i in range(reps + 1):                                          # run 0 is untimed (allocations)
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = sharding.run(make(), comm)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if dist is not None:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            if i > 0:
                best = ms if best is None else min(best, ms)
        return res, best

    out = {"nuclei": n, "k": k, "radius_px": RADIUS, "world": world}
    if world > 1:
        edges, t_edges = timed(lambda: sharding.equal_count_edges(l_xy[:, 0].contiguous(), world, 0.0, float(side)))
        part, t_part = timed(lambda: sharding.partition_by_strips(eng, l_xy, l_ty, l_gid, edges, rank, world))
        s_xy, s_ty, s_gid = part
        strip = sharding.strips_from_edges(edges)[rank]
        out["partition_ms"] = t_edges + t_part
    else:
        s_xy, s_ty, s_gid = l_xy, l_ty, l_gid
        strip = sharding.Strip(0.0, float(side), True, True)
        out["partition_ms"] = 0.0
    del l_xy, l_ty
    if os.environ.get("PG_C5_SORT", "1") != "0":
        # the strip keeps its points in cell order (rows are keyed by global id, so the order is the strip's own business)
        (s_xy, s_ty, s_gid), t_sort = timed(lambda: iter_value(sharding.spatial_sort(eng, s_xy, s_ty, s_gid, radius_cell(RADIUS), bounds)))
        out["partition_ms"] += t_sort
        out["spatial_sort_ms"] = t_sort
    slot = torch.arange(1, k + 1, device=dev, dtype=torch.int64)

    def builds(peer):
        """both sharded builds (timed) -> order-independent checksums of this rank's outputs"""
        rg, t_r = timed(lambda: sharding.sharded_radius_graph(eng, s_xy, s_ty, s_gid, RADIUS, strip, rank, world, bounds=bounds, peer=peer))
        sm = {"radius_edges": int(rg["edges"].shape[0]), "radius_edge_hash": checksum_edges(rg["edges"]),
              "radius_degree_hash": int(((s_gid.long() + 1) * rg["degree"].long()).sum().item()),
              "radius_nbr_hash": int(((s_gid.long() + 1)[:, None] * rg["nbr_count"].long()).sum().item())}
        del rg
        kg, t_k = timed(lambda: sharding.sharded_knn_graph(eng, s_xy, s_ty, s_gid, k, strip, rank, world, n_global=n, bounds=bounds, peer=peer))
        sm.update({"knn_idx_hash": int((((s_gid.long() + 1)[:, None] * 31 + slot[None, :]) * (kg["knn_idx"].long() + 1)).sum().item()),
                   "knn_dist_hash": int(((kg["dist"].view(torch.int64) >> 11) * slot[None, :]).sum().item()),
                   "union_edges": int(kg["edges"].shape[0]), "union_edge_hash": checksum_edges(kg["edges"]),
                   "union_weight_hash": int((kg["weight"].view(torch.int64) >> 11).sum().item()),
                   "union_degree_hash": int(((s_gid.long() + 1) * kg["degree"].long()).sum().item())})
        return sm, t_r, t_k, kg["halo"], kg["n_ghost"]

    sums, t_rad, t_knn, halo, ghosts = builds(None)
    # the exchange step of the kNN build alone (pack kernel + the two all-gathers + the host read of the counts)
    t_halo = timed(lambda: sharding.exchange_halo(eng, s_xy, s_ty, s_gid, strip, 2.0 * halo, rank, world))[1] if world > 1 else 0.0
    out["halo_path"] = "nccl all-gather" if world > 1 else "none (one rank)"
    if world > 1 and os.environ.get("PG_C5_PEER", "1") != "0":
        # the same two builds with the halo exchange as one pack+store kernel over NVLink peer memory (sharding.PeerHalo);
        # taken as the stage's time only if every rank reproduces the NCCL path's checksums
        try:
            peer = sharding.PeerHalo(int(os.environ.get("PG_C5_PEER_CAP", 262144)), dev)
            ok_t = torch.ones((1,), device=dev, dtype=torch.int32)
        except Exception as exc:                                           # symmetric memory unavailable on this box
            peer, ok_t = None, torch.zeros((1,), device=dev, dtype=torch.int32)
            out["peer_memory_error"] = repr(exc)[:200]
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
        if int(ok_t.item()) == 1:
            p_sums, p_rad, p_knn, _, _ = builds(peer)
            same = torch.tensor([int(p_sums == sums)], device=dev, dtype=torch.int32)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            ranges = [(strip.lo - 2 * halo, strip.hi + 2 * halo)]
            p_halo = timed(lambda: iter_value(peer.exchange(eng, s_xy, s_ty, s_gid, strip, 2.0 * halo, ranges)))[1]
            out["nvlink_peer_halo"] = {"radius_ms": p_rad, "knn_union_ms": p_knn, "halo_exchange_and_merge_ms": p_halo,
                                       "identical_to_nccl_path": bool(same.item()), "slab_records_per_rank": peer.cap,
                                       "nccl_path": {"radius_ms": t_rad, "knn_union_ms": t_knn, "halo_exchange_ms": t_halo}}
            if bool(same.item()) and p_rad + p_knn < t_rad + t_knn:
                t_rad, t_knn = p_rad, p_knn
                out["halo_path"] = "pg_halo_push over NVLink peer memory (pack + all-gather in one kernel)"
        del peer
    torch.cuda.empty_cache()
    keys = sorted(sums)
    vec = torch.tensor([sums[q] for q in keys], dtype=torch.int64, device=dev)
    if dist is not None:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)        # int64 sums wrap the same way on every world size
    total = dict(zip(keys, vec.tolist()))
    out.update({"radius_ms": t_rad, "knn_union_ms": t_knn, "total_ms": out["partition_ms"] + t_rad + t_knn,
                "nuclei_per_s": n / ((t_rad + t_knn) / 1e3), "halo_px": halo, "ghosts_rank0": ghosts, "halo_exchange_ms": t_halo,
                "radius_edges": total["radius_edges"], "union_edges": total["union_edges"],
                "timing": "CUDA events around each sharded build (halo exchange, host reads of counts included), max over ranks, best of %d" % reps})
    if rank == 0:
        if world > 1:
            # single-GPU build of the whole slide: the checksums every world size must reproduce
            d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
            gid = torch.arange(n, dtype=torch.int64, device=dev)
            eng.grid_build(d_xy, d_ty, None, radius_cell(RADIUS), bounds)
            ref = eng.radius_graph(RADIUS, upper=True, n_types=N_TYPES, want_edges=True)
            want = {"radius_edges": int(ref["edges"].shape[0]), "radius_edge_hash": checksum_edges(ref["edges"]),
                    "radius_degree_hash": int(((gid + 1) * ref["degree"].long()).sum().item()),
                    "radius_nbr_hash": int(((gid + 1)[:, None] * ref["nbr_count"].long()).sum().item())}
            del ref
            eng.grid_build(d_xy, d_ty, None, default_knn_cell(n, float(side) ** 2, k), bounds)
            kn = eng.knn(k, dist_dtype=torch.float64)
            want.update({"knn_idx_hash": int((((gid + 1)[:, None] * 31 + slot[None, :]) * (kn["knn_idx"].long() + 1)).sum().item()),
                         "knn_dist_hash": int(((kn["dist"].view(torch.int64) >> 11) * slot[None, :]).sum().item())})
            un = eng.knn_union(kn["knn_idx"], kn["dist"], types=d_ty, n_types=N_TYPES, symmetric_dist=True, hist_len=0)
            want.update({"union_edges": int(un["edges"].shape[0]), "union_edge_hash": checksum_edges(un["edges"]),
                         "union_weight_hash": int((un["edge_w"].view(torch.int64) >> 11).sum().item()),
                         "union_degree_hash": int(((gid + 1) * un["degree"].long()).sum().item())})
            del un, kn, d_xy, d_ty
            torch.cuda.empty_cache()
            bad = [q for q in keys if total[q] != want[q]]
            out["bit_identical_to_single_gpu"] = not bad
            if bad:
                out["mismatch"] = bad
        else:
            out["bit_identical_to_single_gpu"] = True   # this IS the single-GPU build
        out["checksums"] = {q: total[q] for q in ("radius_edge_hash", "union_edge_hash", "knn_idx_hash")}
    return out


def c4_stage(dev, local_rank, dist, rank, world, n_slides=64, n=500_000, lanes=4, staging="float"):
    """BASELINE config 4: 64 slides x 500k nuclei from page-locked HOST tables, slide-parallel over the ranks
    (sharding.assign_slides), `lanes` slides in flight per GPU. Device time between the first enqueue and the last
    completion, max over ranks; the digest of all per-slide summaries must not depend on the number of GPUs."""
    import torch

    from path_gene_multimodal_b200 import cohort, sharding, synth

    mine = sharding.assign_slides(n_slides, world, sizes=[n] * n_slides)[rank]
    cache, tables = {}, {}
    for sl in mine:
        tables[sl] = cohort.pin_table(synth.make_cohort_slide(sl, n), cache, staging=staging)
    runner = cohort.CohortRunner(local_rank, lanes=lanes)
    runner.run(mine[:lanes], tables.__getitem__)                        # warm-up: allocations, first launches
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    res, ms = runner.run(mine, tables.__getitem__)
    runner.close()
    h2d = sum(cohort.table_bytes(tables[sl]) for sl in mine)
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        res = {}
        for d in gathered:
            res.update(d)
    assert sorted(res) == list(range(n_slides))
    return {"slides": n_slides, "nuclei_per_slide": n, "world": world, "lanes": lanes, "ms": ms,
            "nuclei_per_s": n_slides * n / (ms / 1e3), "ms_per_slide_per_gpu": ms / max(len(mine), 1),
            "h2d_bytes_per_slide": h2d // max(len(mine), 1), "digest": cohort.cohort_checksum(res),
            "polygon_staging": "float32 pixels (8 B / vertex)" if staging == "float" else "int16 half-pixels (4 B / vertex), widened on the device",
            "note": "slides dealt from 4 base tables (synth.make_cohort_slide); every slide = H2D of its table + map + morphology "
                    "+ kNN-8 union + radius-50 graph + summary read; CUDA events, max over ranks"}


def run_ours(args, rank, world, local_rank):
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    from path_gene_multimodal_b200 import _host, build_radius_graph, synth
    from path_gene_multimodal_b200.engine import get_engine

    eng = get_engine(local_rank)
    peak, peak_src = measured_peak()
    n = N_NUCLEI
    slide = C2Slide(eng, dev, n, synth.SEEDS["C2"] + rank)              # one slide per rank (weak scaling)
    e_und, cells = slide.e_und, slide.cells
    h_xy = _host.pinned_empty((n, 2), np.float64); h_xy[...] = slide.xy_np   # pinned host copies: the e2e input
    h_ty = _host.pinned_empty((n,), np.int32); h_ty[...] = slide.types_np
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    sampler = ClockSampler(world)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    slide.step()
    launches_per_step = eng.launches - l0
    # the step replayed as ONE CUDA graph (same five kernels, same programmatic-dependent-launch edges): host jitter
    # between the launches of a step (8 ranks + a sampler on one VM) cannot open gaps inside the timed region
    try:
        graph = eng.capture(slide.step)
        run_step, how = graph.replay, "one CUDA graph replay per step (5 kernels, programmatic dependent launch edges kept)"
    except Exception as exc:  # noqa: BLE001
        run_step, how = slide.step, f"eager launches (graph capture failed: {type(exc).__name__})"
    timed_steps(run_step, flush, 0, warm)
    eng.check_overflow()
    barrier()
    step_ms = timed_steps(run_step, flush, args.steps, 0)
    barrier()
    dump = last_step_outputs(slide) if args.dump_outputs and rank == 0 else None
    launches = launches_per_step * args.steps
    eng.check_overflow()
    total_ms = float(sum(step_ms))
    assert int(slide.out["row_ptr"][-1]) == e_und
    if dist is not None:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * n * args.steps / (total_ms / 1e3)

    # ---- e2e: public host API, pinned host inputs, H2D + kernels + D2H inside the timed region
    def e2e(outputs, count_dtype=np.int32):
        res = None
        kw = {"count_dtype": count_dtype} if outputs == "compact" else {}
        for _ in range(3):
            res = build_radius_graph(h_xy, r=RADIUS, types=h_ty, n_types=N_TYPES, bounds=slide.bounds, device=local_rank, outputs=outputs, **kw)
        assert res["edges"].shape[0] == e_und
        barrier()
        steps = max(3, min(args.steps, 20))
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = build_radius_graph(h_xy, r=RADIUS, types=h_ty, n_types=N_TYPES, bounds=slide.bounds, device=local_rank, outputs=outputs, **kw)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        wall = (time.perf_counter() - t0) * 1e3
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        if outputs == "compact":
            d2h = res["edges"].nbytes + res["dist"].nbytes + res["degree"].nbytes + res["nbr_count"].nbytes + 32 + 64 * 4 + 4
        else:
            d2h = res["edge_index"].nbytes + res["edge_attr"].nbytes + res["degree"].nbytes + res["nbr_count"].nbytes + 32 + 64 * 4
        return {"value": world * n * steps / (ms / 1e3), "unit": "nuclei/s", "h2d_bytes_per_step": int(h_xy.nbytes + h_ty.nbytes),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": ms / steps, "wall_ms_per_step": wall / steps, "steps": steps}

    e2e_c = e2e("compact", np.uint8)
    e2e_c["api"] = ("path_gene_multimodal_b200.build_radius_graph(host coords, r, types, outputs='compact', count_dtype=uint8) -> host edges "
                    "int32 [E,2] / dist float32 [E] / degree uint8 [N] / nbr_count uint8 [N,5] / degree_stats")
    e2e_c32 = e2e("compact")
    e2e_c32["api"] = "the same call with int32 degree / nbr_count"
    e2e_n = e2e("notebook")
    e2e_n["api"] = "the same call with outputs='notebook': host edge_index int64 [2,2E] / edge_attr float32 [2E,1] / degree / nbr_count"
    clocks = sampler.stop() if rank == 0 else None
    if dump is not None:
        write_outputs(args.dump_outputs, dump)

    line = {
        "metric": METRIC, "value": value, "unit": "nuclei/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nuclei_per_gpu": n, "nuclei_per_step": n, "radius_px": RADIUS, "n_types": N_TYPES,
                   "undirected_edges": e_und, "grid_cells": cells, "parallelism": f"slide-parallel x{world} (one slide per GPU, no data-path collective)",
                   "l2": "512 MB buffer written between timed steps (L2 flush)", "timing": "CUDA events per step, summed, max over ranks",
                   "launch": how,
                   "outputs": "pre-sized (capacity 1.25 E from one exact pass before the timed region): a step is one enqueue, no host read; "
                              "callers without E take count -> total -> fill (see e2e)"},
        "clocks": clocks, "e2e": e2e_c, "e2e_compact_int32_counts": e2e_c32, "e2e_notebook": e2e_n, "gpu_launches": int(launches),
    }

    # ---- host-link ceiling with every rank copying at once, then e2e as a fraction of it
    link = link_ceiling(dev, dist)
    floor_ms = (e2e_c["h2d_bytes_per_step"] / link["h2d_GBs_per_rank"] + e2e_c["d2h_bytes_per_step"] / link["d2h_GBs_per_rank"]) / 1e6
    line["host_link"] = dict(link, e2e_copy_floor_ms=floor_ms, e2e_frac_of_copy_floor=floor_ms / e2e_c["ms_per_step"],
                             note="pinned cudaMemcpyAsync, all ranks at once; e2e_copy_floor = this step's H2D + D2H bytes at those rates, "
                                  "one after the other as the call issues them")

    # ---- the two multi-GPU workloads of BASELINE configs[3..4] under this process's clock
    stages_mg = {}
    del flush
    torch.cuda.empty_cache()
    try:
        stages_mg["c5_strip_sharded"] = c5_stage(eng, dev, dist, rank, world)
    except Exception as exc:  # noqa: BLE001 - the headline line must still be printed
        stages_mg["c5_strip_sharded"] = {"error": f"{type(exc).__name__}: {exc}"}
    torch.cuda.empty_cache()
    try:
        # the cohort twice: polygons staged as float32 pixels and as int16 half-pixels (the lattice find_contours emits);
        # the second is the stage's figure only if its digest equals the first's
        c4_f = c4_stage(dev, local_rank, dist, rank, world)
        torch.cuda.empty_cache()
        c4_h = c4_stage(dev, local_rank, dist, rank, world, staging="halfpx16")
        same = c4_h["digest"] == c4_f["digest"]
        c4_h["digest_equals_float32_staging"] = same
        stages_mg["c4_cohort"] = c4_h if same else c4_f
        stages_mg["c4_cohort_float32_tables"] = c4_f
    except Exception as exc:  # noqa: BLE001
        stages_mg["c4_cohort"] = {"error": f"{type(exc).__name__}: {exc}"}
    torch.cuda.empty_cache()
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)

    if rank == 0:
        # ---- per-kernel timing inside the library (CUDA events on the launching stream), L2 flushed
        eng.profile(True)
        reps = 10
        for _ in range(reps):
            flush.zero_()
            slide.step()
        recs = eng.profile_records()
        eng.profile(False)
        per = {}
        for name, ms in recs:
            per.setdefault(name, []).append(ms)
        avg = {k: sum(v) / len(v) for k, v in per.items()}
        share = {k: sum(v) / reps for k, v in per.items()}  # ms per step
        dom = max(share, key=share.get)
        step_sum = sum(share.values())
        alg = algorithmic_bytes(n, 2 * e_und)
        line["kernels_ms_per_step"] = {k: round(v, 5) for k, v in sorted(share.items(), key=lambda kv: -kv[1])}
        ach = alg / (avg[dom] / 1e3) / 1e9
        traffic, traffic_src = ncu_traffic(dom)
        kb = kernel_bytes(dom, n, e_und, cells)
        line["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "traffic": traffic, "traffic_source": traffic_src,
                            "algorithmic_bytes_per_launch": int(alg), "avg_launch_ms": avg[dom],
                            "share_of_step": share[dom] / step_sum, "peak_source": peak_src,
                            "kernel_own_bytes_per_launch": int(kb) if kb else None,
                            "kernel_own_frac": (kb / (avg[dom] / 1e3) / 1e9 / peak) if kb else None,
                            "note": "SURVEY 8(d): achieved = the step's algorithmic bytes (48 N + 8 E_dir: every boundary array once) over the "
                                    "dominant kernel's launch time; kernel_own_* = that kernel's own inputs + outputs (intermediates included) "
                                    "over the same time. The kernel is issue / L2-latency bound (ncu: ~60 % issue, DRAM 10 %), not DRAM bound"}
        ach_step = alg / (total_ms / args.steps / 1e3) / 1e9
        line["roofline_step"] = {"bound": "hbm", "achieved": ach_step, "peak": peak, "unit": "GB/s", "frac": ach_step / peak,
                                 "algorithmic_bytes_per_step": int(alg), "bytes_per_nucleus": alg / n,
                                 "note": "SURVEY 8(d): 48 N + 8 E_dir over the whole step (all kernels + launch gaps)"}
        # ---- the same step at other slide sizes (same density): where the fraction saturates
        sweep = {}
        for nn in (250_000, 1_000_000, 4_000_000, 16_000_000):
            sl = slide if nn == n else C2Slide(eng, dev, nn, synth.SEEDS["C2"])
            ms = statistics.median(timed_steps(sl.step, flush, 8, 3))
            a = algorithmic_bytes(nn, 2 * sl.e_und)
            sweep[str(nn)] = {"ms_per_step": ms, "undirected_edges": sl.e_und, "nuclei_per_s": nn / ms * 1e3,
                              "achieved_GBs": a / ms / 1e6, "frac": a / ms / 1e6 / peak}
            if sl is not slide:
                del sl
                torch.cuda.empty_cache()
        line["roofline_sweep"] = sweep
        line["stages"] = dict(other_stages(eng, dev, flush, peak), **stages_mg)
        if world == 1:
            t0 = time.perf_counter()
            ne, _, _ = reference_pipeline(slide.xy_np, slide.types_np, RADIUS)
            dt = time.perf_counter() - t0
            assert ne == e_und
            line["cpu_baseline"] = {
                "value": n / dt, "unit": "nuclei/s", "cores": 1, "kind": "port",
                "sample": "the full 1M-nuclei slide once: scipy cKDTree + query_ball_tree + the notebook's i<j Python loop + "
                          "np.linalg.norm + numpy composition/degree (oracle/graph.py); same edges as the GPU run",
                "seconds": dt, "host_cores_available": len(os.sched_getaffinity(0))}
            line["cpu_stages"] = cpu_stage_timings()
            line["table_api_e2e"] = table_api_timings(local_rank)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def other_stages(eng, dev, flush, peak):
    """Device-resident timings of the other hot-path stages (informational; not the headline)."""
    import torch

    from path_gene_multimodal_b200 import synth
    from path_gene_multimodal_b200.engine import default_knn_cell, radius_cell

    def timed(fn, reps=5):
        ms = []
        for i in range(reps + 2):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ms.append(e0.elapsed_time(e1))
        return statistics.median(ms)

    out = {}
    # C3: 2M polygons x 32 vertices, fused tile->WSI shift + morphology, float32 vertices
    n3 = 2_000_000
    off, xy = synth.make_polygons(n3, synth.SEEDS["C3"], v_fixed=32)
    rng = np.random.default_rng(3)
    side = 73
    tile_x = torch.from_numpy(((np.arange(side * side) % side) * 508).astype(np.int32)).to(dev)
    tile_y = torch.from_numpy(((np.arange(side * side) // side) * 508).astype(np.int32)).to(dev)
    nuc_tile = torch.from_numpy(rng.integers(0, side * side, size=n3).astype(np.int32)).to(dev)
    cen = torch.from_numpy(rng.random((n3, 2)) * 508).to(dev)
    bb = torch.from_numpy(rng.integers(0, 508, size=(n3, 4)).astype(np.int32)).to(dev)
    d_off, d_xy = torch.from_numpy(off).to(dev), torch.from_numpy(xy).to(dev)
    res = {}

    def morph():
        nonlocal res
        res = eng.map_morph(d_off, d_xy, nuc_tile, tile_x, tile_y, cen, bb, write_polygons=True, out=res)

    ms = timed(morph)
    m = int(xy.shape[0])
    b3 = 16 * m + 84 * n3
    out["C3_map_morph_2Mx32_f32"] = {"ms": ms, "polygons_per_s": n3 / ms * 1e3, "algorithmic_bytes": b3,
                                     "achieved_GBs": b3 / ms / 1e6, "frac_of_peak": b3 / ms / 1e6 / peak}
    del d_xy, res, cen, bb
    # C1-style kNN k=8 + undirected union + composition on the 1M slide
    xy1, ty1, side1 = synth.make_points(N_NUCLEI, synth.SEEDS["C2"])
    dx, dt_ = torch.from_numpy(xy1).to(dev), torch.from_numpy(ty1).to(dev)
    cellk = default_knn_cell(N_NUCLEI, float(side1) ** 2, 8)
    kres = {}

    def knn():
        nonlocal kres
        eng.grid_build(dx, dt_, None, cellk, (0.0, 0.0, float(side1), float(side1)))
        kres = eng.knn(8, dist_dtype=torch.float32, out=kres)

    ms = timed(knn)
    out["knn_k8_1M_grid+query"] = {"ms": ms, "nuclei_per_s": N_NUCLEI / ms * 1e3}

    def knn_union():
        knn()
        eng.knn_union(kres["knn_idx"], kres["dist32"], types=dt_, n_types=N_TYPES, want_edges=False, symmetric_dist=True)

    ms = timed(knn_union, reps=3)
    out["knn_k8_1M_full(grid+query+union+composition)"] = {"ms": ms, "nuclei_per_s": N_NUCLEI / ms * 1e3}
    del dx, dt_, kres

    # C1 (100k nuclei, V ~ U{8..32}) and one C4 slide (500k): the whole nuclei-table pass, device-resident -
    # tile->WSI map + morphology (ragged float32 rings), kNN k=8 + undirected union + i<j edges + composition and,
    # for C4, the r=50 px radius graph on the WSI centroids the map kernel just produced
    for name, n_s, seed, with_radius in (("C1_100k", 100_000, synth.SEEDS["C1"], False),
                                          ("C4_slide_500k", 500_000, synth.SEEDS["C4"], True)):
        tab = synth.make_table(n_s, seed)
        side_px = float(tab.n_tiles_side * 508)
        t_off, t_xy = torch.from_numpy(tab.poly_off).to(dev), torch.from_numpy(tab.poly_xy).to(dev)
        t_tile = torch.from_numpy(tab.nuc_tile).to(dev)
        t_tx, t_ty = torch.from_numpy(tab.tile_x).to(dev), torch.from_numpy(tab.tile_y).to(dev)
        t_cen, t_bb = torch.from_numpy(tab.centroid).to(dev), torch.from_numpy(tab.bbox).to(dev)
        t_types = torch.from_numpy(tab.types).to(dev)
        cell_k = default_knn_cell(n_s, side_px ** 2, 8)
        bnd = (0.0, 0.0, side_px, side_px)
        keep = {}

        def slide():
            mm = eng.map_morph(t_off, t_xy, t_tile, t_tx, t_ty, t_cen, t_bb, write_polygons=True, out=keep.get("mm"))
            keep["mm"] = mm
            wsi = mm["wsi_centroid"]
            eng.grid_build(wsi, t_types, None, cell_k, bnd)
            kn = eng.knn(8, dist_dtype=torch.float32, out=keep.get("kn"))
            keep["kn"] = kn
            # outputs sized by their bounds / by the capacity of an earlier exact pass: the whole table pass is one
            # enqueue, no host read in between
            keep["un"] = eng.knn_union(kn["knn_idx"], kn["dist32"], types=t_types, n_types=N_TYPES, symmetric_dist=True, presized=True)
            if with_radius:
                eng.grid_build(wsi, t_types, None, radius_cell(RADIUS), bnd)
                if "rg_cap" not in keep:
                    keep["rg_cap"] = int(int(eng.radius_graph(RADIUS, upper=True, n_types=N_TYPES, want_edges=True)["total"]) * 1.25) + 1024
                keep["rg"] = eng.radius_graph(RADIUS, upper=True, n_types=N_TYPES, want_dist32=True, want_edges=True,
                                              capacity=keep["rg_cap"], out=keep.get("rg"))

        ms = timed(slide, reps=3)
        m_s = int(tab.poly_xy.shape[0])
        entry = {"ms": ms, "nuclei_per_s": n_s / ms * 1e3, "vertices": m_s}
        try:   # the same pass replayed as ONE CUDA graph (it reads nothing back, so it can be captured whole)
            graph = eng.capture(slide)
            g_ms = timed(graph.replay, reps=5)
            entry.update({"cuda_graph_ms": g_ms, "cuda_graph_nuclei_per_s": n_s / g_ms * 1e3})
            del graph
        except Exception as exc:  # noqa: BLE001
            entry["cuda_graph_error"] = f"{type(exc).__name__}: {exc}"[:200]
        out[name + "_table_pass(map+morph+kNN8 union" + ("+radius50)" if with_radius else ")")] = entry
        del t_off, t_xy, keep
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0's slide) as DIR/<name>.npy, float32 / float64")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs writes the outputs of --impl ours")
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
