"""K16 (pg_pair_dist_hist) on the C2 slide (1 M nuclei, seed 1002, T = 5) with 50 thresholds up to 200 px and up to
400 px, and on the C5-sized slide (20 M, seed 1005, T = 5) up to 200 px, one GPU.

Timing: the histogram call alone (on a grid already built for t_max, as co_occurrence builds it) between CUDA events,
after a 512 MB write that flushes L2; 3 warm-ups, median and p10 / p90 of 10 runs. Rates: candidate pairs visited
(the records of every query point's (2R+1)^2 block, self included) and pairs counted (ordered pairs within t_max) per
second. Kernel shares come from one further call with pg_profile on. The C2 histogram at 200 px is compared with the
oracle (oracle/cooccurrence.py) bit for bit, and the host path users have without this kernel - scipy's
cKDTree.count_neighbors once per type pair - is timed on the same machine on a band of the C2 slide (a tenth of its width) and extrapolated
to the whole slide (labelled as such). The hull area ripley() uses by default (K14 over one 1 M-vertex ring) is timed
too.

    python profiles/cooccurrence_stage.py [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import cooccurrence as oc  # noqa: E402
from path_gene_multimodal_b200 import synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine, pair_hist_cell  # noqa: E402
from profiles.enrichment_stage import device_info  # noqa: E402

WARMUP, RUNS, T, N_THR = 3, 10, 5, 50


def timed(fn, flush):
    times = []
    for i in range(WARMUP + RUNS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= WARMUP:
            times.append(e0.elapsed_time(e1))
    return times


def candidates(xy, info, t_max):
    """Records in every point's (2R+1)^2 block (R as pg_ring_radius), counted from the cell histogram on the host."""
    nx, ny, cell, x0, y0 = info["nx"], info["ny"], info["cell"], info["x0"], info["y0"]
    cover = max(nx, ny)
    r = int(min(np.ceil(t_max / cell * (1 + 1e-9) + 1e-9 + 4.0 * cover * np.finfo(float).eps), cover))
    cx = np.clip(np.floor((xy[:, 0] - x0) * (1.0 / cell)).astype(np.int64), 0, nx - 1)
    cy = np.clip(np.floor((xy[:, 1] - y0) * (1.0 / cell)).astype(np.int64), 0, ny - 1)
    grid = np.zeros((nx + 1, ny + 1), dtype=np.int64)
    np.add.at(grid, (cx + 1, cy + 1), 1)
    s = grid.cumsum(0).cumsum(1)                                  # 2-D prefix sums
    xa, xb = np.maximum(cx - r, 0), np.minimum(cx + r, nx - 1) + 1
    ya, yb = np.maximum(cy - r, 0), np.minimum(cy + r, ny - 1) + 1
    return int((s[xb, yb] - s[xa, yb] - s[xb, ya] + s[xa, ya]).sum())


def run(eng, flush, name, n, seed, t_max):
    xy, types, _ = synth.make_points(n, seed)
    thr = np.linspace(0.0, t_max, N_THR)
    dev = eng.device
    d_xy, d_t = torch.from_numpy(xy).to(dev), torch.from_numpy(types).to(dev)
    span = np.ptp(xy, axis=0)
    b = (float(xy[:, 0].min()), float(xy[:, 1].min()), float(xy[:, 0].max()), float(xy[:, 1].max()))
    eng.grid_build(d_xy, d_t, None, pair_hist_cell(t_max, n, span[0] * span[1]), b)
    times = timed(lambda: eng.pair_dist_hist(thr, T), flush)
    flush.zero_()
    eng.profile(True)
    res = eng.pair_dist_hist(thr, T)
    recs = eng.profile_records()
    eng.profile(False)
    hist = res["hist"].cpu().numpy()
    info = eng.grid_info()
    cand = candidates(xy, info, t_max)
    ms = float(np.median(times))
    per = {}
    for k, v in recs:
        per.setdefault(k, [0, 0.0])
        per[k][0] += 1
        per[k][1] += v
    total = sum(v[1] for v in per.values())
    row = {"slide": name, "nuclei": n, "n_types": T, "n_thresholds": N_THR, "t_max_px": t_max,
           "cell_px": round(info["cell"], 3), "ms": round(ms, 3),
           "ms_p10_p90": [round(float(np.percentile(times, q)), 3) for q in (10, 90)],
           "candidates": cand, "pairs_counted": int(hist.sum()),
           "candidates_per_s": float(f"{cand / (ms * 1e-3):.4g}"),
           "pairs_counted_per_s": float(f"{hist.sum() / (ms * 1e-3):.4g}"),
           "kernels": {k: {"launches": v[0], "ms": round(v[1], 3), "share": round(v[1] / total, 3)} for k, v in per.items()}}
    print(json.dumps(row), flush=True)
    return row, xy, types, thr, hist


def count_neighbors_s(xy, types, thr, frac):
    """(points, seconds) of the host path on the band x <= the frac quantile of x (the slide's density, so its pairs
    within t_max scale with its points): cKDTree.count_neighbors per type pair."""
    from scipy.spatial import cKDTree

    band = xy[:, 0] <= np.quantile(xy[:, 0], frac)
    x, t = xy[band], types[band]
    t0 = time.perf_counter()
    trees = {a: cKDTree(x[t == a]) for a in range(1, T + 1)}
    for a in range(1, T + 1):
        for c in range(1, T + 1):
            trees[a].count_neighbors(trees[c], thr, cumulative=False)
    return int(band.sum()), time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cooccurrence_stage.py needs the GPU")
    eng = get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=eng.device)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20, "runs_timed": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}), flush=True)

    row, xy, types, thr, hist = run(eng, flush, "C2", 1_000_000, synth.SEEDS["C2"], 200.0)
    result["runs_timed"].append(row)
    result["c2_200px_bit_equal_to_oracle"] = bool(np.array_equal(hist, oc.pair_hist(xy, types, thr, T)))
    n_pre, s_pre = count_neighbors_s(xy, types, thr, 0.1)
    result["host_count_neighbors_c2_200px"] = {"band_nuclei": n_pre, "s_band": round(s_pre, 3),
                                               "s_whole_slide_extrapolated": round(s_pre * len(xy) / n_pre, 2),
                                               "host_cpu_count": os.cpu_count()}
    d_xy = torch.from_numpy(xy).to(eng.device)
    off = torch.tensor([0, len(xy)], dtype=torch.int32, device=eng.device)
    hull_ms = float(np.median(timed(lambda: eng.ring_hull(off, d_xy), flush)))
    result["hull_area_1m_vertex_ring_ms"] = round(hull_ms, 3)
    print(json.dumps({k: result[k] for k in ("c2_200px_bit_equal_to_oracle", "host_count_neighbors_c2_200px",
                                             "hull_area_1m_vertex_ring_ms")}), flush=True)
    del xy, types, hist, d_xy
    row, *_ = run(eng, flush, "C2", 1_000_000, synth.SEEDS["C2"], 400.0)
    result["runs_timed"].append(row)
    row, *_ = run(eng, flush, "C5", 20_000_000, synth.SEEDS["C5"], 200.0)
    result["runs_timed"].append(row)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
