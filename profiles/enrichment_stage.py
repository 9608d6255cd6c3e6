"""K15 (pg_nhood_enrichment) on the C2 slide (1 M nuclei, seed 1002, r = 50, T = 5) at P = 100 and 1000 and on the
C5-sized slide (20 M, seed 1005, r = 50) at P = 1000, one GPU.

Timing: the enrichment call alone (labels, counts and finish kernels) between CUDA events, after a 512 MB write that
flushes L2 (the C2 inputs, about 16 MB, would otherwise stay resident); 3 warm-ups, median and p10 / p90 of 10 runs.
Rate = directed entries (2 E) x permutations per second. Kernel shares come from one further call with pg_profile on
(per-kernel CUDA events; the events themselves stretch the timeline a little). The C2 result at P = 20 is compared
with the oracle (oracle/enrichment.py) bit for bit, and numpy's version of squidpy's procedure (rng.permutation of
the labels, two bincounts) is timed on the same machine's host for comparison.

    python profiles/enrichment_stage.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import enrichment as oe  # noqa: E402
from path_gene_multimodal_b200 import build_radius_graph, synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine  # noqa: E402

WARMUP, RUNS, T, R = 3, 10, 5, 50.0


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({e})"
    return info


def numpy_squidpy_per_perm(edges, types, reps=10):
    """Seconds per permutation of squidpy's procedure in numpy: permute the labels, count with two bincounts."""
    rng = np.random.default_rng(0)
    e0, e1 = edges[:, 0].astype(np.int64), edges[:, 1].astype(np.int64)
    lab = types.astype(np.int64) - 1
    t0 = time.perf_counter()
    for _ in range(reps):
        tp = lab[rng.permutation(len(lab))]
        a, b = tp[e0], tp[e1]
        c = np.bincount(a * T + b, minlength=T * T) + np.bincount(b * T + a, minlength=T * T)
    assert c.sum() == 2 * len(edges)
    return (time.perf_counter() - t0) / reps


def time_slide(eng, flush, name, n, seed, perms_list):
    xy, types, _ = synth.make_points(n, seed)
    g = build_radius_graph(xy, r=R, types=types, outputs="compact", device=0)
    edges = g["edges"]
    n_edges = len(edges)
    dev = eng.device
    d_e = torch.from_numpy(np.ascontiguousarray(edges, dtype=np.int32)).to(dev)
    d_t = torch.from_numpy(types).to(dev)
    rows = []
    for p in perms_list:
        times = []
        for i in range(WARMUP + RUNS):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.nhood_enrichment(d_e, d_t, T, p, 0)
            e1.record()
            torch.cuda.synchronize()
            if i >= WARMUP:
                times.append(e0.elapsed_time(e1))
        flush.zero_()
        eng.profile(True)
        eng.nhood_enrichment(d_e, d_t, T, p, 0)
        recs = eng.profile_records()
        eng.profile(False)
        per = {}
        for k, ms in recs:
            per.setdefault(k, [0, 0.0])
            per[k][0] += 1
            per[k][1] += ms
        total = sum(v[1] for v in per.values())
        ms = float(np.median(times))
        row = {"slide": name, "nuclei": n, "edges": n_edges, "n_types": T, "n_perms": p, "ms": round(ms, 3),
               "ms_p10_p90": [round(float(np.percentile(times, q)), 3) for q in (10, 90)],
               "updates_per_s": float(f"{2.0 * n_edges * p / (ms * 1e-3):.4g}"),
               "kernels": {k: {"launches": v[0], "ms": round(v[1], 3), "share": round(v[1] / total, 3)}
                           for k, v in per.items()}}
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows, edges, types


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("enrichment_stage.py needs the GPU")
    eng = get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=eng.device)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20, "runs_timed": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}), flush=True)

    rows, edges, types = time_slide(eng, flush, "C2", 1_000_000, synth.SEEDS["C2"], (100, 1000))
    result["runs_timed"] += rows
    from path_gene_multimodal_b200 import neighbourhood_enrichment

    got = neighbourhood_enrichment(edges, types, n_types=T, n_perms=20, seed=0, device=0)
    ref = oe.nhood_enrichment(edges, types, T, 20, 0)
    result["c2_p20_bit_equal_to_oracle"] = bool(all(np.array_equal(got[k], ref[k])
                                                    for k in ("count", "zscore", "perm_mean", "perm_std")))
    result["c2_p20_zscore"] = got["zscore"].round(3).tolist()
    result["numpy_squidpy_s_per_perm_c2"] = round(numpy_squidpy_per_perm(edges, types), 4)
    result["host_cpu_count"] = os.cpu_count()
    print(json.dumps({k: result[k] for k in ("c2_p20_bit_equal_to_oracle", "numpy_squidpy_s_per_perm_c2",
                                             "host_cpu_count")}), flush=True)
    del edges, types
    rows, _, _ = time_slide(eng, flush, "C5", 20_000_000, synth.SEEDS["C5"], (1000,))
    result["runs_timed"] += rows
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
