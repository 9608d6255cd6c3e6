"""K19 through cell_clusters (radius CSR by K6, pg_dbscan, pg_cluster_props, K14 hulls of the member sets) on the C2
slide (1 M nuclei, seed 1002): all types at eps = 50 (mean degree 2.9, below the continuum percolation threshold) and
eps = 75 (6.6: one giant cluster), inflammatory only (type 2) at eps = 50 and 100; and a C5-sized slide (20 M nuclei,
seed 1005) at eps = 50. min_samples = 5, hull on. One GPU.

Timing: the whole call (host to host: copies, the one read-back of the cluster count, the DataFrame) between CUDA
events, after a 512 MB write that flushes L2; every configuration is warmed up 3 times, then the median and p10 / p90
of 10 runs. Kernel shares come from one further call with pg_profile on (the per-kernel event times of every library
launch in the call). The host baseline is sklearn.cluster.DBSCAN(algorithm="kd_tree", n_jobs=-1) on the same
machine's host, on the same points (labels only, no table), one timed run per configuration; its labels must equal the
GPU's.

    python profiles/clusters_stage.py [--out FILE.json]
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
from path_gene_multimodal_b200 import cell_clusters, synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine  # noqa: E402

WARMUP, RUNS, MIN_SAMPLES = 3, 10, 5


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({e})"
    return info


def time_config(eng, flush, name, xy, types, eps, keep, sklearn_ok):
    call = lambda: cell_clusters(xy, eps, MIN_SAMPLES, types=types, keep_types=keep, device=0)  # noqa: E731
    times = []
    for i in range(WARMUP + RUNS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = call()
        e1.record()
        torch.cuda.synchronize()
        if i >= WARMUP:
            times.append(e0.elapsed_time(e1))
    flush.zero_()
    eng.profile(True)
    call()
    recs = eng.profile_records()
    eng.profile(False)
    per = {}
    for k, ms in recs:
        per.setdefault(k, [0, 0.0])
        per[k][0] += 1
        per[k][1] += ms
    total = sum(v[1] for v in per.values())
    sel = np.flatnonzero(np.isin(types, keep)) if keep is not None else np.arange(len(xy))
    df = res["clusters"]
    ms = float(np.median(times))
    row = {"slide": name, "nuclei": len(xy), "clustered": int(len(sel)), "eps": eps,
           "keep_types": list(keep) if keep is not None else "all", "min_samples": MIN_SAMPLES,
           "n_clusters": res["n_clusters"], "largest_cluster": int(df["n_nuclei"].max()) if len(df) else 0,
           "noise": int((res["labels"][sel] < 0).sum()),
           "ms": round(ms, 3), "ms_p10_p90": [round(float(np.percentile(times, q)), 3) for q in (10, 90)],
           "kernel_ms_sum": round(total, 3),
           "kernels": {k: {"launches": v[0], "ms": round(v[1], 3), "share_of_kernel_time": round(v[1] / total, 3)}
                       for k, v in sorted(per.items(), key=lambda kv: -kv[1][1])}}
    if sklearn_ok:
        from sklearn.cluster import DBSCAN

        t0 = time.perf_counter()
        sk = DBSCAN(eps=eps, min_samples=MIN_SAMPLES, algorithm="kd_tree", n_jobs=-1).fit(xy[sel])
        s = time.perf_counter() - t0
        row["sklearn_host_s"] = round(s, 3)
        row["sklearn_labels_equal"] = bool(np.array_equal(sk.labels_, res["labels"][sel]))
        row["speedup_vs_sklearn_host"] = round(s * 1e3 / ms, 1)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clusters_stage.py needs the GPU")
    eng = get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=eng.device)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20,
              "host_cpu_count": os.cpu_count(), "runs_timed": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}), flush=True)
    try:
        import sklearn  # noqa: F401
        sklearn_ok = True
    except ImportError:
        sklearn_ok = False
    xy, types, _ = synth.make_points(1_000_000, synth.SEEDS["C2"])
    for eps, keep in ((50.0, None), (75.0, None), (50.0, (2,)), (100.0, (2,))):
        result["runs_timed"].append(time_config(eng, flush, "C2", xy, types, eps, keep, sklearn_ok))
    xy, types, _ = synth.make_points(20_000_000, synth.SEEDS["C5"])
    result["runs_timed"].append(time_config(eng, flush, "C5", xy, types, 50.0, None, sklearn_ok))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
