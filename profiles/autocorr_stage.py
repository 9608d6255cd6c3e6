"""K17 (pg_spatial_autocorr) on the C2 slide (1 M nuclei, seed 1002, radius graph r = 50 as a symmetric CSR) with the
10 morphology columns (polygon_morphology.CONT_COLS) and with 16 columns (those + the 5 neighbour-type fractions + the
degree), P = 100 and 1000, Moran and Geary, row-standardised weights; and on a 20 M-nucleus slide (seed 1005, points
only, 10 synthetic columns) at P = 100. One GPU.

Timing: the call alone (all K17 kernels) between CUDA events, after a 512 MB write that flushes L2; every shape is
warmed up 3 times, then the median and p10 / p90 of 10 runs. Kernel shares come from one further call with pg_profile
on. Bytes: what the kernels move if nothing hits L2 (computed from the shapes, see bytes_moved), over the median time.
The C2 result at P = 20 is compared with the oracle (oracle/autocorr.py) against its per-value bound, and squidpy's
procedure - one scipy.sparse product W @ X[perm] per permutation - is timed on the same machine's host on 5
permutations and extrapolated (labelled as such).

    python profiles/autocorr_stage.py [--out FILE.json]
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
from oracle import autocorr as oa  # noqa: E402
from path_gene_multimodal_b200 import build_radius_graph, nuclei_morphology_table, synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine  # noqa: E402
from path_gene_multimodal_b200.polygon_morphology import CONT_COLS  # noqa: E402

WARMUP, RUNS, R = 3, 10, 50.0


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({e})"
    return info


def bytes_moved(n, e_dir, n_feat, p):
    """Bytes the kernels read and write if nothing hits L2: per labelling the int32 index (write 4n); per labelling and
    4-column group the row pass's row_ptr / col (4n + 4E), the indices of the rows and of their entries (4n + 4E) and
    one 32-byte sector of centred values per row and per entry (32n + 32E); plus the prep, degree and weight passes."""
    g = (n_feat + 3) // 4
    labellings = p + 1
    row_pass = labellings * g * (8 * n + 8 * e_dir + 32 * n + 32 * e_dir)
    once = 3 * 8 * n_feat * n + 32 * g * n + 2 * (4 * n + 4 * e_dir) + 4 * n
    return labellings * 4 * n + row_pass + once


def host_squidpy_per_perm(rp, col, x, reps=5):
    """Seconds per permutation of squidpy's procedure on the host: permute the rows of X, one sparse product with the
    row-normalised W, the Moran numerator per column."""
    n = x.shape[0]
    w = oa.weight_matrix(rp, col, n, True)
    z = oa.centred(x)
    rng = np.random.default_rng(0)
    t0 = time.perf_counter()
    for _ in range(reps):
        zp = z[rng.permutation(n)]
        num = (zp * (w @ zp)).sum(axis=0)
    assert num.shape == (x.shape[1],)
    return (time.perf_counter() - t0) / reps


def time_config(eng, flush, name, d, n_feat, p, mode):
    n, e_dir = d["n"], d["e_dir"]
    feat = d["feat"][:n_feat].contiguous()
    times = []
    for i in range(WARMUP + RUNS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.spatial_autocorr(d["rp"], d["col"], feat, mode, True, p, 0)
        e1.record()
        torch.cuda.synchronize()
        if i >= WARMUP:
            times.append(e0.elapsed_time(e1))
    flush.zero_()
    eng.profile(True)
    eng.spatial_autocorr(d["rp"], d["col"], feat, mode, True, p, 0)
    recs = eng.profile_records()
    eng.profile(False)
    per = {}
    for k, ms in recs:
        per.setdefault(k, [0, 0.0])
        per[k][0] += 1
        per[k][1] += ms
    total = sum(v[1] for v in per.values())
    ms = float(np.median(times))
    b = bytes_moved(n, e_dir, n_feat, p)
    row = {"slide": name, "nuclei": n, "csr_entries": e_dir, "n_feat": n_feat, "n_perms": p, "mode": mode,
           "transformation": "row", "ms": round(ms, 3),
           "ms_p10_p90": [round(float(np.percentile(times, q)), 3) for q in (10, 90)],
           "bytes_if_no_l2_hit": b, "effective_tb_per_s": round(b / (ms * 1e-3) / 1e12, 2),
           "us_per_perm_and_group": round(ms * 1e3 / ((p + 1) * ((n_feat + 3) // 4)), 2),
           "kernels": {k: {"launches": v[0], "ms": round(v[1], 3), "share": round(v[1] / total, 3)}
                       for k, v in per.items()}}
    print(json.dumps(row), flush=True)
    return row


def to_dev(eng, rp, col, x):
    dev = eng.device
    return {"n": len(rp) - 1, "e_dir": len(col), "rp": torch.from_numpy(rp.astype(np.int32)).to(dev),
            "col": torch.from_numpy(col.astype(np.int32)).to(dev),
            "feat": torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autocorr_stage.py needs the GPU")
    eng = get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=eng.device)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20, "runs_timed": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}), flush=True)

    tab = synth.make_table(1_000_000, synth.SEEDS["C2"])
    df = nuclei_morphology_table(tab.poly_xy, poly_off=tab.poly_off, hull=True, device=0)
    g = build_radius_graph(tab.wsi_centroids(), r=R, types=tab.types, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    deg = np.maximum(g["degree"], 1).astype(np.float64)
    x = np.column_stack([df[CONT_COLS].to_numpy(), g["nbr_count"] / deg[:, None], g["degree"].astype(np.float64)])
    assert x.shape[1] == 16 and np.isfinite(x).all()
    d = to_dev(eng, rp, col, x)
    for n_feat in (10, 16):
        for p in (100, 1000):
            for mode in ("moran", "geary"):
                result["runs_timed"].append(time_config(eng, flush, "C2", d, n_feat, p, mode))

    got = {k: v.cpu().numpy() for k, v in eng.spatial_autocorr(d["rp"], d["col"], d["feat"][:10].contiguous(), "moran",
                                                               True, 20, 0, want_sims=True).items()}
    ref = oa.spatial_autocorr(rp, col, x[:, :10], "moran", True, 20, 0)
    result["c2_p20_stat_err_over_bound_max"] = float((np.abs(got["stat"] - ref["stat"]) / ref["bound"]).max())
    result["c2_p20_sims_err_over_bound_max"] = float((np.abs(got["sims"] - ref["sims"]) / ref["sims_bound"]).max())
    result["c2_moran_I"] = dict(zip(CONT_COLS, got["stat"].round(4).tolist()))
    s = host_squidpy_per_perm(rp, col, x[:, :10])
    result["host_squidpy_procedure_c2_f10"] = {"s_per_perm_measured_on_5": round(s, 4),
                                               "s_for_1000_perms_extrapolated": round(1000 * s, 1)}
    result["host_cpu_count"] = os.cpu_count()
    print(json.dumps({k: result[k] for k in ("c2_p20_stat_err_over_bound_max", "c2_p20_sims_err_over_bound_max",
                                             "host_squidpy_procedure_c2_f10", "host_cpu_count")}), flush=True)
    del d, tab, df, g, rp, col, x

    xy, _, _ = synth.make_points(20_000_000, synth.SEEDS["C5"])
    g = build_radius_graph(xy, r=R, symmetric_csr=True, device=0)
    rng = np.random.default_rng(5)
    span = float(np.ptp(xy[:, 0]))
    cols = [np.sin(2 * np.pi * (k + 1) * xy[:, k % 2] / span) + rng.normal(size=len(xy)) for k in range(10)]
    d = to_dev(eng, g["row_ptr"], g["col"], np.column_stack(cols))
    del g, xy, cols
    result["runs_timed"].append(time_config(eng, flush, "20M", d, 10, 100, "moran"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
