"""K18 (pg_local_autocorr) on the C2 slide (1 M nuclei, seed 1002, radius graph r = 50 as a symmetric CSR) with the
10 morphology columns (polygon_morphology.CONT_COLS), P = 99 and 999, local Moran and Gi*, row-standardised weights;
and on a 20 M-nucleus slide (seed 1005, points only, 10 synthetic columns) at P = 99. One GPU.

Timing: the call alone (all K18 kernels) between CUDA events, after a 512 MB write that flushes L2; every shape is
warmed up 3 times, then the median and p10 / p90 of 10 runs. Kernel shares come from one further call with pg_profile
on. Selected adds: P x F x sum d_i (one neighbour value selected and added per permutation, column and CSR entry) over
the median time. The C2 result at P = 20 is compared with the oracle (oracle/local_autocorr.py) against its per-value
bound on a node sample, and the oracle's vectorised conditional permutation (esda's procedure: one gather and sum per
node, permutation and neighbour) is timed on the same machine's host on a node sample and extrapolated to the slide
(labelled as such).

    python profiles/local_autocorr_stage.py [--out FILE.json]
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
from oracle import local_autocorr as ol  # noqa: E402
from path_gene_multimodal_b200 import build_radius_graph, nuclei_morphology_table, synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine  # noqa: E402
from path_gene_multimodal_b200.polygon_morphology import CONT_COLS  # noqa: E402

WARMUP, RUNS, R = 3, 10, 50.0
API = {"moran": ("moran", True), "gi_star": ("getis_ord", True)}


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({e})"
    return info


def call(eng, d, feat, mode, p):
    api, star = API[mode]
    return eng.local_autocorr(d["rp"], d["col"], feat, api, True, star, p, 0)


def time_config(eng, flush, name, d, n_feat, p, mode):
    feat = d["feat"][:n_feat].contiguous()
    times = []
    for i in range(WARMUP + RUNS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call(eng, d, feat, mode, p)
        e1.record()
        torch.cuda.synchronize()
        if i >= WARMUP:
            times.append(e0.elapsed_time(e1))
    flush.zero_()
    eng.profile(True)
    call(eng, d, feat, mode, p)
    recs = eng.profile_records()
    eng.profile(False)
    per = {}
    for k, ms in recs:
        per.setdefault(k, [0, 0.0])
        per[k][0] += 1
        per[k][1] += ms
    total = sum(v[1] for v in per.values())
    ms = float(np.median(times))
    adds = p * n_feat * d["sum_d"]
    row = {"slide": name, "nuclei": d["n"], "csr_entries": d["e_dir"], "sum_d": d["sum_d"], "max_d": d["max_d"],
           "n_feat": n_feat, "n_perms": p, "mode": mode, "transformation": "row", "ms": round(ms, 3),
           "ms_p10_p90": [round(float(np.percentile(times, q)), 3) for q in (10, 90)],
           "selected_adds": adds, "selected_adds_per_s": float(f"{adds / (ms * 1e-3):.4g}"),
           "kernels": {k: {"launches": v[0], "ms": round(v[1], 3), "share": round(v[1] / total, 3)}
                       for k, v in per.items()}}
    print(json.dumps(row), flush=True)
    return row


def to_dev(eng, rp, col, x):
    dev = eng.device
    deg = ol.degrees(rp, col, len(rp) - 1)
    return {"n": len(rp) - 1, "e_dir": len(col), "sum_d": int(deg.sum()), "max_d": int(deg.max()),
            "rp": torch.from_numpy(rp.astype(np.int32)).to(dev), "col": torch.from_numpy(col.astype(np.int32)).to(dev),
            "feat": torch.from_numpy(np.ascontiguousarray(x.T)).to(dev)}


def host_conditional_per_node_perm(rp, col, x, nodes, p):
    """Seconds per (node, permutation) of the oracle's vectorised conditional randomisation (all columns at once)."""
    n = x.shape[0]
    z = ol.centred(x)
    d = ol.degrees(rp, col, n)
    r = ol.draws(n, 0, range(p), int(d.max()))
    t0 = time.perf_counter()
    s, _ = ol.permuted_sums(z, np.abs(z), d, nodes, r)
    ol.finish("moran", True, n, d[nodes], z[nodes], (z * z).sum(axis=0), s)
    return (time.perf_counter() - t0) / (len(nodes) * p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("local_autocorr_stage.py needs the GPU")
    eng = get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=eng.device)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20, "runs_timed": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}), flush=True)

    tab = synth.make_table(1_000_000, synth.SEEDS["C2"])
    df = nuclei_morphology_table(tab.poly_xy, poly_off=tab.poly_off, hull=True, device=0)
    g = build_radius_graph(tab.wsi_centroids(), r=R, symmetric_csr=True, device=0)
    rp, col = g["row_ptr"], g["col"]
    x = df[CONT_COLS].to_numpy()
    assert x.shape[1] == 10 and np.isfinite(x).all()
    d = to_dev(eng, rp, col, x)
    for p in (99, 999):
        for mode in ("moran", "gi_star"):
            result["runs_timed"].append(time_config(eng, flush, "C2", d, 10, p, mode))

    nodes = np.random.default_rng(0).choice(d["n"], 20_000, replace=False)
    for mode in ("moran", "gi_star"):
        api, star = API[mode]
        got = {k: v.cpu().numpy() for k, v in eng.local_autocorr(d["rp"], d["col"], d["feat"], api, True, star, 20, 0,
                                                                 want_sims=True).items()}
        ref = ol.local_autocorr(rp, col, x, mode, True, 20, 0, nodes=nodes)
        with np.errstate(invalid="ignore"):
            result[f"c2_p20_{mode}_stat_err_over_bound_max"] = float(np.nanmax(np.abs(got["stat"] - ref["stat"])
                                                                               / ref["bound"]))
            result[f"c2_p20_{mode}_sims_err_over_bound_max"] = float(np.nanmax(
                np.abs(got["sims"][:, :, nodes] - ref["sims"]) / ref["sims_bound"]))
        del got
    s = host_conditional_per_node_perm(rp, col, x, nodes[:5000], 20)
    result["host_oracle_conditional_c2_f10"] = {
        "s_per_node_and_perm_measured_on_5000_nodes_x_20_perms": float(f"{s:.4g}"),
        "s_for_all_nodes_999_perms_extrapolated": round(s * d["n"] * 999, 1)}
    result["host_cpu_count"] = os.cpu_count()
    print(json.dumps({k: v for k, v in result.items() if k.startswith(("c2_p20", "host"))}), flush=True)
    del d, tab, df, g, rp, col, x

    xy, _, _ = synth.make_points(20_000_000, synth.SEEDS["C5"])
    g = build_radius_graph(xy, r=R, symmetric_csr=True, device=0)
    rng = np.random.default_rng(5)
    span = float(np.ptp(xy[:, 0]))
    cols = [np.sin(2 * np.pi * (k + 1) * xy[:, k % 2] / span) + rng.normal(size=len(xy)) for k in range(10)]
    d = to_dev(eng, g["row_ptr"], g["col"], np.column_stack(cols))
    del g, xy, cols
    result["runs_timed"].append(time_config(eng, flush, "20M", d, 10, 99, "moran"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
