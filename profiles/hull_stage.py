"""K14 (pg_ring_hull_*) against K1 (pg_map_morph_*) on the four tables of profiles/morph_dtypes.py.

Both kernels run in the same process, alternating, each after a 512 MB write that flushes L2; CUDA events, 3 warm-ups
and the median of 25 timed runs. K14's algorithmic bytes are sizeof(T) * 2 * M (vertices) + 4 * N (offsets) +
24 * N (three float64 outputs); the fraction is of 6550.7 GB/s, the copy rate measured on the B200 (DESIGN.md).
A seeded sample of 20 000 rings of each timed table is compared with the exact oracle (oracle/hull.py): convex area and
solidity bit for bit, orientation as an axis (modulo pi) where the moments are anisotropic.

    python profiles/hull_stage.py [--out FILE.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import hull as ohull  # noqa: E402
from oracle import morphology as omorph  # noqa: E402
from path_gene_multimodal_b200 import synth  # noqa: E402
from path_gene_multimodal_b200.engine import get_engine  # noqa: E402

PEAK_GBS = 6550.7
WARMUP, RUNS, SAMPLE = 3, 25, 20_000


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hull_stage.py needs the GPU")
    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    result = {**device_info(), "warmup": WARMUP, "runs": RUNS, "l2_flush_bytes": 512 << 20, "tables": []}
    print(json.dumps({k: result[k] for k in ("device", "power_limit")}))
    tables = (("C3 f32", 32, np.float32), ("C3 f64", 32, np.float64), ("ragged f32", None, np.float32),
              ("ragged f64", None, np.float64))
    n = 2_000_000
    for name, vfix, dt in tables:
        off, xy = synth.make_polygons(n, 1003, v_fixed=vfix, dtype=dt)
        rng = np.random.default_rng(3)
        t = 73
        tile_x = torch.from_numpy(((np.arange(t * t) % t) * 508).astype(np.int32)).to(dev)
        tile_y = torch.from_numpy(((np.arange(t * t) // t) * 508).astype(np.int32)).to(dev)
        nuc_tile = torch.from_numpy(rng.integers(0, t * t, size=n).astype(np.int32)).to(dev)
        cen = torch.from_numpy(rng.random((n, 2)) * 508).to(dev)
        bb = torch.from_numpy(rng.integers(0, 508, size=(n, 4)).astype(np.int32)).to(dev)
        d_off, d_p = torch.from_numpy(off).to(dev), torch.from_numpy(xy).to(dev)
        k1_out, k14_out = {}, {}

        def k1():
            k1_out.update(eng.map_morph(d_off, d_p, nuc_tile, tile_x, tile_y, cen, bb, write_polygons=True,
                                        out=k1_out or None))

        def k14():
            k14_out.update(eng.ring_hull(d_off, d_p, out=k14_out or None))

        times = {"K14": [], "K1": []}
        for i in range(WARMUP + RUNS):
            for key, fn in (("K14", k14), ("K1", k1)):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if i >= WARMUP:
                    times[key].append(e0.elapsed_time(e1) * 1e3)
        m = xy.shape[0]
        nbytes = xy.itemsize * 2 * m + 4 * n + 24 * n
        k14_us, k1_us = float(np.median(times["K14"])), float(np.median(times["K1"]))
        sel = np.sort(np.random.default_rng(17).choice(n, SAMPLE, replace=False))
        sub_off = np.concatenate([[0], np.cumsum(np.diff(off)[sel])]).astype(np.int32)
        sub_xy = np.vstack([xy[off[i]:off[i + 1]] for i in sel])
        ref = ohull.ring_hull_csr(sub_off, sub_xy)
        got = {k: v.cpu().numpy()[sel] for k, v in k14_out.items()}
        f = omorph.polygon_features_csr(sub_off, sub_xy)
        aniso = np.isfinite(ref["orientation"]) & (1.0 - f["minor_axis_length"] / f["major_axis_length"] > 1e-3)
        orient_diff = (got["orientation"][aniso] - ref["orientation"][aniso] + np.pi / 2) % np.pi - np.pi / 2
        row = {
            "table": name, "rings": n, "vertices": int(m), "k14_us": round(k14_us, 1), "k1_us": round(k1_us, 1),
            "k14_us_p10_p90": [round(float(np.percentile(times["K14"], q)), 1) for q in (10, 90)],
            "k1_us_p10_p90": [round(float(np.percentile(times["K1"], q)), 1) for q in (10, 90)],
            "k14_bytes": int(nbytes), "k14_gbs": round(nbytes / k14_us / 1e3, 1),
            "k14_fraction_of_copy_peak": round(nbytes / k14_us / 1e3 / PEAK_GBS, 3),
            "byte_floor_us": round(nbytes / PEAK_GBS / 1e3, 1),
            "sample_rings": SAMPLE,
            "sample_convex_area_bit_equal": bool(np.array_equal(got["convex_area"], ref["convex_area"])),
            "sample_solidity_bit_equal": bool(np.array_equal(got["solidity"], ref["solidity"])),
            "sample_orientation_nan_equal": bool(np.array_equal(np.isnan(got["orientation"]), np.isnan(ref["orientation"]))),
            "sample_orientation_max_axis_diff_anisotropic": float(np.max(np.abs(orient_diff))),
        }
        result["tables"].append(row)
        print(json.dumps(row))
        del d_p, k1_out, k14_out
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
