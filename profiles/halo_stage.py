"""K9 (the halo exchange kernels) per kernel: pack, push, unpack_multi over 3 ranges and unpack_slab, at 1 M and 8 M points.

Each library given with --lib runs in a process of its own (PG_LIBPATH); the processes alternate, --rounds of them per
library, --runs timed steps each (after 3 warm-ups), so every library gets rounds x runs samples. A 512 MB write flushes
L2 before every step (the 8 M working set exceeds L2 anyway). Times are the per-kernel CUDA-event records of
Engine.profile(), summed over a step's launches of that kernel (unpack: one launch per range). Every library's outputs
are digested (counts, sum of gids, records equal to the points they name) and the digests of every round of every
library must agree.
Giving one build twice under two labels measures the spread between identical code.

    python profiles/halo_stage.py --lib parent=PATH --lib new=PATH --lib new_again=PATH [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
WARMUP = 3
SIZES = (1_000_000, 8_000_000)


def worker(runs: int) -> dict:
    from path_gene_multimodal_b200 import synth
    from path_gene_multimodal_b200.engine import get_engine

    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    out = {}
    for n in SIZES:
        xy, ty, side = synth.make_points(n, seed=61)
        d_xy, d_ty = torch.from_numpy(xy).to(dev), torch.from_numpy(ty).to(dev)
        gid = torch.arange(n, dtype=torch.int32, device=dev)
        lo, hi = 0.05 * side, 0.95 * side                       # ~10 % of the points are halo
        world, cap = 4, n // 4
        recs, _ = eng.strip_partition(d_xy, d_ty, gid, [])       # every point as a record, in input order
        slab = torch.zeros(world * cap * 24 + 16, dtype=torch.uint8, device=dev)
        slab[:world * cap * 24].view(torch.float64).copy_(recs[:world * cap].reshape(-1))
        slab[world * cap * 24:].view(torch.int32)[:world] = cap
        peers = [torch.zeros(world * cap * 24 + 16, dtype=torch.uint8, device=dev) for _ in range(world)]
        ptrs = torch.tensor([p.data_ptr() for p in peers], dtype=torch.int64, device=dev)
        ranges = [(0.3 * side, 0.7 * side), (0.1 * side, 0.3 * side), (0.7 * side, 0.9 * side)]
        dst = [torch.empty((2 * n, 2), dtype=torch.float64, device=dev), torch.empty(2 * n, dtype=torch.int32, device=dev),
               torch.empty(2 * n, dtype=torch.int32, device=dev)]
        n_base = n // 2

        def digest(counts):      # independent of the append order inside a range
            g = dst[2][n_base:n_base + sum(counts)].long()
            return [counts, int(g.sum()), torch.equal(dst[0][n_base:n_base + sum(counts)], d_xy[g])]

        steps = {
            "pack": lambda: eng.halo_pack(d_xy, d_ty, gid, lo, hi, capacity=n),
            "push": lambda: eng.halo_push(d_xy, d_ty, gid, lo, hi, ptrs.data_ptr(), world, 1, cap),
            "unpack_multi": lambda: eng.halo_unpack_multi(recs, n, 0, n // 4, ranges, dst[0], dst[1], dst[2], n_base),
            "unpack_slab": lambda: eng.halo_unpack_slab(slab, world, 0, cap, ranges, dst[0], dst[1], dst[2], n_base),
        }
        for name, fn in steps.items():
            times = {}
            for i in range(WARMUP + runs):
                flush.zero_()
                torch.cuda.synchronize()
                eng.profile(True)
                res = fn()
                rec = eng.profile_records()
                eng.profile(False)
                if i >= WARMUP:
                    for k, ms in rec:
                        times.setdefault(k, [0.0] * runs)[i - WARMUP] += ms * 1e3
            eng.check_overflow()
            if name == "pack":
                g = _meta_gid(res[0][:int(res[1].item())])
                got = [int(res[1].item()), int(g.sum()), torch.equal(res[0][:g.numel(), :2], d_xy[g])]
            elif name == "push":     # rank 1's slots of peers 0, 2 and 3, and the count it published there
                got = [[int(_meta_gid(p[:world * cap * 24].view(torch.float64).reshape(world, cap, 3)[1]).sum()),
                        int(p[world * cap * 24:].view(torch.int32)[1])] for p in (peers[0], peers[2], peers[3])]
            else:
                got = digest(res.tolist())
            out[f"{name} {n}"] = {"us": times, "digest": got}
        del d_xy, d_ty, gid, recs, slab, peers, dst
        torch.cuda.empty_cache()
    return out


def _meta_gid(recs):
    return recs[:, 2].contiguous().view(torch.int32).reshape(-1, 2)[:, 0].to(torch.int64)


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
    ap.add_argument("--lib", action="append", default=[], help="label=path of a libpathgraph.so build")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("halo_stage.py needs the GPU")
    if args.worker:
        print(json.dumps(worker(args.runs)))
        return
    libs = dict(s.split("=", 1) for s in args.lib) or {"in-tree": str(ROOT / "path_gene_multimodal_b200" / "libpathgraph.so")}
    samples = {label: {} for label in libs}
    digests = {}
    for _ in range(args.rounds):
        for label, path in libs.items():
            r = subprocess.run([sys.executable, __file__, "--worker", "--runs", str(args.runs)], capture_output=True,
                               text=True, env={**os.environ, "PG_LIBPATH": str(Path(path).resolve())})
            if r.returncode != 0:
                raise SystemExit(f"worker for {label} failed:\n{r.stderr}")
            for key, v in json.loads(r.stdout.strip().splitlines()[-1]).items():
                for k, us in v["us"].items():
                    samples[label].setdefault(f"{key} {k}", []).extend(us)
                digests.setdefault(key, set()).add(json.dumps(v["digest"]))
    same = {key: len(ds) == 1 for key, ds in digests.items()}
    result = {**device_info(), "warmup": WARMUP, "runs_per_library": args.rounds * args.runs, "l2_flush_bytes": 512 << 20,
              "libraries": list(libs), "outputs_equal": same,
              "median_us": {label: {k: round(float(np.median(v)), 2) for k, v in s.items()} for label, s in samples.items()}}
    print(json.dumps(result, indent=1))
    if not all(same.values()):
        raise SystemExit(f"outputs differ between libraries or rounds: {digests}")
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
