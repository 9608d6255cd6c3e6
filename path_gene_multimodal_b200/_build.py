"""nvcc build recipe for libpathgraph.so (sm_100a only, in-tree, no JIT cache)."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
INCLUDE = PKG_DIR.parent / "include"
LIB_PATH = PKG_DIR / "libpathgraph.so"
SOURCES = ["pg_handle.cu", "pg_scan.cu", "pg_grid.cu", "pg_radius.cu", "pg_knn.cu", "pg_graph.cu", "pg_shard.cu", "pg_morph.cu", "pg_features.cu", "pg_raster.cu", "pg_contour.cu", "pg_hull.cu", "pg_enrich.cu", "pg_pairhist.cu", "pg_autocorr.cu", "pg_lisa.cu", "pg_cluster.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "--extended-lambda",
    "-Xcompiler", "-fPIC",
    "-diag-suppress", "177",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; libpathgraph.so cannot be built")


def needs_build() -> bool:
    if not LIB_PATH.exists():
        return True
    t = LIB_PATH.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + list(CSRC.glob("*.cuh")) + [INCLUDE / "pathgraph.h"]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines: tuple = (), out: Path | None = None) -> Path:
    """Compile csrc/*.cu for sm_100a and link libpathgraph.so next to this file.

    ``defines`` / ``out``: an experimental variant (-DNAME=VALUE ...) linked to another path; select it at run
    time with PG_LIBPATH (profiles/ uses this to time compile-time alternatives in one GPU session)."""
    lib_path = Path(out) if out else LIB_PATH
    if not force and not out and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    obj_dir = PKG_DIR / "build" / (lib_path.stem if out else "")
    obj_dir.mkdir(exist_ok=True, parents=True)

    def compile_one(src: str) -> Path:
        obj = obj_dir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *[f"-D{d}" for d in defines], f"-I{INCLUDE}", f"-I{CSRC}", "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = lib_path.with_suffix(".so.tmp")
    # static cudart: the library carries its own runtime and shares the primary context (and so
    # the stream handles) with torch's
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *map(str, objs), "-o", str(tmp),
           "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib_path)
    return lib_path


if __name__ == "__main__":
    print(build(force=True, verbose=bool(os.environ.get("PG_VERBOSE"))))
