"""Builds libb200sort.so (the C-ABI library of include/b200sort.h) in-tree with nvcc for sm_100a.

    python simd-radix-sort_b200/build.py [--force]

The library has no torch dependency; it links the CUDA runtime statically and loads NCCL lazily
(multi-GPU entry points only).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libb200sort.so"
# (source, object stem, extra defines): sweep_inst.cu is compiled once per (key bytes, tile geometry)
UNITS = [(CSRC / "b200sort.cu", "b200sort", []), (CSRC / "segmented_inst.cu", "segmented_inst", [])] + [
    (CSRC / "sweep_inst.cu", f"sweep_kb{k}_c{c}", [f"-DSWEEP_KB={k}", f"-DSWEEP_CFG={c}"]) for k in (8, 4, 2, 1) for c in (0, 1)] + [
    (CSRC / "sweep_inst.cu", "sweep_kb4_c2", ["-DSWEEP_KB=4", "-DSWEEP_CFG=2"])]
SOURCES = [CSRC / "b200sort.cu", CSRC / "sweep_inst.cu", CSRC / "segmented_inst.cu"]
HEADERS = [CSRC / "kernels.cuh", CSRC / "hybrid.cuh", CSRC / "mgpu.cuh", CSRC / "segmented.cuh", CSRC / "segmented_host.cuh", CSRC / "sweep_select.cuh", PKG.parent / "include" / "b200sort.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
    "-shared", "-Xcompiler", "-fPIC", "-cudart", "static",
]


def nvcc_path() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found; libb200sort.so cannot be built (there is no CPU fallback)")
    return cand


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(p.exists() and p.stat().st_mtime > t for p in SOURCES + HEADERS)


def build_lib(force: bool = False, verbose: bool = False) -> Path:
    """Compiles every translation unit for sm_100a (in parallel) and links libb200sort.so."""
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor

    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]
    newest_header = max(h.stat().st_mtime for h in HEADERS if h.exists())

    def compile_one(unit) -> Path:
        src, stem, defines = unit
        obj = objdir / (stem + ".o")
        if not force and obj.exists() and obj.stat().st_mtime > max(src.stat().st_mtime, newest_header):
            return obj
        cmd = [nvcc_path(), *compile_flags, *defines, "-c", "-o", str(obj), str(src)]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src.name} {defines}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(compile_one, UNITS))
    cmd = [nvcc_path(), "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB),
           *[str(o) for o in objs], "-ldl"]
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


BENCH = PKG / "sortbench"


def build_sortbench(force: bool = False) -> Path:
    """The native self-check / micro-benchmark driver (a development tool)."""
    src = CSRC / "sortbench.cu"
    if not force and BENCH.exists() and BENCH.stat().st_mtime > max(src.stat().st_mtime, LIB.stat().st_mtime):
        return BENCH
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo", "-o", str(BENCH),
           str(src), "-L", str(PKG), "-lb200sort", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{r.stdout}\n{r.stderr}")
    return BENCH


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose=True))
    print(build_sortbench(force="--force" in sys.argv))
