"""Builds libpbsgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m pbs_plus_b200.build [--force]

The shared library is the product: C ABI in include/pbsgpu.h, kernels in csrc/*.cu.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OBJ = HERE / "_obj"
LIB = HERE / "libpbsgpu.so"
SOURCES = ["scan.cu", "resolve.cu", "sha256.cu", "digestset.cu", "crc32.cu", "xxh3.cu", "corpus.cu", "capi.cu", "capi_set.cu",
           "capi_stream.cu", "capi_aux.cu", "zframe.cu", "zlz.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _deps(src: Path) -> float:
    hdrs = list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.hpp")) + list(CSRC.glob("*.inc")) + [HERE.parent / "include" / "pbsgpu.h"]
    return max([src.stat().st_mtime] + [h.stat().st_mtime for h in hdrs])


def build(force: bool = False, verbose: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    jobs = []
    for name in SOURCES:
        src, obj = CSRC / name, OBJ / (name + ".o")
        if force or not obj.exists() or obj.stat().st_mtime < _deps(src):
            jobs.append([NVCC, *FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-c", str(src), "-o", str(obj)])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=6) as ex:
        for out in ex.map(run, jobs):
            if verbose and out:
                print(out)
    objs = [str(OBJ / (n + ".o")) for n in SOURCES]
    if jobs or not LIB.exists():
        run([NVCC, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
             "-Xcompiler", "-fPIC", "-o", str(LIB), *objs, "-ldl"])
    return LIB


def build_cxx_driver() -> Path:
    """C++ caller of the C ABI through include/pbsgpu.hpp (stands in for the Go caller)."""
    root = HERE.parent
    src, out = root / "tests" / "cxx" / "driver.cpp", root / "tests" / "cxx" / "driver.bin"
    if not src.exists():
        return out
    dep = max(src.stat().st_mtime, (root / "include" / "pbsgpu.hpp").stat().st_mtime,
              (root / "include" / "pbsgpu.h").stat().st_mtime)
    if not out.exists() or out.stat().st_mtime < dep:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", str(out), str(src), f"-L{HERE}", "-lpbsgpu",
                               "-Wl,-rpath,$ORIGIN/../../pbs_plus_b200"])
    return out


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_cxx_driver()
    print(p)
