"""In-tree build of the CUDA library (nvcc, sm_100a only).  `python -m` is not usable with the hyphenated
package name; call build_library() or run this file directly."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgsplat_b200.so")
SOURCES = ["gs_api.cu", "gs_sort.cu", "gs_slab.cu", "gs_pack.cu", "gs_project.cu", "gs_raster.cu"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "--fmad=false",  # no implicit FMA contraction: parity needs the written op order (DESIGN.md)
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "-shared",
]


def stale(out: str = LIB) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "gsplat_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False, out: str = LIB) -> str:
    """Compile libgsplat_b200.so to `out`, by default next to this file (cross-compiles without a GPU)."""
    if not force and not stale(out):
        return out
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("GS_NVCC_EXTRA", "").split()
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        sys.stderr.write(res.stderr)
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
