"""In-tree build of libpcs_b200.so (hand-written CUDA for sm_100a + the C ABI of include/pcs_b200.h).

nvcc cross-compiles without a GPU, so this runs in the CPU-only build container; the resulting .so is
git-ignored but travels to the GPU box with the repository snapshot.
"""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libpcs_b200.so"
SOURCES = ["pcs_core.cu", "pcs_normal.cu", "pcs_solver.cu", "pcs_p2p.cu", "pcs_costfn.cu", "pcs_chol.cu", "pcs_schur.cu", "pcs_gauge.cu", "pcs_cov.cu"]
HEADERS = ["pcs_math.cuh", "pcs_internal.cuh", "../../include/pcs_b200.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-O2",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (cand == "nvcc" or Path(cand).exists()):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    files = [CSRC / s for s in SOURCES] + [CSRC / h for h in HEADERS]
    return any(f.exists() and f.stat().st_mtime > t for f in files)


def build_library(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    procs, objs = [], []
    for s in SOURCES:
        src = CSRC / s
        if not src.exists():
            continue
        obj = objdir / (src.stem + ".o")
        objs.append(str(obj))
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, pr in procs:
        out, _ = pr.communicate()
        if verbose and out:
            print(out)
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + (out or ""))
    link = [nvcc, "-shared", "-o", str(LIB), *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-cudart", "static", "-Xlinker", "--no-undefined"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
