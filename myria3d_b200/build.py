"""Build ``libb200randla.so`` (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

``python -m myria3d_b200.build`` or ``__graft_entry__.build()``.  The shared object lands next to
this file so that it travels with the source tree (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
BUILD_DIR = PKG_DIR / "csrc" / "build"
LIB_PATH = PKG_DIR / "libb200randla.so"
SOURCES = ["runtime.cu", "knn.cu", "knn_grid.cu", "lfa.cu", "lfa_tc.cu", "lfa_tc256.cu", "fold.cu", "pointwise.cu", "linear_rows.cu", "tma_rows.cu", "index_ops.cu", "decimate.cu", "sample_prep.cu", "batch_prep.cu", "stitch.cu", "loss.cu", "tc_selftest.cu", "tc_gemm.cu", "tc_nt.cu", "tc_skinny.cu", "optim.cu"]
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libb200randla.so cannot be built (set NVCC=/path/to/nvcc)")


def _digest() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "b200randla.h"]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(ARCH_FLAGS + NVCC_FLAGS).encode())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> Path:
    """Compile every ``csrc/*.cu`` for sm_100a and link ``libb200randla.so``.  Up-to-date builds are skipped."""
    stamp = BUILD_DIR / "digest.txt"
    digest = _digest()
    if not force and LIB_PATH.exists() and stamp.exists() and stamp.read_text() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    BUILD_DIR.mkdir(parents=True, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]

    def compile_one(src: str) -> Path:
        obj = BUILD_DIR / (Path(src).stem + ".o")
        cmd = [nvcc, *ARCH_FLAGS, *flags, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, *ARCH_FLAGS, "-shared", "-cudart", "shared", "-Xlinker", "-rpath,/usr/local/cuda/lib64",
            "-o", str(LIB_PATH), *map(str, objs)]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
