"""Build ``liboo_b200.so`` (the C-ABI CUDA library, ``include/oo_b200.h``) in-tree with nvcc
for sm_100a.  ``python -m auto_oo_b200.build`` or ``build_library()``.

The library links the CUDA runtime statically and takes the one driver symbol it
needs (``cuTensorMapEncodeTiled``) through ``cudaGetDriverEntryPoint``, so it loads
on a machine without a GPU driver (nvcc cross-compiles; no GPU needed to build).
"""
from __future__ import annotations

import glob
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(OUT_DIR, "liboo_b200.so")
SOURCES = ["api.cu", "dgemm_tn.cu", "dgemm_tri.cu", "dgemm_small.cu", "expm.cu", "contract.cu", "hessian.cu",
           "hessian_operator.cu", "classes.cu", "rdm.cu", "krylov.cu"]
# every header a source may include: an edit to any of them rebuilds the library
HEADERS = (sorted(glob.glob(os.path.join(CSRC, "*.cuh")))
           + [os.path.join(os.path.dirname(HERE), "include", "oo_b200.h")])
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build liboo_b200.so")
    return exe


def _digest():
    h = hashlib.sha256()
    for path in [os.path.join(CSRC, s) for s in SOURCES] + HEADERS:
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_library(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns its path."""
    os.makedirs(OUT_DIR, exist_ok=True)
    stamp = os.path.join(OUT_DIR, "build.sha256")
    if not force and os.path.exists(LIB_PATH) and not os.path.isdir(CSRC):
        return LIB_PATH                       # binary-only deployment: nothing to compare the library with
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        with open(os.path.join(OUT_DIR, src.replace(".cu", ".ptxas.log")), "w") as f:
            f.write(res.stderr)
        if verbose:
            print(res.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-cudart", "static", "-o", LIB_PATH, *objs]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
