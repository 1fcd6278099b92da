"""Builds libicpcuda.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# experiment builds (extra -D flags) go to their own library / object directory: ICPCUDA_LIB_TAG=timing -> libicpcuda_timing.so
_TAG = os.environ.get("ICPCUDA_LIB_TAG", "")
OBJ = os.path.join(HERE, "build" + ("_" + _TAG if _TAG else ""))
LIB = os.path.join(HERE, "libicpcuda" + ("_" + _TAG if _TAG else "") + ".so")
SOURCES = ["api.cu", "bvh.cu", "model.cu", "posterior.cu", "evaluate.cu", "chain.cu", "debug.cu", "gpmm.cu", "svdfactor.cu", "metrics.cu", "bvh_wide.cu", "comm.cu", "jsonlog.cu", "tc_i8.cu", "stats.cu", "stdicp.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr"] + os.environ.get("ICPCUDA_NVCC_EXTRA", "").split()


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _newest_dep():
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", h) for h in ("icpcuda.h", "icpcuda_debug.h")]
    return max(os.path.getmtime(d) for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    newest = _newest_dep()
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest:
        return LIB
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= newest:
            return obj
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
