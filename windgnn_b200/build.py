"""Build the in-tree C-ABI library ``windgnn_b200/lib/libwindgnn_b200.so`` for sm_100a.

    python -m windgnn_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
repo snapshot.  ``graph.cu`` is compiled with ``-fmad=false`` (bit-exact fp64 graph build);
everything else with FMA contraction on.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libwindgnn_b200.so")
# experiment builds (WG_NVCC_FLAGS=-D...) go to their own file so that they never replace the product:
# WG_LIB_SUFFIX=trace -> lib/libwindgnn_b200_trace.so, loaded with WINDGNN_B200_LIB=<that path>
_SUFFIX = os.environ.get("WG_LIB_SUFFIX", "")
if _SUFFIX:
    LIB = os.path.join(LIBDIR, f"libwindgnn_b200_{_SUFFIX}.so")
    BUILD = os.path.join(HERE, f"build_{_SUFFIX}")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]
UNITS = [
    ("abi.cu", ["-ftz=true"]),  # denormals flushed: single-instruction ex2/rcp in the gate math
    ("graph.cu", ["-fmad=false"]),
    ("windows.cu", []),
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the windgnn_b200 CUDA library cannot be built")


def _sources():
    out = []
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                out.append(os.path.join(root, f))
    return out


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    nvcc = _nvcc()
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(BUILD, exist_ok=True)
    objs = []
    for src, extra in UNITS:
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        env_extra = os.environ.get("WG_NVCC_FLAGS", "").split()  # experiment builds, e.g. -DWG_RC_TRACE
        cmd = [nvcc, *ARCH, *COMMON, *extra, *env_extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
