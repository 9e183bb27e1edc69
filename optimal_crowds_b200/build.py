"""Build liboc_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m optimal_crowds_b200.build        # or: from optimal_crowds_b200.build import build_lib

nvcc cross-compiles without a GPU.  The GCFM / rasteriser translation units are compiled with
-fmad=false so that their arithmetic is exactly the sequence of IEEE operations written in the source
(bit-exact parity with the CPU restatement); the HJB unit keeps FMA contraction (its parity bar is 1e-10).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "liboc_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math"]
UNITS = {  # source -> extra flags
    "oc_api.cu": ["-fmad=false"],
    "oc_gcfm.cu": ["-fmad=false"],
    "oc_voronoi.cu": ["-fmad=false"],
    "oc_hjb.cu": [],
    "oc_hjb_dist.cu": [],
}


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force: bool = False, verbose: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "nvcc")
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(HERE, "..", "include", "optimal_crowds.h"))
    objs = []
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src[:-3] + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
    if force or _stale(LIB, objs):
        subprocess.run([nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-ldl", "-lpthread"], check=True)
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
