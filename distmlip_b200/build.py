"""Build libb200mlip.so (sm_100a only) in-tree with nvcc.  `python -m distmlip_b200.build`.

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libb200mlip.so")
SOURCES = ["graph.cu", "kernels.cu", "kernels_tc.cu", "kernels_ac3.cu", "kernels_tn.cu", "engine.cu"]
HEADERS = ["common.cuh", "graph.cuh", "kernels.cuh", "tc_common.cuh", "tn_state.cuh", "peratom.cuh", "engine_tn.inl", os.path.join("..", "..", "include", "b200mlip.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--extended-lambda",
    "-Xcompiler", "-fPIC", "-Wno-deprecated-declarations",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True, cwd=CSRC)
    if force or _stale(OUT, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + ["-ldl"]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return OUT


def build_probes(verbose=False):
    """standalone hardware probes under csrc/tests/ (umma_probe: tcgen05 descriptor variants; gather_probe: gather staging
    and MUFU rates) -> csrc/build/<name>; they are what profiles/r02b_run.sh runs on the GPU box"""
    nvcc = _nvcc()
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    outs = []
    for name in ("umma_probe", "gather_probe"):
        out = os.path.join(objdir, name)
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", out, os.path.join(CSRC, "tests", name + ".cu")]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        outs.append(out)
    return outs


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    if "--probes" in sys.argv:
        print(build_probes(verbose=True))
