"""Build physher_b200/libphysher_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libphysher_b200.so")

CUDA_SOURCES = ["phb_cuda.cu", "phb_nuc4.cu", "phb_dmma.cu", "phb_dwalk.cu", "phb_timetree.cu", "phb_patterns.cu", "phb_branch.cu", "phb_nni.cu",
                "phb_spr.cu"]
C_SOURCES = ["phb_treelikelihood.c", "phb_group.c", "phb_nccl.c"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build the sm_100a extension")


def sources():
    out = [os.path.join(CSRC, f) for f in CUDA_SOURCES + C_SOURCES if os.path.exists(os.path.join(CSRC, f))]
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "physher_b200.h"))
    return out, hdrs


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    srcs, hdrs = sources()
    return any(os.path.getmtime(p) > t for p in srcs + hdrs)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = nvcc_path()
    srcs, _ = sources()
    objs = []
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    common = ["-O3", "-lineinfo", "-Xcompiler", "-fPIC", "-I", CSRC, "-I", os.path.join(os.path.dirname(HERE), "include")]
    procs = []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s) + ".o")
        objs.append(o)
        if s.endswith(".cu"):
            cmd = [nvcc, *ARCH, *common, "-std=c++17", "-Xptxas", "-v" if verbose else "-warn-spills", "-c", s, "-o", o]
        else:
            cmd = [nvcc, *ARCH, *common, "-Xcompiler", "-std=gnu11", "-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(" ".join(cmd) + "\n" + out + "\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [nvcc, *ARCH, "-shared", "-Xcompiler", "-fPIC", "-cudart", "static", "-o", LIB, *objs, "-ldl"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
