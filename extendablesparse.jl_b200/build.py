"""Builds libxsparse_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libxsparse_b200.so")
SOURCES = ["xsb_sort.cu", "xsb_flush.cu", "xsb_colfold.cu", "xsb_group.cu", "xsb_runs.cu", "xsb_preagg.cu", "xsb_route.cu", "xsb_insert.cu", "xsb_values.cu", "xsb_mul.cu", "xsb_algebra.cu", "xsb_spgemm.cu", "xsb_api.cu"]
HEADERS = ["xsb_common.cuh", "xsb_internal.h", "xsb_fold.cuh", "xsb_group_count.cuh", "xsb_chunk.cuh", "xsb_x86nan.cuh", os.path.join("..", "..", "include", "xsparse_b200.h")]

NVCC_FLAGS = [
    "-O3",
    "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",  # emitters must round like the CPU oracle; nothing here is FMA-bound
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libxsparse_b200 needs the CUDA toolkit to build")
    return exe


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    objdir = os.path.join(CSRC, "_obj")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for s in SOURCES:
        o = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(o)
        # XSB_NVCC_EXTRA: tuning experiments only (e.g. "-DXSB_GP_W=1024"); use with --force
        cmd = [nvcc(), *NVCC_FLAGS, *os.environ.get("XSB_NVCC_EXTRA", "").split(), "-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        log.append(f"== {s}\n{out}")
        failed |= p.returncode != 0
    text = "\n".join(log)
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write(text)
    if failed:
        sys.stderr.write(text)
        raise RuntimeError("nvcc failed")
    if verbose:
        print(text)
    link = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-Xcompiler", "-fPIC"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
