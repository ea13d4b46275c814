"""Builds libgl_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the tree)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgl_b200.so")
SOURCES = ["gl_b200.cu", "ntt_kernels.cu", "ntt_tma.cu", "hash_kernels.cu", "fri_kernels.cu", "host_staging.cu", "quotient_kernels.cu",
           "permutation_kernels.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "--threads", "4",
]


def _deps():
    out = [os.path.join(HERE, "..", "include", "gl_b200.h")]
    for f in os.listdir(CSRC):
        out.append(os.path.join(CSRC, f))
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
