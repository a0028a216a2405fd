"""Build jackalope_b200/libjlp_b200.so in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libjlp_b200.so")
SOURCES = ["jlp_api.cu", "jlp_kernels.cu", "jlp_bgzf.cu", "jlp_pacbio.cu", "jlp_mutate.cu", "jlp_pacbio.cpp", "jlp_host.cpp", "jlp_deflate.cpp"]
HEADERS = ["jlp_draws.h", "jlp_host.h", "jlp_kernels.cuh", "jlp_deflate.h", "jlp_pacbio.h", os.path.join("..", "..", "include", "jlp_b200.h")]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    if os.environ.get("JLP_NO_BUILD") and os.path.exists(LIB):      # use the library as shipped (measuring an older build)
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function", "-shared", "-o", LIB]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += os.environ.get("JLP_NVCC_EXTRA", "").split()
    cmd += [os.path.join(CSRC, f) for f in SOURCES] + ["-lz"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libjlp_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    build(force=True, verbose=True)
    print(LIB)
