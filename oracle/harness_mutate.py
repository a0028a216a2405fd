"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the create_haplotypes oracle (oracle/mutate_oracle.c).

The library is compiled on first use (gcc, the flags of the Illumina oracle) next to its source, or into a
temporary directory when the tree is read-only.  Importable from tests/ only; nothing under jackalope_b200/ imports
this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "mutate_oracle.c")
u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint32, C.c_uint64, C.c_double))

_lib = None


def build():
    """Compile mutate_oracle.c unless an up-to-date library exists; returns its path."""
    for d in (HERE, os.path.join(tempfile.gettempdir(), "jlp_mutate_oracle_%d" % os.getuid())):
        path = os.path.join(d, "libjlp_mutate_oracle.so")
        if os.path.exists(path) and os.path.getmtime(path) >= os.path.getmtime(SRC):
            return path
        if d == HERE and not os.access(HERE, os.W_OK):
            continue
        try:
            os.makedirs(d, exist_ok=True)
            tmp = path + ".%d.tmp" % os.getpid()
            subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-Wextra",
                            "-o", tmp, SRC, "-lm"], check=True)
            os.replace(tmp, path)
            return path
        except (OSError, subprocess.CalledProcessError):
            if d != HERE:
                raise
    raise RuntimeError("cannot build the create_haplotypes oracle")


def oracle():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.orc_mut_draw.restype = C.c_uint64
        lib.orc_mut_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint32]
        lib.orc_mutate.argtypes = [C.c_uint64, C.c_char_p, u64p, C.c_uint64, C.c_uint32, C.POINTER(C.c_int32), C.c_uint32,
                                   C.c_double, f64p, C.c_uint32, u32p, u64p, u64p, C.c_char_p, C.c_uint64]
        _lib = lib
    return _lib


def mut_draw(seed, chrom, site, node):
    return oracle().orc_mut_draw(int(seed) & (2 ** 64 - 1), chrom, site, node)


def mutate(reference, tree, sub, seed):
    """The oracle's create_haplotypes: per tip and chromosome (positions uint64[], new bases bytes).  P of every
    (node, category) comes from the product's jlp_transition_matrix (tested against scipy on its own), so both
    sides decide against the same thresholds."""
    from jackalope_b200.mutate import transition_matrix
    bases, off = reference.flat()
    bases = np.ascontiguousarray(bases)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    nn, K, nt, nc = tree.n_nodes, sub.rates.size, len(tree.tip_names), reference.n_chroms()
    P = np.zeros((nn, K, 16))
    for v in range(1, nn):
        for k in range(K):
            P[v, k] = transition_matrix(sub.Q, sub.rates[k] * tree.branch_len[v]).reshape(16)
    P = np.ascontiguousarray(P)
    counts = np.zeros(nt * nc, dtype=np.uint64)
    cap = max(1024, int(bases.size * nt // 50))
    while True:
        pos = np.zeros(cap, dtype=np.uint64)
        nuc = C.create_string_buffer(cap)
        rc = oracle().orc_mutate(int(seed) & (2 ** 64 - 1), bases.tobytes(), off.ctypes.data_as(u64p), nc, nn,
                                 tree.parent.ctypes.data_as(C.POINTER(C.c_int32)), K, float(sub.invariant),
                                 P.ctypes.data_as(f64p), nt, tree.tip_node.ctypes.data_as(u32p),
                                 counts.ctypes.data_as(u64p), pos.ctypes.data_as(u64p), nuc, cap)
        if rc == -2:
            cap = int(counts.sum())
            continue
        assert rc == 0, rc
        break
    out, k, raw = [], 0, nuc.raw
    for t in range(nt):
        row = []
        for c in range(nc):
            m = int(counts[t * nc + c])
            row.append((pos[k:k + m].copy(), raw[k:k + m]))
            k += m
        out.append(row)
    return out
