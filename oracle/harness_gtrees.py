"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the create_haplotypes oracle along gene trees (oracle/gtrees_oracle.c,
which includes oracle/mutate_oracle.c), and an independent reading of ms-format text: the tree lines of each `//` block
parsed with the product's Python parse_newick, the regions computed here in Python integers.

The library is compiled on first use (gcc, the flags of the other oracles) next to its source, or into a temporary
directory when the tree is read-only.  Importable from tests/ only; nothing under jackalope_b200/ imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "gtrees_oracle.c")
DEPS = (SRC, os.path.join(HERE, "mutate_oracle.c"))
u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint32, C.c_uint64, C.c_double))

_lib = None


def build():
    """Compile gtrees_oracle.c unless an up-to-date library exists; returns its path."""
    newest = max(os.path.getmtime(f) for f in DEPS)
    for d in (HERE, os.path.join(tempfile.gettempdir(), "jlp_gtrees_oracle_%d" % os.getuid())):
        path = os.path.join(d, "libjlp_gtrees_oracle.so")
        if os.path.exists(path) and os.path.getmtime(path) >= newest:
            return path
        if d == HERE and not os.access(HERE, os.W_OK):
            continue
        try:
            os.makedirs(d, exist_ok=True)
            tmp = path + ".%d.tmp" % os.getpid()
            subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-Wextra",
                            "-I", HERE, "-o", tmp, SRC, "-lm"], check=True)
            os.replace(tmp, path)
            return path
        except (OSError, subprocess.CalledProcessError):
            if d != HERE:
                raise
    raise RuntimeError("cannot build the create_haplotypes gene-tree oracle")


def oracle():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.orc_mutate_gtrees.argtypes = [C.c_uint64, C.c_char_p, u64p, C.c_uint64, u64p, u64p, u64p, u32p, C.c_uint32,
                                          u64p, C.POINTER(C.c_int32), u32p, C.c_uint32, C.c_double, f64p, C.c_uint32,
                                          u64p, u64p, C.c_char_p, C.c_uint64]
        _lib = lib
    return _lib


def _unpack(nt, nc, counts, pos, raw):
    out, k = [], 0
    for t in range(nt):
        row = []
        for c in range(nc):
            m = int(counts[t * nc + c])
            row.append((pos[k:k + m].copy(), raw[k:k + m]))
            k += m
        out.append(row)
    return out


def ms_blocks(text):
    """ms-format text -> per `//` block the tree lines as (n or None, Newick text), read here on its own"""
    blocks = None
    for line in text.split("\n"):
        line = line.rstrip("\r")
        if line.startswith("//"):
            blocks = (blocks or []) + [[]]
        elif blocks is not None and line[:1] in ("[", "("):
            n = None
            if line[0] == "[" and "]" in line:
                inner = line[1:line.index("]")]
                if inner and all(ch in "0123456789" for ch in inner):
                    n, line = int(inner), line[line.index("]") + 1:]
            blocks[-1].append((n, line))
    return blocks or []


def regions(lengths, L):
    """[floor(L c_{k-1} / S), floor(L c_k / S)) for the prefix sums c_k of the lengths (None: one tree, the whole
    chromosome), empty regions dropped: (start, end, index in the block)"""
    lens = [1 if n is None else n for n in lengths]
    S, cum, start, out = sum(lens), 0, 0, []
    for k, n in enumerate(lens):
        cum += n
        end = L * cum // S
        if end > start:
            out.append((start, end, k))
        start = end
    return out


def mutate_gtrees(reference, text, names, sub, seed):
    """The oracle's create_haplotypes along gene trees: the trees read with parse_newick, the regions computed here,
    every site walked with its region's tree; P from jlp_transition_matrix as in mutate()."""
    from jackalope_b200.mutate import parse_newick, transition_matrix
    bases, off = reference.flat()
    bases = np.ascontiguousarray(bases)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    nc, K, nt = reference.n_chroms(), sub.rates.size, len(names)
    blocks = ms_blocks(text)
    assert len(blocks) == nc
    trees, reg_off, rs, re_, rt = [], [0], [], [], []
    for c, b in enumerate(blocks):
        base = len(trees)
        for s0, e0, k in regions([n for n, _ in b], int(reference.seqs[c].size)):
            rs.append(s0), re_.append(e0), rt.append(base + k)
        trees += [parse_newick(nw) for _, nw in b]
        reg_off.append(len(rs))
    node_off = np.concatenate(([0], np.cumsum([t.n_nodes for t in trees]))).astype(np.uint64)
    parent = np.ascontiguousarray(np.concatenate([t.parent for t in trees]), dtype=np.int32)
    tip_node = np.zeros(len(trees) * nt, dtype=np.uint32)
    P = np.zeros((int(node_off[-1]), K, 16))
    for i, t in enumerate(trees):
        where = {nm: int(v) for nm, v in zip(t.tip_names, t.tip_node)}
        tip_node[i * nt:(i + 1) * nt] = [where[nm] for nm in names]
        if not any(rt_ == i for rt_ in rt):
            continue
        for v in range(1, t.n_nodes):
            for k in range(K):
                P[int(node_off[i]) + v, k] = transition_matrix(sub.Q, sub.rates[k] * t.branch_len[v]).reshape(16)
    P = np.ascontiguousarray(P)
    arr = lambda x, dt: np.ascontiguousarray(np.asarray(x, dtype=dt))
    reg_off, rs, re_, rt = arr(reg_off, np.uint64), arr(rs, np.uint64), arr(re_, np.uint64), arr(rt, np.uint32)
    counts = np.zeros(nt * nc, dtype=np.uint64)
    cap = max(1024, int(bases.size * nt // 50))
    while True:
        pos = np.zeros(cap, dtype=np.uint64)
        nuc = C.create_string_buffer(cap)
        rc = oracle().orc_mutate_gtrees(int(seed) & (2 ** 64 - 1), bases.tobytes(), off.ctypes.data_as(u64p), nc,
                                        reg_off.ctypes.data_as(u64p), rs.ctypes.data_as(u64p), re_.ctypes.data_as(u64p),
                                        rt.ctypes.data_as(u32p), len(trees), node_off.ctypes.data_as(u64p),
                                        parent.ctypes.data_as(C.POINTER(C.c_int32)), tip_node.ctypes.data_as(u32p), K,
                                        float(sub.invariant), P.ctypes.data_as(f64p), nt, counts.ctypes.data_as(u64p),
                                        pos.ctypes.data_as(u64p), nuc, cap)
        if rc == -2:
            cap = int(counts.sum())
            continue
        assert rc == 0, rc
        break
    return _unpack(nt, nc, counts, pos, nuc.raw)
