"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the create_haplotypes oracle with insertions and deletions
(oracle/indel_oracle.c, which includes oracle/mutate_oracle.c).

The library is compiled on first use (gcc, the flags of the other oracles, without floating-point contraction) next to
its source, or into a temporary directory when the tree is read-only.  Importable from tests/ only; nothing under
jackalope_b200/ imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "indel_oracle.c")
DEPS = (SRC, os.path.join(HERE, "mutate_oracle.c"))
u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint32, C.c_uint64, C.c_double))

_lib = None


class IndelResult(C.Structure):
    _fields_ = [("seq_off", u64p), ("seq", C.POINTER(C.c_char)), ("rec_off", u64p), ("old_pos", u64p),
                ("new_pos", u64p), ("nuc_off", u64p), ("size_mod", C.POINTER(C.c_int64)), ("pool_off", u64p),
                ("pool", C.POINTER(C.c_char)), ("n_steps", C.c_uint64), ("steps", u64p), ("n_events", C.c_uint64),
                ("events", u64p)]


def build():
    """Compile indel_oracle.c unless an up-to-date library exists; returns its path."""
    newest = max(os.path.getmtime(f) for f in DEPS)
    for d in (HERE, os.path.join(tempfile.gettempdir(), "jlp_indel_oracle_%d" % os.getuid())):
        path = os.path.join(d, "libjlp_indel_oracle.so")
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
    raise RuntimeError("cannot build the create_haplotypes indel oracle")


def oracle():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.orc_indels.restype = C.POINTER(IndelResult)
        lib.orc_indels.argtypes = [C.c_uint64, C.c_char_p, u64p, C.c_uint64, C.c_uint32, C.POINTER(C.c_int32), f64p,
                                   C.c_uint32, C.c_double, f64p, f64p, C.c_double, f64p, C.c_uint32, C.c_double, f64p,
                                   C.c_uint32, C.c_double, C.c_uint32, u32p, C.POINTER(C.c_int64), C.c_uint64]
        lib.orc_indel_free.argtypes = [C.POINTER(IndelResult)]
        lib.orc_indel_free.restype = None
        _lib = lib
    return _lib


def _tables(tree, sub):
    from jackalope_b200.mutate import transition_matrix
    nn, K = tree.n_nodes, sub.rates.size
    P = np.zeros((nn, K, 16))
    for v in range(1, nn):
        for k in range(K):
            P[v, k] = transition_matrix(sub.Q, sub.rates[k] * tree.branch_len[v]).reshape(16)
    return np.ascontiguousarray(P)


class IndelOracle:
    """What orc_indels returns: tips[t][c] = (tip sequence bytes, records (old_pos, new_pos, nuc_off, size_mod,
    pool bytes)); steps: rows (chrom, node, step, L, events); events: rows (chrom, node, step, pos, ins, length)."""

    def __init__(self, tips, steps, events):
        self.tips, self.steps, self.events = tips, steps, events


def indels(reference, tree, sub, ins, dele, epsilon, seed, events=None, pi=None):
    """The oracle's create_haplotypes with indels (ins / dele: IndelModel or None; events: None to draw them, else
    rows (chrom, node, step, pos, 1 insertion / 0 deletion, length) sorted in that order; pi: the inserted columns'
    birth distribution, sub.pi by default)."""
    bases, off = reference.flat()
    bases = np.ascontiguousarray(bases)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    nn, K, nt, nc = tree.n_nodes, sub.rates.size, len(tree.tip_names), reference.n_chroms()
    P = _tables(tree, sub)
    pi = np.ascontiguousarray(sub.pi if pi is None else pi, dtype=np.float64)
    wi = np.ascontiguousarray(ins.rel_rates if ins is not None else [1.0], dtype=np.float64)
    wd = np.ascontiguousarray(dele.rel_rates if dele is not None else [1.0], dtype=np.float64)
    ri = ins.rate if ins is not None else 0.0
    rd = dele.rate if dele is not None else 0.0
    ev = None if events is None else np.ascontiguousarray(np.asarray(events, dtype=np.int64).reshape(-1, 6))
    bl = np.ascontiguousarray(tree.branch_len, dtype=np.float64)
    res = oracle().orc_indels(int(seed) & (2 ** 64 - 1), bases.tobytes(), off.ctypes.data_as(u64p), nc, nn,
                              tree.parent.ctypes.data_as(C.POINTER(C.c_int32)), bl.ctypes.data_as(f64p), K,
                              float(sub.invariant), P.ctypes.data_as(f64p), pi.ctypes.data_as(f64p), ri,
                              wi.ctypes.data_as(f64p), wi.size, rd, wd.ctypes.data_as(f64p), wd.size, float(epsilon), nt,
                              tree.tip_node.ctypes.data_as(u32p),
                              None if ev is None else ev.ctypes.data_as(C.POINTER(C.c_int64)), 0 if ev is None else len(ev))
    assert res, "orc_indels failed"
    try:
        r = res.contents
        n = nt * nc
        arr = lambda ptr, k, dt=np.uint64: np.ctypeslib.as_array(ptr, shape=(k,)).astype(dt) if k else np.zeros(0, dt)
        so, ro, po = arr(r.seq_off, n + 1), arr(r.rec_off, n + 1), arr(r.pool_off, n + 1)
        seq = C.string_at(r.seq, int(so[-1])) if so[-1] else b""
        pool = C.string_at(r.pool, int(po[-1])) if po[-1] else b""
        NR = int(ro[-1])
        old, new, nuc = arr(r.old_pos, NR), arr(r.new_pos, NR), arr(r.nuc_off, NR)
        sm = arr(r.size_mod, NR, np.int64)
        tips = []
        for t in range(nt):
            row = []
            for c in range(nc):
                i = t * nc + c
                a, b = int(ro[i]), int(ro[i + 1])
                row.append((seq[int(so[i]):int(so[i + 1])],
                            (old[a:b], new[a:b], nuc[a:b], sm[a:b], pool[int(po[i]):int(po[i + 1])])))
            tips.append(row)
        steps = arr(r.steps, int(r.n_steps) * 5).reshape(-1, 5)
        events = arr(r.events, int(r.n_events) * 6).reshape(-1, 6)
    finally:
        oracle().orc_indel_free(res)
    return IndelOracle(tips, steps, events)
