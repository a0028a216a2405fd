"""jlp_add_haplotype with enough mutations (>= 2^16 in all) that its host store is built by several threads: a failing
chromosome is reported as the lowest failing chromosome, whatever thread finishes first, and leaves no haplotype."""
import ctypes as C

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200 import _lib

pytestmark = pytest.mark.gpu

N_CHROMS, CHROM_LEN, SUBS = 5, 100_000, 30_000


def add(ctx, muts, sizes):
    """muts[c]: (old_pos, new_pos, pool) of chromosome c, or None; returns (rc, hap_index, last error)"""
    nc = len(muts)
    empty = np.zeros(0, np.uint64)
    arrs = [m if m is not None else (empty, empty, np.zeros(0, np.uint8)) for m in muts]
    offs = [np.arange(len(o), dtype=np.uint64) for o, _, _ in arrs]       # substitutions: one pool byte each
    n_muts = np.array([len(o) for o, _, _ in arrs], np.uint64)
    pool_len = np.array([len(p) for _, _, p in arrs], np.uint64)
    sizes = np.array(sizes, np.uint64)
    ptrs = lambda xs: (_lib.u64p * nc)(*[x.ctypes.data_as(_lib.u64p) for x in xs])
    pools = (C.c_void_p * nc)(*[p.ctypes.data for _, _, p in arrs])
    idx = C.c_uint64(99)
    rc = ctx.lib.jlp_add_haplotype(ctx.h, b"h", n_muts.ctypes.data_as(_lib.u64p), ptrs([o for o, _, _ in arrs]),
                                   ptrs([n for _, n, _ in arrs]), ptrs(offs), pools, pool_len.ctypes.data_as(_lib.u64p),
                                   sizes.ctypes.data_as(_lib.u64p), C.byref(idx))
    return rc, idx.value, ctx.lib.jlp_last_error(ctx.h).decode()


def test_threaded_store_reports_the_lowest_failing_chromosome_and_adds_nothing():
    g = J.random_genome(N_CHROMS, CHROM_LEN, seed=3)
    rng = np.random.default_rng(4)
    subs = []
    for _ in range(N_CHROMS):
        pos = np.sort(rng.choice(CHROM_LEN, SUBS, replace=False)).astype(np.uint64)
        subs.append((pos, pos.copy(), rng.choice(np.frombuffer(b"TCAG", np.uint8), SUBS)))
    good = [subs[0], None, subs[2], subs[3], subs[4]]
    ctx = J.Context(0)
    try:
        ctx.set_genome(g)
        assert add(ctx, good, [CHROM_LEN] * N_CHROMS)[:2] == (0, 0)
        old, new, pool = subs[3]
        new = new.copy()
        new[[100, 101]] = new[[101, 100]]                                 # chromosome 3: not sorted by new_pos
        bad = [subs[0], None, subs[2], (old, new, pool), subs[4]]
        sizes = [CHROM_LEN, CHROM_LEN + 1, CHROM_LEN, CHROM_LEN, CHROM_LEN]  # chromosome 1: no mutations, another size
        rc, _, msg = add(ctx, bad, sizes)
        assert rc == _lib.JLP_ERR_ARG
        assert msg == "chromosome without mutations must keep the reference size"
        assert add(ctx, good, [CHROM_LEN] * N_CHROMS)[:2] == (0, 1)       # the failed haplotype was not added
    finally:
        ctx.close()
