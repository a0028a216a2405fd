"""The state a context is left in: after a genome setter fails, and when jlp_ctx_create_multi is given one device."""
import ctypes as C

import pytest

import jackalope_b200 as J
from jackalope_b200 import _lib

pytestmark = pytest.mark.gpu

KW = dict(seq_sys="HS25", prob_dup=0.1, read_pool_size=50, ins_prob1=0.002, del_prob2=0.003)


@pytest.mark.parametrize("devices", [None, [0, 0]], ids=["plain", "dev00"])
def test_a_failed_set_genome_leaves_no_genome(ctx, devices):
    m = J.Context(0) if devices is None else J.Context(devices=devices)
    try:
        # one chromosome of 2^44 bases: allocating 16 TB fails with an ordinary error return; the deferred form copies
        # nothing from the one-byte `bases`
        bases = C.create_string_buffer(1)
        off = (C.c_uint64 * 2)(0, 1 << 44)
        names = (C.c_char_p * 1)(b"big")
        rc = m.lib.jlp_set_genome_async(m.h, C.cast(bases, C.c_void_p), off, 1, names, b"REF")
        assert rc == _lib.JLP_ERR_CUDA, m.lib.jlp_last_error(m.h)
        n = C.c_uint64(0)
        assert m.lib.jlp_get_genome(m.h, None, 0, C.byref(n)) == _lib.JLP_ERR_ARG
        assert m.lib.jlp_last_error(m.h).decode() == "no reference genome has been set"
        # a valid genome afterwards: the context works as a fresh one does
        g = J.random_genome(3, [30_000, 8_000, 20_000], seed=301)
        want = J.illumina(g, "", 6_000, 100, True, seed=11, ctx=ctx, sink="memory", batch_pairs=700, **KW)
        got = J.illumina(g, "", 6_000, 100, True, seed=11, ctx=m, sink="memory", batch_pairs=700, **KW)
        assert got[0] == want[0] and got[1] == want[1]
    finally:
        m.close()


def test_a_one_device_multi_context_is_a_plain_context(ctx):
    m = J.Context(devices=[0])
    try:
        assert m.n_devices == 1
        g = J.random_genome(4, 25_000, seed=302)
        r1, r2, st = J.illumina(g, "", 10_000, 120, True, seed=12, ctx=m, sink="memory", batch_pairs=900, **KW)
        q1, q2, sq = J.illumina(g, "", 10_000, 120, True, seed=12, ctx=ctx, sink="memory", batch_pairs=900, **KW)
        assert r1 == q1 and r2 == q2
        # no size pass: the same batches and launches as the plain context
        for k in ("pairs", "batches", "kernel_launches", "bytes_out", "d2h_bytes"):
            assert st[k] == sq[k], k
    finally:
        m.close()
