"""Pins the CPU oracle (oracle/jlp_oracle.c) to the UNMODIFIED reference built from
/root/reference into oracle/_ref/ (oracle/Makefile):

* replay: the oracle lists, per read, the draws in the order the reference consumes
  them (SURVEY.md Appendix A.1); libjlp_ref_replay.so feeds that ledger to the
  reference's own sample_indels / append_pools / fill_read_qual / fill_fq_lines through a
  scripted pcg64 and must produce byte-identical FASTQ while consuming exactly the
  ledger's number of draws per read;
* haplotype materialisation: random edits through the reference's HapChrom::add_* vs the
  oracle's get_chrom_full restatement (the reference's own differential test,
  tests/testthat/test-R_classes.R:195-244);
* alias tables, quality->error map, reverse complement, the long-double uniform
  expressions.

Skipped where neither /root/reference nor a prebuilt oracle/_ref exists.
The replay tests are not: without the reference they check the oracle against the reference's FASTQ stored for the
same scenario (tests/golden, written by make_golden.py only where the reference consumed exactly the draw ledger).
"""
import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200 import _lib
from oracle import harness as H
from golden.cases import assert_oracle_reproduces
from oracle.compare import hap_sequences, oracle_run

HAVE_REF = H.have_ref(True) and H.have_ref(False)
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref not built")


def genome_with_n(seed=1, n=3, length=5000):
    g = J.random_genome(n, length, seed=seed)
    s = g.seqs[0].copy()
    s[100:160] = ord("N")
    s[1000] = ord("x")          # cmp_map -> NUL -> 'N' (SURVEY.md Appendix F.5)
    g.seqs[0] = s
    return g


def to_ref_haps(haps, edits, replay):
    """Build the reference HapSet by replaying the generator's edits through add_*."""
    ref = H.RefGenomeH(haps.reference.names, [haps.reference.chrom(c) for c in range(haps.n_chroms())], replay=replay)
    hs = H.HapSetH(ref, haps.hap_names)
    for h, eh in enumerate(edits):
        for c, ec in enumerate(eh):
            for kind, pos, payload in ec:
                if kind == "sub":
                    hs.add_sub(h, c, payload, pos)
                elif kind == "ins":
                    hs.add_ins(h, c, payload, pos)
                else:
                    hs.add_del(h, c, payload, pos)
    return hs


def replay_check(obj, n_reads, L, paired, seed, ref_obj=None, **kw):
    o = oracle_run(obj, n_reads, L, paired, seed, want_ledger=True, **kw)
    p = o["params"]
    prof1, prof2 = o["profiles"]
    is_hap = isinstance(obj, J.Haplotypes)
    nc = o["n_chroms"]
    if ref_obj is None:
        ref_obj = H.RefGenomeH(obj.names, [obj.chrom(c) for c in range(nc)], replay=True)
    plan = np.concatenate(o["plan"])
    ledger = np.concatenate(o["ledger"])
    cnt = np.concatenate(o["ledger_cnt"])
    nb = obj.n_haps() if is_hap else 1
    r = H.ref_replay(ref_obj, is_hap=is_hap, paired=bool(p.paired), matepair=bool(p.matepair), prof1=prof1, prof2=prof2,
                     ins_prob=[p.ins_prob1, p.ins_prob2], del_prob=[p.del_prob1, p.del_prob2],
                     barcodes=[p.barcodes[i] for i in range(nb)],
                     hap=plan[:, 0] // nc, chrom=plan[:, 0] % nc, frag_len=plan[:, 1], frag_start=plan[:, 2],
                     script=ledger)
    assert np.array_equal(r["consumed"], cnt), "the reference consumed a different number of draws"
    assert r["r1"] == o["r1"]
    assert r["r2"] == o["r2"]
    return o


@pytest.mark.parametrize("paired,matepair", [(False, False), (True, False), (True, True)])
def test_replay_ref_default_args(paired, matepair):
    if not HAVE_REF:
        assert_oracle_reproduces({False: "se100_default", True: "mp100_default" if matepair else "pe100_default"}[paired])
        return
    replay_check(genome_with_n(), 1200, 100, paired, seed=11, matepair=matepair)


def test_replay_pe150_hs25():
    if not HAVE_REF:
        assert_oracle_reproduces("pe150_hs25")
        return
    replay_check(genome_with_n(seed=2, n=4, length=9000), 1500, 150, True, seed=12, seq_sys="HS25")


def test_replay_high_indels_dups_barcode():
    if not HAVE_REF:
        assert_oracle_reproduces("pe100_indels_dups_barcode")
        return
    replay_check(genome_with_n(seed=4), 1500, 100, True, seed=13, ins_prob1=0.02, del_prob1=0.03, ins_prob2=0.05,
                 del_prob2=0.01, prob_dup=0.4, read_pool_size=14, barcodes=["ACGTTG"])


def test_replay_short_fragments_and_chromosomes():
    if not HAVE_REF:
        assert_oracle_reproduces("pe100_short_fragments")
        return
    g = J.RefGenome(["a", "b", "c"], [J.random_genome(1, 60, seed=5).seqs[0], J.random_genome(1, 4000, seed=6).seqs[0],
                                      J.random_genome(1, 130, seed=7).seqs[0]])
    replay_check(g, 1500, 100, True, seed=14, frag_mean=120, frag_sd=40, frag_len_min=20, ins_prob1=0.01,
                 del_prob1=0.01)


def test_replay_haplotypes():
    if not HAVE_REF:
        assert_oracle_reproduces("hap_pe100_pooled")
        assert_oracle_reproduces("hap_se100_sep_files")
        return
    g = J.random_genome(3, 6000, seed=8)
    haps, edits = J.random_haplotypes(g, 3, sub_rate=0.02, indel_rate=0.005, seed=9, return_edits=True)
    hs = to_ref_haps(haps, edits, replay=True)
    replay_check(haps, 1500, 100, True, seed=15, ref_obj=hs, haplotype_probs=[1, 2, 4], barcodes=["AC", "GT", "TT"])
    replay_check(haps, 900, 100, False, seed=16, ref_obj=hs, sep_files=True)


@needs_ref
def test_materialize_matches_reference():
    g = J.random_genome(3, 20000, seed=3)
    haps, edits = J.random_haplotypes(g, 3, sub_rate=0.02, indel_rate=0.01, seed=5, return_edits=True)
    hs = to_ref_haps(haps, edits, replay=False)
    want = hap_sequences(haps)
    for h in range(3):
        for c in range(3):
            full = hs.chrom_full(h, c)
            assert hs.chrom_size(h, c) == haps.muts[h][c].chrom_size
            assert full == want[h][c]
            # and the flat arrays our generator wrote are the ones the reference holds
            op, npos, no, nl, pool = hs.muts(h, c)
            m = haps.muts[h][c]
            assert np.array_equal(op, m.old_pos) and np.array_equal(npos, m.new_pos)
            assert np.array_equal(nl, m.nuc_len) and pool == m.pool.tobytes()


@needs_ref
def test_materialize_random_edit_order():
    """The reference's differential test applies edits in random order at random
    haplotype positions (tests/testthat/test-R_classes.R:195-244); mirror it with a
    plain-Python string model and check oracle == reference == model."""
    rng = np.random.default_rng(7)
    g = J.random_genome(2, 400, seed=21)
    ref = H.RefGenomeH(g.names, [g.chrom(c) for c in range(2)])
    hs = H.HapSetH(ref, ["h0", "h1"])
    model = [[bytearray(g.chrom(c)) for c in range(2)] for _ in range(2)]
    for h in range(2):
        for c in range(2):
            for _ in range(100):
                s = model[h][c]
                kind = rng.integers(0, 3)
                pos = int(rng.integers(0, len(s)))
                if kind == 0:
                    nt = b"TCAG"[rng.integers(0, 4)]
                    hs.add_sub(h, c, bytes([nt]), pos)
                    s[pos] = nt
                elif kind == 1:
                    ins = bytes(b"TCAG"[i] for i in rng.integers(0, 4, size=int(rng.integers(1, 11))))
                    hs.add_ins(h, c, ins, pos)
                    s[pos + 1:pos + 1] = ins
                else:
                    size = int(min(rng.integers(1, 11), len(s) - pos))
                    if size >= len(s):
                        continue
                    hs.add_del(h, c, size, pos)
                    del s[pos:pos + size]
            full = hs.chrom_full(h, c)
            assert full == bytes(model[h][c])
            op, npos, no, nl, pool = hs.muts(h, c)
            assert H.materialize(g.chrom(c), op, npos, no, pool, len(full)) == full


@needs_ref
def test_alias_tables_and_error_map_match_reference():
    for L, seq_sys in ((100, "HS25"), (150, "HS25"), (36, "GA1")):
        for read in (1, 2):
            flat = J.flatten_profile(J.read_profile(None, seq_sys, L, read))
            _, nq, probs, quals = flat
            off = 0
            for n in nq[::7]:      # every 7th table keeps this fast
                pr = probs[off:off + n]
                P0, A0 = H.alias_build(pr)
                P1, A1 = H.ref_alias_build(pr)
                assert np.array_equal(P0, P1) and np.array_equal(A0, A1)
                off += int(nq[0]) * 0 + int(n)
            ref_map = np.zeros(256)
            n = H.ref_lib().jref_qual_prob_map(L, H._ptr(nq, H.u32p), H._ptr(probs, H.f64p), H._ptr(quals, H.u8p),
                                               H._ptr(ref_map, H.f64p), 256)
            assert n > 0
            assert np.array_equal(H.qual_prob_map(flat)[:n], ref_map[:n])


@needs_ref
def test_rev_comp_matches_reference():
    rng = np.random.default_rng(3)
    import ctypes as C
    for n in (0, 1, 2, 7, 100, 151):
        s = bytes(rng.choice(np.frombuffer(b"TCAGNxn", np.uint8), size=n))
        a, b = C.create_string_buffer(s, max(n, 1)), C.create_string_buffer(s, max(n, 1))
        H.oracle().orc_rev_comp(a, n)
        H.ref_lib().jref_rev_comp(b, n)
        assert a.raw[:n] == b.raw[:n]


@needs_ref
def test_uniform_expressions_match_reference():
    """oracle (literal long double), product (integer restatement, jlp_unif_expr /
    jlp_threshold) and the reference's own expressions agree on random and edge draws."""
    lib, orc, ref = _lib.lib(), H.oracle(), H.ref_lib()
    rng = np.random.default_rng(5)
    xs = [0, 1, 2, 2 ** 63 - 1, 2 ** 63, 2 ** 64 - 2, 2 ** 64 - 1] + [int(x) for x in rng.integers(0, 2 ** 64, size=3000, dtype=np.uint64)]
    # products sitting on an integer boundary: x+1 = ceil(k * 2^64 / n)
    for n in (3, 4, 8, 10, 22, 999901):
        for k in range(1, min(n, 12)):
            b = -(-(k << 64) // n)
            xs += [b - 2, b - 1, b]
    for x in xs:
        x &= 2 ** 64 - 1
        for n in (3, 4, 8, 10, 22, 999901):
            want = ref.jref_unif_expr(0, x, 0.0, n)
            assert orc.orc_unif_expr(0, x, 0.0, n) == want
            assert lib.jlp_unif_expr(0, x, 0.0, n) == want
            w5 = ref.jref_unif_expr(5, x, 0.0, n)
            assert orc.orc_unif_expr(5, x, 0.0, n) == w5 and lib.jlp_unif_expr(5, x, 0.0, n) == w5
        assert orc.orc_unif_expr(4, x, 0.0, 0) == ref.jref_unif_expr(4, x, 0.0, 0) == lib.jlp_unif_expr(4, x, 0.0, 0)
    # thresholds: count of x satisfying the predicate, checked on both sides of the edge
    import ctypes as C
    for p in (0.0, 1.0, 0.5, 0.02, 9e-5, 2e-4, 1e-4 + 9e-5, 10 ** -4.1, 10 ** -0.2, 0.9999999, 1e-300, 0.3333333333333333):
        for kind, expr, truth in ((1, 1, 1), (2, 2, 0), (3, 3, 1)):
            thr, al = C.c_uint64(), C.c_int()
            assert lib.jlp_threshold(kind, p, C.byref(thr), C.byref(al)) == 0
            t = thr.value
            if al.value:
                assert ref.jref_unif_expr(expr, 2 ** 64 - 1, p, 0) == truth
                continue
            if t > 0:
                assert ref.jref_unif_expr(expr, t - 1, p, 0) == truth
            assert ref.jref_unif_expr(expr, t, p, 0) == 1 - truth


@needs_ref
def test_pair_geometry_known_answers_through_the_reference():
    """tests/testthat/test-sequencer.R:81-161 run on the unmodified reference end to end
    (real pcg64): chromosome C25 N150 T25, fragment forced to 200, error-free profile."""
    import os
    import tempfile
    chrom = b"C" * 25 + b"N" * 150 + b"T" * 25
    ref = H.RefGenomeH(["chrom0"], [chrom])
    L = 100
    nq = np.ones(4 * L, dtype=np.uint32)
    flat = (L, nq, np.ones(4 * L), np.full(4 * L, 255, dtype=np.uint8))
    for matepair, want in ((False, {b"C" * 25 + b"N" * 75, b"A" * 25 + b"N" * 75}),
                           (True, {b"N" * 75 + b"T" * 25, b"N" * 75 + b"G" * 25})):
        with tempfile.TemporaryDirectory() as d:
            pre = os.path.join(d, "t")
            H.ref_illumina_ref(ref, paired=True, matepair=matepair, out_prefix=pre, n_reads=200, prob_dup=0.02,
                               n_threads=1, read_pool_size=1000, shape=100.0, scale=2.0, frag_len_min=200,
                               frag_len_max=200, prof1=flat, prof2=flat, ins_prob=[0, 0], del_prob=[0, 0])
            for k in (1, 2):
                lines = open("%s_R%d.fq" % (pre, k), "rb").read().split(b"\n")
                assert set(lines[1::4]) - {b""} == want


@needs_ref
@pytest.mark.parametrize("pi", [[0.25, 0.25, 0.25, 0.25], [0.1, 0.2, 0.3, 0.4], [0, 1, 0, 3], [5, 1, 1, 1]])
def test_create_genome_replay(pi):
    """create_genome: the reference's sampling loop (AliasSampler::sample per base,
    src/create_sequences.cpp:129-132) fed with the oracle's draw ledger gives the oracle's chromosome."""
    for chrom, n in ((0, 1), (3, 4097), (7, 20000)):
        seq, led = H.create_chrom(99, chrom, n, pi, want_ledger=True)
        ref_seq, used = H.ref_create_chrom_replay(pi, n, led)
        assert used == 2 * n and ref_seq == seq
    lib = _lib.lib()
    assert all(lib.jlp_genome_draw(99, 3, p, w) == H.oracle().orc_genome_draw(99, 3, p, w)
               for p in list(range(0, 200)) + [2 ** 33 + 5] for w in (0, 1))
