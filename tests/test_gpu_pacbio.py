"""PacBio reads (SURVEY.md section 8f rank 3) on the GPU through the C ABI, byte-compared with the oracle.

The library reports what it drew per read before the per-base work (jlp_pacbio_read_plan: group, read length, pass
split -- the statistical tier, tests/test_pacbio_samplers.py); those values are injected into the oracle, which the
unmodified reference replays byte for byte (tests/test_pacbio_oracle.py), and everything after them -- error
probabilities and qualities, the insertion / deletion / substitution walk, template start, strand, extraction,
reverse complement, the edits, the FASTQ record -- must then be identical."""
import gzip

import numpy as np
import pytest

import jackalope_b200 as J
from common import first_diff, hap_sequences
from oracle import harness_pacbio as P

pytestmark = pytest.mark.gpu


def oracle_for(obj, plan, seed, prob_dup=0.0, pool_reads=100, **model):
    if isinstance(obj, J.Haplotypes):
        hs = hap_sequences(obj)
        seqs = [hs[h][c] for h in range(obj.n_haps()) for c in range(len(obj.reference.names))]
        names = [n for _ in range(obj.n_haps()) for n in obj.reference.names]
        gnames = [h for h in obj.hap_names for _ in obj.reference.names]
    else:
        seqs, names, gnames = [bytes(s) for s in obj.seqs], list(obj.names), "REF"
    counts = np.bincount(plan["group"].astype(np.int64), minlength=len(seqs))
    assert (np.diff(plan["group"].astype(np.int64)) >= 0).all()
    return P.generate(names, seqs, gnames, counts, plan["read_len"], plan["split_pos"], plan["passes_left"],
                      plan["passes_right"], seed, want_ledger=False, beyond_template_is_n=True, prob_dup=prob_dup,
                      pool_reads=pool_reads, **model)["fastq"]


def check(ctx, obj, n_reads, seed, **kw):
    fq, st, plan = J.pacbio(obj, "", n_reads, seed=seed, ctx=ctx, sink="memory", want_plan=True, **kw)
    model = {k: kw[k] for k in ("sqrt_params", "norm_params", "prob_thresh", "ins_prob", "del_prob", "sub_prob") if k in kw}
    want = oracle_for(obj, plan, seed, prob_dup=kw.get("prob_dup", 0.0), pool_reads=kw.get("read_pool_size", 100), **model)
    d = first_diff(fq, want)
    assert d is None, "differs at byte %d: gpu=%r oracle=%r" % (d, fq[max(0, d - 60):d + 40], want[max(0, d - 60):d + 40])
    assert st["pairs"] == n_reads and (fq.count(b"\n") == 4 * n_reads or kw.get("prob_dup", 0) > 0)
    return fq, st, plan


def genome(seed, n, length, with_n=True):
    g = J.random_genome(n, length, seed=seed)
    if with_n:
        s = g.seqs[0].copy()
        s[100:160] = ord("N")
        s[1000] = ord("x")
        g.seqs[0] = s
    return g


def test_pacbio_ref_defaults(ctx):
    fq, st, plan = check(ctx, genome(1, 3, 60000), 300, seed=11)
    assert 3000 < plan["read_len"].mean() < 15000


def test_pacbio_several_batches_and_custom_lengths(ctx):
    g = genome(2, 4, 30000)
    a, _, _ = check(ctx, g, 500, seed=12, custom_read_lengths=[[200, 1], [1500, 2], [4000, 1]], batch_reads=64)
    b, _, _ = check(ctx, g, 500, seed=12, custom_read_lengths=[[200, 1], [1500, 2], [4000, 1]])
    assert a == b                                      # output does not depend on the batch size


def test_pacbio_reads_as_long_as_chromosomes(ctx):
    # reads limited by short chromosomes: no spare template for deletions, read_chrom_space == chrom_len, start 0
    g = J.RefGenome(["a", "b", "c"], [J.random_genome(1, n, seed=5 + n).seqs[0] for n in (300, 1200, 5000)])
    check(ctx, g, 400, seed=13, custom_read_lengths=[[250, 1], [1300, 1], [6000, 1]])


def test_pacbio_high_error_rates_and_tail_branch(ctx):
    g = genome(3, 2, 20000)
    check(ctx, g, 200, seed=14, ins_prob=0.3, del_prob=0.25, sub_prob=0.2, custom_read_lengths=[900, 2500])
    check(ctx, g, 200, seed=15, norm_params=(-10.0, 0.1), custom_read_lengths=[900, 2500])


def test_pacbio_haplotypes_pooled_and_sep_files(ctx, tmp_path):
    g = genome(4, 3, 40000, with_n=False)
    haps = J.random_haplotypes(g, 3, sub_rate=0.01, indel_rate=0.002, seed=6)
    kw = dict(haplotype_probs=[1, 2, 3], custom_read_lengths=[[800, 1], [3000, 1]])
    fq, _, _ = check(ctx, haps, 300, seed=16, **kw)
    # one writer thread and the default batches; four writer threads (mapped files, zlib in slices) and small batches
    for i, files_kw in enumerate([{}, dict(n_threads=4, batch_reads=64)]):
        pre = str(tmp_path / ("pb%d" % i))
        J.pacbio(haps, pre, 300, seed=16, ctx=ctx, sep_files=True, **kw, **files_kw)
        assert b"".join(open("%s_%s_R1.fq" % (pre, h), "rb").read() for h in haps.hap_names) == fq
        J.pacbio(haps, pre + "z", 300, seed=16, ctx=ctx, compress=True, **kw, **files_kw)      # BGZF written by the GPU
        assert gzip.decompress(open(pre + "z_R1.fq.gz", "rb").read()) == fq
        J.pacbio(haps, pre + "h", 300, seed=16, ctx=ctx, compress=9, **kw, **files_kw)         # zlib on the host
        assert gzip.decompress(open(pre + "h_R1.fq.gz", "rb").read()) == fq
    pre = str(tmp_path / "pb0")
    with pytest.raises(J.JackalopeError, match="already exists"):
        J.pacbio(haps, pre, 300, seed=16, ctx=ctx, sep_files=True, **kw)


def test_pacbio_end_to_end_statistics_against_the_reference(ctx, tmp_path):
    """The whole generator against the unmodified reference run end to end on its own pcg64 streams (two-sample
    tests, alpha = 1e-3): read lengths, the two quality characters of a read and where they split, strand, reads per
    chromosome, and the observed mismatch-free fraction of short exact k-mers as a proxy for the error rates."""
    import ctypes as C
    from scipy import stats
    from oracle import harness as H
    if not H.have_ref(False):
        pytest.skip("oracle/_ref not built")
    g = genome(21, 4, 200000, with_n=False)
    n = 6000
    fq, _, _ = J.pacbio(g, "", n, seed=31, ctx=ctx, sink="memory", want_plan=True)
    lib = H.ref_lib(False)
    f64p, u64p = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
    lib.jrefpb_pacbio_ref.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_double] * 5 + \
        [f64p, u64p, C.c_uint64, C.c_uint64, f64p, f64p, f64p, f64p] + [C.c_double] * 4 + [C.c_char_p, C.c_uint64]
    rg = H.RefGenomeH(g.names, [bytes(s) for s in g.seqs])
    D = P.DEFAULTS
    arr = lambda x: np.ascontiguousarray(x, dtype=np.float64)
    cn, cs, sq, nm = arr(D["chi2_params_n"]), arr(D["chi2_params_s"]), arr(D["sqrt_params"]), arr(D["norm_params"])
    ln = D["lognorm_read_length"]
    err = C.create_string_buffer(256)
    lib.jref_set_r_seed(12345)
    pre = str(tmp_path / "ref")
    assert lib.jrefpb_pacbio_ref(rg.h, pre.encode(), n, 1, 100, 0.0, ln[2], ln[0], ln[1], 50.0, None, None, 0, 40,
                                 cn.ctypes.data_as(f64p), cs.ctypes.data_as(f64p), sq.ctypes.data_as(f64p),
                                 nm.ctypes.data_as(f64p), 0.2, 0.11, 0.04, 0.01, err, 256) == 0, err.value
    ref = open(pre + "_R1.fq", "rb").read()

    def features(b):
        L = b.split(b"\n")[:-1]
        ids, seqs, quals = L[0::4], L[1::4], L[3::4]
        lens = np.array([len(s) for s in seqs], dtype=float)
        strand = np.array([i.endswith(b"-R") for i in ids])
        chrom = np.array([int(i.split(b"-")[1][5:]) for i in ids])
        ql = np.array([q[0] for q in quals]); qr = np.array([q[-1] for q in quals])
        split = np.array([len(q) - len(q.lstrip(bytes([q[0]]))) if q[0] != q[-1] else len(q) for q in quals]) / lens
        return lens, strand, chrom, ql, qr, split

    a, b = features(fq), features(ref)
    assert len(a[0]) == len(b[0]) == n
    assert stats.ks_2samp(a[0], b[0]).pvalue > 1e-3                                              # read lengths
    assert stats.chi2_contingency([[a[1].sum(), (~a[1]).sum()], [b[1].sum(), (~b[1]).sum()]])[1] > 1e-3   # strand
    # reads per chromosome: a deliberate deviation.  PacBioOneGenome never decrements chrom_reads (src/hts_pacbio.cpp:147,
    # :200 look for the first chromosome with reads left; nothing takes them away, unlike IlluminaOneGenome,
    # src/hts_illumina.cpp:404-406, and PacBioHaplotypes), so with a reference genome the reference takes EVERY read from
    # the first chromosome; here the reads are apportioned by chromosome length, as add_n_reads intends.
    ca, cb = np.bincount(a[2], minlength=4), np.bincount(b[2], minlength=4)
    assert cb[0] == n and cb[1:].sum() == 0
    assert stats.chisquare(ca).pvalue > 1e-3                                                     # four equal chromosomes
    for k in (3, 4):                                                                              # quality characters
        vals = np.union1d(a[k], b[k])
        ta, tb = np.array([(a[k] == v).sum() for v in vals]), np.array([(b[k] == v).sum() for v in vals])
        keep = (ta + tb) >= 20
        assert stats.chi2_contingency([np.append(ta[keep], ta[~keep].sum() + 1), np.append(tb[keep], tb[~keep].sum() + 1)])[1] > 1e-3
    assert stats.ks_2samp(a[5], b[5]).pvalue > 1e-3                                              # where the quality changes


def test_pacbio_duplicates(ctx):
    """prob_dup > 0 (ReadWriterOneThread::create_reads + PacBioOneGenome::re_read): chains inside pools, the chain's
    chromosome, read length and start, new passes / errors / strand; batches are whole pools."""
    g = genome(7, 3, 30000)
    kw = dict(prob_dup=0.4, read_pool_size=7, custom_read_lengths=[[300, 1], [1500, 2], [4000, 1]])
    a, _, plan = check(ctx, g, 600, seed=41, batch_reads=64, **kw)
    b, _, _ = check(ctx, g, 600, seed=41, **kw)
    assert a == b
    ids = a.split(b"\n")[0::4][:-1]
    starts = [i.rsplit(b"-", 2)[1] for i in ids]
    same = sum(starts[k] == starts[k - 1] for k in range(1, len(starts)))
    assert 0.25 * 600 < same < 0.5 * 600                       # about prob_dup * (1 - 1/pool) of the reads repeat a start
    haps = J.random_haplotypes(genome(8, 2, 20000, with_n=False), 2, seed=9)
    check(ctx, haps, 300, seed=42, prob_dup=0.3, read_pool_size=10, custom_read_lengths=[700, 2500])


def test_pacbio_duplicates_of_chromosome_long_reads(ctx):
    """Duplicates whose own walk needs more template than the chain's start leaves: deletions are given up from the
    back until it fits, and a read that still does not fit is not written (fewer than n_reads records)."""
    g = J.RefGenome(["a", "b", "c"], [J.random_genome(1, n, seed=50 + n).seqs[0] for n in (700, 400, 900)])
    fq, st, plan = check(ctx, g, 600, seed=43, prob_dup=0.6, read_pool_size=9, custom_read_lengths=[[1000, 3], [650, 1]])
    n_rec = fq.count(b"\n") // 4
    assert 400 < n_rec < 600                                   # some duplicates cannot be written
    check(ctx, g, 300, seed=44, prob_dup=0.5, read_pool_size=5, custom_read_lengths=[[1000, 1]], ins_prob=0.05, del_prob=0.2,
          sub_prob=0.02)                                       # many deletions to give up


def test_pacbio_shards_concatenate(ctx):
    """One process per GPU takes shard (k, n) of every job: whole pools, so chains of duplicates stay inside a shard; the
    shards' outputs concatenate to the unsharded run."""
    g = genome(9, 3, 30000)
    kw = dict(prob_dup=0.3, read_pool_size=11, custom_read_lengths=[[300, 1], [2000, 2]])
    whole, _ = J.pacbio(g, "", 500, seed=45, ctx=ctx, sink="memory", **kw)
    parts = [J.pacbio(g, "", 500, seed=45, ctx=ctx, sink="memory", shard=(k, 3), **kw)[0] for k in range(3)]
    assert all(len(p) > 0 for p in parts) and b"".join(parts) == whole
    haps = J.random_haplotypes(genome(10, 2, 20000, with_n=False), 3, seed=11)
    hk = dict(sep_files=True, haplotype_probs=[3, 2, 1], custom_read_lengths=[900, 2500])
    whole, _ = J.pacbio(haps, "", 400, seed=46, ctx=ctx, sink="memory", **hk)
    parts = [J.pacbio(haps, "", 400, seed=46, ctx=ctx, sink="memory", shard=(k, 2), **hk)[0] for k in range(2)]
    # with sep_files every job (haplotype) is split: shard 0 holds the first halves, in haplotype order
    assert sum(len(p) for p in parts) == len(whole) and sorted(b"".join(parts).split(b"@")) == sorted(whole.split(b"@"))


def test_pacbio_callbacks(ctx):
    """jlp_pacbio_params.progress_cb / abort_cb (Progress::increment / check_abort of the shared driver,
    /root/reference/src/hts.h:396-399,414): progress adds up to n_reads over the batches; an abort request ends the
    run with JLP_ERR_ABORTED."""
    import ctypes as C
    from jackalope_b200 import _lib
    from jackalope_b200.pacbio import _params
    from oracle.harness_pacbio import DEFAULTS as D
    g = J.random_genome(2, 40_000, seed=51)
    ctx.set_genome(g)
    p, keep = _params(g, "", 900, D["chi2_params_s"], D["chi2_params_n"], D["max_passes"], D["sqrt_params"], D["norm_params"],
                      D["prob_thresh"], D["ins_prob"], D["del_prob"], D["sub_prob"], D["min_read_length"], D["lognorm_read_length"],
                      None, 0.0, None, False, 0, "bgzip", 2, 100, 77, 200, "auto")
    seen = [0, 0]

    def progress(_u, n):
        seen[0] += n
        seen[1] += 1

    p.progress_cb = _lib.PROGRESS_CB(progress)
    p.abort_cb = _lib.ABORT_CB(lambda _u: 0)
    st, n = _lib.RunStats(), C.c_uint64()
    assert ctx.lib.jlp_pacbio_to_memory(ctx.h, 0, C.byref(p), None, 0, C.byref(n), C.byref(st)) == 0
    assert seen == [900, 5]
    calls = [0]

    def abort(_u):
        calls[0] += 1
        return 1 if calls[0] > 2 else 0

    p.abort_cb = _lib.ABORT_CB(abort)
    assert ctx.lib.jlp_pacbio_to_memory(ctx.h, 0, C.byref(p), None, 0, C.byref(n), C.byref(st)) == _lib.JLP_ERR_ABORTED
    assert seen[0] == 900 + 2 * 200


def _c_params(ctx, out_prefix):
    """jlp_pacbio_params of a small reference run, set up as test_pacbio_callbacks sets them up."""
    from jackalope_b200.pacbio import _params
    from oracle.harness_pacbio import DEFAULTS as D
    g = J.random_genome(2, 40_000, seed=51)
    ctx.set_genome(g)
    return _params(g, out_prefix, 900, D["chi2_params_s"], D["chi2_params_n"], D["max_passes"], D["sqrt_params"], D["norm_params"],
                   D["prob_thresh"], D["ins_prob"], D["del_prob"], D["sub_prob"], D["min_read_length"], D["lognorm_read_length"],
                   None, 0.0, None, False, 0, "bgzip", 2, 100, 77, 200, "auto")


def test_pacbio_rejects_an_unknown_comp_engine(ctx, tmp_path):
    """comp_engine is checked as for Illumina and VCF: 7 is an argument error, not zlib output."""
    import ctypes as C
    from jackalope_b200 import _lib
    p, keep = _c_params(ctx, str(tmp_path / "pb"))
    p.compress, p.comp_engine = 6, 7
    assert ctx.lib.jlp_pacbio(ctx.h, 0, C.byref(p), C.byref(_lib.RunStats())) == _lib.JLP_ERR_ARG
    assert b"comp_engine" in ctx.lib.jlp_last_error(ctx.h)
    assert not (tmp_path / "pb_R1.fq.gz").exists()


def test_pacbio_bad_shard_leaves_existing_file(ctx, tmp_path):
    """shard_index >= shard_count is rejected before the job's file is opened (and truncated)."""
    import ctypes as C
    from jackalope_b200 import _lib
    prefix = tmp_path / "pb"
    p, keep = _c_params(ctx, str(prefix))
    p.shard_index, p.shard_count = 2, 2
    old = tmp_path / "pb_R1.fq"
    old.write_bytes(b"@earlier run\nACGT\n+\nIIII\n")
    assert ctx.lib.jlp_pacbio(ctx.h, 0, C.byref(p), C.byref(_lib.RunStats())) == _lib.JLP_ERR_ARG
    assert b"shard_index" in ctx.lib.jlp_last_error(ctx.h)
    assert old.read_bytes() == b"@earlier run\nACGT\n+\nIIII\n"
