"""write_vcf on the GPU: the uncompressed file byte-identical to the oracle's (create_haplotypes with and without
indels, random_haplotypes, hand-written records, N runs, several chromosomes, haploid / diploid / triploid matrices,
4096 samples), independent of the batch size, the device file applied back to the reference, compressed files, a
multi-device context, determinism, and the C ABI's errors."""
import ctypes as C
import gzip

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200 import _lib
from oracle import vcf_oracle as V
from test_vcf_host import CASES, R, haps_of

pytestmark = pytest.mark.gpu

DATE = "20261021"


def genome_with_n_runs(lens, seed):
    g = J.random_genome(len(lens), lens, seed=seed)
    rng = np.random.default_rng(seed)
    seqs = []
    for s in g.seqs:
        s = s.copy()
        for _ in range(3):
            a = int(rng.integers(0, s.size))
            s[a:a + int(rng.integers(1, 3000))] = ord("N")
        s[:min(7, s.size)] = np.frombuffer(b"nNRacgt", dtype=np.uint8)[:min(7, s.size)]
        seqs.append(s)
    return J.RefGenome(g.names, seqs)


def gpu_vcf(ctx, haps, path, **kw):
    st = J.write_vcf(haps, str(path), ctx=ctx, file_date=DATE, overwrite=True, **kw)
    fn = str(path) + (".vcf.gz" if kw.get("compress") else ".vcf")
    with open(fn, "rb") as f:
        return f.read(), st


def same_as_oracle(ctx, haps, tmp_path, sample_matrix=None, **kw):
    got, st = gpu_vcf(ctx, haps, tmp_path / "o", sample_matrix=sample_matrix, **kw)
    want = V.vcf(haps, sample_matrix=sample_matrix, file_date=DATE)
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        raise AssertionError("differs at byte %d: got %r want %r" % (i, got[i - 80:i + 80], want[i - 80:i + 80]))
    assert st["text_bytes"] == len(want) == st["file_bytes"]
    assert st["lines"] == sum(1 for ln in want.split(b"\n") if ln and not ln.startswith(b"#"))
    return got, st


@pytest.mark.parametrize("n_tips", [2, 40, 1024])
def test_substitutions_only(ctx, tmp_path, n_tips):
    g = genome_with_n_runs([30_011, 8_193, 5], seed=n_tips)
    haps = J.create_haplotypes(g, J.haps_theta(0.02, n_tips), J.sub_TN93([0.1, 0.2, 0.3, 0.4], 3, 1.2, 0.5, gamma_shape=0.5),
                               seed=3, ctx=ctx)
    same_as_oracle(ctx, haps, tmp_path)


@pytest.mark.parametrize("kinds", ["ins", "del", "both"])
def test_with_indels(ctx, tmp_path, kinds):
    g = genome_with_n_runs([40_003, 777, 9_000], seed=4)
    ins = J.indels(0.05, max_length=12) if kinds in ("ins", "both") else None
    dele = J.indels(0.05, max_length=12) if kinds in ("del", "both") else None
    haps = J.create_haplotypes(g, J.haps_theta(0.05, 12), J.sub_HKY85([0.1, 0.2, 0.3, 0.4], 2, 0.5), ins=ins, del_=dele,
                               epsilon=0.03, seed=5, ctx=ctx)
    same_as_oracle(ctx, haps, tmp_path)
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=[[0, 3], [11, 11], [5, 0]])


def test_a_chromosome_lost_entirely(ctx, tmp_path):
    g = J.random_genome(3, [3_000, 6, 2_000], seed=7)
    info, sub = J.haps_phylo("(a:3,(b:0.01,c:2):0.5);"), J.sub_JC69(1.0)
    for seed in range(100, 200):
        haps = J.create_haplotypes(g, info, sub, ins=J.indels(0.01), del_=J.indels(1.5, max_length=4), epsilon=0.05, seed=seed,
                                   ctx=ctx)
        if any(haps.muts[h][1].chrom_size == 0 for h in range(3)):
            break
    got, _ = same_as_oracle(ctx, haps, tmp_path)
    assert b"<DEL>" in got


def test_random_haplotypes_and_matrices(ctx, tmp_path):
    g = genome_with_n_runs([20_000, 1, 15_000, 3], seed=8)
    haps = J.random_haplotypes(g, 7, sub_rate=0.01, indel_rate=0.003, seed=9)
    haps.muts[3][2] = J.HapChromMuts.empty(15_000)            # a chromosome without records in one haplotype
    same_as_oracle(ctx, haps, tmp_path)
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=[[1, 1], [6, 0], [2, 5]])
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=[[4, 4, 4], [0, 3, 6]])
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=[[5]])


def test_hand_written_records(ctx, tmp_path):
    for per_hap, _ in CASES:
        same_as_oracle(ctx, haps_of(R, per_hap), tmp_path)
    # no lines at all: the header alone
    got, st = same_as_oracle(ctx, haps_of(R, [[("sub", 3, b"T")], []]), tmp_path)
    assert st["lines"] == 0 and got.endswith(b"FORMAT\th0\th1\n")


def test_more_than_nine_alts_and_4096_samples(ctx, tmp_path):
    ref = b"ACGT" * 50
    per_hap = [[("ins", 10, b"G" * (h + 1)), ("sub", 40 + h % 3, b"A")] for h in range(14)] + [[]]
    haps = haps_of(ref, per_hap)
    rng = np.random.default_rng(1)
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=rng.integers(0, 15, size=(4096, 2)))
    same_as_oracle(ctx, haps, tmp_path, sample_matrix=rng.integers(0, 15, size=(33, 3)))


def big_haps(ctx):
    g = genome_with_n_runs([200_003, 50_000, 7], seed=10)
    return J.create_haplotypes(g, J.haps_theta(0.05, 20), J.sub_JC69(1.0), ins=J.indels(0.02), del_=J.indels(0.02),
                               epsilon=0.03, seed=11, ctx=ctx)


def test_batches_round_trip_compression(ctx, tmp_path):
    haps = big_haps(ctx)
    plain, st = same_as_oracle(ctx, haps, tmp_path)
    small, st2 = gpu_vcf(ctx, haps, tmp_path / "b", batch_bytes=1000)
    assert small == plain and st2["batches"] > 20 * st["batches"]
    # the device file applied to the reference gives every haplotype as the context materialises it
    for h in range(haps.n_haps()):
        seq = V.apply(plain, haps.reference, h)
        for c, n in enumerate(haps.reference.names):
            assert seq[n] == ctx.haplotype_chrom(h, c), (h, c)
    for level, engine in ((1, "auto"), (6, "auto"), (9, "auto"), (3, "host")):
        z, zs = gpu_vcf(ctx, haps, tmp_path / ("z%d" % level), compress=level, comp_engine=engine, batch_bytes=50_000)
        assert gzip.decompress(z) == plain and zs["file_bytes"] == len(z) < len(plain) / 2
        if level <= 6 and engine == "auto":
            assert zs["bgzf_ms"] > 0 and z.endswith(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))


def test_multi_device_determinism_after_illumina(ctx, tmp_path):
    haps = big_haps(ctx)
    a, _ = gpu_vcf(ctx, haps, tmp_path / "a", sample_matrix=[[0, 1], [2, 19]])
    b, _ = gpu_vcf(ctx, haps, tmp_path / "b", sample_matrix=[[0, 1], [2, 19]])
    assert a == b
    J.illumina(haps, "", 2000, 150, True, seq_sys="HS25", seed=1, ctx=ctx, sink="memory")
    c, _ = gpu_vcf(ctx, haps, tmp_path / "c", sample_matrix=[[0, 1], [2, 19]])
    assert c == a
    m = J.Context(devices=[0, 0])
    try:
        d, _ = gpu_vcf(m, haps, tmp_path / "d", sample_matrix=[[0, 1], [2, 19]])
    finally:
        m.close()
    assert d == a


def test_c_abi_errors(tmp_path):
    ctx = J.Context(0)
    try:
        L = ctx.lib
        S = np.zeros(1, dtype=np.uint64)
        names = (C.c_char_p * 1)(b"s")

        def call(path, hap):
            S[0] = hap
            p = _lib.VcfParams(path=str(path).encode(), n_samples=1, ploidy=1, sample_haps=S.ctypes.data_as(_lib.u64p),
                               sample_names=names, file_date=DATE.encode(), compress=0, comp_method=b"bgzip", comp_engine=0,
                               n_threads=1, batch_bytes=0)
            return L.jlp_write_vcf(ctx.h, C.byref(p), C.byref(_lib.VcfStats()))

        haps = haps_of(R, [[("sub", 3, b"A")], []])
        ctx.set_genome(haps.reference)
        assert call(tmp_path / "n.vcf", 0) == _lib.JLP_ERR_ARG and b"haplotypes" in L.jlp_last_error(ctx.h)
        ctx.set_haplotypes(haps)
        assert call(tmp_path / "r.vcf", 2) == _lib.JLP_ERR_ARG and b"out of range" in L.jlp_last_error(ctx.h)
        assert call(tmp_path / "no" / "dir" / "x.vcf", 0) == _lib.JLP_ERR_IO
        assert call(tmp_path / "ok.vcf", 0) == 0
        assert (tmp_path / "ok.vcf").read_bytes() == V.vcf(haps, sample_matrix=[[0]], sample_names=["s"], file_date=DATE)
    finally:
        ctx.close()
