"""haps_vcf on the GPU: the records equal the oracle's (DESIGN.md section 12) for write_vcf output of create_haplotypes
(substitutions, indels, gene trees), random haplotypes with sample matrices, the hand-written cases, 4096 diploid
samples and a wide file of mostly 0|0 fields; write_vcf output read back materialises the same haplotypes; plain, BGZF
and gzip input, batch sizes and thread counts give the same records; reads from the VCF haplotypes equal reads from the
same records added through set_haplotypes; and malformed files give the oracle's line and reason."""
import gzip
import os
import re
import struct
import zlib

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200.mutate import kingman
from oracle import vcf_oracle as V
from oracle import vcf_read_oracle as O
from test_gpu_vcf import genome_with_n_runs
from test_vcf_host import CASES, R, haps_of
from test_vcf_read_host import REJECT, ln, vcf

pytestmark = pytest.mark.gpu

DATE = "20261022"


def read(ctx, g, path, **kw):
    return J.create_haplotypes(g, J.haps_vcf(str(path)), seed=1, ctx=ctx, **kw)


def same_as_oracle(got, text, g):
    """got's records (size_modifier derived from new_pos, as the packed layout holds it) against the oracle's."""
    refs = [g.chrom(c) for c in range(g.n_chroms())]
    names, recs, st = O.read(text, g.names, refs)
    assert got.hap_names == names
    for h in range(len(names)):
        for c in range(g.n_chroms()):
            m, w = got.muts[h][c], recs[h][c]
            assert m.old_pos.tolist() == w["old_pos"] and m.new_pos.tolist() == w["new_pos"], (h, c)
            assert m.nuc_off.tolist() == w["nuc_off"] and m.pool.tobytes() == w["pool"], (h, c)
            assert m.chrom_size == w["size"], (h, c)
            assert V.size_modifiers(m, len(refs[c])).tolist() == w["size_modifier"], (h, c)
    for k in ("lines", "samples", "haplotypes", "calls", "records", "overlaps_skipped", "symbolic_calls", "missing_calls"):
        assert got.stats[k] == st[k], k
    assert got.stats["text_bytes"] == len(text)
    return names


def write_and_read(ctx, haps, tmp_path, sample_matrix=None, **kw):
    J.write_vcf(haps, str(tmp_path / "w"), ctx=ctx, file_date=DATE, overwrite=True, sample_matrix=sample_matrix)
    fn = tmp_path / "w.vcf"
    text = fn.read_bytes()
    got = read(ctx, haps.reference, fn, **kw)
    same_as_oracle(got, text, haps.reference)
    return got, text


def materialised(ctx, haps):
    ctx.set_haplotypes(haps)
    return [[ctx.haplotype_chrom(h, c) for c in range(haps.n_chroms())] for h in range(haps.n_haps())]


def round_trip(ctx, haps, tmp_path):
    want = materialised(ctx, haps)
    got, _ = write_and_read(ctx, haps, tmp_path)
    assert got.hap_names == haps.hap_names
    assert [list(got.sizes(h)) for h in range(got.n_haps())] == [list(haps.sizes(h)) for h in range(haps.n_haps())]
    assert materialised(ctx, got) == want
    J.write_vcf(got, str(tmp_path / "again"), ctx=ctx, file_date=DATE, overwrite=True)
    again = (tmp_path / "again.vcf").read_bytes()
    g = haps.reference
    for h in sorted({0, 1, haps.n_haps() - 1} & set(range(haps.n_haps()))):      # applying the text is slow in Python
        assert [V.apply(again, g, h)[n] for n in g.names] == want[h]
    return got


@pytest.mark.parametrize("n_tips", [2, 40, 1024])
def test_substitutions(ctx, tmp_path, n_tips):
    g = genome_with_n_runs([20_011, 8_193, 5], seed=n_tips)
    haps = J.create_haplotypes(g, J.haps_theta(0.02, n_tips), J.sub_TN93([0.1, 0.2, 0.3, 0.4], 3, 1.2, 0.5), seed=3, ctx=ctx)
    round_trip(ctx, haps, tmp_path)


def test_indels_and_sample_matrix(ctx, tmp_path):
    g = genome_with_n_runs([40_003, 777, 9_000], seed=4)
    haps = J.create_haplotypes(g, J.haps_theta(0.05, 12), J.sub_HKY85([0.1, 0.2, 0.3, 0.4], 2, 0.5),
                               ins=J.indels(0.05, max_length=12), del_=J.indels(0.05, max_length=12), seed=5, ctx=ctx)
    round_trip(ctx, haps, tmp_path)
    write_and_read(ctx, haps, tmp_path, sample_matrix=[[0, 3], [11, 11], [5, 0]])
    write_and_read(ctx, haps, tmp_path, sample_matrix=[[0, 3, 7], [1, 2, 4]])


@pytest.mark.parametrize("n_tips", [2, 40, 1024])
def test_gene_trees(ctx, tmp_path, n_tips):
    rng = np.random.default_rng(n_tips)
    g = J.random_genome(2, [12_000, 3_001], seed=n_tips)
    blocks = [["[%d]%s" % (int(rng.integers(1, 50)), kingman(n_tips, rng).scaled(0.05).newick()) for _ in range(3)]
              for _ in range(2)]
    haps = J.create_haplotypes(g, J.haps_gtrees(obj=blocks), J.sub_JC69(1.0), seed=6, ctx=ctx)
    round_trip(ctx, haps, tmp_path)


@pytest.mark.parametrize("matrix", [None, [[0], [3], [1]], [[0, 1], [2, 2], [4, 0]], [[0, 1, 2], [3, 4, 0]]])
def test_random_haplotypes(ctx, tmp_path, matrix):
    g = J.random_genome(3, [30_000, 7_001, 50], seed=7)
    haps = J.random_haplotypes(g, 5, sub_rate=0.02, indel_rate=0.005, seed=8)
    write_and_read(ctx, haps, tmp_path, sample_matrix=matrix)


def hand_written():
    yield vcf(["a", "b"], ln(b"c1", 2, b"C", b"T,*,GG", "1/2", "3|."), ln(b"c1", 5, b"A", b".", "0|.", "."))
    yield vcf(["a", "b"], ln(b"c1", 4, b"T", b"A", "1", "0|1|1"), ln(b"c1", 6, b"C", b"G", "1", "1"))
    yield vcf(["a"], ln(b"c1", 2, b"CGT", b"C", "1"), ln(b"c1", 3, b"GTACG", b"G", "1"), ln(b"c1", 4, b"T", b"G", "1"),
              ln(b"c1", 5, b"A", b"C", "1"))
    yield vcf(["a"], ln(b"c1", 2, b"C", b"T", "1"), ln(b"c1", 2, b"CGTAC", b"C", "1"), ln(b"c1", 3, b"G", b"A", "1"))
    yield vcf(["a", "b", "c"], ln(b"c1", 2, b"CGT", b"<DEL>", "1", "0", "0"),
              ln(b"c1", 6, b"CG", b"<DEL>", "0", "1", "0", info=b"SVTYPE=DEL;SVLEN=-2"),
              ln(b"c1", 9, b"A", b"<INS>,A[c1:3[", "0", "0", "1|2"))
    yield vcf(["a", "b", "c", "d"], ln(b"c1", 1, b"A", b"GGA,<DEL>", "1", "2", "0", "0"),
              ln(b"c1", 7, b"GTAC", b"G,<DEL>", "0", "0", "1", "0"), ln(b"c2", 1, b"ACGT", b"<DEL>", "1", "1", "0", "1"))
    yield vcf(["a"], ln(b"c2", 2, b"C", b"T", "1"), ln(b"c1", 3, b"G", b"C", "1"), ln(b"c1", 3, b"G", b"A", "1"), crlf=True)
    yield vcf(["a"], ln(b"c1", 4, b"T", b"A", "1"))[:-1]
    yield vcf(["a", "b"])


@pytest.mark.parametrize("k", range(9))
def test_hand_written_cases(ctx, tmp_path, k):
    text = list(hand_written())[k]
    g = J.RefGenome(["c1", "c2"], [R, b"acgt"])
    fn = tmp_path / "h.vcf"
    fn.write_bytes(text)
    same_as_oracle(read(ctx, g, fn), text, g)


@pytest.mark.parametrize("k", range(len(CASES)))
def test_write_vcf_cases_round_trip(ctx, tmp_path, k):
    round_trip(ctx, haps_of(R, CASES[k][0]), tmp_path)             # CASES[6] loses its chromosome


def test_4096_diploid_samples(ctx, tmp_path):
    g = J.random_genome(2, [20_000, 3_000], seed=9)
    haps = J.random_haplotypes(g, 64, sub_rate=0.003, indel_rate=0.0005, seed=10)
    S = np.random.default_rng(11).integers(0, 64, size=(4096, 2))
    got, _ = write_and_read(ctx, haps, tmp_path, sample_matrix=S)
    assert got.n_haps() == 8192


def wide_text(g, n_samples, n_lines, seed):
    """Diploid samples over chromosome 0 of g: mostly 0|0, alleles from a 1/i frequency spectrum."""
    rng = np.random.default_rng(seed)
    L = g.seqs[0].size
    pos = np.sort(rng.choice(L - 5, size=n_lines, replace=False))
    N = 2 * n_samples
    p = 1.0 / np.arange(1, N)
    ac = rng.choice(np.arange(1, N), size=n_lines, p=p / p.sum())
    bases = np.frombuffer(b"TCAG", dtype=np.uint8)
    lines = [b"\t".join([b"#CHROM", b"POS", b"ID", b"REF", b"ALT", b"QUAL", b"FILTER", b"INFO", b"FORMAT"] +
                        [b"s%d" % i for i in range(n_samples)])]
    for x, a in zip(pos.tolist(), ac.tolist()):
        ref = bytes([g.seqs[0][x]])
        alt = bytes([bases[(np.flatnonzero(bases == g.seqs[0][x])[0] + 1) % 4]]) if ref in b"TCAG" else b"A"
        gt = np.zeros(N, dtype=np.uint8)
        gt[rng.choice(N, size=a, replace=False)] = 1
        f = np.full((n_samples, 4), ord("|"), dtype=np.uint8)
        f[:, 0] = ord("0") + gt[0::2]
        f[:, 2] = ord("0") + gt[1::2]
        f[:, 3] = ord("\t")
        lines.append(b"\t".join([g.names[0].encode(), b"%d" % (x + 1), b".", ref, alt, b".", b"PASS", b".", b"GT"]) + b"\t" +
                     f.tobytes()[:-1])
    return b"\n".join(lines) + b"\n"


def test_wide_file(ctx, tmp_path):
    g = J.random_genome(1, 200_000, seed=12)
    text = wide_text(g, 1200, 400, seed=13)
    fn = tmp_path / "wide.vcf"
    fn.write_bytes(text)
    got = read(ctx, g, fn)
    same_as_oracle(got, text, g)
    small = read(ctx, g, fn, batch_bytes=100_000)             # lines across batches, a line longer than a batch
    assert small.stats["batches"] > 1 and all(same(a, b) for a, b in zip(got.muts, small.muts))


def same(a, b):
    return all(x.old_pos.tolist() == y.old_pos.tolist() and x.new_pos.tolist() == y.new_pos.tolist() and
               x.nuc_off.tolist() == y.nuc_off.tolist() and x.pool.tobytes() == y.pool.tobytes() and
               x.chrom_size == y.chrom_size for x, y in zip(a, b))


def test_formats_batches_threads_and_devices(ctx, tmp_path):
    g = genome_with_n_runs([60_011, 9_000], seed=14)
    haps = J.random_haplotypes(g, 6, sub_rate=0.02, indel_rate=0.004, seed=15)
    S = [[0, 1], [2, 3], [4, 5], [5, 0]]
    J.write_vcf(haps, str(tmp_path / "p"), ctx=ctx, file_date=DATE, sample_matrix=S)
    J.write_vcf(haps, str(tmp_path / "b"), ctx=ctx, file_date=DATE, sample_matrix=S, compress=True)
    text = (tmp_path / "p.vcf").read_bytes()
    with gzip.open(tmp_path / "g.vcf.gz", "wb") as f:
        f.write(text)
    base = read(ctx, g, tmp_path / "p.vcf")
    same_as_oracle(base, text, g)
    runs = [read(ctx, g, tmp_path / "b.vcf.gz"), read(ctx, g, tmp_path / "g.vcf.gz"),
            read(ctx, g, tmp_path / "b.vcf.gz", n_threads=8), read(ctx, g, tmp_path / "b.vcf.gz", n_threads=1),
            read(ctx, g, tmp_path / "p.vcf", batch_bytes=4096), read(ctx, g, tmp_path / "b.vcf.gz", batch_bytes=70_000),
            read(ctx, g, tmp_path / "p.vcf", batch_bytes=100), read(ctx, g, tmp_path / "p.vcf")]
    for r in runs:
        assert r.hap_names == base.hap_names and all(same(a, b) for a, b in zip(base.muts, r.muts))
        assert r.stats["text_bytes"] == len(text)
    assert runs[4].stats["batches"] > 10
    multi = J.Context(devices=[0, 0])
    try:
        m = read(multi, g, tmp_path / "b.vcf.gz")
        assert all(same(a, b) for a, b in zip(base.muts, m.muts))
        assert materialised(multi, m) == materialised(ctx, base)
    finally:
        multi.close()


def test_reads_equal_those_of_added_haplotypes(ctx, tmp_path):
    g = J.random_genome(3, 40_000, seed=16)
    src = J.create_haplotypes(g, J.haps_theta(0.01, 6), J.sub_JC69(1.0), ins=J.indels(0.01), del_=J.indels(0.01), seed=17, ctx=ctx)
    got, _ = write_and_read(ctx, src, tmp_path)
    copy = J.Haplotypes(g, got.hap_names, got.muts)                # the same records through jlp_add_haplotype
    for obj in (got, copy):
        ctx.set_haplotypes(obj)
    r_vcf = J.illumina(got, "", 4000, 100, True, seed=42, ctx=ctx, sink="memory", haplotype_probs=[1] * 6)
    r_add = J.illumina(copy, "", 4000, 100, True, seed=42, ctx=ctx, sink="memory", haplotype_probs=[1] * 6)
    assert r_vcf[0] == r_add[0] and r_vcf[1] == r_add[1]
    p_vcf = J.pacbio(got, "", 200, seed=43, ctx=ctx, sink="memory")
    p_add = J.pacbio(copy, "", 200, seed=43, ctx=ctx, sink="memory")
    assert p_vcf[0] == p_add[0]


@pytest.mark.parametrize("k", range(len(REJECT)))
def test_rejections(ctx, tmp_path, k):
    text, line, reason = REJECT[k]
    g = J.RefGenome(["c1", "c2"], [R, b"ACGT"])
    fn = tmp_path / "bad.vcf"
    fn.write_bytes(text)
    with pytest.raises(J.JackalopeError, match=re.escape("line %d: %s" % (line, reason))):
        read(ctx, g, fn)


def test_smallest_bad_line_wins_truncation_and_random_bytes(ctx, tmp_path):
    g = J.random_genome(1, 100_000, seed=18)
    haps = J.random_haplotypes(g, 4, sub_rate=0.01, indel_rate=0.001, seed=19)
    J.write_vcf(haps, str(tmp_path / "w"), ctx=ctx, file_date=DATE)
    lines = (tmp_path / "w.vcf").read_bytes().split(b"\n")
    n_head = sum(1 for x in lines if x.startswith(b"#"))
    bad = list(lines)
    for i in (n_head + 700, n_head + 50, n_head + 900):
        bad[i] = bad[i].replace(b"\t", b"\tx", 1)                  # POS is no longer a number
    fn = tmp_path / "bad.vcf"
    fn.write_bytes(b"\n".join(bad))
    for bb in (0, 3000):
        with pytest.raises(J.JackalopeError, match="line %d: %s" % (n_head + 51, O.POS)):
            read(ctx, g, fn, batch_bytes=bb)
    text = b"\n".join(lines)
    cut = text[:text.rfind(b"\t")]                                 # the last line loses its last column
    fn.write_bytes(cut)
    with pytest.raises(J.JackalopeError, match="line %d: %s" % (len(lines) - 1, O.COLUMNS)):
        read(ctx, g, fn)
    rng = np.random.default_rng(20)
    for k in range(3):
        junk = text[:text.find(b"\n", len(text) // 3)] + b"\n" + rng.integers(0, 256, size=20_000, dtype=np.uint8).tobytes()
        fn.write_bytes(junk)
        with pytest.raises(O.VcfError) as want:
            O.read(junk, g.names, [g.chrom(0)])
        with pytest.raises(J.JackalopeError, match=re.escape(str(want.value))):     # an error, not a device fault
            read(ctx, g, fn, batch_bytes=4096 * (k + 1))
    fn.write_bytes(gzip.compress(text)[:-100])
    with pytest.raises(RuntimeError, match="inflate|truncated"):
        read(ctx, g, fn)
    z = bytearray(bgzf(text))                                      # a member whose ISIZE claims 4 GiB
    z[bsize(z, 0) - 4:bsize(z, 0)] = struct.pack("<I", 0xfffffff0)
    fn.write_bytes(bytes(z))
    with pytest.raises(RuntimeError, match="damaged member"):
        read(ctx, g, fn)
    assert os.path.exists(fn)


def bgzf(text, block=65280):
    """text as BGZF members of `block` input bytes and the end-of-file member."""
    out = []
    for i in range(0, len(text), block):
        blk = text[i:i + block]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        d = c.compress(blk) + c.flush()
        out.append(struct.pack("<4BI2BH2BHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(d) + 25) + d +
                   struct.pack("<II", zlib.crc32(blk), len(blk)))
    return b"".join(out) + bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bsize(z, at):
    """the length of the BGZF member at byte `at`"""
    return struct.unpack("<H", bytes(z[at + 16:at + 18]))[0] + 1


@pytest.mark.parametrize("compressed", [False, True])
def test_consecutive_lines_longer_than_a_batch(ctx, tmp_path, compressed):
    # lines of 150-330 KB (a long INFO) at batch_bytes 100: each batch carries a line's start much longer than a batch
    rng = np.random.default_rng(21)
    g = J.random_genome(1, 5_000, seed=22)
    lines = []
    for k, x in enumerate(sorted(rng.choice(4_990, size=20, replace=False).tolist())):
        ref = bytes([g.seqs[0][x]])
        info = b"X=" + b"7" * int(rng.integers(150_000, 330_000))
        lines.append(ln(b"chrom0", x + 1, ref, b"A" if ref != b"A" else b"C", "1|0", "%d|1" % (k % 2), info=info))
    text = vcf(["a", "b"], *lines)
    fn = tmp_path / ("long.vcf.gz" if compressed else "long.vcf")
    fn.write_bytes(bgzf(text) if compressed else text)
    for bb in (100, 70_000, 0):
        got = read(ctx, g, fn, batch_bytes=bb)
        same_as_oracle(got, text, g)
        assert got.stats["batches"] > 1 if bb else got.stats["batches"] == 1
