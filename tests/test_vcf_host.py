"""write_vcf without a GPU: the format's definitions (DESIGN.md section 11) on hand-written records through the oracle,
the oracle's VCF applied back to the reference, and write_vcf's argument errors."""
import numpy as np
import pytest

import jackalope_b200 as J
from oracle import harness
from oracle import harness_indels as HI
from oracle import vcf_oracle as V


def muts(ref, edits):
    """HapChromMuts from sorted edits on `ref`: ("sub", pos, base), ("ins", pos, inserted bytes; the pool gets the anchor
    first), ("del", pos, length), ("raw", pos, pool bytes, size_modifier)."""
    op, npos, no, nl, pool, shift = [], [], [], [], b"", 0
    for e in edits:
        kind, p = e[0], e[1]
        if kind == "sub":
            b, d = e[2], 0
        elif kind == "ins":
            b, d = ref[p:p + 1] + e[2], len(e[2])
        elif kind == "del":
            b, d = b"", -e[2]
        else:
            b, d = e[2], e[3]
        op.append(p); npos.append(p + shift); no.append(len(pool)); nl.append(len(b))
        pool += b
        shift += d
    return J.HapChromMuts(op, npos, no, nl, pool, len(ref) + shift)


def haps_of(ref, per_hap, names=None):
    g = J.RefGenome(["c1"], [ref])
    names = names or ["h%d" % i for i in range(len(per_hap))]
    return J.Haplotypes(g, names, [[muts(ref, e)] for e in per_hap])


def body(haps, **kw):
    text = V.vcf(haps, **kw)
    return b"".join(ln + b"\n" for ln in text.split(b"\n") if ln and not ln.startswith(b"#"))


def line(pos, ref, alt, *gts):
    return b"\t".join([b"c1", str(pos).encode(), b".", ref, alt, b".", b"PASS", b".", b"GT"] + [g.encode() for g in gts]) + b"\n"


R = b"ACGTACGTAC"


CASES = [
    ([[("sub", 3, b"A")], [("sub", 3, b"A")], []], line(4, b"T", b"A", "1", "1", "0")),                       # shared SNP
    ([[("sub", 3, b"A")], [("sub", 3, b"C")], []], line(4, b"T", b"A,C", "1", "2", "0")),                     # two ALTs
    ([[("ins", 3, b"GG")], [("sub", 3, b"C")], []], line(4, b"T", b"TGG,C", "1", "2", "0")),                  # ins + sub
    ([[("del", 4, 2)], [("sub", 5, b"T")], []], line(4, b"TAC", b"T,TAT", "1", "2", "0")),                    # del over SNP
    ([[("del", 0, 2)], []], line(1, b"ACG", b"G", "1", "0")),                                                 # del at 0
    ([[("del", 7, 3)], []], line(7, b"GTAC", b"G", "1", "0")),                                                # del to the end
    ([[("del", 0, 10)], [("sub", 5, b"T")]], line(1, R, b"<DEL>,ACGTATGTAC", "1", "2")),                      # chromosome lost
    ([[("sub", 3, b"A")], [("sub", 4, b"C")]], line(4, b"T", b"A", "1", "0") + line(5, b"A", b"C", "0", "1")),  # adjacent SNPs
    ([[("raw", 0, b"TT", 1)], []], line(1, b"A", b"TT", "1", "0")),                                           # leading gap
    ([[("sub", 3, b"T")], []], b""),                                                                          # sub == REF
]


@pytest.mark.parametrize("per_hap, want", CASES)
def test_hand_written_cases(per_hap, want):
    assert body(haps_of(R, per_hap)) == want


def test_n_and_lowercase_reference_bytes():
    ref = b"ACNNacgtAC"
    h = haps_of(ref, [[("sub", 2, b"A"), ("del", 5, 1)], [("sub", 5, b"T")]])
    assert body(h) == (b"c1\t3\t.\tN\tA\t.\tPASS\t.\tGT\t1\t0\n" +
                       b"c1\t5\t.\tac\ta,aT\t.\tPASS\t.\tGT\t1\t2\n")


def test_diploid_matrix_repeated_and_left_out_haplotypes():
    h = haps_of(R, [[("sub", 3, b"A")], [("sub", 7, b"C")], [("sub", 5, b"G"), ("sub", 8, b"C")]])
    S = [[2, 0], [0, 0]]
    want = (line(4, b"T", b"A", "0|1", "1|1") + line(6, b"C", b"G", "1|0", "0|0") + line(9, b"A", b"C", "1|0", "0|0"))
    assert body(h, sample_matrix=S) == want
    text = V.vcf(h, sample_matrix=S, file_date="20261021")
    assert text.startswith(b"##fileformat=VCFv4.3\n##fileDate=20261021\n##source=jackalope_b200\n##contig=<ID=c1,length=10>\n")
    assert b"\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsample1\tsample2\n" in text


def test_alt_order_follows_the_sample_matrix():
    h = haps_of(R, [[("sub", 3, b"A")], [("sub", 3, b"C")], [("sub", 3, b"G")]])
    assert body(h, sample_matrix=[[2, 1], [0, 2]]) == line(4, b"T", b"G,C,A", "1|2", "3|1")


def round_trip(haps, S, seqs):
    """Apply the oracle's VCF for every slot of S and compare with the expected sequences seqs[h][c]."""
    text = V.vcf(haps, sample_matrix=S)
    P = np.asarray(S).shape[1]
    for i, row in enumerate(np.asarray(S).tolist()):
        for k, h in enumerate(row):
            got = V.apply(text, haps.reference, i * P + k)
            for c, n in enumerate(haps.reference.names):
                assert got[n] == seqs[h][c], (i, k, c)


def test_round_trip_random_haplotypes():
    g = J.random_genome(3, [3000, 1, 2500], seed=3)
    haps = J.random_haplotypes(g, 5, sub_rate=0.02, indel_rate=0.01, seed=4)
    seqs = [[harness.materialize(g.chrom(c), m.old_pos, m.new_pos, m.nuc_off, m.pool.tobytes(), m.chrom_size)
             for c, m in enumerate(haps.muts[h])] for h in range(5)]
    round_trip(haps, [[0], [1], [2], [3], [4]], seqs)
    round_trip(haps, [[4, 1, 1], [0, 3, 4]], seqs)


def oracle_haps(g, o, names):
    muts_ = []
    for t in o.tips:
        row = []
        for seq, (old, new, nuc, sm, pool) in t:
            nl = np.diff(np.concatenate((nuc, [len(pool)]))).astype(np.uint32)
            row.append(J.HapChromMuts(old, new, nuc, nl, pool, len(seq)))
        muts_.append(row)
    return J.Haplotypes(g, names, muts_)


def test_round_trip_indel_tips():
    g = J.random_genome(2, [4000, 7], seed=5)
    info, sub = J.haps_phylo("(a:0.3,(b:0.1,c:0.6):0.2,d:2);"), J.sub_JC69(0.3)
    ins, dele = J.indels(0.05), J.indels(0.08, max_length=5)
    o = HI.indels(g, info.tree(sub, 9), sub, ins, dele, 0.05, 9)
    haps = oracle_haps(g, o, ["a", "b", "c", "d"])
    seqs = [[t[c][0] for c in range(2)] for t in o.tips]
    for h in range(4):
        for c in range(2):
            m = haps.muts[h][c]
            assert harness.materialize(g.chrom(c), m.old_pos, m.new_pos, m.nuc_off, m.pool.tobytes(), m.chrom_size) == seqs[h][c]
    round_trip(haps, [[0], [1], [2], [3]], seqs)
    round_trip(haps, [[3, 0], [2, 2]], seqs)


# ------------------------------------------------------------------ argument errors ---

@pytest.fixture
def small_haps():
    return haps_of(R, [[("sub", 3, b"A")], [("sub", 4, b"C")]])


@pytest.mark.parametrize("kw, par", [
    (dict(sample_matrix=[[0, 1], [1]]), "sample_matrix"),
    (dict(sample_matrix=[[0, 2]]), "sample_matrix"),
    (dict(sample_matrix=[[0, -1]]), "sample_matrix"),
    (dict(sample_matrix=[[0.0, 1.0]]), "sample_matrix"),
    (dict(sample_matrix=[0, 1]), "sample_matrix"),
    (dict(compress=0), "compress"), (dict(compress=10), "compress"), (dict(compress="yes"), "compress"),
    (dict(comp_method="zip"), "comp_method"),
])
def test_argument_errors(tmp_path, small_haps, kw, par):
    with pytest.raises(J.JackalopeError, match="`write_vcf` function.*`%s`" % par):
        J.write_vcf(small_haps, str(tmp_path / "x"), **kw)


def test_existing_file_and_names(tmp_path, small_haps):
    (tmp_path / "x.vcf").write_bytes(b"")
    with pytest.raises(J.JackalopeError, match="File .*x.vcf already exists"):
        J.write_vcf(small_haps, str(tmp_path / "x"))
    (tmp_path / "y.vcf.gz").write_bytes(b"")
    with pytest.raises(J.JackalopeError, match="File .*y.vcf.gz already exists"):
        J.write_vcf(small_haps, str(tmp_path / "y"), compress=True)
    bad = haps_of(R, [[("sub", 3, b"A")], []], names=["ok", "a\tb"])
    with pytest.raises(J.JackalopeError, match="tabs or line breaks"):
        J.write_vcf(bad, str(tmp_path / "z"))
    g = J.RefGenome(["chr 1"], [R])
    with pytest.raises(J.JackalopeError, match="whitespace"):
        J.write_vcf(J.Haplotypes(g, ["a"], [[J.HapChromMuts.empty(len(R))]]), str(tmp_path / "w"))
