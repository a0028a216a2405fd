"""haps_vcf without a GPU: the reading rules of DESIGN.md section 12 through the oracle -- its records applied to the
reference equal vcf_oracle.apply() for VCFs of every shape write_vcf makes, hand-written cases for each rule, and each
rejection -- and haps_vcf's argument errors."""
import numpy as np
import pytest

import jackalope_b200 as J
from oracle import vcf_oracle as V
from oracle import vcf_read_oracle as O
from test_vcf_host import CASES, R, haps_of

HEAD = b"##fileformat=VCFv4.3\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"


def vcf(samples, *lines, crlf=False):
    text = HEAD + b"".join(b"\t" + s.encode() for s in samples) + b"\n" + b"".join(lines)
    return text.replace(b"\n", b"\r\n") if crlf else text


def ln(chrom, pos, ref, alt, *gts, info=b".", fmt=b"GT"):
    return b"\t".join([chrom, str(pos).encode(), b".", ref, alt, b".", b"PASS", info, fmt] + [g.encode() for g in gts]) + b"\n"


def seqs_of(text, names, refs):
    hn, recs, st = O.read(text, names, refs)
    return hn, {h: [O.sequence(refs[c], recs[i][c]) for c in range(len(refs))] for i, h in enumerate(hn)}, recs, st


def check_against_apply(haps, sample_matrix=None):
    ref = haps.reference
    text = V.vcf(haps, sample_matrix=sample_matrix)
    refs = [ref.chrom(c) for c in range(ref.n_chroms())]
    hn, seqs, _, st = seqs_of(text, ref.names, refs)
    S = np.arange(haps.n_haps()).reshape(-1, 1) if sample_matrix is None else np.asarray(sample_matrix)
    assert len(hn) == S.size
    for slot in range(S.size):
        want = V.apply(text, ref, slot)
        assert seqs[hn[slot]] == [want[n] for n in ref.names]
    return hn, st


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_haplotypes_read_back(seed):
    g = J.random_genome(3, [3000, 701, 50], seed=seed)
    haps = J.random_haplotypes(g, 5, sub_rate=0.02, indel_rate=0.01, seed=seed)
    hn, st = check_against_apply(haps)
    assert hn == haps.hap_names and st["overlaps_skipped"] == 0
    for h in range(haps.n_haps()):                       # and the sequences the records describe
        for c in range(g.n_chroms()):
            m = haps.muts[h][c]
            want = V.apply(V.vcf(haps), g, h)[g.names[c]]
            assert len(want) == m.chrom_size


@pytest.mark.parametrize("matrix", [[[0], [3], [1]], [[0, 1], [2, 2], [4, 0]], [[0, 1, 2], [3, 4, 0]]])
def test_sample_matrices_read_back(matrix):
    g = J.random_genome(2, [2000, 333], seed=7)
    haps = J.random_haplotypes(g, 5, sub_rate=0.03, indel_rate=0.01, seed=8)
    hn, st = check_against_apply(haps, matrix)
    P = len(matrix[0])
    assert hn == (["sample%d" % (i + 1) for i in range(len(matrix))] if P == 1 else
                  ["sample%d__%d" % (i + 1, k + 1) for i in range(len(matrix)) for k in range(P)])


@pytest.mark.parametrize("per_hap, want", CASES)
def test_write_vcf_cases_read_back(per_hap, want):
    check_against_apply(haps_of(R, per_hap))


def test_multi_allelic_star_missing_and_unphased():
    text = vcf(["a", "b"], ln(b"c1", 2, b"C", b"T,*,GG", "1/2", "3|."), ln(b"c1", 5, b"A", b".", "0|.", "."))
    hn, seqs, recs, st = seqs_of(text, ["c1"], [R])
    assert hn == ["a__1", "a__2", "b__1", "b__2"]
    assert seqs["a__1"] == [b"ATGTACGTAC"] and seqs["a__2"] == [R] and seqs["b__1"] == [b"AGGGTACGTAC"]
    assert seqs["b__2"] == [R]
    assert st["missing_calls"] == 3 and st["calls"] == 2 and st["symbolic_calls"] == 0


def test_mixed_ploidy_and_short_gt():
    text = vcf(["a", "b"], ln(b"c1", 4, b"T", b"A", "1", "0|1|1"), ln(b"c1", 6, b"C", b"G", "1", "1"))
    hn, seqs, _, st = seqs_of(text, ["c1"], [R])
    assert hn == ["a", "b__1", "b__2", "b__3"]
    assert seqs["a"] == [b"ACGAAGGTAC"] and seqs["b__1"] == [b"ACGTAGGTAC"]
    assert seqs["b__2"] == seqs["b__3"] == [b"ACGAACGTAC"]


def test_overlaps_skipped_and_skipped_calls_do_not_advance_the_end():
    # line 1 covers [1, 4); line 2 starts inside it (skipped); line 3 starts at 3, inside [1, 4) too; line 4 starts at 4
    text = vcf(["a"], ln(b"c1", 2, b"CGT", b"C", "1"), ln(b"c1", 3, b"GTACG", b"G", "1"), ln(b"c1", 4, b"T", b"G", "1"),
               ln(b"c1", 5, b"A", b"C", "1"))
    hn, seqs, _, st = seqs_of(text, ["c1"], [R])
    assert seqs["a"] == [b"ACCCGTAC"] and st["overlaps_skipped"] == 2 and st["calls"] == 2
    # a skipped call leaves the end of the applied line: the next line after it is judged against that end
    text = vcf(["a"], ln(b"c1", 2, b"C", b"T", "1"), ln(b"c1", 2, b"CGTAC", b"C", "1"), ln(b"c1", 3, b"G", b"A", "1"))
    hn, seqs, _, st = seqs_of(text, ["c1"], [R])
    assert seqs["a"] == [b"ATATACGTAC"] and st["overlaps_skipped"] == 1


def test_both_meanings_of_del_and_symbolic_alleles():
    text = vcf(["a", "b", "c"], ln(b"c1", 2, b"CGT", b"<DEL>", "1", "0", "0"),
               ln(b"c1", 6, b"CG", b"<DEL>", "0", "1", "0", info=b"SVTYPE=DEL;SVLEN=-2"),
               ln(b"c1", 9, b"A", b"<INS>,A[c1:3[", "0", "0", "1|2"))
    hn, seqs, _, st = seqs_of(text, ["c1"], [R])
    assert seqs["a"] == [b"AACGTAC"] and seqs["b"] == [R] and seqs["c__1"] == seqs["c__2"] == [R]
    assert st["symbolic_calls"] == 3


def test_lowercase_reference_and_ref_differing_in_case():
    ref = b"acgtACGTac"
    text = vcf(["a"], ln(b"c1", 1, b"AC", b"aG", "1"), ln(b"c1", 5, b"a", b"aTT", "1"), ln(b"c1", 9, b"A", b"t", "1"))
    hn, seqs, recs, _ = seqs_of(text, ["c1"], [ref])
    assert seqs["a"] == [b"aGgtATTCGTtc"]
    r = recs[0][0]
    assert r["old_pos"] == [1, 4, 8] and r["pool"] == b"GATTt" and r["size_modifier"] == [0, 2, 0]


def test_edges_of_the_chromosome():
    text = vcf(["a", "b", "c", "d"], ln(b"c1", 1, b"A", b"GGA,<DEL>", "1", "2", "0", "0"),
               ln(b"c1", 7, b"GTAC", b"G,<DEL>", "0", "0", "1", "0"))
    hn, seqs, recs, _ = seqs_of(text, ["c1"], [R])
    assert seqs["a"] == [b"GGACGTACGTAC"] and seqs["b"] == [b"CGTACGTAC"] and seqs["c"] == [b"ACGTACG"]
    assert recs[1][0]["old_pos"] == [0] and recs[1][0]["size_modifier"] == [-1]       # deletion at 0: the leading form
    text = vcf(["a"], ln(b"c1", 1, R, b"<DEL>", "1"))                                    # a chromosome deleted entirely
    hn, seqs, recs, _ = seqs_of(text, ["c1"], [R])
    assert seqs["a"] == [b""] and recs[0][0]["size"] == 0 and recs[0][0]["size_modifier"] == [-10]


def test_missing_chromosomes_blocks_in_any_order_crlf_and_no_final_newline():
    refs = [b"AAAA", b"CCCC", b"GGGG"]
    text = vcf(["a"], ln(b"z", 2, b"G", b"T", "1"), ln(b"x", 3, b"A", b"C", "1"), ln(b"x", 3, b"A", b"G", "1"))
    for t in (text, text[:-1], vcf(["a"], *[x + b"\n" for x in text.split(b"\n")[2:-1]], crlf=True)):
        hn, seqs, _, st = seqs_of(t, ["x", "y", "z"], refs)
        assert seqs["a"] == [b"AACA", b"CCCC", b"GTGG"] and st["lines"] == 3 and st["overlaps_skipped"] == 1


def test_header_only_file():
    hn, seqs, recs, st = seqs_of(vcf(["a", "b"]), ["c1"], [R])
    assert hn == ["a", "b"] and seqs["a"] == [R] and st["lines"] == 0 and recs[1][0]["old_pos"] == []


REJECT = [
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1", "0")), 3, O.COLUMNS),
    (vcf(["a"], ln(b"c3", 4, b"T", b"A", "1")), 3, O.CHROM),
    (vcf(["a"], ln(b"c1", 0, b"A", b"T", "1")), 3, O.POS),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1"), ln(b"c1", 4, b"T.", b"A", "1")), 4, O.REF_LETTERS),
    (vcf(["a"], ln(b"c1", 9, b"ACG", b"A", "1")), 3, O.REF_RANGE),
    (vcf(["a"], ln(b"c1", 4, b"A", b"T", "1")), 3, O.REF_DIFF),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A,", "1")), 3, O.ALT),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1", fmt=b"DS:GT")), 3, O.FORMAT),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1||0")), 3, O.GT),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "|".join("0" * 9))), 3, O.PLOIDY),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "2")), 3, O.INDEX),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1"), ln(b"c2", 1, b"A", b"C", "1"), ln(b"c1", 6, b"C", b"A", "1")), 5, O.CONTIG),
    (vcf(["a"], ln(b"c1", 4, b"T", b"A", "1"), ln(b"c1", 3, b"G", b"A", "1")), 4, O.ORDER),
    (b"##x\nc1\t1\n", 2, O.NO_HEADER),
    (b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFMT\ta\n", 1, O.HEADER),
    (vcf(["a", "a"]), 2, O.SAMPLE),
    (vcf(["a b"]), 2, O.SAMPLE),
]


@pytest.mark.parametrize("text, line, reason", REJECT)
def test_rejections(text, line, reason):
    with pytest.raises(O.VcfError) as e:
        O.read(text, ["c1", "c2"], [R, b"ACGT"])
    assert (e.value.line, e.value.reason) == (line, reason)


def test_first_check_of_a_line_decides_its_reason():
    # a wrong column count comes before every other check; a bad ALT before a bad GT
    t = vcf(["a"], ln(b"zz", 0, b"T", b"A", "1", "x"))
    with pytest.raises(O.VcfError, match=O.COLUMNS):
        O.read(t, ["c1"], [R])
    with pytest.raises(O.VcfError, match="line 3: ALT"):
        O.read(vcf(["a"], ln(b"c1", 4, b"T", b"1", "x")), ["c1"], [R])


def test_haps_vcf_arguments(tmp_path):
    with pytest.raises(J.JackalopeError):
        J.haps_vcf(str(tmp_path / "missing.vcf"))
    fn = tmp_path / "a.vcf"
    fn.write_bytes(vcf(["a"]))
    info = J.haps_vcf(str(fn))
    g = J.RefGenome(["c1"], [R])
    with pytest.raises(J.JackalopeError, match="must be NULL"):
        J.create_haplotypes(g, info, J.sub_JC69(1.0))
    with pytest.raises(J.JackalopeError, match="sub"):
        J.create_haplotypes(g, J.haps_theta(0.1, 3))       # other haps_info still need a model
