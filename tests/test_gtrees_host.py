"""create_haplotypes along gene trees without a GPU: the library's ms parser (through the C ABI) and haps_gtrees'
reading, the region rule, the oracle's gene-tree walk against its one-tree walk, and the law of two regions with
contrasting trees against exact pattern probabilities."""
import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200.mutate import ms_regions, parse_newick
from oracle import harness_gtrees as HG
from oracle import harness_mutate as HM
from test_mutate_host import chi2_fit

MS = """ms 3 2 -T -r 10 1000
31415 92653 58979

//
[3](1:0.5,('2':0.25,3:0.25)[&&NHX:x=1]:0.25);
[5]  ( 2:0.5 , (1:0.25, 3:0.25):0.25 ) ;
[2](3:1.5e-1,(2:0.1,1:0.1):0.05);
segsites: 2
positions: 0.1 0.7
01
10
11

//
((1:1,2:1):1,3:2);
segsites: 0
"""


def test_the_parser_reads_ms_output():
    regs, n_trees = ms_regions(MS, [100, 7], ["1", "2", "3"])
    assert n_trees == 4
    assert regs == [(0, 0, 30, 0), (0, 30, 80, 1), (0, 80, 100, 2), (1, 0, 7, 3)]
    # Python reads the first tree and orders integer labels numerically
    info = J.haps_gtrees(obj=[["[3](10:0.5,(2:0.25,1:0.25):0.25);"]])
    assert info.names == ["1", "2", "10"]
    assert J.haps_gtrees(obj=[["(b:1,a:1);"]]).names == ["b", "a"]
    # the harness reads the same text its own way
    blocks = HG.ms_blocks(MS)
    assert [[n for n, _ in b] for b in blocks] == [[3, 5, 2], [None]]
    assert sorted(parse_newick(blocks[0][0][1]).tip_names) == ["1", "2", "3"]


def test_haps_gtrees_reads_a_file_and_checks_its_arguments(tmp_path):
    fn = tmp_path / "trees.ms"
    fn.write_text(MS)
    info = J.haps_gtrees(fn=str(fn))
    assert info.names == ["1", "2", "3"] and info.text == MS
    with pytest.raises(J.JackalopeError, match="haps_gtrees.*obj"):
        J.haps_gtrees()
    with pytest.raises(J.JackalopeError, match="haps_gtrees.*obj"):
        J.haps_gtrees(obj=[["(a:1,b:1);"]], fn=str(fn))
    with pytest.raises(J.JackalopeError, match="fn"):
        J.haps_gtrees(fn=str(tmp_path / "missing"))
    with pytest.raises(J.JackalopeError, match="obj"):
        J.haps_gtrees(obj="(a:1,b:1);")
    with pytest.raises(J.JackalopeError, match="no trees"):
        J.haps_gtrees(obj=[["segsites: 0"]])


@pytest.mark.parametrize("text, what", [
    ("//\n[2](1:1,2:1);\n(1:1,2:1);\n", "mixes trees with and without"),
    ("//\n(1:1,2:1);\n(2:1,1:1);\n", "2 trees without a \\[n\\] prefix"),
    ("//\n[0](1:1,2:1);\n", "positive integer, not \\[0\\]"),
    ("//\n[1](1:1,3:1);\n", "tip label '3' is not one of"),
    ("//\n[1](1:1,(2:1,1:1):1);\n", "duplicate tip label '1'"),
    ("//\n(1:1,2:1);\n//\n(1:1,2:1);\n//\n(1:1,2:1);\n", "3 blocks \\('//' lines\\), the reference has 1"),
    ("ms 2 1\n1 2 3\n", "no trees"),
    ("//\nsegsites: 0\n//\n(1:1,2:1);\n", "block 1 has no trees"),
    ("//\n[1](1:1,2:-1);\n", "negative branch length"),
    ("//\n[1](1:1,2);\n", "has no branch length"),
    ("//\n[1](1:1,2:1)\n", "must end with ';'"),
    ("//\n[1](1:1,2:x);\n", "not a number"),
])
def test_the_parser_rejects(text, what):
    lens = [50, 50] if text.count("//") == 2 else [50]
    with pytest.raises(J.JackalopeError, match=what):
        ms_regions(text, lens, ["1", "2"])


def test_the_region_rule():
    rng = np.random.default_rng(5)
    for case in range(200):
        m = int(rng.integers(1, 12))
        lens = [int(x) for x in rng.integers(1, 50 if case % 3 else 4, size=m)]
        if case % 5 == 0:
            lens = [x * 10 ** 12 for x in lens]               # S far beyond L: exact integer arithmetic
        L = int(rng.integers(1, 40)) if case % 4 or case % 5 == 0 else sum(lens)
        text = "//\n" + "".join("[%d](1:1,2:1);\n" % n for n in lens)
        regs, _ = ms_regions(text, [L], ["1", "2"])
        want = HG.regions(lens, L)
        assert [(s, e, k) for _, s, e, k in regs] == want
        assert want[0][0] == 0 and want[-1][1] == L and all(s < e for s, e, _ in want)
        if L == sum(lens):
            assert [e - s for s, e, _ in want] == lens         # S = L: the lengths as written
    # dropped empty regions: 1 + 1 + 98 over 10 sites
    regs, _ = ms_regions("//\n[1](1:1,2:1);\n[1](1:1,2:1);\n[98](1:1,2:1);\n", [10], ["1", "2"])
    assert regs == [(0, 0, 10, 2)]


def test_indels_with_gene_trees_are_refused():
    g = J.random_genome(1, 100, seed=1)
    info = J.haps_gtrees(obj=[["(1:1,2:1);"]])
    with pytest.raises(J.JackalopeError, match="not supported.*haps_gtrees"):
        J.create_haplotypes(g, info, J.sub_JC69(1.0), ins=J.indels(0.1), seed=1)


def test_oracle_gene_tree_walk_with_one_region_is_the_one_tree_walk():
    g = J.random_genome(2, [20_011, 3_333], seed=3)
    nw = "((a:0.1,b:0.25)x:0.05,(c:0.02,d:0.4):0.3);"
    m = J.sub_HKY85([0.1, 0.2, 0.3, 0.4], 2.0, 0.5, invariant=0.2, gamma_shape=0.8, gamma_k=3)
    tree = parse_newick(nw)
    want = HM.mutate(g, tree, m, seed=9)
    for text in ("//\n%s\n//\n%s\n" % (nw, nw), "//\n[3]%s\n[4]%s\n//\n[1]%s\n" % (nw, nw, nw)):
        got = HG.mutate_gtrees(g, text, tree.tip_names, m, seed=9)
        for t in range(4):
            for c in range(2):
                assert np.array_equal(got[t][c][0], want[t][c][0]) and got[t][c][1] == want[t][c][1]


def test_law_two_regions_with_contrasting_trees():
    t1, t2 = "((a:0.3,b:0.2):0.01,c:0.4);", "((a:0.3,c:0.4):0.01,b:0.2);"
    m = J.sub_TN93([0.1, 0.2, 0.3, 0.4], 2.0, 1.0, 0.5, invariant=0.1, gamma_shape=0.9, gamma_k=3)
    L = 3_000_000
    g = J.random_genome(1, L, seed=41)
    names = ["a", "b", "c"]
    recs = HG.mutate_gtrees(g, "//\n[1]%s\n[2]%s\n" % (t1, t2), names, m, seed=4242)
    lut = np.full(256, 255, dtype=np.uint8)
    lut[np.frombuffer(b"TCAG", dtype=np.uint8)] = np.arange(4, dtype=np.uint8)
    ref = lut[g.seqs[0]]
    states = {}
    for t, nm in enumerate(names):
        s = ref.astype(np.int64).copy()
        pos, nuc = recs[t][0]
        s[pos.astype(np.int64)] = lut[np.frombuffer(nuc, dtype=np.uint8)]
        states[nm] = s
    for (lo, hi), nw in (((0, L // 3), t1), ((L // 3, L), t2)):
        tree = parse_newick(nw)
        pat = np.zeros(hi - lo, dtype=np.int64)
        for nm in tree.tip_names:                         # the tree's tip order: tip 0 most significant
            pat = pat * 4 + states[nm][lo:hi]
        keep = ref[lo:hi] < 4
        assert chi2_fit(ref[lo:hi][keep], pat[keep], tree, m) > 0.001
    # and the other tree does not fit region 1: the contrast is visible at this size
    tree = parse_newick(t2)
    pat = np.zeros(L // 3, dtype=np.int64)
    for nm in tree.tip_names:
        pat = pat * 4 + states[nm][:L // 3]
    keep = ref[:L // 3] < 4
    assert chi2_fit(ref[:L // 3][keep], pat[keep], tree, m) < 1e-6


def test_gtree_structs_match_the_header():
    import os
    import re
    from jackalope_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "jlp_b200.h")).read()
    for struct, cls in (("jlp_gtree_params", _lib.GtreeParams), ("jlp_gtree_stats", _lib.GtreeStats)):
        body = hdr[hdr.index("typedef struct " + struct):hdr.index("} " + struct + ";")]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S).split("{", 1)[1]
        names = [re.findall(r"([A-Za-z_][A-Za-z_0-9]*)\s*$", d.strip())[0] for d in body.split(";") if d.strip()]
        assert names == [f[0] for f in cls._fields_]
