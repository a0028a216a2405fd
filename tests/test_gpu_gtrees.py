"""create_haplotypes along gene trees on the GPU: records byte-identical to the oracle's per-site walk with each
region's tree, the one-tree case equal to haps_phylo, windows, determinism, several devices, the device-built
transition tables against jlp_transition_matrix, and the haplotypes through illumina() / write_vcf()."""
import os
import tempfile

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200.mutate import kingman, transition_matrix, transition_tables
from oracle import harness_gtrees as HG
from oracle import vcf_oracle as V
from oracle.compare import first_diff, oracle_run
from test_gpu_mutate import MODELS, genome_with_n_runs

pytestmark = pytest.mark.gpu


def ms_tree(n, rng, scale=0.05):
    """a Kingman tree of n tips labelled 1..n as ms labels them, Newick text"""
    t = kingman(n, rng).scaled(scale)
    return J.Tree(t.parent, t.branch_len, t.tip_node, [str(i + 1) for i in range(n)]).newick()


def ms_text(blocks):
    """blocks: per chromosome a list of (n or None, Newick)"""
    out = ["ms %d 1 -T\n1 2 3\n" % 2]
    for b in blocks:
        out.append("\n//\n")
        out += ["%s%s\n" % ("" if n is None else "[%d]" % n, nw) for n, nw in b]
        out.append("segsites: 0\n")
    return "".join(out)


def random_blocks(lens, n_tips, rng, per_chrom):
    return [[(int(rng.integers(1, 2000)), ms_tree(n_tips, rng)) for _ in range(per_chrom)] for _ in lens]


def check(ctx, g, text, sub, seed, **kw):
    with tempfile.TemporaryDirectory() as d:
        fn = os.path.join(d, "trees.ms")
        with open(fn, "w") as f:
            f.write(text)
        info = J.haps_gtrees(fn=fn)
    haps = J.create_haplotypes(g, info, sub, seed=seed, ctx=ctx, **kw)
    want = HG.mutate_gtrees(g, text, info.names, sub, seed)
    assert haps.tree is None and haps.hap_names == info.names
    n_rec = 0
    for h in range(haps.n_haps()):
        for c in range(g.n_chroms()):
            m = haps.muts[h][c]
            pos, nuc = want[h][c]
            assert np.array_equal(m.old_pos, pos) and m.pool.tobytes() == nuc, (h, c)
            assert np.array_equal(m.new_pos, m.old_pos) and np.array_equal(m.nuc_off, np.arange(pos.size))
            assert m.chrom_size == g.seqs[c].size
            n_rec += pos.size
    assert haps.stats["records"] == n_rec
    return haps


def same_records(a, b):
    return all(np.array_equal(a.muts[h][c].old_pos, b.muts[h][c].old_pos) and
               a.muts[h][c].pool.tobytes() == b.muts[h][c].pool.tobytes()
               for h in range(a.n_haps()) for c in range(a.n_chroms()))


@pytest.mark.parametrize("model", sorted(MODELS))
def test_records_equal_the_oracle_every_model(ctx, model):
    rng = np.random.default_rng(len(model))
    g = genome_with_n_runs([150_001, 9_999, 40_123], seed=3)
    sub = MODELS[model](invariant=0.15, gamma_shape=0.6, gamma_k=4)
    haps = check(ctx, g, ms_text(random_blocks(g.seqs, 40, rng, 7)), sub, seed=11)
    assert haps.stats["n_trees"] == 21 and haps.stats["n_regions"] <= 21


@pytest.mark.parametrize("n_tips", [2, 40, 1024])
def test_records_equal_the_oracle_tips(ctx, n_tips):
    rng = np.random.default_rng(n_tips)
    g = genome_with_n_runs([30_011, 20_000], seed=n_tips)
    per = 2 if n_tips == 1024 else 5
    check(ctx, g, ms_text(random_blocks(g.seqs, n_tips, rng, per)), MODELS["HKY85"](gamma_shape=0.5), seed=13)


def test_boundaries_inside_blocks_short_regions_and_n_runs(ctx):
    L = 40_000
    g = genome_with_n_runs([L], seed=5)
    seq = g.seqs[0].copy()
    seq[4090:4110] = ord("N")                       # an N run across the boundary at 4097
    seq[12340:12350] = ord("N")
    g = J.RefGenome(g.names, [seq])
    cuts = [1, 4, 4097, 4098, 4101, 8191, 12345, 12346, 20000, 20003, L]      # regions of 1 and 3 sites
    rng = np.random.default_rng(1)
    lens = np.diff([0] + cuts).tolist()               # S = L: the lengths as written
    text = ms_text([[(n, ms_tree(6, rng, 0.5)) for n in lens]])
    haps = check(ctx, g, text, MODELS["GTR"](invariant=0.1), seed=17)
    assert haps.stats["n_regions"] == len(cuts)


def test_more_than_a_thousand_regions_and_a_tiny_table_budget(ctx):
    rng = np.random.default_rng(2)
    g = genome_with_n_runs([300_007, 5_003], seed=6)
    text = ms_text([[(int(rng.integers(1, 600)), ms_tree(5, rng, 0.3)) for _ in range(1500)],
                    [(int(rng.integers(1, 600)), ms_tree(5, rng, 0.3)) for _ in range(3)]])
    sub = MODELS["F84"](gamma_shape=0.7)
    a = check(ctx, g, text, sub, seed=19)
    assert a.stats["n_regions"] > 1000 and a.stats["windows"] == 1
    b = check(ctx, g, text, sub, seed=19, table_budget=4096)
    assert b.stats["windows"] > 100 and same_records(a, b)


def test_one_tree_everywhere_is_haps_phylo(ctx):
    g = genome_with_n_runs([100_003, 17, 50_000], seed=7)
    nw = "((1:0.1,2:0.25):0.05,(3:0.02,(4:1e-3,5:0.7):0.1):0.4);"
    sub = MODELS["UNREST"](invariant=0.2, gamma_shape=1.5, gamma_k=3)
    ref = J.create_haplotypes(g, J.haps_phylo(nw), sub, seed=23, ctx=ctx)
    rng = np.random.default_rng(3)
    for text in (ms_text([[(None, nw)]] * 3),
                 ms_text([[(int(rng.integers(1, 9)), nw) for _ in range(int(rng.integers(1, 40)))] for _ in range(3)])):
        got = J.create_haplotypes(g, J.haps_gtrees(obj=[[ln for ln in blk.split("\n") if ln[:1] in "[("]
                                                        for blk in text.split("//")[1:]]),
                                  sub, seed=23, ctx=ctx)
        assert got.hap_names == ref.hap_names and same_records(got, ref)


def test_determinism_and_independence_of_other_chromosomes(ctx):
    rng = np.random.default_rng(4)
    g = J.random_genome(3, 200_000, seed=8)
    blocks = random_blocks(g.seqs, 6, rng, 4)
    sub = MODELS["K80"](gamma_shape=0.5)
    info = J.haps_gtrees(obj=[["[%d]%s" % b for b in blk] for blk in blocks])
    a = J.create_haplotypes(g, info, sub, seed=21, ctx=ctx)
    b = J.create_haplotypes(g, info, sub, seed=21, ctx=ctx)
    c = J.create_haplotypes(g, info, sub, seed=22, ctx=ctx)
    assert same_records(a, b) and not same_records(a, c)
    other = J.random_genome(2, [123_457, 50_000], seed=9)
    gab = J.RefGenome(["A", "B"], [g.seqs[0], g.seqs[1]])
    gac = J.RefGenome(["A", "C"], [g.seqs[0], other.seqs[1]])
    x = J.create_haplotypes(gab, J.haps_gtrees(obj=[["[%d]%s" % b for b in blk] for blk in blocks[:2]]), sub, seed=21, ctx=ctx)
    y = J.create_haplotypes(gac, J.haps_gtrees(obj=[["[%d]%s" % b for b in blocks[0]], ["(1:1,(2:1,(3:1,(4:1,(5:1,6:1):1):1):1):1);"]]),
                            sub, seed=21, ctx=ctx)
    for h in range(6):
        assert np.array_equal(x.muts[h][0].old_pos, y.muts[h][0].old_pos)
        assert x.muts[h][0].pool.tobytes() == y.muts[h][0].pool.tobytes()
        assert np.array_equal(x.muts[h][0].old_pos, a.muts[h][0].old_pos)


def test_block_count_must_match(ctx):
    g = J.random_genome(2, 1000, seed=1)
    with pytest.raises(J.JackalopeError, match="1 blocks.*2 chromosomes"):
        J.create_haplotypes(g, J.haps_gtrees(obj=[["(1:1,2:1);"]]), MODELS["JC69"](), seed=1, ctx=ctx)


def test_multi_gpu_context_gives_the_same_haplotypes(ctx):
    rng = np.random.default_rng(5)
    g = J.random_genome(4, 100_003, seed=10)
    info = J.haps_gtrees(obj=[["[%d]%s" % b for b in blk] for blk in random_blocks(g.seqs, 5, rng, 3)])
    sub = MODELS["TN93"](invariant=0.1)
    one = J.create_haplotypes(g, info, sub, seed=31, ctx=ctx)
    multi = J.Context(devices=[0, 0])
    try:
        two = J.create_haplotypes(g, info, sub, seed=31, ctx=multi)
        assert same_records(one, two)
        r1, r2, _ = J.illumina(two, "", 4000, 100, True, seed=5, ctx=multi, sink="memory", seq_sys="HS25")
        s1, s2, _ = J.illumina(one, "", 4000, 100, True, seed=5, ctx=ctx, sink="memory", seq_sys="HS25")
        assert r1 == s1 and r2 == s2
    finally:
        multi.close()


def host_tables(Q, ts):
    P = np.array([transition_matrix(Q, t) for t in ts])
    thr = np.zeros((len(ts), 4, 3), dtype=np.uint64)
    for i in range(len(ts)):
        for a in range(4):
            p = np.where(P[i, a] > 0, P[i, a], 0.0)
            s, c = 0.0, 0.0
            for j in range(4):
                s += p[j]
            for j in range(3):
                c += p[j] / s
                thr[i, a, j] = 0 if not c > 0 else (2 ** 64 - 1 if c >= 1 else int(np.ldexp(c, 64)))
    return P, thr


def test_device_tables_equal_the_host_bit_for_bit(ctx):
    rng = np.random.default_rng(6)
    for trial in range(6):
        Q = rng.exponential(1.0, (4, 4)) * (10.0 ** rng.uniform(-2, 1))
        if trial == 0:
            Q = MODELS["UNREST"]().Q
        np.fill_diagonal(Q, 0)
        ts = np.concatenate(([0.0, 1e-8], 10 ** rng.uniform(-8, 2, 3000)))
        P, thr, nh = transition_tables(Q, ts, ctx=ctx)
        Ph, thrh = host_tables(Q, ts)
        assert np.array_equal(P.view(np.uint64), Ph.view(np.uint64)), trial
        assert np.array_equal(thr, thrh), trial
    # t with ||Q t||_1 = 2^k (1 + 2^-52): the scaling exponent is left to the host
    Q = MODELS["GTR"]().Q.copy()
    np.fill_diagonal(Q, 0)
    A = Q.copy()
    np.fill_diagonal(A, -Q.sum(axis=1))
    norm1 = np.abs(A).sum(axis=0).max()
    ts = []
    for k in range(-1, 9):
        t = np.ldexp(1.0, k) * (1 + 2.0 ** -52) / norm1
        for step in range(-3, 4):                      # neighbours, until the rounded norm lands there
            x = np.nextafter(t, np.inf) if step > 0 else t
            for _ in range(abs(step)):
                x = np.nextafter(x, np.inf if step > 0 else -np.inf)
            ts.append(x)
    ts = np.array(ts)
    P, thr, nh = transition_tables(Q, ts, ctx=ctx)
    Ph, thrh = host_tables(Q, ts)
    assert nh > 0
    assert np.array_equal(P.view(np.uint64), Ph.view(np.uint64)) and np.array_equal(thr, thrh)


def test_illumina_and_write_vcf_on_gene_tree_haplotypes(ctx, tmp_path):
    rng = np.random.default_rng(7)
    g = genome_with_n_runs([60_000, 30_011, 40_000], seed=12)
    info = J.haps_gtrees(obj=[["[%d]%s" % b for b in blk] for blk in random_blocks(g.seqs, 4, rng, 6)])
    haps = J.create_haplotypes(g, info, MODELS["TN93"](gamma_shape=0.5), seed=41, ctx=ctx)
    r1, r2, st = J.illumina(haps, "", 6000, 150, True, seed=42, ctx=ctx, sink="memory", seq_sys="HS25")
    o = oracle_run(haps, 6000, 150, True, seed=42, seq_sys="HS25")
    assert first_diff(r1, o["r1"]) is None and first_diff(r2, o["r2"]) is None
    J.write_vcf(haps, str(tmp_path / "o"), ctx=ctx, file_date="20261022", overwrite=True)
    got = (tmp_path / "o.vcf").read_bytes()
    assert got == V.vcf(haps, file_date="20261022")
