"""create_haplotypes on the GPU: records byte-identical to the oracle's per-site walk, determinism, edge cases,
and the haplotypes through illumina() / pacbio()."""
import numpy as np
import pytest
from scipy import stats

import jackalope_b200 as J
from jackalope_b200.mutate import haplotype_muts, parse_newick
from oracle import harness_mutate as HM
from oracle.compare import first_diff, oracle_run

pytestmark = pytest.mark.gpu

PI = [0.1, 0.2, 0.3, 0.4]
MODELS = {
    "JC69": lambda **kw: J.sub_JC69(0.5, **kw),
    "K80": lambda **kw: J.sub_K80(2.0, 0.5, **kw),
    "F81": lambda **kw: J.sub_F81(PI, **kw),
    "HKY85": lambda **kw: J.sub_HKY85(PI, 2.0, 0.5, **kw),
    "F84": lambda **kw: J.sub_F84(PI, 0.4, 1.5, **kw),
    "TN93": lambda **kw: J.sub_TN93(PI, 3.0, 1.2, 0.5, **kw),
    "GTR": lambda **kw: J.sub_GTR(PI, [1, 2, 3, 4, 5, 6], **kw),
    "UNREST": lambda **kw: J.sub_UNREST([[0, 0.1, 0.7, 0.2], [0.3, 0, 0.05, 0.9], [0.6, 0.2, 0, 0.4], [0.1, 1.1, 0.3, 0]], **kw),
}


def genome_with_n_runs(lens, seed):
    g = J.random_genome(len(lens), lens, seed=seed)
    rng = np.random.default_rng(seed)
    seqs = []
    for s in g.seqs:
        s = s.copy()
        for _ in range(3):
            a = int(rng.integers(0, s.size))
            s[a:a + int(rng.integers(1, 3000))] = ord("N")
        s[:7] = np.frombuffer(b"nNRacgt", dtype=np.uint8)
        seqs.append(s)
    return J.RefGenome(g.names, seqs)


def check_against_oracle(ctx, g, info, sub, seed):
    haps = J.create_haplotypes(g, info, sub, seed=seed, ctx=ctx)
    tree = info.tree(sub, seed)
    want = HM.mutate(g, tree, sub, seed)
    assert haps.hap_names == tree.tip_names and sorted(parse_newick(haps.tree).tip_names) == sorted(tree.tip_names)
    n_rec = 0
    for h in range(haps.n_haps()):
        for c in range(g.n_chroms()):
            m = haps.muts[h][c]
            pos, nuc = want[h][c]
            assert np.array_equal(m.old_pos, pos) and m.pool.tobytes() == nuc, (h, c)
            assert np.array_equal(m.new_pos, m.old_pos) and np.all(m.nuc_len == 1)
            assert np.array_equal(m.nuc_off, np.arange(pos.size)) and m.chrom_size == g.seqs[c].size
            assert np.all(np.diff(m.old_pos.astype(np.int64)) > 0)
            ref = g.seqs[c][m.old_pos.astype(np.int64)]
            assert np.all(np.isin(ref, np.frombuffer(b"TCAG", np.uint8))) and np.all(np.isin(m.pool, np.frombuffer(b"TCAG", np.uint8)))
            assert np.all(ref != m.pool)
            n_rec += pos.size
    assert haps.stats["records"] == n_rec
    return haps


@pytest.mark.parametrize("model", sorted(MODELS))
def test_records_equal_the_oracle_every_model(ctx, model):
    g = genome_with_n_runs([150_001, 9_999, 40_123], seed=3)
    sub = MODELS[model](invariant=0.15, gamma_shape=0.6, gamma_k=4)
    haps = check_against_oracle(ctx, g, J.haps_theta(0.05, 40), sub, seed=11)
    for h in (0, 17, 39):
        for c in range(g.n_chroms()):
            m = haps.muts[h][c]
            want = g.seqs[c].copy()
            want[m.old_pos.astype(np.int64)] = m.pool
            assert ctx.haplotype_chrom(h, c) == want.tobytes()


def test_records_equal_the_oracle_tiles_cross(ctx):
    g = genome_with_n_runs([2_500_003, 2_499_999, 2_600_000], seed=4)
    info = J.haps_phylo("(left:0.02,right:0.3);")
    check_against_oracle(ctx, g, info, MODELS["TN93"](gamma_shape=1.0, gamma_k=5), seed=12)


def test_records_equal_the_oracle_1024_tips(ctx):
    g = genome_with_n_runs([20_011], seed=5)
    haps = check_against_oracle(ctx, g, J.haps_theta(0.1, 1024), MODELS["HKY85"](), seed=13)
    assert haps.n_haps() == 1024
    with pytest.raises(J.JackalopeError, match="4096"):
        J.create_haplotypes(g, J.haps_theta(0.1, 4097), MODELS["HKY85"](), seed=1, ctx=ctx)


def test_multifurcation_zero_branch_and_long_branch_tree(ctx):
    g = genome_with_n_runs([300_007, 77], seed=6)
    info = J.haps_phylo("((A:0.1,B:0.25)x:0.05,(C:0.02,D:0,E:0.6,(F:1e-3,G:2)y:0):0.4)r;")
    check_against_oracle(ctx, g, info, MODELS["GTR"](invariant=0.3), seed=14)


def test_determinism_and_independence_of_other_chromosomes(ctx):
    g = J.random_genome(3, 200_000, seed=7)
    info, sub = J.haps_theta(0.02, 6), MODELS["F84"](gamma_shape=0.5)
    a = J.create_haplotypes(g, info, sub, seed=21, ctx=ctx)
    b = J.create_haplotypes(g, info, sub, seed=21, ctx=ctx)
    c = J.create_haplotypes(g, info, sub, seed=22, ctx=ctx)
    same = lambda x, y: all(np.array_equal(x.muts[h][k].old_pos, y.muts[h][k].old_pos) and
                            np.array_equal(x.muts[h][k].pool, y.muts[h][k].pool)
                            for h in range(x.n_haps()) for k in range(x.n_chroms()))
    assert same(a, b) and not same(a, c) and a.tree == b.tree and a.tree != c.tree
    # genome [A, B] against [A, C]: chromosome A's records do not change
    other = J.random_genome(2, [123_457, 50_000], seed=8)
    gab = J.RefGenome(["A", "B"], [g.seqs[0], g.seqs[1]])
    gac = J.RefGenome(["A", "C"], [g.seqs[0], other.seqs[1]])
    x = J.create_haplotypes(gab, info, sub, seed=21, ctx=ctx)
    y = J.create_haplotypes(gac, info, sub, seed=21, ctx=ctx)
    for h in range(6):
        assert np.array_equal(x.muts[h][0].old_pos, y.muts[h][0].old_pos)
        assert np.array_equal(x.muts[h][0].pool, y.muts[h][0].pool)
        assert np.array_equal(x.muts[h][0].old_pos, a.muts[h][0].old_pos)


def test_multi_gpu_context_gives_the_same_haplotypes(ctx):
    g = J.random_genome(4, 100_003, seed=9)
    info, sub = J.haps_theta(0.03, 5), MODELS["UNREST"](invariant=0.1)
    one = J.create_haplotypes(g, info, sub, seed=31, ctx=ctx)
    multi = J.Context(devices=[0, 0])
    try:
        two = J.create_haplotypes(g, info, sub, seed=31, ctx=multi)
        for h in range(5):
            for c in range(4):
                assert np.array_equal(one.muts[h][c].old_pos, two.muts[h][c].old_pos)
                assert np.array_equal(one.muts[h][c].pool, two.muts[h][c].pool)
        r1, r2, _ = J.illumina(two, "", 4000, 100, True, seed=5, ctx=multi, sink="memory", seq_sys="HS25")
        s1, s2, _ = J.illumina(one, "", 4000, 100, True, seed=5, ctx=ctx, sink="memory", seq_sys="HS25")
        assert r1 == s1 and r2 == s2
    finally:
        multi.close()


def test_zero_branches_give_no_records_long_branches_reach_stationarity(ctx):
    g = J.random_genome(2, 400_000, seed=10)
    haps = J.create_haplotypes(g, J.haps_phylo("((a:0,b:0):0,c:0);"), MODELS["JC69"](), seed=3, ctx=ctx)
    assert all(haps.muts[h][c].old_pos.size == 0 for h in range(3) for c in range(2))
    assert haps.stats["records"] == 0
    sub = MODELS["UNREST"]()
    haps = J.create_haplotypes(g, J.haps_phylo("(a:60,b:80);"), sub, seed=4, ctx=ctx)
    for h in range(2):
        tip = np.concatenate([g.seqs[c].copy() for c in range(2)])
        off = 0
        for c in range(2):
            m = haps.muts[h][c]
            tip[off + m.old_pos.astype(np.int64)] = m.pool
            off += g.seqs[c].size
        obs = np.array([np.sum(tip == ord(b)) for b in "TCAG"])
        assert stats.chisquare(obs, sub.pi * obs.sum()).pvalue > 0.001


def test_end_to_end_illumina_and_pacbio(ctx):
    g = J.random_genome(3, 60_000, seed=12)
    haps = J.create_haplotypes(g, J.haps_theta(0.02, 4), MODELS["TN93"](gamma_shape=0.5), seed=41, ctx=ctx)
    assert ctx._haps is haps
    for kw in (dict(seq_sys="HS25"), dict(seq_sys="HS25", sep_files=True, haplotype_probs=[1, 2, 3, 4])):
        r1, r2, st = J.illumina(haps, "", 6000, 150, True, seed=42, ctx=ctx, sink="memory", **kw)
        o = oracle_run(haps, 6000, 150, True, seed=42, **kw)
        assert first_diff(r1, o["r1"]) is None and first_diff(r2, o["r2"]) is None
    fq, _ = J.pacbio(haps, "", 200, seed=7, ctx=ctx, sink="memory")
    assert fq.count(b"\n") == 4 * 200


def test_get_haplotype_muts_returns_what_add_haplotype_stored(ctx):
    g = J.random_genome(3, 50_000, seed=13)
    haps = J.random_haplotypes(g, 3, sub_rate=0.01, indel_rate=0.002, seed=14)
    ctx.set_haplotypes(haps)
    for h in range(3):
        for c in range(3):
            got, m = haplotype_muts(ctx, h, c), haps.muts[h][c]
            assert np.array_equal(got.old_pos, m.old_pos) and np.array_equal(got.new_pos, m.new_pos)
            assert np.array_equal(got.nuc_off, m.nuc_off) and got.pool.tobytes() == m.pool.tobytes()
            assert np.array_equal(got.nuc_len, m.nuc_len) and got.chrom_size == m.chrom_size
