"""create_haplotypes with insertions and deletions on the GPU: records and materialised haplotypes byte-identical to
the oracle, indels(0) equal to None, determinism, multi-GPU contexts, and the haplotypes through illumina() / pacbio()."""
import numpy as np
import pytest

import jackalope_b200 as J
from oracle import harness_indels as HI
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
        s[:min(7, s.size)] = np.frombuffer(b"nNRacgt", dtype=np.uint8)[:min(7, s.size)]
        seqs.append(s)
    return J.RefGenome(g.names, seqs)


def check(ctx, g, info, sub, ins, dele, eps, seed):
    haps = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, epsilon=eps, seed=seed, ctx=ctx)
    tree = info.tree(sub, seed)
    o = HI.indels(g, tree, sub, ins, dele, eps, seed)
    n_rec = 0
    for h in range(haps.n_haps()):
        for c in range(g.n_chroms()):
            m = haps.muts[h][c]
            seq, (old, new, nuc, sm, pool) = o.tips[h][c]
            assert np.array_equal(m.old_pos, old) and np.array_equal(m.new_pos, new), (h, c)
            assert np.array_equal(m.nuc_off, nuc) and m.pool.tobytes() == pool, (h, c)
            assert m.chrom_size == len(seq), (h, c)
            assert ctx.haplotype_chrom(h, c) == seq, (h, c)
            n_rec += old.size
    assert haps.stats["records"] == n_rec
    ev = o.events
    assert haps.stats["insertions"] == int(np.sum(ev[:, 4] == 1)) and haps.stats["deletions"] == int(np.sum(ev[:, 4] == 0))
    assert haps.stats["inserted_bases"] == int(ev[ev[:, 4] == 1, 5].sum()) and haps.stats["steps"] == len(o.steps)
    return haps, o


@pytest.mark.parametrize("model", sorted(MODELS))
def test_records_equal_the_oracle_every_model(ctx, model):
    g = genome_with_n_runs([60_001, 9_999, 20_123], seed=3)
    sub = MODELS[model](invariant=0.15, gamma_shape=0.6, gamma_k=4)
    check(ctx, g, J.haps_theta(0.05, 40), sub, J.indels(0.01, max_length=8), J.indels(0.012, a=1.2), 0.03, 11)


@pytest.mark.parametrize("kinds", ["ins", "del", "both"])
def test_insertions_only_deletions_only_both(ctx, kinds):
    g = genome_with_n_runs([100_003, 777], seed=4)
    ins = J.indels(0.05, rel_rates=[1, 2, 0, 1]) if kinds in ("ins", "both") else None
    dele = J.indels(0.05) if kinds in ("del", "both") else None
    check(ctx, g, J.haps_phylo("((a:0.1,b:0.25)x:0.05,(c:0.02,d:0,e:0.6)y:0.4);"), MODELS["HKY85"](gamma_shape=1.0),
          ins, dele, 0.03, 12)


@pytest.mark.parametrize("n_tips", [2, 1024])
def test_records_equal_the_oracle_tip_counts(ctx, n_tips):
    g = genome_with_n_runs([20_011, 8_193], seed=5)
    check(ctx, g, J.haps_theta(0.1, n_tips), MODELS["TN93"](gamma_shape=0.5), J.indels(0.02), J.indels(0.02), 0.03, 13)


def test_several_steps_per_branch_and_tiles_crossing_chromosome_ends(ctx):
    g = genome_with_n_runs([30_001, 8_192, 8_193, 16_383], seed=6)
    haps, o = check(ctx, g, J.haps_phylo("(left:0.2,(m:0.1,right:0.3):0.4);"), MODELS["GTR"](invariant=0.3),
                    J.indels(0.1, max_length=20), J.indels(0.1, max_length=30, a=0.8), 0.002, 14)
    assert o.steps[:, 2].max() >= 20


def test_a_small_chromosome_lost_entirely(ctx):
    g = J.random_genome(2, [40_000, 6], seed=7)
    info, sub = J.haps_phylo("(a:3,(b:0.01,c:2):0.5);"), MODELS["JC69"]()
    ins, dele = J.indels(0.01), J.indels(1.5, max_length=4)
    seed = next(s for s in range(100, 200)
                if any(len(t[1][0]) == 0 for t in HI.indels(g, info.tree(sub, s), sub, ins, dele, 0.05, s).tips))
    haps, _ = check(ctx, g, info, sub, ins, dele, 0.05, seed)
    assert any(haps.muts[h][1].chrom_size == 0 for h in range(3))


def test_zero_rates_equal_none_and_determinism(ctx):
    g = J.random_genome(3, 150_000, seed=8)
    info, sub = J.haps_theta(0.02, 6), MODELS["F84"](gamma_shape=0.5)
    a = J.create_haplotypes(g, info, sub, seed=21, ctx=ctx)
    b = J.create_haplotypes(g, info, sub, ins=J.indels(0), del_=J.indels(0), seed=21, ctx=ctx)
    fields = ("old_pos", "new_pos", "nuc_off", "pool")
    same = lambda x, y, k=None: all(np.array_equal(getattr(x.muts[h][c], f), getattr(y.muts[h][c], f)) and
                                    x.muts[h][c].chrom_size == y.muts[h][c].chrom_size
                                    for h in range(x.n_haps()) for c in (range(x.n_chroms()) if k is None else [k])
                                    for f in fields)
    assert same(a, b)
    ins, dele = J.indels(0.01), J.indels(0.01)
    x = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=21, ctx=ctx)
    y = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=21, ctx=ctx)
    z = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=22, ctx=ctx)
    assert same(x, y) and not same(x, z) and x.stats["indel_records"] > 0
    # genome [A, B] against [A, C]: chromosome A's records do not change
    other = J.random_genome(2, [123_457, 50_000], seed=9)
    gab = J.RefGenome(["A", "B"], [g.seqs[0], g.seqs[1]])
    gac = J.RefGenome(["A", "C"], [g.seqs[0], other.seqs[1]])
    p = J.create_haplotypes(gab, info, sub, ins=ins, del_=dele, seed=21, ctx=ctx)
    q = J.create_haplotypes(gac, info, sub, ins=ins, del_=dele, seed=21, ctx=ctx)
    assert same(p, q, 0) and same(p, x, 0)


def test_multi_gpu_illumina_add_haplotype_and_pacbio(ctx):
    g = J.random_genome(4, 60_003, seed=10)
    info, sub = J.haps_theta(0.03, 5), MODELS["UNREST"](invariant=0.1)
    ins, dele = J.indels(0.02), J.indels(0.02, a=1.1)
    one = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=31, ctx=ctx)
    assert one.stats["indel_records"] > 0
    kw = dict(seq_sys="HS25")
    s1, s2, _ = J.illumina(one, "", 4000, 100, True, seed=5, ctx=ctx, sink="memory", **kw)
    o = oracle_run(one, 4000, 100, True, seed=5, **kw)
    assert first_diff(s1, o["r1"]) is None and first_diff(s2, o["r2"]) is None
    multi = J.Context(devices=[0, 0])
    fresh = J.Context(0)
    try:
        two = J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=31, ctx=multi)
        for h in range(5):
            for c in range(4):
                for f in ("old_pos", "new_pos", "nuc_off", "pool"):
                    assert np.array_equal(getattr(one.muts[h][c], f), getattr(two.muts[h][c], f))
        r1, r2, _ = J.illumina(two, "", 4000, 100, True, seed=5, ctx=multi, sink="memory", **kw)
        assert r1 == s1 and r2 == s2
        fresh.set_haplotypes(one)          # jlp_add_haplotype: size_modifier from the records
        f1, f2, _ = J.illumina(one, "", 4000, 100, True, seed=5, ctx=fresh, sink="memory", **kw)
        assert f1 == s1 and f2 == s2
    finally:
        multi.close()
        fresh.close()
    J.create_haplotypes(g, info, sub, ins=ins, del_=dele, seed=31, ctx=ctx)
    fq, _ = J.pacbio(ctx._haps, "", 200, seed=7, ctx=ctx, sink="memory")
    assert fq.count(b"\n") == 4 * 200
