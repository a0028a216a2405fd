"""The kernels' exact-draw fallbacks on the GPU, reached on purpose: create_haplotypes records and tip chromosomes,
and Illumina FASTQ, byte-identical to the oracles on the cases test_draw_fallbacks_host.py constructs and proves.
Each test asserts that proof again (ties present on both sides, exact ties, flips) before it compares, so a case
that stops reaching its fallback fails instead of passing without testing it."""
import numpy as np
import pytest

import jackalope_b200 as J
from oracle import harness_indels as HI
from oracle import harness_mutate as HM
from oracle.compare import explain_diff, first_diff
from test_draw_fallbacks_host import (ALL_N_KW, ALL_N_PAIRS, ALL_N_SEED, INS_KIDS, SLOT_KW, SLOT_PAIRS, SLOT_SEED,
                                      all_n_genome, all_n_oracle, prove_category_tie, prove_transition_ties,
                                      slot_genome, slot_oracle, tie_case)

pytestmark = pytest.mark.gpu


def check_mutate(ctx, case):
    """Records and materialised tips of create_haplotypes equal the oracle's (substitutions only)."""
    g = case.genome
    haps = J.create_haplotypes(g, J.haps_phylo(case.newick), case.sub, seed=case.seed, ctx=ctx)
    want = HM.mutate(g, case.tree, case.sub, case.seed)
    n_rec = 0
    for h in range(haps.n_haps()):
        m = haps.muts[h][0]
        pos, nuc = want[h][0]
        assert np.array_equal(m.old_pos, pos) and m.pool.tobytes() == nuc, h
        tip = g.seqs[0].copy()
        tip[pos.astype(np.int64)] = np.frombuffer(nuc, np.uint8)
        assert ctx.haplotype_chrom(h, 0) == tip.tobytes(), h
        n_rec += pos.size
    assert haps.stats["records"] == n_rec
    return haps


def check_indels(ctx, case):
    """Records and materialised tips of create_haplotypes with indels equal the oracle's."""
    g = case.genome
    haps = J.create_haplotypes(g, J.haps_phylo(case.newick), case.sub, ins=case.ins, del_=case.dele, epsilon=case.eps,
                               seed=case.seed, ctx=ctx)
    o = HI.indels(g, case.tree, case.sub, case.ins, case.dele, case.eps, case.seed)
    for h in range(haps.n_haps()):
        m = haps.muts[h][0]
        seq, (old, new, nuc, _, pool) = o.tips[h][0]
        assert np.array_equal(m.old_pos, old) and np.array_equal(m.new_pos, new), h
        assert np.array_equal(m.nuc_off, nuc) and m.pool.tobytes() == pool, h
        assert ctx.haplotype_chrom(h, 0) == seq, h
    return haps


@pytest.mark.parametrize("name,smem", [("smem", 1), ("global", 0)])
def test_transition_ties(ctx, name, smem):
    case = tie_case(name)
    c = prove_transition_ties(case)
    assert c["exact"] >= 3 and sum(case.tree.parent[t.node] != 0 for t in case.ties) == 16
    haps = check_mutate(ctx, case)
    assert haps.stats["table_in_smem"] == smem


def test_transition_ties_with_indels(ctx):
    case = tie_case("indels")
    c = prove_transition_ties(case)
    assert c["ties"] == 168 and c["exact"] >= 1
    haps = check_indels(ctx, case)
    assert haps.stats["insertions"] > 0 and haps.stats["deletions"] > 0


def test_ins_walk_ties(ctx):
    case = tie_case("ins_walk")
    c = prove_transition_ties(case)
    assert c["ties"] == INS_KIDS and c["exact"] >= 1
    check_indels(ctx, case)


@pytest.mark.parametrize("name,evolves", [("cat0_exact", 1), ("cat0_below", 1), ("cat0_above", 0),
                                          ("cat1_lo", 2), ("cat1_hi", 1)])
def test_category_ties(ctx, name, evolves):
    case = tie_case(name)
    assert prove_category_tie(case) == evolves
    check_mutate(ctx, case)


def test_n_qualities_undecided_on_24_bits(ctx):
    o = all_n_oracle()
    assert o["fallback"]["nqual_flipped"] >= 2
    r1, r2, _ = J.illumina(all_n_genome(), "", 2 * ALL_N_PAIRS, 150, True, seed=ALL_N_SEED, ctx=ctx, sink="memory",
                           **ALL_N_KW)
    assert first_diff(r1, o["r1"]) is None, explain_diff(r1, o["r1"])
    assert first_diff(r2, o["r2"]) is None, explain_diff(r2, o["r2"])


def test_alias_slot_and_substitution_carries(ctx):
    slices, fb = slot_oracle()
    assert fb["slot_flipped"] >= 3 and fb["sub_flipped"] >= 3
    r1, r2, _ = J.illumina(slot_genome(), "", 2 * SLOT_PAIRS, 150, True, seed=SLOT_SEED, ctx=ctx, sink="memory",
                           **SLOT_KW)
    lines1, lines2 = r1.split(b"\n"), r2.split(b"\n")
    assert len(lines1) == len(lines2) == 4 * SLOT_PAIRS + 1
    for lo, hi, o1, o2 in slices:
        got1, got2 = b"\n".join(lines1[4 * lo:4 * hi]) + b"\n", b"\n".join(lines2[4 * lo:4 * hi]) + b"\n"
        assert first_diff(got1, o1) is None, explain_diff(got1, o1)
        assert first_diff(got2, o2) is None, explain_diff(got2, o2)
