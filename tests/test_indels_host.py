"""create_haplotypes with insertions and deletions, without a GPU: indels() and the argument errors, hand-written event
lists through the oracle, the oracle's records materialised by a restatement of get_char, and the model's law on the
oracle (chi-square at alpha = 0.001)."""
import math

import numpy as np
import pytest
from scipy import stats

import jackalope_b200 as J
from jackalope_b200.mutate import kingman, parse_newick
from oracle import harness_indels as HI

ALPHA = 1e-3


# ------------------------------------------------------------------ indels() and arguments ---

def test_indels_weights():
    u = np.arange(1, 11)
    m = J.indels(0.01)
    assert m.rate == 0.01 and m.max_length == 10 and np.allclose(m.rel_rates, np.exp(-u))
    m = J.indels(0.2, max_length=4, a=1.5)
    L, u4 = 4, np.arange(1, 5.0)
    assert np.allclose(m.rel_rates, (u4 * L / (L - u4 + 1)) ** -1.5)
    m = J.indels(0, max_length=3, a=2, rel_rates=[0, 2, 1, 5])
    assert m.max_length == 4 and np.array_equal(m.rel_rates, [0, 2, 1, 5]) and np.allclose(m.probs().sum(), 1)


@pytest.mark.parametrize("kw, par", [
    (dict(rate=-1), "rate"), (dict(rate=float("nan")), "rate"), (dict(rate=True), "rate"),
    (dict(rate=1, max_length=0), "max_length"), (dict(rate=1, max_length=2.5), "max_length"),
    (dict(rate=1, a=0), "`a`"), (dict(rate=1, a=-2), "`a`"),
    (dict(rate=1, rel_rates=[0, 0]), "rel_rates"), (dict(rate=1, rel_rates=[1, -1]), "rel_rates"),
    (dict(rate=1, rel_rates=[]), "rel_rates"), (dict(rate=1, rel_rates="ab"), "rel_rates"),
])
def test_indels_argument_errors(kw, par):
    with pytest.raises(J.JackalopeError, match="`indels` function.*%s" % par.strip("`")):
        J.indels(**kw)


def test_create_haplotypes_argument_errors():
    g = J.random_genome(1, 100, seed=1)
    info, sub = J.haps_theta(0.01, 3), J.sub_JC69(1)
    with pytest.raises(J.JackalopeError, match="argument `epsilon` must be a single number > 0"):
        J.create_haplotypes(g, info, sub, ins=J.indels(0.1), epsilon=0, seed=1)
    with pytest.raises(J.JackalopeError, match="argument `epsilon` must be a single number > 0"):
        J.create_haplotypes(g, info, sub, del_=J.indels(0.1), epsilon=0, seed=1)
    with pytest.raises(J.JackalopeError, match="argument `ins` must be NULL or an \"indel_info\""):
        J.create_haplotypes(g, info, sub, ins=0.1, seed=1)
    with pytest.raises(J.JackalopeError, match="argument `del_` must be NULL or an \"indel_info\""):
        J.create_haplotypes(g, info, sub, del_="x", seed=1)
    with pytest.raises(J.JackalopeError, match="argument `epsilon`"):
        J.create_haplotypes(g, info, sub, ins=J.indels(0.1), epsilon=1, seed=1)


# ------------------------------------------------------------- hand-written event lists ---

REF = b"TTCCAATTCC"          # no G: an inserted column (pi = G only, no substitutions) reads G


def hand(events, newick="(x:1,y:1);", ref=REF):
    """The oracle on given events: no substitutions (JC69 rate 0), every inserted column G, one step per branch."""
    return HI.indels(J.RefGenome(["c"], [ref]), parse_newick(newick), J.sub_JC69(0), J.indels(0.1), J.indels(0.1), 0.5, 1,
                     events=events, pi=[0, 0, 0, 1])


def recs(o, t):
    seq, (old, new, nuc, sm, pool) = o.tips[t][0]
    return seq, list(zip(old.tolist(), new.tolist(), nuc.tolist(), sm.tolist())), pool


# rows: (chrom, node, step, pos, 1 insertion / 0 deletion, length); nodes of "(x:1,y:1);": x = 1, y = 2
@pytest.mark.parametrize("name, events, seq, want, pool", [
    ("overlapping deletions", [(0, 1, 0, 2, 0, 3), (0, 1, 0, 3, 0, 4)], b"TTTCC",
     [(2, 2, 0, -5)], b""),
    ("insertion after a deleted position", [(0, 1, 0, 2, 0, 3), (0, 1, 0, 3, 1, 2)], b"TTGGATTCC",
     [(1, 1, 0, 2), (2, 4, 3, -3)], b"TGG"),
    ("deletion clipped at the end", [(0, 1, 0, 8, 0, 9)], b"TTCCAATT",
     [(8, 8, 0, -2)], b""),
    ("insertion after the last base", [(0, 1, 0, 9, 1, 3)], b"TTCCAATTCCGGG",
     [(9, 9, 0, 3)], b"CGGG"),
    ("chromosome deleted entirely", [(0, 1, 0, 0, 0, 4), (0, 1, 0, 3, 0, 10)], b"",
     [(0, 0, 0, -10)], b""),
    ("leading deletion", [(0, 1, 0, 0, 0, 1)], b"TCCAATTCC", [(0, 0, 0, -1)], b""),
])
def test_hand_written_events(name, events, seq, want, pool):
    o = hand(events)
    s, r, p = recs(o, 0)
    assert (s, r, p) == (seq, want, pool), name
    assert recs(o, 1) == (REF, [], b"")


def test_leading_gap_encoding():
    # column 0 kept: an insertion after it is an ordinary insertion record (pool[0] = its base)
    s, r, p = recs(hand([(0, 1, 0, 0, 1, 2)]), 0)
    assert s == b"TGGTCCAATTCC" and r == [(0, 0, 0, 2)] and p == b"TGG"
    # the same with column 0 (and 1 and 2) deleted: one position starts one event, so the deletion starts at 0 and
    # the insertion is at position 1 -- both after the deleted column 0
    s, r, p = recs(hand([(0, 1, 0, 0, 0, 3), (0, 1, 0, 1, 1, 2)]), 0)
    assert s == b"GGCAATTCC" and r == [(0, 0, 0, 1), (1, 2, 2, -2)] and p == b"GG"
    # everything deleted but inserted columns
    s, r, p = recs(hand([(0, 1, 0, 0, 0, 10), (0, 1, 0, 9, 1, 3)]), 0)
    assert s == b"GGG" and r == [(0, 0, 0, 2), (1, 3, 3, -9)] and p == b"GGG"


def test_insertion_inherited_then_partly_deleted():
    # root -> a (node 1) -> tips x (2), y (3): GGGG inserted after position 4 on the branch to a; on the branch to x the
    # last two inserted columns and the reference column 5 go (positions 7..9 of a's sequence)
    newick = "((x:1,y:1)a:1,z:1);"
    o = hand([(0, 1, 0, 4, 1, 4), (0, 2, 0, 7, 0, 3)], newick)
    assert recs(o, 0) == (b"TTCCAGGTTCC", [(4, 4, 0, 2), (5, 7, 3, -1)], b"AGG")
    assert recs(o, 1) == (b"TTCCAGGGGATTCC", [(4, 4, 0, 4)], b"AGGGG")
    assert recs(o, 2) == (REF, [], b"")


# ------------------------------------------------- the records materialise to the tips ---

def get_char_all(ref, old, new, nuc, pool, size):
    """HapChrom::get_chrom_full restated: size_modifier from neighbouring records, as jlp_add_haplotype computes it."""
    M = old.size
    old, new, nuc = old.astype(np.int64), new.astype(np.int64), nuc.astype(np.int64)
    sm = np.array([((new[i + 1] - old[i + 1]) if i + 1 < M else size - len(ref)) + old[i] - new[i] for i in range(M)],
                  dtype=np.int64)
    out = bytearray()
    i = -1
    for p in range(size):
        while i + 1 < M and new[i + 1] <= p:
            i += 1
        if i < 0:
            out.append(ref[p])
            continue
        ind = p - new[i]
        out.append(ref[ind + old[i] - sm[i]] if ind > sm[i] else pool[nuc[i] + ind])
    return bytes(out), sm


@pytest.mark.parametrize("case", range(12))
def test_oracle_records_materialise_to_its_tips(case):
    rng = np.random.default_rng(case)
    n = int(rng.integers(2, 9))
    tree = kingman(n, rng).scaled(float(rng.uniform(0.1, 1.5)))
    seqs = [J.random_genome(1, int(rng.integers(1, 300)), seed=case * 7 + k).seqs[0].copy() for k in range(3)]
    if seqs[0].size >= 5:
        seqs[0][:5] = np.frombuffer(b"nNacg", dtype=np.uint8)
    ref = J.RefGenome(["a", "b", "c"], seqs)
    sub = J.sub_HKY85([0.1, 0.2, 0.3, 0.4], 2, 1, invariant=0.2, gamma_shape=0.7)
    o = HI.indels(ref, tree, sub, J.indels(float(rng.uniform(0, 0.4)), max_length=6),
                  J.indels(float(rng.uniform(0, 0.4)), a=1.3), float(rng.choice([0.3, 0.02])), 100 + case)
    for t in range(n):
        for c in range(3):
            seq, (old, new, nuc, sm, pool) = o.tips[t][c]
            assert np.all(np.diff(old.astype(np.int64)) > 0) and np.all(np.diff(new.astype(np.int64)) >= 0)
            got, sm2 = get_char_all(ref.seqs[c].tobytes(), old, new, nuc, pool, len(seq))
            assert got == seq and np.array_equal(sm, sm2), (t, c)


# ------------------------------------------------------------------------------- the law ---

def chisq_counts(obs, probs):
    """chi-square p-value of counts against probabilities, bins with expected count < 5 merged into their neighbour"""
    obs, exp = np.asarray(obs, float), np.asarray(probs, float) * np.sum(obs)
    o2, e2, ao, ae = [], [], 0.0, 0.0
    for o, e in zip(obs, exp):
        ao += o
        ae += e
        if ae >= 5:
            o2.append(ao); e2.append(ae); ao = ae = 0.0
    if ae > 0:
        o2[-1] += ao; e2[-1] += ae
    e2 = np.array(e2) * (np.sum(o2) / np.sum(e2))
    return stats.chisquare(o2, e2).pvalue


def star(n, t):
    return parse_newick("(" + ",".join("t%d:%r" % (i, t) for i in range(n)) + ");")


@pytest.fixture(scope="module")
def star_run():
    # 64 one-step branches from the root over 16 chromosomes of 2000 N: 2.05e6 positions, all at the same (L, p);
    # the inserted columns are born on the tip branches, so the tips' T/C/A/G are their birth states
    ref = J.RefGenome(["c%d" % i for i in range(16)], [b"N" * 2000] * 16)
    sub = J.sub_F81([0.1, 0.2, 0.3, 0.4])
    ins, dele = J.indels(0.3), J.indels(0.2, max_length=7, a=1.4)
    t, eps = 0.1, 1.0
    return ref, sub, ins, dele, t, HI.indels(ref, star(64, t), sub, ins, dele, eps, 77)


def test_law_events_per_step_binomial(star_run):
    ref, sub, ins, dele, t, o = star_run
    R = ins.rate + dele.rate
    p = -math.expm1(-R * t)
    assert np.all(o.steps[:, 3] == 2000) and len(o.steps) == 64 * 16
    cnt = o.steps[:, 4].astype(int)
    k = np.arange(cnt.max() + 1)
    probs = stats.binom.pmf(k, 2000, p)
    probs[-1] += stats.binom.sf(k[-1], 2000, p)
    assert chisq_counts(np.bincount(cnt, minlength=k.size), probs) > ALPHA


def test_law_kinds_and_lengths(star_run):
    ref, sub, ins, dele, t, o = star_run
    ev = o.events
    n_ins = int(np.sum(ev[:, 4] == 1))
    R = ins.rate + dele.rate
    assert stats.binomtest(n_ins, len(ev), ins.rate / R).pvalue > ALPHA
    for kind, m in ((1, ins), (0, dele)):
        lens = ev[ev[:, 4] == kind, 5].astype(int)
        assert lens.min() >= 1 and lens.max() <= m.max_length
        assert chisq_counts(np.bincount(lens, minlength=m.max_length + 1)[1:], m.probs()) > ALPHA


def test_law_rel_rates_lengths():
    ref = J.RefGenome(["c%d" % i for i in range(8)], [b"A" * 2000] * 8)
    ins, dele = J.indels(0.4, rel_rates=[3, 0, 1, 2, 0.5]), J.indels(0.0)
    o = HI.indels(ref, star(64, 0.1), J.sub_JC69(0), ins, dele, 1.0, 5)
    ev = o.events
    assert np.all(ev[:, 4] == 1) and len(ev) > 20000
    obs = np.bincount(ev[:, 5].astype(int), minlength=6)[1:]
    assert obs[1] == 0
    keep = ins.probs() > 0
    assert chisq_counts(obs[keep], ins.probs()[keep]) > ALPHA


def test_law_inserted_bases_follow_pi(star_run):
    ref, sub, ins, dele, t, o = star_run
    counts = np.zeros(4)
    for tip in o.tips:
        for seq, _ in tip:
            a = np.frombuffer(seq, np.uint8)
            counts += [np.sum(a == ord(b)) for b in "TCAG"]
    assert counts.sum() > 20000
    assert stats.chisquare(counts, sub.pi * counts.sum()).pvalue > ALPHA


def test_law_steps_per_branch():
    tree = parse_newick("((a:0.5,b:0.013)x:0.2,(c:1e-4,d:0)y:2.5);")
    ref = J.RefGenome(["c"], [b"ACGT" * 50])
    ins, dele, eps = J.indels(0.3), J.indels(0.1), 0.01
    o = HI.indels(ref, tree, J.sub_JC69(1), ins, dele, eps, 9)
    R = ins.rate + dele.rate
    got = np.bincount(o.steps[:, 1].astype(int), minlength=tree.n_nodes)
    for v in range(1, tree.n_nodes):
        assert got[v] == max(1, math.ceil(R * tree.branch_len[v] / eps)), v
