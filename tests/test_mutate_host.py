"""create_haplotypes without a GPU: substitution models, transition matrices, discrete Gamma rates, the Newick
parser, the coalescent sampler, argument checks, and the law of the oracle's per-site walk against exact
probabilities (pruning over internal states and rate categories with P from scipy)."""
import itertools
import math
import os
import re

import numpy as np
import pytest
from scipy import integrate, linalg, stats

import jackalope_b200 as J
from jackalope_b200 import _lib
from jackalope_b200.mutate import Tree, discrete_gamma_rates, kingman, parse_newick, transition_matrix
from oracle import harness as H
from oracle import harness_mutate as HM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PI = np.array([0.1, 0.2, 0.3, 0.4])
T, C_, A, G = 0, 1, 2, 3


def models():
    """(model, expected off-diagonal Q written out by hand, reversible?)"""
    pT, pC, pA, pG = PI
    pY, pR = pT + pC, pA + pG
    out = []
    out.append((J.sub_JC69(0.3), np.full((4, 4), 0.3), True))
    a, b = 2.0, 0.5
    out.append((J.sub_K80(a, b), np.array([[0, a, b, b], [a, 0, b, b], [b, b, 0, a], [b, b, a, 0]]), True))
    out.append((J.sub_F81(PI * 7), np.array([[0, pC, pA, pG], [pT, 0, pA, pG], [pT, pC, 0, pG], [pT, pC, pA, 0]]), True))
    out.append((J.sub_HKY85(PI, a, b), np.array([[0, a * pC, b * pA, b * pG], [a * pT, 0, b * pA, b * pG],
                                                 [b * pT, b * pC, 0, a * pG], [b * pT, b * pC, a * pA, 0]]), True))
    be, ka = 0.4, 1.5
    y, r = be * (1 + ka / pY), be * (1 + ka / pR)
    out.append((J.sub_F84(PI, be, ka), np.array([[0, y * pC, be * pA, be * pG], [y * pT, 0, be * pA, be * pG],
                                                  [be * pT, be * pC, 0, r * pG], [be * pT, be * pC, r * pA, 0]]), True))
    a1, a2 = 3.0, 1.2
    out.append((J.sub_TN93(PI, a1, a2, b), np.array([[0, a1 * pC, b * pA, b * pG], [a1 * pT, 0, b * pA, b * pG],
                                                      [b * pT, b * pC, 0, a2 * pG], [b * pT, b * pC, a2 * pA, 0]]), True))
    ra, rb, rc, rd, re_, rf = 1.0, 2.0, 3.0, 4.0, 5.0, 6.0      # TC, TA, TG, CA, CG, AG
    out.append((J.sub_GTR(PI, [ra, rb, rc, rd, re_, rf]),
                np.array([[0, ra * pC, rb * pA, rc * pG], [ra * pT, 0, rd * pA, re_ * pG],
                          [rb * pT, rd * pC, 0, rf * pG], [rc * pT, re_ * pC, rf * pA, 0]]), True))
    U = np.array([[9, 0.1, 0.7, 0.2], [0.3, 9, 0.05, 0.9], [0.6, 0.2, 9, 0.4], [0.1, 1.1, 0.3, 9]])
    out.append((J.sub_UNREST(U), U * (1 - np.eye(4)), False))
    return out


@pytest.mark.parametrize("i", range(8))
def test_q_builders_match_hand_written_matrices(i):
    m, off, reversible = models()[i]
    want = off * (1 - np.eye(4))
    np.fill_diagonal(want, -want.sum(axis=1))
    np.testing.assert_allclose(m.Q, want, rtol=1e-14, atol=0)
    np.testing.assert_allclose(m.Q.sum(axis=1), 0, atol=1e-14)
    if reversible:
        np.testing.assert_allclose(m.pi @ m.Q, 0, atol=1e-14)
        pi = PI if m.name not in ("JC69", "K80") else np.full(4, 0.25)
        np.testing.assert_allclose(m.pi, pi, atol=1e-12)
        # detailed balance
        np.testing.assert_allclose(m.pi[:, None] * m.Q, (m.pi[:, None] * m.Q).T, atol=1e-14)
    np.testing.assert_allclose(m.pi @ m.Q, 0, atol=1e-12)
    assert abs(m.pi.sum() - 1) < 1e-12


@pytest.mark.parametrize("i", range(8))
def test_transition_matrix_matches_scipy(i):
    m = models()[i][0]
    for t in (0, 1e-8, 1e-3, 0.1, 1, 10, 100):
        P = transition_matrix(m.Q, t)
        np.testing.assert_allclose(P, linalg.expm(m.Q * t), rtol=0, atol=1e-12, err_msg="t=%g" % t)
        if t == 0:
            assert np.array_equal(P, np.eye(4))
        np.testing.assert_allclose(P.sum(axis=1), 1, atol=1e-13)


def test_transition_matrix_jc69_closed_form_and_diagonal_ignored():
    lam = 0.7
    m = J.sub_JC69(lam)
    for t in (1e-6, 0.01, 0.5, 3, 40):
        e = math.exp(-4 * lam * t)
        want = np.full((4, 4), 0.25 - 0.25 * e)
        np.fill_diagonal(want, 0.25 + 0.75 * e)
        np.testing.assert_allclose(transition_matrix(m.Q, t), want, rtol=0, atol=1e-13)
    q = m.Q.copy()
    np.fill_diagonal(q, 123.0)                 # the library takes the diagonal as minus the row sum
    np.testing.assert_array_equal(transition_matrix(q, 0.3), transition_matrix(m.Q, 0.3))
    P = np.zeros(16)
    assert _lib.lib().jlp_transition_matrix(m.Q.reshape(16).copy().ctypes.data_as(_lib.f64p), -1.0,
                                            P.ctypes.data_as(_lib.f64p)) == _lib.JLP_ERR_ARG


@pytest.mark.parametrize("shape,k", [(0.5, 4), (1.0, 5), (2.3, 3), (0.2, 10), (7.0, 2)])
def test_discrete_gamma_rates_are_bin_means(shape, k):
    r = discrete_gamma_rates(shape, k)
    edges = stats.gamma.ppf(np.arange(k + 1) / k, a=shape, scale=1 / shape)
    for j in range(k):
        num = integrate.quad(lambda x: x * stats.gamma.pdf(x, a=shape, scale=1 / shape), edges[j], edges[j + 1],
                             limit=200)[0]
        assert abs(r[j] - num * k) < 1e-7 * max(1, r[j]), (j, r[j], num * k)
    assert abs(r.mean() - 1) < 1e-12
    assert np.all(np.diff(r) > 0)
    np.testing.assert_allclose(discrete_gamma_rates(0.5, 4), [0.0334, 0.2519, 0.8203, 2.8944], atol=1e-4)   # Yang (1994)
    m = J.sub_JC69(1, gamma_shape=shape, gamma_k=k)
    np.testing.assert_array_equal(m.rates, r)
    assert np.array_equal(J.sub_JC69(1).rates, [1.0])


# --------------------------------------------------------------------------- Newick ---

def test_newick_parser_accepts_the_grammar():
    t = parse_newick(" ( (A:0.1 , B:2e-1)x:5E-2,\n(C:1e-2,D:0,E:3)  :0.4 ) root:99 ;\n")
    assert t.tip_names == ["A", "B", "C", "D", "E"]
    assert list(t.parent) == [-1, 0, 1, 1, 0, 4, 4, 4]
    np.testing.assert_array_equal(t.branch_len, [0, 0.05, 0.1, 0.2, 0.4, 0.01, 0, 3])
    assert list(t.tip_node) == [2, 3, 5, 6, 7]
    assert all(t.parent[i] < i for i in range(1, t.n_nodes))
    # round trip through the writer
    t2 = parse_newick(t.newick())
    assert t2.tip_names == t.tip_names and np.array_equal(t2.parent, t.parent)
    np.testing.assert_array_equal(t2.branch_len, t.branch_len)
    # quoted labels, comments, a root without a length, a deep caterpillar
    t3 = parse_newick("('a b':1,[comment]'it''s':2);")
    assert t3.tip_names == ["a b", "it's"]
    cat = "t0:1"
    for i in range(1, 3000):
        cat = "(%s,t%d:1):1" % (cat, i)
    t4 = parse_newick(cat + ";")
    assert len(t4.tip_names) == 3000 and all(t4.parent[i] < i for i in range(1, t4.n_nodes))


@pytest.mark.parametrize("bad,what", [
    ("(A:1,B);", "no branch length"), ("(A:1,B:-1);", "negative"), ("(A:1,A:2);", "duplicate"),
    ("(A:1,B:1)", "end with"), ("(A:1,B:1);(C:1);", "one tree"), ("(A:1,:1);", "label"), ("(A:1,B:x);", "not a number"),
    ("(A:1,B:1;", "unexpected"), ("A:1;", "start with"), ("", "start with"), ("(A:1,B:inf);", "not finite"),
    ("((A:1,B:1),C:1);", "no branch length"), ("(A:1,B:1)):1;", "end with"), ("(A:1,()B:1);", "label"),
    ("(A:1,B:1)[open;", "comment"), ("('A:1,B:1);", "quoted"),
])
def test_newick_parser_rejects_malformed_input(bad, what):
    with pytest.raises(J.JackalopeError, match=what):
        parse_newick(bad)


def test_haps_phylo_reads_a_file(tmp_path):
    fn = tmp_path / "tree.nwk"
    fn.write_text("((h1:0.1,h2:0.1):0.2,h3:0.3);\n")
    info = J.haps_phylo(fn=str(fn))
    assert info.tree(None, 0).tip_names == ["h1", "h2", "h3"]
    with pytest.raises(J.JackalopeError, match="haps_phylo"):
        J.haps_phylo()
    with pytest.raises(J.JackalopeError, match="haps_phylo"):
        J.haps_phylo("(a:1,b:1);", fn=str(fn))
    with pytest.raises(J.JackalopeError, match="fn"):
        J.haps_phylo(fn=str(tmp_path / "missing.nwk"))


# ------------------------------------------------------------------------ coalescent ---

@pytest.mark.parametrize("n", [2, 5, 12])
def test_kingman_sampler_moments(n):
    tm, tot = [], []
    for seed in range(3000):
        t = kingman(n, np.random.default_rng(seed))
        assert len(t.tip_names) == n and t.n_nodes == 2 * n - 1
        assert t.tip_names == ["hap%d" % i for i in range(n)]
        assert all(t.parent[i] < i for i in range(1, t.n_nodes))
        depth = np.zeros(t.n_nodes)
        for v in range(1, t.n_nodes):
            depth[v] = depth[t.parent[v]] + t.branch_len[v]
        np.testing.assert_allclose(depth[t.tip_node], depth[t.tip_node][0], rtol=1e-12)    # ultrametric
        tm.append(depth[t.tip_node[0]])
        tot.append(t.branch_len[1:].sum())
    tm, tot = np.array(tm), np.array(tot)
    assert abs(tm.mean() - 2 * (1 - 1 / n)) < 5 * tm.std() / math.sqrt(tm.size)
    want_tot = 2 * sum(1 / i for i in range(1, n))
    assert abs(tot.mean() - want_tot) < 5 * tot.std() / math.sqrt(tot.size)


def test_haps_theta_scale():
    m = J.sub_TN93(PI, 2, 1, 0.5, invariant=0.3, gamma_shape=0.8)
    info = J.haps_theta(0.01, 6)
    mu = -np.sum(m.pi * np.diag(m.Q))
    assert abs(info.scale(m) - 0.01 / (2 * mu * 0.7)) < 1e-15
    t = info.tree(m, 11)
    base = kingman(6, np.random.default_rng(11))
    np.testing.assert_allclose(t.branch_len, base.branch_len * info.scale(m), rtol=1e-15)
    assert t.tip_names == ["hap%d" % i for i in range(6)]
    # UNREST: mu_bar from the left null vector
    u = models()[7][0]
    assert abs(u.mu_bar() + np.sum(u.pi * np.diag(u.Q))) < 1e-15 and np.allclose(u.pi @ u.Q, 0, atol=1e-12)


# ------------------------------------------------------------------- argument checks ---

def test_argument_validation():
    g = J.random_genome(1, 100, seed=1)
    info, m = J.haps_theta(0.01, 3), J.sub_JC69(1)
    with pytest.raises(J.JackalopeError, match="`create_haplotypes` .* argument `reference`"):
        J.create_haplotypes("ACGT", info, m)
    with pytest.raises(J.JackalopeError, match="argument `haps_info`"):
        J.create_haplotypes(g, "(a:1,b:1);", m)
    with pytest.raises(J.JackalopeError, match="argument `sub`"):
        J.create_haplotypes(g, info, np.eye(4))
    with pytest.raises(J.JackalopeError, match="not built yet"):
        J.create_haplotypes(g, info, m, ins=0.1)
    with pytest.raises(J.JackalopeError, match="not built yet"):
        J.create_haplotypes(g, info, m, del_=0.1)
    for eps in (-0.1, 1, float("nan")):
        with pytest.raises(J.JackalopeError, match="argument `epsilon`"):
            J.create_haplotypes(g, info, m, epsilon=eps)
    with pytest.raises(J.JackalopeError, match="argument `n_threads`"):
        J.create_haplotypes(g, info, m, n_threads=0)
    with pytest.raises(J.JackalopeError, match="argument `show_progress`"):
        J.create_haplotypes(g, info, m, show_progress="yes")
    for bad in (dict(invariant=1), dict(invariant=-0.1), dict(gamma_shape=0), dict(gamma_shape=1, gamma_k=1),
                dict(gamma_shape=1, gamma_k=256), dict(gamma_k=2.5)):
        with pytest.raises(J.JackalopeError, match="`sub_JC69`"):
            J.sub_JC69(1, **bad)
    with pytest.raises(J.JackalopeError, match="argument `lambda`"):
        J.sub_JC69(-1)
    with pytest.raises(J.JackalopeError, match="argument `pi_tcag`"):
        J.sub_F81([0.5, 0.5, 0.5])
    with pytest.raises(J.JackalopeError, match="argument `pi_tcag`"):
        J.sub_HKY85([0, 0, 0, 0], 1, 1)
    with pytest.raises(J.JackalopeError, match="argument `abcdef`"):
        J.sub_GTR(PI, [1, 2, 3])
    with pytest.raises(J.JackalopeError, match="argument `Q`"):
        J.sub_UNREST(-np.ones((4, 4)))
    with pytest.raises(J.JackalopeError, match="argument `pi_tcag`"):
        J.sub_F84([0, 0, 0.5, 0.5], 1, 1)
    with pytest.raises(J.JackalopeError, match="argument `theta`"):
        J.haps_theta(0, 4)
    with pytest.raises(J.JackalopeError, match="argument `n_haps`"):
        J.haps_theta(0.1, 1)


def test_mutation_structs_match_the_header():
    hdr = open(os.path.join(ROOT, "include", "jlp_b200.h")).read()

    def fields(struct):
        body = hdr[hdr.index("typedef struct " + struct):hdr.index("} " + struct + ";")]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        out = []
        for decl in body.split("{", 1)[1].split(";"):
            names = re.findall(r"([A-Za-z_][A-Za-z_0-9]*)\s*(?:\[[0-9]+\])?\s*(?:,|$)", decl.strip())
            out += [n for n in names if n]
        return out

    assert fields("jlp_mutation_params") == [f[0] for f in _lib.MutationParams._fields_]
    assert fields("jlp_mutation_stats") == [f[0] for f in _lib.MutationStats._fields_]


# --------------------------------------------------------------------- the law, on the oracle ---

def exact_pattern_probs(tree: Tree, m, root_base):
    """P(tip states = pattern | root = root_base) over all 4^n_tips patterns (pattern index: tip 0 most significant),
    summed over rate categories (and the invariant class) and internal states, with P from scipy."""
    nt = len(tree.tip_names)
    kids = tree.children()
    tip_idx = {int(v): i for i, v in enumerate(tree.tip_node)}
    out = np.zeros(4 ** nt)
    K = m.rates.size
    for k in range(K):
        Ps = [None] + [linalg.expm(m.Q * m.rates[k] * tree.branch_len[v]) for v in range(1, tree.n_nodes)]

        # partial likelihood vector over tip patterns: L[v][s] = distribution of the tips below v given state s
        def below(v):
            if v in tip_idx:
                vec = np.zeros((4, 4))
                np.fill_diagonal(vec, 1.0)
                return vec, [tip_idx[v]]
            acc, tips = None, []
            for c in kids[v]:
                sub, ct = below(c)
                child = Ps[c] @ sub                       # [parent state][patterns of c's tips]
                acc = child if acc is None else (acc[:, :, None] * child[:, None, :]).reshape(4, -1)
                tips += ct
            return acc, tips

        dist, order = below(0)
        d = dist[root_base].reshape([4] * nt)
        d = np.transpose(d, np.argsort(order))           # axes in tip order
        out += (1 - m.invariant) / K * d.reshape(-1)
    out[sum(root_base * 4 ** (nt - 1 - i) for i in range(nt))] += m.invariant
    return out


def tip_patterns(genome, tree, recs):
    """per site: reference code and the pattern index of the tips' states"""
    lut = np.full(256, 255, dtype=np.uint8)
    lut[np.frombuffer(b"TCAG", dtype=np.uint8)] = np.arange(4, dtype=np.uint8)
    ref = lut[genome.seqs[0]]
    nt = len(tree.tip_names)
    pat = np.zeros(ref.size, dtype=np.int64)
    for t in range(nt):
        s = ref.astype(np.int64).copy()
        pos, nuc = recs[t][0]
        s[pos.astype(np.int64)] = lut[np.frombuffer(nuc, dtype=np.uint8)]
        assert np.all(s[pos.astype(np.int64)] != ref[pos.astype(np.int64)])
        pat = pat * 4 + s
    return ref, pat


def chi2_fit(ref, pat, tree, m):
    nt = len(tree.tip_names)
    stat, df = 0.0, 0
    for a in range(4):
        obs = np.bincount(pat[ref == a], minlength=4 ** nt).astype(np.float64)
        exp = exact_pattern_probs(tree, m, a) * obs.sum()
        assert abs(exp.sum() - obs.sum()) < 1e-6 * obs.sum()
        big = exp >= 5
        o = np.concatenate((obs[big], [obs[~big].sum()]))
        e = np.concatenate((exp[big], [exp[~big].sum()]))
        keep = e > 0
        stat += np.sum((o[keep] - e[keep]) ** 2 / e[keep])
        df += int(keep.sum()) - 1
    return stats.chi2.sf(stat, df)


def test_law_five_tips_tn93_gamma_invariant():
    tree = parse_newick("((A:0.1,B:0.25)x:0.05,(C:0.02,D:0,E:0.6):0.4)r;")
    m = J.sub_TN93(PI, 2.0, 1.0, 0.5, invariant=0.2, gamma_shape=0.7, gamma_k=4)
    g = J.random_genome(1, 4_000_000, seed=21)
    recs = HM.mutate(g, tree, m, seed=1234)
    ref, pat = tip_patterns(g, tree, recs)
    assert chi2_fit(ref, pat, tree, m) > 0.001


@pytest.mark.parametrize("i", range(8))
def test_law_three_tips_every_model(i):
    m0 = models()[i][0]
    m = J.mutate.SubModel(m0.name, m0.Q, 0.1 if i % 2 else 0.0, 1.3 if i % 3 == 0 else None, 3)
    tree = parse_newick("(A:0.3,(B:0.1,C:0.5):0.2);")
    g = J.random_genome(1, 600_000, seed=30 + i, pi_tcag=(0.4, 0.3, 0.2, 0.1))
    recs = HM.mutate(g, tree, m, seed=77 + i)
    ref, pat = tip_patterns(g, tree, recs)
    assert chi2_fit(ref, pat, tree, m) > 0.001


def test_oracle_walk_only_touches_tcag_and_is_seeded():
    tree = parse_newick("(A:2,B:2);")
    m = J.sub_JC69(1.0)
    seq = np.frombuffer(b"NNNNacgtTCAGRYKM" * 500, dtype=np.uint8)
    g = J.RefGenome(["c0"], [seq])
    r1 = HM.mutate(g, tree, m, seed=5)
    for t in range(2):
        pos, nuc = r1[t][0]
        assert pos.size > 0 and all(chr(seq[p]) in "TCAG" for p in pos)
        assert all(chr(b) in "TCAG" and b != seq[p] for p, b in zip(pos, nuc))
    r2 = HM.mutate(g, tree, m, seed=5)
    r3 = HM.mutate(g, tree, m, seed=6)
    assert all(np.array_equal(r1[t][0][0], r2[t][0][0]) and r1[t][0][1] == r2[t][0][1] for t in range(2))
    assert not np.array_equal(r1[0][0][0], r3[0][0][0])
    # the draws: X(c, b, v) = high word of the MUT block, low word of the MSLOW block
    x = HM.mut_draw(9, 2, 13, 5)
    w = H.philox([13 >> 2, 0, 2, 7 | (5 << 8)], [9, 0])
    v = H.philox([13, 0, 2, 8 | (5 << 8)], [9, 0])
    assert x == (int(w[13 & 3]) << 32) | int(v[0])


def test_itertools_pattern_index_convention():
    # tip 0 is the most significant digit of a pattern index (tip_patterns and exact_pattern_probs agree)
    tree = parse_newick("(A:0.5,B:0.01);")
    m = J.sub_JC69(1.0)
    p = exact_pattern_probs(tree, m, 0).reshape(4, 4)
    PA, PB = linalg.expm(m.Q * 0.5)[0], linalg.expm(m.Q * 0.01)[0]
    for a, b in itertools.product(range(4), range(4)):
        assert abs(p[a, b] - PA[a] * PB[b]) < 1e-14
