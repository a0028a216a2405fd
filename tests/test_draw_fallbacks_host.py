"""Inputs that reach the kernels' exact-draw fallbacks on purpose, with both outcomes, proved on the CPU.

Every random decision is defined on a full 64-bit draw; the kernels decide on its high bits and fetch the rest only
when those leave the answer open (DESIGN.md section 2).  The rarest of these branches are almost never reached by
random inputs, so the cases here are constructed:

  * create_haplotypes, k_mutate's transition decision (`decide()`): branch lengths bisected on the 64-bit comparison
    of threshold T_j(t) and draw X(c, b, v) until the two sit in the same high word, one branch length on each side;
    some of them with T_j == X exactly.  Star trees (tips) and chains root -> x -> y -> two tips of length 0 (ties
    at y, whose row is the state the walk computed at x); with and without indels (k_mutate<*, true>).
  * k_mutate's category decision: `invariant` set to X / 2^64 of a site, one step below and one above
    (cat_thr[0]), and bisected so that cat_thr[1] ties.
  * k_ins_walk: the branch lengths below the birth branch of inserted columns bisected against their IMUT draws.
  * k_reads: the oracle counts the draws whose high bits leave the alias slot, the N quality and the substitution
    index open, and those where the exact answer differs (OrcJob.fallback); pinned seeds keep the counts up.

Each case carries its proof: the draws and thresholds are recomputed here and the tie count and outcomes asserted,
so that a change of draw layout or threshold rule fails this file instead of leaving the GPU tests (in
test_gpu_draw_fallbacks.py, which builds the same cases) testing nothing."""
import functools
import math
import struct

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200.mutate import Tree, parse_newick, transition_matrix
from oracle import harness as H
from oracle import harness_indels as HI
from oracle import harness_mutate as HM
from oracle.compare import oracle_run

M64 = 2 ** 64 - 1
SEED = 0x5EED_F411_BAC5


# ------------------------------------------------------------------------------------------------ draws ---

def philox(c0, c1, c2, c3, seed, rounds=10):
    """Philox4x32-R of arrays of counters (jlp_draws.h): four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c0, c1, c2, c3 = (x.copy() for x in c)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(rounds):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & np.uint64(0xFFFFFFFF),
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & np.uint64(0xFFFFFFFF))
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c0, c1, c2, c3


def mut_draws(seed, chrom, sites, node, hi_plane=7, lo_plane=8):
    """X(chrom, site, node) of create_haplotypes for an array of sites < 2^32 (planes MUT / MSLOW; IMUT / IMSLOW
    with the column id in place of the site)."""
    b = np.asarray(sites, dtype=np.uint64)
    w = philox(b >> np.uint64(2), 0, chrom, hi_plane | (node << 8), seed)
    k = (b & np.uint64(3)).astype(np.int64)
    hi = np.choose(k, w)
    lo = philox(b, 0, chrom, lo_plane | (node << 8), seed)[0]
    return (hi << np.uint64(32)) | lo


def mut_draw(seed, chrom, site, node):
    return int(mut_draws(seed, chrom, [site], node)[0])


def imut_draw(seed, chrom, col, node):
    return int(mut_draws(seed, chrom, [col], node, 11, 12)[0])


def icol_draws(seed, chrom, col):
    """plane ICOL: (category draw, birth-state draw) of inserted column `col`"""
    w = [int(x[0]) for x in philox([col], 0, chrom, 10, seed)]
    return (w[1] << 32) | w[0], (w[3] << 32) | w[2]


# ------------------------------------------------------------------------------------------- thresholds ---

def prob_threshold(c):
    """jlp_host.cpp prob_threshold: floor(c 2^64), 0 for c <= 0, 2^64 - 1 for c >= 1"""
    if not c > 0:
        return 0
    if c >= 1:
        return M64
    return int(math.ldexp(c, 64))


def row_thresholds(row):
    """jlp_host.cpp row_thresholds: clipped at 0, summed in order, c += p[j] / sum"""
    p = [float(x) if x > 0 else 0.0 for x in row]
    s = 0.0
    for x in p:
        s += x
    out, c = [], 0.0
    for j in range(3):
        c += p[j] / s
        out.append(prob_threshold(c))
    return out


def thresholds(sub, t, cat, row):
    return row_thresholds(transition_matrix(sub.Q, sub.rates[cat] * t)[row])


def cat_thresholds(invariant, K):
    return [prob_threshold(invariant)] + [prob_threshold(invariant + j * (1 - invariant) / K) for j in range(1, K)]


def state(X, thr):
    return sum(X >= t for t in thr)


def representable(X):
    return 0 < X < 2 ** 64 and int(float(X)) == X


def _bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def _dbl(i):
    return struct.unpack("<d", struct.pack("<q", i))[0]


def bisect_double(f, lo, hi):
    """Adjacent doubles a < b in [lo, hi] (both >= 0) with f(a) == f(lo) != f(b)."""
    flo = f(lo)
    assert f(hi) != flo
    a, b = _bits(lo), _bits(hi)
    while b - a > 1:
        m = (a + b) // 2
        if f(_dbl(m)) == flo:
            a = m
        else:
            b = m
    return _dbl(a), _dbl(b)


# ------------------------------------------------------------------------------------- transition ties ---

class Tie:
    """One constructed tie: the decision at `node` for site (or inserted column) `site` compares draw X with
    threshold j of `row`; `moves` is whether the state moves past j (T_j <= X)."""

    def __init__(self, node, site, row, j, X, T, cat=0):
        self.node, self.site, self.row, self.j, self.X, self.T, self.cat = node, site, row, j, X, T, cat

    @property
    def moves(self):
        return self.T <= self.X

    @property
    def exact(self):
        return self.T == self.X


def tune_branch(sub, row, X, rank, t_max, cat=0):
    """A branch length at which one threshold of `row` ties X's high word: (t, j, T_j(t)) or None.  rank picks the
    side: even -> T_j <= X (moves past j), odd -> T_j > X; 'exact' -> T_j == X or None."""
    for j in range(3):
        T = lambda t: thresholds(sub, t, cat, row)[j]
        f = lambda t: T(t) <= X
        if f(0.0) == f(t_max):
            continue
        a, b = bisect_double(f, 0.0, t_max)
        Ta, Tb = T(a), T(b)
        if rank == "exact":
            hit = [(t, Tt) for t, Tt in ((a, Ta), (b, Tb)) if Tt == X]
            return (hit[0][0], j, hit[0][1]) if hit else None
        t, Tt = (a, Ta) if f(a) == (rank % 2 == 0) else (b, Tb)
        return (t, j, Tt) if Tt >> 32 == X >> 32 else None
    return None


def star_and_chains(n_star, n_chains):
    """Root -> n_star tips, then n_chains chains root -> x -> y -> (a, b), node ids in preorder (the numbering of
    parse_newick).  Returns (parent, tip nodes, chain (x, y) pairs)."""
    parent, tips, chains = [-1], [], []
    for _ in range(n_star):
        tips.append(len(parent))
        parent.append(0)
    for _ in range(n_chains):
        x = len(parent)
        parent += [0, x, x + 1, x + 1]
        tips += [x + 2, x + 3]
        chains.append((x, x + 1))
    return parent, tips, chains


def make_tree(parent, branch_len, tips):
    """The Tree as create_haplotypes will see it: written with repr'd lengths and parsed back unchanged."""
    tree = Tree(parent, branch_len, tips, ["t%d" % v for v in tips])
    text = tree.newick()
    back = parse_newick(text)
    assert np.array_equal(back.parent, tree.parent) and np.array_equal(back.tip_node, tree.tip_node)
    assert np.array_equal(back.branch_len, tree.branch_len) and back.tip_names == tree.tip_names
    return text, back


class Case:
    """A create_haplotypes input with constructed ties: genome, Newick text, model, indel models, ties."""

    def __init__(self, genome, newick, sub, seed, ties, ins=None, dele=None, eps=0.03):
        self.genome, self.newick, self.sub, self.seed, self.ties = genome, newick, sub, seed, ties
        self.ins, self.dele, self.eps = ins, dele, eps
        self.tree = parse_newick(newick)

    def counts(self):
        return dict(ties=len(self.ties), moves=sum(t.moves for t in self.ties),
                    stays=sum(not t.moves for t in self.ties), exact=sum(t.exact for t in self.ties))


def transition_case(n_star, n_chains, seed=SEED, length=4096, indel_rate=0.0, exact_every=8):
    """Ties of k_mutate's transition decision at every star tip and at the y of every chain.  With indel_rate > 0
    (ins = del_ = indels(rate)) a tie whose site does not survive to its tip in the oracle is replaced by another
    site, and the oracle is run again, until every tie's site survives."""
    sub = J.sub_JC69(1.0)
    g = J.random_genome(1, length, seed=seed & 0xFFFF)
    ref = g.seqs[0]
    code = {ord("T"): 0, ord("C"): 1, ord("A"): 2, ord("G"): 3}
    parent, tips, chains = star_and_chains(n_star, n_chains)
    n = len(parent)
    bl = np.zeros(n)
    for x, _ in chains:
        bl[x] = 0.3
    ties = {}
    sites = np.arange(16, length, dtype=np.uint64)        # clear of the leading-record edge at position 0

    def plan(v, rank, skip):
        x = parent[v]
        X_all = None
        tries = [rank] if not (exact_every and rank % exact_every == 0) else ["exact", rank]
        for r in tries:
            if r == "exact":
                X_all = mut_draws(seed, 0, sites, v)
                cand = [int(s) for s, X in zip(sites, X_all) if representable(int(X))][:3]
            else:
                cand = [int(s) for s in sites[:64]]
            for b in cand:
                if b in skip:
                    continue
                a = code[int(ref[b])]
                if x != 0:                     # the row is the state the walk computed at x
                    a = state(mut_draw(seed, 0, b, x), thresholds(sub, bl[x], 0, a))
                X = mut_draw(seed, 0, b, v) if X_all is None else int(X_all[b - 16])
                got = tune_branch(sub, a, X, r, 40.0)
                if got:
                    t, j, T = got
                    return t, Tie(v, b, a, j, X, T)
        raise AssertionError("no tie for node %d" % v)

    nodes = list(tips[:n_star]) + [y for _, y in chains]
    skip = {v: set() for v in nodes}
    for rank, v in enumerate(nodes):
        bl[v], ties[v] = plan(v, rank, skip[v])
    ins = dele = None
    if indel_rate:
        ins, dele = J.indels(indel_rate, max_length=4), J.indels(indel_rate, max_length=4)
        for _ in range(6):
            _, tree = make_tree(parent, bl, tips)
            o = HI.indels(g, tree, sub, ins, dele, 0.03, seed)
            dead = [v for v in nodes if not all(site_alive(o, tips.index(t), ties[v].site)
                                                for t in tips_below(parent, tips, v))]
            if not dead:
                break
            for v in dead:
                skip[v].add(ties[v].site)
                bl[v], ties[v] = plan(v, nodes.index(v), skip[v])
        else:
            raise AssertionError("tied sites keep dying")
    text, _ = make_tree(parent, bl, tips)
    return Case(g, text, sub, seed, [ties[v] for v in nodes], ins, dele)


def tips_below(parent, tips, v):
    return [t for t in tips if t == v or parent[t] == v or (parent[t] >= 0 and parent[parent[t]] == v)]


def site_alive(o, tip, b, chrom=0):
    """Reference site b is alive at the tip: no deletion record of the oracle covers it."""
    old, _, _, sm, _ = o.tips[tip][chrom][1]
    d = sm < 0
    return not np.any((old[d] <= b) & (b < old[d] - sm[d]))


@functools.lru_cache(maxsize=None)
def tie_case(name):
    """The constructed cases, by name (shared with test_gpu_draw_fallbacks.py)."""
    if name == "smem":
        return transition_case(192, 16)
    if name == "global":
        return transition_case(1500, 16)
    if name == "indels":
        return transition_case(160, 8, indel_rate=0.002)
    if name == "ins_walk":
        return ins_walk_case()
    if name.startswith("cat"):
        return category_case(name)
    raise KeyError(name)


# -------------------------------------------------------------------------------------- category ties ---

CAT_TIPS = 12


def category_site(seed, g, pred, start=16):
    """(b, X) of the sites b >= start whose category draw X satisfies pred(X), in order."""
    X0 = mut_draws(seed, 0, np.arange(start, g.seqs[0].size, dtype=np.uint64), 0)
    for i, X in enumerate(X0):
        if pred(int(X)):
            yield start + i, int(X)


def category_case(name):
    """cat0_{exact, below, above}: invariant = X / 2^64 of a site's category draw, and one double below / above it
    (the site evolves, evolves, does not); cat1_{lo, hi}: gamma_k = 4, invariant bisected so that cat_thr[1] ties
    the draw's high word on either side (category 1 or 0 of the variable sites)."""
    seed = SEED + 1
    g = J.random_genome(1, 4096, seed=7)
    ref = g.seqs[0]
    code = {ord("T"): 0, ord("C"): 1, ord("A"): 2, ord("G"): 3}
    tips = list(range(1, CAT_TIPS + 1))
    bl = np.array([0.0] + [0.7 + 0.1 * k for k in range(CAT_TIPS)])
    text, _ = make_tree([-1] + [0] * CAT_TIPS, bl, tips)
    kind, side = name.split("_")
    if kind == "cat0":
        sub0 = J.sub_JC69(1.0)

        def visible(b):        # the evolving site differs from the reference at some tip
            a = code[int(ref[b])]
            return any(state(mut_draw(seed, 0, b, v), thresholds(sub0, bl[v], 0, a)) != a for v in tips)
        b, X = next((b, X) for b, X in category_site(seed, g, lambda X: representable(X) and X < 2 ** 63)
                    if visible(b))
        inv = float(X) / 2 ** 64
        inv = {"exact": inv, "below": math.nextafter(inv, 0), "above": math.nextafter(inv, 1)}[side]
        sub = J.sub_JC69(1.0, invariant=inv)
        thr = cat_thresholds(inv, 1)
        tie = Tie(0, b, None, 0, X, thr[0])
    else:
        K = 4
        base = J.sub_JC69(1.0, gamma_shape=0.3, gamma_k=K)

        def visible(b):        # category 1 and category 0 give different states at some tip
            a = code[int(ref[b])]
            return any(state(mut_draw(seed, 0, b, v), thresholds(base, bl[v], 0, a)) !=
                       state(mut_draw(seed, 0, b, v), thresholds(base, bl[v], 1, a)) for v in tips)
        for b, X in category_site(seed, g, lambda X: X > 2 ** 62):
            if not visible(b):
                continue
            f = lambda inv: cat_thresholds(inv, K)[1] <= X
            lo, hi = bisect_double(f, 0.0, 0.999)
            inv = lo if side == "lo" else hi
            thr = cat_thresholds(inv, K)
            if thr[1] >> 32 == X >> 32 and X >= thr[0] and (K < 3 or X < thr[2]):
                break
        sub = J.sub_JC69(1.0, invariant=inv, gamma_shape=0.3, gamma_k=K)
        tie = Tie(0, b, None, 1, X, thr[1])
    return Case(g, text, sub, seed, [tie])


# --------------------------------------------------------------------------------------- k_ins_walk ties ---

def columns(tree, events, length, node, chrom=0):
    """The column list at `node` (reference sites b >= 0, inserted columns -(id + 1)), replayed from the oracle's
    events as orc_indels applies them; ids in the order the events were drawn."""
    ev = events[events[:, 0] == chrom]
    first_id, nid = {}, 0
    for k, e in enumerate(ev):
        if e[4] == 1:
            first_id[k] = nid
            nid += int(e[5])
    path, v = [], node
    while v > 0:
        path.append(v)
        v = int(tree.parent[v])
    cols = list(range(length))
    for v in reversed(path):
        rows = [k for k in range(len(ev)) if ev[k, 1] == v]
        for s in sorted({int(ev[k, 2]) for k in rows}):
            step = [k for k in rows if ev[k, 2] == s]
            dead = set()
            for k in step:
                if ev[k, 4] == 0:
                    dead.update(range(int(ev[k, 3]), int(ev[k, 3]) + int(ev[k, 5])))
            ins = {int(ev[k, 3]): k for k in step if ev[k, 4] == 1}
            nx = []
            for i, c in enumerate(cols):
                if i not in dead:
                    nx.append(c)
                if i in ins:
                    k = ins[i]
                    nx += [-(first_id[k] + q) - 1 for q in range(int(ev[k, 5]))]
            cols = nx
    return cols


INS_KIDS = 48


def ins_walk_case():
    """((k1, ..., k48):x, d): insertions on the long branch x, and every k_i's length bisected so that the IMUT
    draw of one inserted column born on x ties a threshold of the row of its birth state at k_i."""
    seed = SEED + 2
    sub = J.sub_JC69(4.0)
    length = 2048
    g = J.random_genome(1, length, seed=11)
    ins, dele = J.indels(0.08, max_length=3), J.indels(0.004, max_length=3)
    parent = [-1, 0] + [1] * INS_KIDS + [0]
    kids = list(range(2, 2 + INS_KIDS))
    tips = kids + [2 + INS_KIDS]
    bl = np.array([0.0, 1.0] + [0.05] * INS_KIDS + [0.2])
    pi_thr = row_thresholds(sub.pi)
    used = {k: set() for k in kids}
    ties = {}
    for _ in range(6):
        _, tree = make_tree(parent, bl, tips)
        o = HI.indels(g, tree, sub, ins, dele, 0.03, seed)
        born = [-c - 1 for c in columns(tree, o.events, length, 1) if c < 0]
        born_on_x = set(born) - {-c - 1 for c in columns(tree, o.events, length, 0) if c < 0}
        stale = [k for k in kids if k not in ties or -ties[k].site - 1 not in columns(tree, o.events, length, k)]
        if not stale:
            break
        for r, k in enumerate(kids):
            if k not in stale:
                continue
            if k in ties:
                used[k].add(ties[k].site)
            cand = sorted(i for i in born_on_x if i not in used[k])
            want = ["exact", r] if r % 4 == 0 else [r]
            done = False
            for rank in want:
                pool = [i for i in cand if representable(imut_draw(seed, 0, i, k))] if rank == "exact" else cand
                for i in pool[:8]:
                    s = state(icol_draws(seed, 0, i)[1], pi_thr)
                    X = imut_draw(seed, 0, i, k)
                    got = tune_branch(sub, s, X, rank, 10.0)
                    if got:
                        bl[k], ties[k] = got[0], Tie(k, -i - 1, s, got[1], X, got[2])
                        done = True
                        break
                if done:
                    break
            assert done, k
    else:
        raise AssertionError("no fixed point of the inserted columns' ties")
    text, _ = make_tree(parent, bl, tips)
    return Case(g, text, sub, seed, [ties[k] for k in kids], ins, dele)


# ------------------------------------------------------------------------------------------ the proofs ---

def prove_transition_ties(case):
    """Recompute every tie of a case from its final tree: draw, threshold, same high word, outcome."""
    tree, sub, seed = case.tree, case.sub, case.seed
    for t in case.ties:
        if t.site >= 0:
            assert mut_draw(seed, 0, t.site, t.node) == t.X
        else:
            assert imut_draw(seed, 0, -t.site - 1, t.node) == t.X
        T = thresholds(sub, tree.branch_len[t.node], t.cat, t.row)
        assert T[t.j] == t.T and T[t.j] >> 32 == t.X >> 32, (t.node, t.site)
    c = case.counts()
    assert c["moves"] > 0 and c["stays"] > 0
    return c


def prove_category_tie(case):
    (t,) = case.ties
    assert mut_draw(case.seed, 0, t.site, 0) == t.X
    thr = cat_thresholds(case.sub.invariant, case.sub.rates.size)
    assert thr[t.j] == t.T and t.T >> 32 == t.X >> 32
    return state(t.X, thr)


def test_numpy_draws_equal_the_oracles():
    sites = np.array([0, 1, 2, 3, 4, 5, 1023, 4097, 2 ** 31 + 7], dtype=np.uint64)
    for node in (0, 1, 77, 1500):
        X = mut_draws(SEED, 3, sites, node)
        assert [int(x) for x in X] == [HM.mut_draw(SEED, 3, int(b), node) for b in sites]
    w = philox([5], [0], [2], [11 | (9 << 8)], SEED)
    assert [int(x[0]) for x in w] == [int(x) for x in H.philox([5, 0, 2, 11 | (9 << 8)], [SEED & 0xFFFFFFFF, SEED >> 32])]


def test_row_thresholds_restate_the_library():
    sub = J.sub_UNREST([[0, 0.1, 0.7, 0.2], [0.3, 0, 0.05, 0.9], [0.6, 0.2, 0, 0.4], [0.1, 1.1, 0.3, 0]])
    P = transition_matrix(sub.Q, 0.37)
    for a in range(4):
        T = row_thresholds(P[a])
        assert T == sorted(T) and T[2] < M64
        assert all(abs(T[j] / 2 ** 64 - P[a][:j + 1].sum() / P[a].sum()) < 1e-15 for j in range(3))
    assert row_thresholds([1, 0, 0, 0]) == [M64] * 3 and row_thresholds([0, 0, -1e-18, 1]) == [0, 0, 0]
    assert prob_threshold(0.5) == 2 ** 63 and prob_threshold(1 - 2 ** -53) == 2 ** 64 - 2 ** 11


def _tip_bases_follow_the_ties(case):
    """In the oracle's records, every tie's tip carries the state its outcome gives."""
    tree = case.tree
    want = HM.mutate(case.genome, tree, case.sub, case.seed)
    tips = [int(v) for v in tree.tip_node]
    ref = case.genome.seqs[0]
    for t in case.ties:
        s = state(t.X, thresholds(case.sub, tree.branch_len[t.node], 0, t.row))
        for tip in [t.node] if t.node in tips else [v for v in tips if tree.parent[v] == t.node]:
            pos, nuc = want[tips.index(tip)][0]
            k = np.searchsorted(pos, t.site)
            base = nuc[k] if k < pos.size and pos[k] == t.site else int(ref[t.site])
            assert base == b"TCAG"[s], (t.node, t.site)


@pytest.mark.parametrize("name", ["smem", "global"])
def test_transition_ties(name):
    case = tie_case(name)
    c = prove_transition_ties(case)
    n_star = 192 if name == "smem" else 1500
    assert c["ties"] == n_star + 16 and c["exact"] >= 3
    internal = [t for t in case.ties if case.tree.parent[t.node] != 0]
    assert len(internal) == 16 and any(t.moves for t in internal) and any(not t.moves for t in internal)
    # rows x 16 B against the 64 KiB of shared memory k_mutate stages the table in
    assert (case.tree.n_nodes * 4 * 16 <= 64 << 10) == (name == "smem")
    _tip_bases_follow_the_ties(case)


def test_transition_ties_with_indels_survive():
    case = tie_case("indels")
    c = prove_transition_ties(case)
    assert c["ties"] == 168 and c["exact"] >= 1
    o = HI.indels(case.genome, case.tree, case.sub, case.ins, case.dele, case.eps, case.seed)
    assert (o.events[:, 4] == 0).any() and (o.events[:, 4] == 1).any()
    tips = [int(v) for v in case.tree.tip_node]
    for t in case.ties:
        for tip in [t.node] if t.node in tips else [v for v in tips if case.tree.parent[v] == t.node]:
            assert site_alive(o, tips.index(tip), t.site)


def test_ins_walk_ties():
    case = tie_case("ins_walk")
    c = prove_transition_ties(case)
    assert c["ties"] == INS_KIDS and c["exact"] >= 1
    o = HI.indels(case.genome, case.tree, case.sub, case.ins, case.dele, case.eps, case.seed)
    at_x = set(columns(case.tree, o.events, case.genome.seqs[0].size, 1))
    pi_thr = row_thresholds(case.sub.pi)
    for t in case.ties:
        assert t.site in at_x and t.site not in columns(case.tree, o.events, case.genome.seqs[0].size, 0)
        assert t.site in columns(case.tree, o.events, case.genome.seqs[0].size, t.node)
        assert state(icol_draws(case.seed, 0, -t.site - 1)[1], pi_thr) == t.row


@pytest.mark.parametrize("name,evolves", [("cat0_exact", 1), ("cat0_below", 1), ("cat0_above", 0),
                                          ("cat1_lo", 2), ("cat1_hi", 1)])
def test_category_ties(name, evolves):
    case = tie_case(name)
    assert prove_category_tie(case) == evolves
    if name == "cat0_exact":
        assert case.ties[0].exact


# ------------------------------------------------------------------------------------ k_reads fallbacks ---

ALL_N_PAIRS = 30_000
ALL_N_SEED = 11


def all_n_genome():
    """Every read base takes base_rare's N branch: 'N' and a few other non-T/C/A/G bytes."""
    s = np.full(60_000, ord("N"), dtype=np.uint8)
    s[::997] = ord("R")
    s[5::1009] = ord("n")
    s[7::1013] = ord("-")
    return J.RefGenome(["allN"], [s])


ALL_N_KW = dict(seq_sys="HS25", ins_prob1=0, del_prob1=0, ins_prob2=0, del_prob2=0)
# Alias-slot flips are rare (about one in 6 x 10^4 HS25 PE150 pairs: HS25's tables are small, and a slot whose
# deficit is k of n flips only when the draw's low 40 bits reach k / n); the oracle runs on slices of a large run
# that hold them.
SLOT_KW = dict(seq_sys="HS25")
SLOT_PAIRS = 400_000
SLOT_SEED = 3
SLOT_SLICES = ((65_000, 66_000), (72_000, 75_000), (171_000, 172_000))


def slot_genome():
    return J.random_genome(3, [70_001, 50_000, 33_333], seed=17)


def nqual_recount(seed, n_pairs, L):
    """N qualities whose 24 high bits leave u * 10 + 33 open, recounted from the QUAL plane (base_rare)."""
    j = np.repeat(np.arange(n_pairs, dtype=np.uint64), L // 2)
    blk = np.tile(np.arange(L // 2, dtype=np.uint64), n_pairs)
    n = 0
    for e in (0, 1):
        w = philox(j, j >> np.uint64(32), blk, 2 | (e << 8), seed, rounds=7)
        for h in (0, 2):
            dn = (w[h] >> np.uint64(8)) << np.uint64(8)
            n += int(np.sum(((dn * np.uint64(10) + np.uint64(2560)) & np.uint64(0xFFFFFFFF)) < 2560))
    return n


@functools.lru_cache(maxsize=None)
def all_n_oracle():
    return oracle_run(all_n_genome(), 2 * ALL_N_PAIRS, 150, True, seed=ALL_N_SEED, **ALL_N_KW)


@functools.lru_cache(maxsize=None)
def slot_oracle():
    """The oracle on SLOT_SLICES of the run: [(lo, hi, r1, r2)] and the slices' fallback counts."""
    out, fb = [], dict.fromkeys(H.FALLBACK_KINDS, 0)
    for lo, hi in SLOT_SLICES:
        o = oracle_run(slot_genome(), 2 * SLOT_PAIRS, 150, True, seed=SLOT_SEED, lo=lo, hi=hi, **SLOT_KW)
        out.append((lo, hi, o["r1"], o["r2"]))
        for k, v in o["fallback"].items():
            fb[k] += v
    return out, fb


def test_n_quality_counter_equals_the_recount():
    o = all_n_oracle()
    fb = o["fallback"]
    assert o["r1"].count(b"\n") == 4 * ALL_N_PAIRS
    assert set(o["r1"].split(b"\n")[1::4]) == {b"N" * 150}
    assert fb["nqual_ambiguous"] == nqual_recount(o["params"].seed, ALL_N_PAIRS, 150)
    assert fb["nqual_flipped"] >= 2 and fb["slot_ambiguous"] == 0 and fb["sub_ambiguous"] == 0


def test_slot_and_substitution_flips():
    fb = slot_oracle()[1]
    assert fb["slot_flipped"] >= 3 and fb["sub_flipped"] >= 3 and fb["nqual_ambiguous"] == 0
    assert fb["slot_ambiguous"] >= fb["slot_flipped"] and fb["sub_ambiguous"] > fb["sub_flipped"]

