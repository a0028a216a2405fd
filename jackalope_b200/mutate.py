"""``create_haplotypes()`` -- haplotypes evolved from the reference along a tree, substitutions only.

jackalope's middle step (reference -> haplotypes -> reads) with the per-site work on the GPU
(``jlp_create_haplotypes``, ``csrc/jlp_mutate.cu``).  The definitions this module implements are the
project's own (DESIGN.md section 10):

* States in the order T, C, A, G; ``Q`` rows are the "from" state, ``q_ii = -sum_{j != i} q_ij``; Q is not
  normalised.  The ``sub_*`` functions below build Q as their docstrings say.
* Every site draws one rate, shared by all branches: 0 with probability ``invariant``, otherwise one of
  ``gamma_k`` equally likely categories of Yang's (1994) discrete Gamma (shape = rate = ``gamma_shape``, each
  category the mean of its equal-probability bin), or 1 when ``gamma_shape`` is None.
* The root state is the reference base; a child's state is drawn from row ``parent state`` of
  ``expm(Q * rate * branch_length)``.  Only T/C/A/G sites evolve.  A haplotype's records are the sites where its
  tip differs from the reference.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
import os

import numpy as np

from .genome import HapChromMuts, Haplotypes, RefGenome
from .profiles import JackalopeError

BASES = "TCAG"
# index pairs of GTR's exchangeabilities (TC, TA, TG, CA, CG, AG)
GTR_PAIRS = ((0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3))


def _bad(fun, par, what):
    raise JackalopeError("\nFor the `%s` function in jackalope, argument `%s` must be %s." % (fun, par, what))


def _is_number(x):
    return isinstance(x, numbers.Real) and not isinstance(x, bool) and math.isfinite(float(x))


def _is_int(x):
    return isinstance(x, numbers.Real) and not isinstance(x, bool) and math.isfinite(float(x)) and float(x) == int(x)


# ------------------------------------------------------------------ substitution models ---

def discrete_gamma_rates(shape, k):
    """Yang's (1994) discrete Gamma: k equal-probability bins of Gamma(shape, rate = shape), each category's
    rate the mean of its bin (so the mean rate is 1)."""
    from scipy import special, stats
    edges = stats.gamma.ppf(np.arange(1, k) / k, a=shape, scale=1.0 / shape)
    cdf1 = special.gammainc(shape + 1.0, shape * np.concatenate(([0.0], edges, [np.inf])))
    return k * np.diff(cdf1)


def stationary(Q):
    """The stationary distribution of Q: the left null vector, summing to 1."""
    Q = np.asarray(Q, dtype=np.float64)
    A = np.vstack([Q.T, np.ones(4)])
    b = np.zeros(5)
    b[4] = 1.0
    pi = np.linalg.lstsq(A, b, rcond=None)[0]
    return np.clip(pi, 0.0, None) / np.clip(pi, 0.0, None).sum()


class SubModel:
    """A substitution model: rate matrix ``Q`` (T, C, A, G; diagonal = minus the row sum), the site-rate
    categories ``rates`` of the variable sites and the ``invariant`` probability."""

    def __init__(self, name, Q, invariant, gamma_shape, gamma_k):
        Q = np.array(Q, dtype=np.float64)
        np.fill_diagonal(Q, 0.0)
        np.fill_diagonal(Q, -Q.sum(axis=1))
        self.name, self.Q = name, Q
        self.invariant = float(invariant)
        self.gamma_shape = None if gamma_shape is None else float(gamma_shape)
        self.gamma_k = int(gamma_k)
        self.rates = np.ones(1) if gamma_shape is None else discrete_gamma_rates(self.gamma_shape, self.gamma_k)
        self.pi = stationary(Q)

    def mu_bar(self):
        """Mean substitution rate at stationarity, -sum_i pi_i q_ii."""
        return float(-np.sum(self.pi * np.diag(self.Q)))

    def __repr__(self):
        return "<sub_info %s, invariant %g, %d rate categor%s>" % (self.name, self.invariant, self.rates.size,
                                                                  "y" if self.rates.size == 1 else "ies")


def _site_args(fun, invariant, gamma_shape, gamma_k):
    if not (_is_number(invariant) and 0 <= invariant < 1):
        _bad(fun, "invariant", "a single number >= 0 and < 1")
    if gamma_shape is not None and not (_is_number(gamma_shape) and gamma_shape > 0):
        _bad(fun, "gamma_shape", "NULL or a single number > 0")
    if not (_is_int(gamma_k) and 2 <= gamma_k <= 255):
        _bad(fun, "gamma_k", "a single integer in range [2, 255]")


def _rate(fun, par, x):
    if not (_is_number(x) and x >= 0):
        _bad(fun, par, "a single number >= 0")
    return float(x)


def _pi(fun, pi_tcag):
    try:
        pi = np.asarray(pi_tcag, dtype=np.float64)
    except (TypeError, ValueError):
        pi = None
    if pi is None or pi.shape != (4,) or not np.all(np.isfinite(pi)) or np.any(pi < 0) or not np.any(pi > 0):
        _bad(fun, "pi_tcag", "a numeric vector of length 4, where no number can be < 0 and at least one must be > 0")
    return pi / pi.sum()


def _is_transition(i, j):
    return {i, j} in ({0, 1}, {2, 3})


def _from_pi(pi, trans, transv):
    """q_ij = (trans(i, j) or transv) * pi_j"""
    Q = np.zeros((4, 4))
    for i in range(4):
        for j in range(4):
            if i != j:
                Q[i, j] = (trans(i, j) if _is_transition(i, j) else transv) * pi[j]
    return Q


def sub_JC69(lambda_, invariant=0, gamma_shape=None, gamma_k=5):
    """JC69: every off-diagonal rate is ``lambda_``."""
    f = "sub_JC69"
    lam = _rate(f, "lambda", lambda_)
    _site_args(f, invariant, gamma_shape, gamma_k)
    return SubModel("JC69", np.full((4, 4), lam), invariant, gamma_shape, gamma_k)


def sub_K80(alpha, beta, invariant=0, gamma_shape=None, gamma_k=5):
    """K80: transitions ``alpha``, transversions ``beta``."""
    f = "sub_K80"
    a, b = _rate(f, "alpha", alpha), _rate(f, "beta", beta)
    _site_args(f, invariant, gamma_shape, gamma_k)
    Q = np.array([[a if _is_transition(i, j) else b for j in range(4)] for i in range(4)])
    return SubModel("K80", Q, invariant, gamma_shape, gamma_k)


def sub_F81(pi_tcag, invariant=0, gamma_shape=None, gamma_k=5):
    """F81: q_ij = pi_j."""
    f = "sub_F81"
    pi = _pi(f, pi_tcag)
    _site_args(f, invariant, gamma_shape, gamma_k)
    return SubModel("F81", _from_pi(pi, lambda i, j: 1.0, 1.0), invariant, gamma_shape, gamma_k)


def sub_HKY85(pi_tcag, alpha, beta, invariant=0, gamma_shape=None, gamma_k=5):
    """HKY85: transitions alpha * pi_j, transversions beta * pi_j."""
    f = "sub_HKY85"
    pi = _pi(f, pi_tcag)
    a, b = _rate(f, "alpha", alpha), _rate(f, "beta", beta)
    _site_args(f, invariant, gamma_shape, gamma_k)
    return SubModel("HKY85", _from_pi(pi, lambda i, j: a, b), invariant, gamma_shape, gamma_k)


def sub_F84(pi_tcag, beta, kappa, invariant=0, gamma_shape=None, gamma_k=5):
    """F84: T<->C beta (1 + kappa / pi_Y) pi_j, A<->G beta (1 + kappa / pi_R) pi_j, transversions beta pi_j."""
    f = "sub_F84"
    pi = _pi(f, pi_tcag)
    b, k = _rate(f, "beta", beta), _rate(f, "kappa", kappa)
    _site_args(f, invariant, gamma_shape, gamma_k)
    pi_y, pi_r = pi[0] + pi[1], pi[2] + pi[3]
    if pi_y == 0 or pi_r == 0:
        _bad(f, "pi_tcag", "a vector with pi_T + pi_C > 0 and pi_A + pi_G > 0 for F84")
    Q = _from_pi(pi, lambda i, j: b * (1 + k / (pi_y if i < 2 else pi_r)), b)
    return SubModel("F84", Q, invariant, gamma_shape, gamma_k)


def sub_TN93(pi_tcag, alpha_1, alpha_2, beta, invariant=0, gamma_shape=None, gamma_k=5):
    """TN93: T<->C alpha_1 pi_j, A<->G alpha_2 pi_j, transversions beta pi_j."""
    f = "sub_TN93"
    pi = _pi(f, pi_tcag)
    a1, a2, b = _rate(f, "alpha_1", alpha_1), _rate(f, "alpha_2", alpha_2), _rate(f, "beta", beta)
    _site_args(f, invariant, gamma_shape, gamma_k)
    return SubModel("TN93", _from_pi(pi, lambda i, j: a1 if i < 2 else a2, b), invariant, gamma_shape, gamma_k)


def sub_GTR(pi_tcag, abcdef, invariant=0, gamma_shape=None, gamma_k=5):
    """GTR: q_ij = r_ij pi_j, ``abcdef`` the exchangeabilities of (TC, TA, TG, CA, CG, AG) (Yang's layout)."""
    f = "sub_GTR"
    pi = _pi(f, pi_tcag)
    try:
        r = np.asarray(abcdef, dtype=np.float64)
    except (TypeError, ValueError):
        r = None
    if r is None or r.shape != (6,) or not np.all(np.isfinite(r)) or np.any(r < 0):
        _bad(f, "abcdef", "a numeric vector of length 6, where no number can be < 0")
    _site_args(f, invariant, gamma_shape, gamma_k)
    Q = np.zeros((4, 4))
    for (i, j), x in zip(GTR_PAIRS, r):
        Q[i, j], Q[j, i] = x * pi[j], x * pi[i]
    return SubModel("GTR", Q, invariant, gamma_shape, gamma_k)


def sub_UNREST(Q, invariant=0, gamma_shape=None, gamma_k=5):
    """UNREST: the given 4 x 4 matrix (T, C, A, G; rows = "from"); its diagonal is ignored."""
    f = "sub_UNREST"
    try:
        q = np.array(Q, dtype=np.float64)
    except (TypeError, ValueError):
        q = None
    if q is None or q.shape != (4, 4):
        _bad(f, "Q", "a 4 x 4 numeric matrix")
    np.fill_diagonal(q, 0.0)
    if not np.all(np.isfinite(q)) or np.any(q < 0):
        _bad(f, "Q", "a 4 x 4 matrix with no off-diagonal value < 0")
    _site_args(f, invariant, gamma_shape, gamma_k)
    return SubModel("UNREST", q, invariant, gamma_shape, gamma_k)


def transition_matrix(Q, t):
    """P = expm(Q t) as the library computes it (jlp_transition_matrix)."""
    from . import _lib
    q = np.ascontiguousarray(np.asarray(Q, dtype=np.float64).reshape(16))
    P = np.zeros(16)
    if _lib.lib().jlp_transition_matrix(q.ctypes.data_as(_lib.f64p), float(t), P.ctypes.data_as(_lib.f64p)) != 0:
        raise JackalopeError("jlp_transition_matrix: invalid arguments")
    return P.reshape(4, 4)


# ------------------------------------------------------------------------------- trees ---

class Tree:
    """A rooted tree in preorder: ``parent[0] = -1``, ``parent[i] < i``, ``branch_len[i]`` the branch above node i;
    tip i of the haplotypes is node ``tip_node[i]``, named ``tip_names[i]``."""

    def __init__(self, parent, branch_len, tip_node, tip_names, labels=None):
        self.parent = np.ascontiguousarray(parent, dtype=np.int32)
        self.branch_len = np.ascontiguousarray(branch_len, dtype=np.float64)
        self.tip_node = np.ascontiguousarray(tip_node, dtype=np.uint32)
        self.tip_names = [str(x) for x in tip_names]
        self.labels = labels

    @property
    def n_nodes(self):
        return int(self.parent.size)

    def children(self):
        kids = [[] for _ in range(self.n_nodes)]
        for i in range(1, self.n_nodes):
            kids[self.parent[i]].append(i)
        return kids

    def scaled(self, f):
        return Tree(self.parent, self.branch_len * f, self.tip_node, self.tip_names, self.labels)

    def newick(self):
        kids = self.children()
        name = {int(v): n for v, n in zip(self.tip_node, self.tip_names)}
        text = [None] * self.n_nodes
        for v in range(self.n_nodes - 1, -1, -1):           # children come after their parent in preorder
            lab = name.get(v, (self.labels[v] if self.labels and self.labels[v] else ""))
            s = ("(" + ",".join(text[c] for c in kids[v]) + ")" if kids[v] else "") + _quote(lab)
            if v:
                s += ":%r" % float(self.branch_len[v])
            text[v] = s
        return text[0] + ";"


def _quote(label):
    if label and any(ch in label for ch in "()[]':;, \t\n"):
        return "'" + label.replace("'", "''") + "'"
    return label


def parse_newick(text):
    """One rooted Newick tree -> Tree.  Branch lengths are required on every node but the root (whose length is
    ignored) and must be >= 0; tip labels (the haplotype names, in order of appearance) are required and unique.
    Multifurcations, internal labels, quoted labels, [comments], whitespace and scientific notation are accepted."""
    s, n = str(text), len(str(text))
    parent, length, label = [], [], []
    i = 0

    def err(msg):
        raise JackalopeError("\nNewick tree: %s (at character %d)." % (msg, i))

    def skip():
        nonlocal i
        while i < n:
            if s[i].isspace():
                i += 1
            elif s[i] == "[":
                j = s.find("]", i)
                if j < 0:
                    err("unterminated comment")
                i = j + 1
            else:
                break

    def read_label():
        nonlocal i
        skip()
        if i < n and s[i] == "'":
            out = []
            i += 1
            while True:
                if i >= n:
                    err("unterminated quoted label")
                if s[i] == "'":
                    if i + 1 < n and s[i + 1] == "'":
                        out.append("'")
                        i += 2
                        continue
                    i += 1
                    break
                out.append(s[i])
                i += 1
            return "".join(out)
        j = i
        while i < n and s[i] not in "(),:;[]'" and not s[i].isspace():
            i += 1
        return s[j:i]

    def read_length(v):
        nonlocal i
        skip()
        if i < n and s[i] == ":":
            i += 1
            skip()
            j = i
            while i < n and s[i] not in "(),:;[]'" and not s[i].isspace():
                i += 1
            tok = s[j:i]
            try:
                x = float(tok)
            except ValueError:
                err("branch length %r is not a number" % tok)
            if not math.isfinite(x):
                err("branch length %r is not finite" % tok)
            length[v] = x

    def new(par):
        parent.append(par)
        length.append(None)
        label.append("")
        return len(parent) - 1

    skip()
    if i >= n or s[i] != "(":
        err("the tree must start with '(' (a tree of more than one node)")
    stack = [new(-1)]
    i += 1
    while True:                      # at the start of a child of stack[-1]
        skip()
        if i < n and s[i] == "(":
            stack.append(new(stack[-1]))
            i += 1
            continue
        v = new(stack[-1])
        label[v] = read_label()
        if not label[v]:
            err("every tip needs a label")
        read_length(v)
        while True:                  # after a child
            skip()
            if i >= n:
                err("unexpected end of the tree")
            if s[i] == ",":
                i += 1
                break
            if s[i] != ")":
                err("unexpected character %r" % s[i])
            i += 1
            v = stack.pop()
            label[v] = read_label()
            read_length(v)
            if not stack:
                break
        if not stack:
            break
    skip()
    if i >= n or s[i] != ";":
        err("the tree must end with ';'")
    i += 1
    skip()
    if i != n:
        err("text after the tree's ';' (one tree only)")
    nn = len(parent)
    has_kid = np.zeros(nn, dtype=bool)
    for v in range(1, nn):
        has_kid[parent[v]] = True
        if length[v] is None:
            raise JackalopeError("\nNewick tree: node %r has no branch length." % (label[v] or "#%d" % v))
        if length[v] < 0:
            raise JackalopeError("\nNewick tree: node %r has a negative branch length." % (label[v] or "#%d" % v))
    tips = [v for v in range(nn) if not has_kid[v]]
    names = [label[v] for v in tips]
    if len(set(names)) != len(names):
        dup = sorted({x for x in names if names.count(x) > 1})
        raise JackalopeError("\nNewick tree: duplicate tip labels %s." % ", ".join(map(repr, dup)))
    bl = np.array([0.0] + [length[v] for v in range(1, nn)])
    return Tree(parent, bl, tips, names, labels=label)


def kingman(n, rng):
    """Kingman coalescent of n tips named hap0..: while k lineages remain, wait Exp(k(k-1)/2), then merge a
    uniformly chosen pair.  Unscaled (coalescent units); node 0 the root, preorder."""
    height = [0.0] * n
    kids = [[] for _ in range(n)]
    lineages = list(range(n))
    t = 0.0
    for k in range(n, 1, -1):
        t += rng.exponential(2.0 / (k * (k - 1)))
        a, b = sorted(rng.choice(k, size=2, replace=False).tolist())
        x, y = lineages[a], lineages[b]
        del lineages[b]
        del lineages[a]
        height.append(t)
        kids.append([x, y])
        lineages.append(len(height) - 1)
    root = lineages[0]
    order, stack = [], [root]
    while stack:
        v = stack.pop()
        order.append(v)
        stack.extend(reversed(kids[v]))
    pre = {v: i for i, v in enumerate(order)}
    parent = np.full(len(order), -1, dtype=np.int32)
    bl = np.zeros(len(order))
    for v in order:
        for c in kids[v]:
            parent[pre[c]] = pre[v]
            bl[pre[c]] = height[v] - height[c]
    return Tree(parent, bl, [pre[h] for h in range(n)], ["hap%d" % h for h in range(n)])


class HapsInfo:
    """Where the haplotypes' tree comes from (``haps_phylo`` or ``haps_theta``)."""

    def tree(self, sub, seed):
        raise NotImplementedError


class HapsPhylo(HapsInfo):
    def __init__(self, tree: Tree):
        self._tree = tree

    def tree(self, sub, seed):
        return self._tree

    def __repr__(self):
        return "<haps_info phylo, %d haplotypes>" % len(self._tree.tip_names)


class HapsTheta(HapsInfo):
    def __init__(self, theta, n_haps):
        self.theta, self.n_haps = float(theta), int(n_haps)

    def scale(self, sub: SubModel):
        """Coalescent units -> branch lengths: theta / (2 mu_bar (1 - invariant)), so that the expected number of
        substitutions per site between two haplotypes is theta."""
        mu = sub.mu_bar()
        if not mu > 0:
            raise JackalopeError("\nFor `haps_theta`, the substitution model must have a mean rate > 0.")
        return self.theta / (2.0 * mu * (1.0 - sub.invariant))

    def tree(self, sub, seed):
        return kingman(self.n_haps, np.random.default_rng(int(seed))).scaled(self.scale(sub))

    def __repr__(self):
        return "<haps_info theta = %g, %d haplotypes>" % (self.theta, self.n_haps)


def haps_phylo(phy=None, fn=None):
    """One rooted Newick tree (text ``phy``, or the file ``fn``), used for every chromosome."""
    if (phy is None) == (fn is None):
        _bad("haps_phylo", "phy", "a Newick string when `fn` is NULL (exactly one of `phy` and `fn` is given)")
    if fn is not None:
        if not isinstance(fn, str) or not os.path.isfile(os.path.expanduser(fn)):
            _bad("haps_phylo", "fn", "the name of an existing file holding one Newick tree")
        with open(os.path.expanduser(fn)) as f:
            phy = f.read()
    if not isinstance(phy, str):
        _bad("haps_phylo", "phy", "a single string (one Newick tree)")
    return HapsPhylo(parse_newick(phy))


def haps_theta(theta, n_haps):
    """A Kingman coalescent tree of ``n_haps`` haplotypes, drawn by create_haplotypes from its seed and scaled so
    that two haplotypes differ at ``theta`` substitutions per site in expectation."""
    if not (_is_number(theta) and theta > 0):
        _bad("haps_theta", "theta", "a single number > 0")
    if not (_is_int(n_haps) and n_haps >= 2):
        _bad("haps_theta", "n_haps", "a single integer >= 2")
    return HapsTheta(theta, n_haps)


# -------------------------------------------------------------------- create_haplotypes ---

def create_haplotypes(reference, haps_info, sub, ins=None, del_=None, epsilon=0.03, n_threads=1,
                      show_progress=False, *, seed=None, ctx=None, device=0):
    """Haplotypes evolved from ``reference`` along the tree of ``haps_info`` under the substitution model ``sub``,
    generated on the GPU.  Returns a ``Haplotypes`` object (substitution records only; the tree as Newick text in
    ``.tree``, the call's figures in ``.stats``) and leaves it resident in the context, so a following
    ``illumina()`` / ``pacbio()`` on it uploads nothing.  ``epsilon`` (validated, unused: substitutions are drawn
    exactly from P(t)), ``n_threads`` and ``show_progress`` are accepted for compatibility.  ``seed`` (keyword-only)
    addresses every draw; None draws one from numpy's global RNG."""
    from . import _lib
    from .illumina import default_context

    f = "create_haplotypes"
    if not isinstance(reference, RefGenome):
        _bad(f, "reference", "a \"ref_genome\" object")
    if not isinstance(haps_info, HapsInfo):
        _bad(f, "haps_info", "a \"haps_info\" object (from `haps_phylo` or `haps_theta`)")
    if not isinstance(sub, SubModel):
        _bad(f, "sub", "a \"sub_info\" object (from one of the `sub_*` functions)")
    if ins is not None or del_ is not None:
        raise JackalopeError("\nFor the `create_haplotypes` function in jackalope, insertions and deletions along a "
                             "tree are not built yet: arguments `ins` and `del_` must be NULL.")
    if not (_is_number(epsilon) and 0 <= epsilon < 1):
        _bad(f, "epsilon", "a single number >= 0 and < 1")
    if not (_is_int(n_threads) and n_threads >= 1):
        _bad(f, "n_threads", "a single integer >= 1")
    if not isinstance(show_progress, (bool, np.bool_)):
        _bad(f, "show_progress", "a single logical")
    if seed is None:
        seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
    tree = haps_info.tree(sub, seed)
    ctx = ctx or default_context(device)
    ctx.set_genome(reference)

    p = _lib.MutationParams()
    p.Q[:] = [float(x) for x in sub.Q.reshape(16)]
    p.invariant = sub.invariant
    rates = np.ascontiguousarray(sub.rates, dtype=np.float64)
    p.n_rates, p.rates = rates.size, rates.ctypes.data_as(_lib.f64p)
    p.n_nodes = tree.n_nodes
    p.parent = tree.parent.ctypes.data_as(C.POINTER(C.c_int32))
    p.branch_len = tree.branch_len.ctypes.data_as(_lib.f64p)
    p.n_tips = len(tree.tip_names)
    p.tip_node = tree.tip_node.ctypes.data_as(_lib.u32p)
    names = (C.c_char_p * len(tree.tip_names))(*[n.encode() for n in tree.tip_names])
    p.tip_names = names
    p.seed = int(seed) & (2 ** 64 - 1)
    st = _lib.MutationStats()
    ctx._haps = None
    ctx._check(ctx.lib.jlp_create_haplotypes(ctx.h, C.byref(p), C.byref(st)), "jlp_create_haplotypes")

    muts = [[haplotype_muts(ctx, h, c) for c in range(reference.n_chroms())] for h in range(len(tree.tip_names))]
    haps = Haplotypes(reference, tree.tip_names, muts)
    haps.tree = tree.newick()
    haps.stats = st.as_dict()
    ctx._haps = haps
    return haps


def haplotype_muts(ctx, hap, chrom) -> HapChromMuts:
    """The records the context holds for (haplotype, chromosome) (jlp_get_haplotype_muts)."""
    from . import _lib
    n, pl, size = C.c_uint64(), C.c_uint64(), C.c_uint64()
    ctx._check(ctx.lib.jlp_get_haplotype_muts(ctx.h, hap, chrom, None, None, None, None, 0, 0, C.byref(n), C.byref(pl),
                                              C.byref(size)), "jlp_get_haplotype_muts")
    M = n.value
    old = np.empty(M, dtype=np.uint64)
    new = np.empty(M, dtype=np.uint64)
    off = np.empty(M, dtype=np.uint64)
    pool = np.empty(pl.value, dtype=np.uint8)
    if M or pl.value:
        ctx._check(ctx.lib.jlp_get_haplotype_muts(ctx.h, hap, chrom, old.ctypes.data_as(_lib.u64p),
                                                  new.ctypes.data_as(_lib.u64p), off.ctypes.data_as(_lib.u64p),
                                                  pool.ctypes.data_as(C.c_void_p), M, pool.size, C.byref(n),
                                                  C.byref(pl), C.byref(size)), "jlp_get_haplotype_muts")
    if M == 0:
        return HapChromMuts.empty(size.value) if pl.value == 0 else HapChromMuts(old, new, off, np.zeros(0, np.uint32), pool, size.value)
    nuc_len = np.diff(np.concatenate((off, [pool.size]))).astype(np.uint32)
    return HapChromMuts(old, new, off, nuc_len, pool, size.value)
