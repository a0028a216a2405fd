"""Host-side genome data model handed to the C ABI.

``RefGenome`` mirrors the reference's RefGenome/RefChrom (name + nucleotide
string per chromosome, /root/reference/src/ref_classes.h:36-140) and
``Haplotypes`` its HapSet/HapGenome/HapChrom/AllMutations (sorted mutation
records ``old_pos``, ``new_pos``, ``nucleos`` per chromosome plus the mutated
size, src/hap_classes.h:100-104,287-296,540).  The objects only *hold* data;
they are flattened into plain arrays before crossing into the library.

``create_genome`` below makes a reference on the GPU; ``create_haplotypes``
(mutate.py) evolves haplotypes from it along a tree under a substitution model
and optional insertion / deletion models, also on the GPU.
``random_genome`` and ``random_haplotypes`` below exist so that tests and the
benchmark have inputs of the named shapes; they are input generators, not
restatements: their mutations are scattered uniformly and the haplotypes share
no ancestry.
"""
from __future__ import annotations

import numpy as np

from .profiles import JackalopeError


class RefGenome:
    """Chromosome names and sequences (bytes / uint8 arrays of ASCII)."""

    name = "REF"   # src/ref_classes.h:138

    def __init__(self, names, seqs):
        if len(names) != len(seqs) or len(names) == 0:
            raise JackalopeError("RefGenome needs one name per chromosome and at least one chromosome")
        self.names = [n.decode() if isinstance(n, bytes) else str(n) for n in names]
        self.seqs = [np.frombuffer(s, dtype=np.uint8) if isinstance(s, (bytes, bytearray))
                     else np.ascontiguousarray(s, dtype=np.uint8) for s in seqs]

    def n_chroms(self):
        return len(self.seqs)

    def sizes(self):
        return np.array([s.size for s in self.seqs], dtype=np.uint64)

    def chrom(self, i) -> bytes:
        return self.seqs[i].tobytes()

    def flat(self):
        """(concatenated bases uint8[], offsets uint64[n+1])"""
        off = np.concatenate(([0], np.cumsum(self.sizes()))).astype(np.uint64)
        return np.ascontiguousarray(np.concatenate(self.seqs)), off


class HapChromMuts:
    """AllMutations of one haplotype chromosome as flat arrays."""

    __slots__ = ("old_pos", "new_pos", "nuc_off", "nuc_len", "pool", "chrom_size")

    def __init__(self, old_pos, new_pos, nuc_off, nuc_len, pool, chrom_size):
        self.old_pos = np.ascontiguousarray(old_pos, dtype=np.uint64)
        self.new_pos = np.ascontiguousarray(new_pos, dtype=np.uint64)
        self.nuc_off = np.ascontiguousarray(nuc_off, dtype=np.uint64)
        self.nuc_len = np.ascontiguousarray(nuc_len, dtype=np.uint32)
        self.pool = np.frombuffer(pool, dtype=np.uint8) if isinstance(pool, (bytes, bytearray)) \
            else np.ascontiguousarray(pool, dtype=np.uint8)
        self.chrom_size = int(chrom_size)

    @staticmethod
    def empty(ref_size):
        z = np.zeros(0, dtype=np.uint64)
        return HapChromMuts(z, z, z, np.zeros(0, dtype=np.uint32), b"", ref_size)


class Haplotypes:
    """A set of named haplotypes over one reference."""

    def __init__(self, reference: RefGenome, hap_names, muts):
        """muts[h][c] is a HapChromMuts."""
        self.reference = reference
        self.hap_names = [str(n) for n in hap_names]
        if len(muts) != len(self.hap_names) or any(len(m) != reference.n_chroms() for m in muts):
            raise JackalopeError("Haplotypes needs mutations for every haplotype and chromosome")
        self.muts = muts

    def n_haps(self):
        return len(self.hap_names)

    def n_chroms(self):
        return self.reference.n_chroms()

    def sizes(self, h):
        return np.array([m.chrom_size for m in self.muts[h]], dtype=np.uint64)


# ------------------------------------------------------------ input generators

def random_genome(n_chroms, chrom_len, seed=0, pi_tcag=(0.25, 0.25, 0.25, 0.25)):
    """Uniform random chromosomes named chrom0.. (the shape create_genome makes
    with len_sd = 0, R/create_genome.R:24-28, src/create_sequences.cpp:178-181)."""
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"TCAG", dtype=np.uint8)
    lens = chrom_len if np.ndim(chrom_len) else [int(chrom_len)] * n_chroms
    if tuple(pi_tcag) == (0.25, 0.25, 0.25, 0.25):
        seqs = [lut[rng.integers(0, 4, size=int(l), dtype=np.uint8)] for l in lens]
    else:
        seqs = [lut[rng.choice(4, size=int(l), p=np.asarray(pi_tcag) / np.sum(pi_tcag)).astype(np.uint8)] for l in lens]
    return RefGenome(["chrom%d" % i for i in range(n_chroms)], seqs)


def random_mutations(ref_seq: np.ndarray, rng, sub_rate, indel_rate, max_indel=10, want_edits=True):
    """Sorted, non-overlapping substitutions / insertions / deletions on one
    chromosome, written directly in AllMutations form (vectorised: usable at 500 Mb).
    Indel sizes 1..max_indel with weights exp(-size) (the relative rates `indels()`
    uses, R/mevo.R:660-699).  Returns (HapChromMuts, edits) where `edits` (only if
    want_edits) is the list of (kind, hap_pos, payload) that replays the same edits
    through HapChrom::add_* in ascending order."""
    n = ref_seq.size
    n_sub = int(rng.binomial(n, sub_rate))
    n_ind = int(rng.binomial(n, indel_rate))
    n_slots = n // (max_indel + 2)
    m = min(n_sub + n_ind, max(0, n_slots))
    if m == 0:
        return HapChromMuts.empty(n), []
    # sites spaced so that a deletion never reaches the next site
    if m * 4 < n_slots:
        slots = np.unique(rng.integers(0, n_slots, size=int(m * 1.05) + 16))
        if slots.size > m:
            slots = np.sort(rng.choice(slots, size=m, replace=False))
        m = slots.size
    else:
        slots = np.sort(rng.choice(n_slots, size=m, replace=False))
    old_pos = slots.astype(np.int64) * (max_indel + 2)
    kinds = np.zeros(m, dtype=np.int8)
    ind_idx = rng.choice(m, size=min(n_ind, m), replace=False)
    kinds[ind_idx] = rng.integers(1, 3, size=ind_idx.size)      # 1 insertion, 2 deletion
    w = np.exp(-np.arange(1, max_indel + 1, dtype=np.float64))
    sizes = rng.choice(np.arange(1, max_indel + 1), size=m, p=w / w.sum()).astype(np.int64)
    is_ins, is_del, is_sub = kinds == 1, kinds == 2, kinds == 0
    sizes[is_del] = np.minimum(sizes[is_del], n - old_pos[is_del])
    delta = np.where(is_ins, sizes, np.where(is_del, -sizes, 0))
    shift_before = np.concatenate(([0], np.cumsum(delta)[:-1]))
    new_pos = old_pos + shift_before
    nuc_len = np.where(is_sub, 1, np.where(is_ins, 1 + sizes, 0)).astype(np.int64)
    nuc_off = np.concatenate(([0], np.cumsum(nuc_len)[:-1]))
    bases = np.frombuffer(b"TCAG", dtype=np.uint8)
    pool = bases[rng.integers(0, 4, size=int(nuc_len.sum()), dtype=np.uint8)]
    # substitutions: a base different from the reference's (any base where the reference is not T/C/A/G)
    ref_at = ref_seq[old_pos]
    lut = np.full(256, 255, dtype=np.uint8)
    lut[bases] = np.arange(4, dtype=np.uint8)
    cur = lut[ref_at[is_sub]]
    alt_idx = np.where(cur < 4, (cur.astype(np.int64) + 1 + rng.integers(0, 3, size=cur.size)) % 4,
                       rng.integers(0, 4, size=cur.size))
    pool[nuc_off[is_sub]] = bases[alt_idx]
    pool[nuc_off[is_ins]] = ref_at[is_ins]                      # the anchor base of an insertion
    muts = HapChromMuts(old_pos, new_pos, nuc_off, nuc_len, pool, n + int(delta.sum()))
    edits = []
    if want_edits:
        pb = pool.tobytes()
        for o, np_, k, sz, no in zip(old_pos.tolist(), new_pos.tolist(), kinds.tolist(), sizes.tolist(), nuc_off.tolist()):
            if k == 0:
                edits.append(("sub", np_, pb[no:no + 1]))
            elif k == 1:
                edits.append(("ins", np_, pb[no + 1:no + 1 + sz]))
            else:
                edits.append(("del", np_, sz))
    return muts, edits


def random_haplotypes(reference: RefGenome, n_haps, sub_rate=0.01, indel_rate=0.001, seed=0, names=None,
                      return_edits=False):
    rng = np.random.default_rng(seed)
    muts, edits = [], []
    for _ in range(n_haps):
        mh, eh = [], []
        for seq in reference.seqs:
            mm, ee = random_mutations(seq, rng, sub_rate, indel_rate, want_edits=return_edits)
            mh.append(mm)
            eh.append(ee)
        muts.append(mh)
        edits.append(eh)
    haps = Haplotypes(reference, names or ["hap%d" % i for i in range(n_haps)], muts)
    return (haps, edits) if return_edits else haps


def create_genome(n_chroms, len_mean, len_sd=0, pi_tcag=(0.25, 0.25, 0.25, 0.25), n_threads=1, *, seed=None, ctx=None, device=0):
    """``create_genome()`` of the reference (R/create_genome.R:24-58, create_genome_cpp,
    src/create_sequences.cpp:162-184) with the chromosomes generated on the GPU: lengths from
    Gamma(mean, sd) truncated to integers >= 1 (or all ``len_mean`` when ``len_sd`` is 0), nucleotides
    alias-sampled from ``pi_tcag`` (T, C, A, G), names ``chrom0..``.  The genome stays resident in the
    context's HBM, so a following ``illumina()`` on the returned object uploads nothing.
    ``n_threads`` is accepted for compatibility.  There is no CPU path."""
    import ctypes as C
    import numbers

    from . import _lib
    from .illumina import default_context

    def bad(par, what):
        raise JackalopeError("\nFor the `create_genome` function in jackalope, argument `%s` must be %s." % (par, what))
    if not (isinstance(n_chroms, numbers.Real) and float(n_chroms) == int(n_chroms) and n_chroms >= 1):
        bad("n_chroms", "a single integer >= 1")
    if not (isinstance(len_mean, numbers.Real) and len_mean >= 1):
        bad("len_mean", "a single number >= 1")
    if not (isinstance(len_sd, numbers.Real) and len_sd >= 0):
        bad("len_sd", "a single number >= 0")
    pi = np.asarray(pi_tcag, dtype=np.float64)
    if pi.shape != (4,) or np.any(pi < 0) or np.all(pi == 0) or np.any(np.isnan(pi)):
        bad("pi_tcag", "a numeric vector of length 4, where no number can be < 0 and at least one must be > 0")
    if not (isinstance(n_threads, numbers.Real) and float(n_threads) == int(n_threads) and n_threads >= 1):
        bad("n_threads", "a single integer >= 1")
    if seed is None:
        seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
    n_chroms = int(n_chroms)
    if len_sd > 0:
        rng = np.random.default_rng(seed)
        shape, scale = (len_mean / len_sd) ** 2, len_sd ** 2 / len_mean      # src/create_sequences.cpp:78-79
        lens = np.maximum(rng.gamma(shape, scale, size=n_chroms).astype(np.uint64), 1)
    else:
        lens = np.full(n_chroms, int(len_mean), dtype=np.uint64)
    ctx = ctx or default_context(device)
    ctx._check(ctx.lib.jlp_create_genome(ctx.h, n_chroms, lens.ctypes.data_as(_lib.u64p), pi.ctypes.data_as(_lib.f64p),
                                         int(seed) & (2 ** 64 - 1), None, b"REF"), "jlp_create_genome")
    total = int(lens.sum())
    flat = np.empty(total, dtype=np.uint8)
    n = C.c_uint64()
    ctx._check(ctx.lib.jlp_get_genome(ctx.h, flat.ctypes.data_as(C.c_void_p), total, C.byref(n)), "jlp_get_genome")
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    g = RefGenome(["chrom%d" % i for i in range(n_chroms)], [flat[off[i]:off[i + 1]] for i in range(n_chroms)])
    g.flat = lambda: (flat, off.astype(np.uint64))
    ctx._genome, ctx._haps = g, None           # already resident
    return g
