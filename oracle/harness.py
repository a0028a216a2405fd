"""TEST INFRASTRUCTURE ONLY -- ctypes bindings for the CPU oracle
(oracle/libjlp_oracle.so) and for the unmodified reference built from
/root/reference (oracle/_ref/libjlp_ref{,_replay}.so).

Importable from tests/, bench.py's cpu_baseline / --impl reference legs and
__graft_entry__.smoke() only.  Nothing under jackalope_b200/ imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
u8p, u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_double))


def build(quiet=True):
    """Compile the oracle (and, where /root/reference exists, oracle/_ref)."""
    subprocess.run(["make", "-C", HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def _ptr(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def _strs(items):
    arr = (C.c_char_p * max(1, len(items)))()
    for i, s in enumerate(items):
        arr[i] = s if isinstance(s, bytes) else s.encode()
    return arr


# ----------------------------------------------------------------- oracle ---

class OrcJob(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("paired", C.c_int32), ("matepair", C.c_int32),
        ("job_lo", C.c_uint64), ("job_hi", C.c_uint64), ("pool_pairs", C.c_uint64),
        ("prob_dup", C.c_double), ("L", C.c_uint64),
        ("ins_prob", C.c_double * 2), ("del_prob", C.c_double * 2),
        ("nq", u32p * 2), ("probs", f64p * 2), ("quals", u8p * 2),
        ("frag_cdf", u64p), ("frag_cdf_n", C.c_uint64), ("frag_min", C.c_uint64),
        ("n_groups", C.c_uint64), ("group_off", u64p),
        ("group_seq", C.POINTER(C.c_char_p)), ("group_len", u64p),
        ("group_genome_name", C.POINTER(C.c_char_p)),
        ("group_chrom_name", C.POINTER(C.c_char_p)),
        ("group_barcode", C.POINTER(C.c_char_p)),
        ("fallback", u64p),
    ]


_orc = None

# OrcJob.fallback, in its order: (slot, N quality, substitution index) x (ambiguous, flipped)
FALLBACK_KINDS = ("slot_ambiguous", "slot_flipped", "nqual_ambiguous", "nqual_flipped", "sub_ambiguous", "sub_flipped")


def oracle():
    global _orc
    if _orc is None:
        path = os.path.join(HERE, "libjlp_oracle.so")
        if not os.path.exists(path):
            build()
        lib = C.CDLL(path)
        lib.orc_draw_pair.restype = C.c_uint64
        lib.orc_draw_pair.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
        lib.orc_draw_pos.restype = C.c_uint64
        lib.orc_draw_pos.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        lib.orc_unif_expr.restype = C.c_uint64
        lib.orc_unif_expr.argtypes = [C.c_int, C.c_uint64, C.c_double, C.c_uint64]
        lib.orc_alias_build.argtypes = [f64p, C.c_uint64, f64p, u64p]
        lib.orc_philox4x32_10.argtypes = [u32p, u32p, u32p]
        lib.orc_rev_comp.argtypes = [C.c_char_p, C.c_uint64]
        lib.orc_qual_prob_map.argtypes = [C.c_uint64, u32p, f64p, u8p, f64p]
        lib.orc_materialize.argtypes = [C.c_char_p, C.c_uint64, C.c_uint64, u64p, u64p, u64p,
                                        C.c_char_p, C.c_uint64, C.c_char_p]
        lib.orc_genome_draw.restype = C.c_uint64
        lib.orc_genome_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_int]
        lib.orc_create_chrom.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, f64p, C.c_char_p, u64p]
        lib.orc_generate.argtypes = [C.POINTER(OrcJob), C.c_uint64, C.c_uint64,
                                     C.c_char_p, C.c_uint64, u64p, C.c_char_p, C.c_uint64, u64p,
                                     u64p, u64p, C.c_uint64, u64p, u64p]
        _orc = lib
    return _orc


def philox(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    oracle().orc_philox4x32_10(_ptr(c, u32p), _ptr(k, u32p), _ptr(out, u32p))
    return out


def alias_build(probs):
    p = np.ascontiguousarray(probs, dtype=np.float64)
    P = np.zeros(p.size, dtype=np.float64)
    A = np.zeros(p.size, dtype=np.uint64)
    assert oracle().orc_alias_build(_ptr(p, f64p), p.size, _ptr(P, f64p), _ptr(A, u64p)) == 0
    return P, A


def qual_prob_map(flat):
    L, nq, probs, quals = flat
    out = np.zeros(256, dtype=np.float64)
    assert oracle().orc_qual_prob_map(L, _ptr(nq, u32p), _ptr(probs, f64p), _ptr(quals, u8p), _ptr(out, f64p)) == 0
    return out


def create_chrom(seed, chrom, length, pi_tcag, want_ledger=False):
    """One chromosome of create_genome from the oracle (bytes[, ledger of draws])."""
    pi = np.ascontiguousarray(pi_tcag, dtype=np.float64)
    out = C.create_string_buffer(max(1, length))
    led = np.zeros(max(1, 2 * length), dtype=np.uint64) if want_ledger else None
    assert oracle().orc_create_chrom(seed, chrom, length, _ptr(pi, f64p), out, _ptr(led, u64p)) == 0
    return (out.raw[:length], led[:2 * length]) if want_ledger else out.raw[:length]


def ref_create_chrom_replay(pi_tcag, length, script):
    """The reference's own sampling loop (create_chromosomes_) fed with `script`."""
    lib = ref_lib(True)
    pi = np.ascontiguousarray(pi_tcag, dtype=np.float64)
    sc = np.ascontiguousarray(script, dtype=np.uint64)
    out = C.create_string_buffer(max(1, length))
    used = C.c_uint64()
    rc = lib.jref_create_chrom_replay(_ptr(pi, f64p), length, _ptr(sc, u64p), sc.size, out, C.byref(used))
    assert rc == 0
    return out.raw[:length], used.value


def materialize(ref: bytes, old_pos, new_pos, nuc_off, pool: bytes, chrom_size: int) -> bytes:
    op = np.ascontiguousarray(old_pos, dtype=np.uint64)
    npos = np.ascontiguousarray(new_pos, dtype=np.uint64)
    no = np.ascontiguousarray(nuc_off, dtype=np.uint64)
    out = C.create_string_buffer(max(1, chrom_size))
    assert oracle().orc_materialize(ref, len(ref), op.size, _ptr(op, u64p), _ptr(npos, u64p),
                                    _ptr(no, u64p), pool, chrom_size, out) == 0
    return out.raw[:chrom_size]


class Groups:
    """(haplotype, chromosome) groups in the order the reference exhausts them."""

    def __init__(self, counts, seqs, genome_names, chrom_names, barcodes, lens=None):
        """`lens`: the chromosomes' sizes when some of `seqs` are placeholders (b"": a group the requested
        pair range cannot touch -- the oracle reads a group's bases only when it places a read there)."""
        self.counts = np.asarray(counts, dtype=np.uint64)
        self.off = np.concatenate(([0], np.cumsum(self.counts))).astype(np.uint64)
        self.seqs = [bytes(s) for s in seqs]
        self.lens = np.array([len(s) for s in self.seqs] if lens is None else lens, dtype=np.uint64)
        self.genome_names = list(genome_names)
        self.chrom_names = list(chrom_names)
        self.barcodes = list(barcodes)


def generate(*, seed, paired, matepair, groups: Groups, prof1, prof2, ins_prob, del_prob,
             prob_dup, pool_pairs, frag_cdf, frag_min, lo=None, hi=None, job_lo=0, job_hi=None,
             want_ledger=False, want_plan=False):
    """Run the oracle for pair instances [lo, hi) of job [job_lo, job_hi).
    prof1/prof2 are flattened profiles (L, nq, probs, quals).  res["fallback"]: the counts of draws that k_reads
    decides with its exact-draw fallbacks (FALLBACK_KINDS; OrcJob.fallback in jlp_oracle.c)."""
    lib = oracle()
    n_total = int(groups.off[-1])
    job_hi = n_total if job_hi is None else job_hi
    lo = job_lo if lo is None else lo
    hi = job_hi if hi is None else hi
    n = hi - lo
    L = prof1[0]
    J = OrcJob()
    J.seed, J.paired, J.matepair = seed, int(paired), int(matepair)
    J.job_lo, J.job_hi, J.pool_pairs, J.prob_dup, J.L = job_lo, job_hi, pool_pairs, prob_dup, L
    keep = []
    for e, pr in enumerate([prof1, prof2] if paired else [prof1]):
        J.ins_prob[e], J.del_prob[e] = ins_prob[e], del_prob[e]
        J.nq[e], J.probs[e], J.quals[e] = _ptr(pr[1], u32p), _ptr(pr[2], f64p), _ptr(pr[3], u8p)
        keep.append(pr)
    cdf = np.ascontiguousarray(frag_cdf, dtype=np.uint64)
    J.frag_cdf, J.frag_cdf_n, J.frag_min = _ptr(cdf, u64p), cdf.size, frag_min
    ng = len(groups.seqs)
    J.n_groups, J.group_off = ng, _ptr(groups.off, u64p)
    seqs = _strs(groups.seqs)
    glen = groups.lens
    gn, cn, bc = _strs(groups.genome_names), _strs(groups.chrom_names), _strs(groups.barcodes)
    J.group_seq, J.group_len = seqs, _ptr(glen, u64p)
    J.group_genome_name, J.group_chrom_name, J.group_barcode = gn, cn, bc
    fallback = np.zeros(len(FALLBACK_KINDS), dtype=np.uint64)
    J.fallback = _ptr(fallback, u64p)
    max_name = max(len(a) + len(b) for a, b in zip(groups.genome_names, groups.chrom_names)) if ng else 0
    cap = n * (max_name + 32 + 2 * L + 8) + 64
    o1, o2 = C.create_string_buffer(cap), C.create_string_buffer(cap if paired else 1)
    l1, l2 = C.c_uint64(0), C.c_uint64(0)
    plan = np.zeros(4 * max(n, 1), dtype=np.uint64) if want_plan else None
    led_cap = n * (8 * L + 64) if want_ledger else 0
    ledger = np.zeros(max(led_cap, 1), dtype=np.uint64) if want_ledger else None
    led_cnt = np.zeros(max(n, 1), dtype=np.uint64) if want_ledger else None
    led_n = C.c_uint64(0)
    rc = lib.orc_generate(C.byref(J), lo, hi, o1, cap, C.byref(l1), o2, cap if paired else 1, C.byref(l2),
                          _ptr(plan, u64p), _ptr(ledger, u64p), led_cap, C.byref(led_n), _ptr(led_cnt, u64p))
    if rc != 0:
        raise RuntimeError("orc_generate failed rc=%d" % rc)
    res = dict(r1=o1.raw[:l1.value], r2=o2.raw[:l2.value] if paired else b"",
               fallback=dict(zip(FALLBACK_KINDS, (int(x) for x in fallback))))
    if want_plan:
        res["plan"] = plan.reshape(-1, 4)[:n]
    if want_ledger:
        res["ledger"] = ledger[:led_n.value]
        res["ledger_cnt"] = led_cnt[:n]
    return res


# -------------------------------------------------------------- reference ---

def have_ref(replay=False):
    return os.path.exists(os.path.join(HERE, "_ref", "libjlp_ref_replay.so" if replay else "libjlp_ref.so"))


_refs = {}


def ref_lib(replay=False):
    if replay not in _refs:
        name = "libjlp_ref_replay.so" if replay else "libjlp_ref.so"
        lib = C.CDLL(os.path.join(HERE, "_ref", name))
        lib.jref_genome_new.restype = C.c_void_p
        lib.jref_genome_new.argtypes = [C.c_uint64, C.POINTER(C.c_char_p), u64p, C.POINTER(C.c_char_p)]
        lib.jref_genome_free.argtypes = [C.c_void_p]
        lib.jref_hapset_new.restype = C.c_void_p
        lib.jref_hapset_new.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p)]
        lib.jref_hapset_free.argtypes = [C.c_void_p]
        lib.jref_add_sub.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_char, C.c_uint64]
        lib.jref_add_ins.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_char_p, C.c_uint64]
        lib.jref_add_del.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]
        lib.jref_add_edits.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, u8p, u64p, u64p, u64p, C.c_char_p]
        for f in ("jref_hap_chrom_size", "jref_hap_n_muts", "jref_hap_nuc_bytes"):
            getattr(lib, f).restype = C.c_uint64
            getattr(lib, f).argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        lib.jref_hap_chrom_full.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_char_p, C.c_uint64]
        lib.jref_hap_get_muts.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, u64p, u64p, u64p, u32p, C.c_char_p]
        lib.jref_alias_build.argtypes = [f64p, C.c_uint64, f64p, u64p]
        lib.jref_qual_prob_map.argtypes = [C.c_uint64, u32p, f64p, u8p, f64p, C.c_uint64]
        lib.jref_rev_comp.argtypes = [C.c_char_p, C.c_uint64]
        lib.jref_reads_per_group.argtypes = [C.c_uint64, f64p, C.c_uint64, u64p]
        lib.jref_set_r_seed.argtypes = [C.c_uint64]
        lib.jref_unif_expr.restype = C.c_uint64
        lib.jref_unif_expr.argtypes = [C.c_int, C.c_uint64, C.c_double, C.c_uint64]
        prof = [C.c_uint64, u32p, f64p, u8p, C.c_double, C.c_double, u32p, f64p, u8p, C.c_double, C.c_double]
        if not replay:
            lib.jref_illumina_ref.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_uint64, C.c_double,
                                              C.c_uint64, C.c_uint64, C.c_double, C.c_double, C.c_uint64,
                                              C.c_uint64] + prof + [C.c_char_p, C.c_char_p, C.c_uint64]
            lib.jref_illumina_hap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_uint64,
                                              C.c_double, C.c_uint64, C.c_uint64, f64p, C.c_double, C.c_double,
                                              C.c_uint64, C.c_uint64] + prof + [C.POINTER(C.c_char_p), C.c_char_p,
                                                                               C.c_uint64]
        else:
            lib.jref_create_chrom_replay.argtypes = [f64p, C.c_uint64, u64p, C.c_uint64, C.c_char_p, u64p]
            lib.jref_replay.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + prof + [
                C.POINTER(C.c_char_p), C.c_uint64, u64p, u64p, u64p, u64p, u64p, C.c_uint64, u64p,
                C.c_char_p, C.c_uint64, u64p, C.c_char_p, C.c_uint64, u64p, C.c_char_p, C.c_uint64]
        _refs[replay] = lib
    return _refs[replay]


class RefGenomeH:
    """A reference `RefGenome` living inside one of the _ref libraries."""

    def __init__(self, names, seqs, replay=False):
        self.lib = ref_lib(replay)
        self.names = [n if isinstance(n, str) else n.decode() for n in names]
        self.seqs = [bytes(s) for s in seqs]
        lens = np.array([len(s) for s in self.seqs], dtype=np.uint64)
        self.h = self.lib.jref_genome_new(len(self.seqs), _strs(self.seqs), _ptr(lens, u64p), _strs(self.names))

    def __del__(self):
        try:
            self.lib.jref_genome_free(self.h)
        except Exception:
            pass


class HapSetH:
    """A reference `HapSet`; mutations are applied by the reference's own
    HapChrom::add_* (src/hap_classes.cpp:298-509)."""

    def __init__(self, ref: RefGenomeH, hap_names):
        self.lib, self.ref = ref.lib, ref
        self.hap_names = list(hap_names)
        self.h = self.lib.jref_hapset_new(ref.h, len(self.hap_names), _strs(self.hap_names))

    def __del__(self):
        try:
            self.lib.jref_hapset_free(self.h)
        except Exception:
            pass

    def add_sub(self, hap, chrom, nt, pos):
        assert self.lib.jref_add_sub(self.h, hap, chrom, nt.encode() if isinstance(nt, str) else nt, pos) == 0

    def add_ins(self, hap, chrom, nts, pos):
        assert self.lib.jref_add_ins(self.h, hap, chrom, nts.encode() if isinstance(nts, str) else nts, pos) == 0

    def add_del(self, hap, chrom, size, pos):
        assert self.lib.jref_add_del(self.h, hap, chrom, size, pos) == 0

    def add_edit_arrays(self, hap, chrom, kind, pos, size, off, payload):
        """many edits in one call (see muts_edit_arrays)"""
        assert self.lib.jref_add_edits(self.h, hap, chrom, len(kind), _ptr(kind, u8p), _ptr(pos, u64p), _ptr(size, u64p),
                                       _ptr(off, u64p), payload) == 0

    def chrom_size(self, hap, chrom):
        return int(self.lib.jref_hap_chrom_size(self.h, hap, chrom))

    def chrom_full(self, hap, chrom) -> bytes:
        n = self.chrom_size(hap, chrom)
        buf = C.create_string_buffer(max(1, n))
        assert self.lib.jref_hap_chrom_full(self.h, hap, chrom, buf, n) == 0
        return buf.raw[:n]

    def muts(self, hap, chrom):
        """(old_pos, new_pos, nuc_off, nuc_len, pool) -- AllMutations as flat arrays."""
        m = int(self.lib.jref_hap_n_muts(self.h, hap, chrom))
        nb = int(self.lib.jref_hap_nuc_bytes(self.h, hap, chrom))
        op, npos, no = (np.zeros(max(m, 1), dtype=np.uint64) for _ in range(3))
        nl = np.zeros(max(m, 1), dtype=np.uint32)
        pool = C.create_string_buffer(max(nb, 1))
        self.lib.jref_hap_get_muts(self.h, hap, chrom, _ptr(op, u64p), _ptr(npos, u64p), _ptr(no, u64p),
                                   _ptr(nl, u32p), pool)
        return op[:m], npos[:m], no[:m], nl[:m], pool.raw[:nb]


def muts_edit_arrays(m, ref_size):
    """AllMutations arrays of one haplotype chromosome (jackalope_b200.genome.HapChromMuts: sorted, non-overlapping
    records) -> the edits that rebuild them through HapChrom::add_* in ascending order, as flat arrays
    (kind u8[], pos u64[], size u64[], pay_off u64[], payload bytes).  Vectorised: usable at 500 Mb."""
    n = m.old_pos.size
    kind = np.where(m.nuc_len == 1, 0, np.where(m.nuc_len > 1, 1, 2)).astype(np.uint8)
    shift = m.new_pos.astype(np.int64) - m.old_pos.astype(np.int64)
    nxt = np.concatenate((shift[1:], [int(m.chrom_size) - int(ref_size)])) if n else shift
    size_mod = nxt - shift                                           # src/hap_classes.h:314-333
    size = np.where(kind == 0, 1, np.where(kind == 1, m.nuc_len.astype(np.int64) - 1, -size_mod)).astype(np.uint64)
    off = (m.nuc_off + (kind == 1)).astype(np.uint64)                # an insertion's payload follows its anchor base
    return kind, np.ascontiguousarray(m.new_pos, dtype=np.uint64), size, off, m.pool.tobytes()


def hapset_from_muts(ref: "RefGenomeH", haps, which=None):
    """A reference HapSet holding haplotypes `which` (default: all) of a jackalope_b200 Haplotypes object."""
    which = list(range(haps.n_haps())) if which is None else list(which)
    hs = HapSetH(ref, [haps.hap_names[h] for h in which])
    for k, h in enumerate(which):
        for c, m in enumerate(haps.muts[h]):
            if m.old_pos.size:
                hs.add_edit_arrays(k, c, *muts_edit_arrays(m, len(ref.seqs[c])))
    return hs


def ref_alias_build(probs, replay=False):
    p = np.ascontiguousarray(probs, dtype=np.float64)
    P = np.zeros(p.size, dtype=np.float64)
    A = np.zeros(p.size, dtype=np.uint64)
    ref_lib(replay).jref_alias_build(_ptr(p, f64p), p.size, _ptr(P, f64p), _ptr(A, u64p))
    return P, A


def _prof_args(paired, prof1, prof2, ins_prob, del_prob):
    L = prof1[0]
    a = [L, _ptr(prof1[1], u32p), _ptr(prof1[2], f64p), _ptr(prof1[3], u8p), ins_prob[0], del_prob[0]]
    if paired:
        a += [_ptr(prof2[1], u32p), _ptr(prof2[2], f64p), _ptr(prof2[3], u8p), ins_prob[1], del_prob[1]]
    else:
        a += [None, None, None, 0.0, 0.0]
    return a


def ref_replay(obj, *, is_hap, paired, matepair, prof1, prof2, ins_prob, del_prob, barcodes,
               hap, chrom, frag_len, frag_start, script):
    """Feed `script` (uint64 draws) to the unmodified reference read model."""
    lib = ref_lib(True)
    n = len(chrom)
    L = prof1[0]
    arrs = [np.ascontiguousarray(x, dtype=np.uint64) for x in (hap, chrom, frag_len, frag_start, script)]
    consumed = np.zeros(max(n, 1), dtype=np.uint64)
    cap = n * (2 * L + 256) + 64
    o1, o2 = C.create_string_buffer(cap), C.create_string_buffer(cap)
    l1, l2 = C.c_uint64(0), C.c_uint64(0)
    err = C.create_string_buffer(512)
    rc = lib.jref_replay(obj.h, int(is_hap), int(paired), int(matepair),
                         *_prof_args(paired, prof1, prof2, ins_prob, del_prob),
                         _strs(barcodes), n, *[_ptr(a, u64p) for a in arrs[:4]],
                         _ptr(arrs[4], u64p), arrs[4].size, _ptr(consumed, u64p),
                         o1, cap, C.byref(l1), o2, cap, C.byref(l2), err, 512)
    if rc != 0:
        raise RuntimeError("jref_replay: " + err.value.decode())
    return dict(r1=o1.raw[:l1.value], r2=o2.raw[:l2.value], consumed=consumed[:n])


def ref_illumina_ref(genome: RefGenomeH, *, paired, matepair, out_prefix, n_reads, prob_dup, n_threads,
                     read_pool_size, shape, scale, frag_len_min, frag_len_max, prof1, prof2, ins_prob,
                     del_prob, barcode="", r_seed=1):
    lib = ref_lib(False)
    lib.jref_set_r_seed(r_seed)
    err = C.create_string_buffer(512)
    rc = lib.jref_illumina_ref(genome.h, int(paired), int(matepair), out_prefix.encode(), n_reads, prob_dup,
                               n_threads, read_pool_size, shape, scale, frag_len_min, frag_len_max,
                               *_prof_args(paired, prof1, prof2, ins_prob, del_prob),
                               barcode.encode(), err, 512)
    if rc != 0:
        raise RuntimeError("illumina_ref_cpp: " + err.value.decode())


def ref_illumina_hap(hs: HapSetH, *, paired, matepair, out_prefix, sep_files, n_reads, prob_dup, n_threads,
                     read_pool_size, hap_probs, shape, scale, frag_len_min, frag_len_max, prof1, prof2,
                     ins_prob, del_prob, barcodes=None, r_seed=1):
    lib = ref_lib(False)
    lib.jref_set_r_seed(r_seed)
    err = C.create_string_buffer(512)
    hp = np.ascontiguousarray(hap_probs, dtype=np.float64)
    bcs = _strs(barcodes if barcodes is not None else [""] * len(hs.hap_names))
    rc = lib.jref_illumina_hap(hs.h, int(paired), int(matepair), out_prefix.encode(), int(sep_files), n_reads,
                               prob_dup, n_threads, read_pool_size, _ptr(hp, f64p), shape, scale,
                               frag_len_min, frag_len_max,
                               *_prof_args(paired, prof1, prof2, ins_prob, del_prob), bcs, err, 512)
    if rc != 0:
        raise RuntimeError("illumina_hap_cpp: " + err.value.decode())


# ------------------------------------------------- Rcpp glue link harness ---
# oracle/_ref/libjlp_glue.so = integration/*.cpp + the stock RcppExports wrappers + oracle/glue_driver.cpp,
# linked with jackalope_b200/libjlp_b200.so (oracle/Makefile).  Calls go wrapper -> glue -> C ABI -> CUDA.

GLUE_SYMBOLS = ["_jackalope_illumina_ref_cpp", "_jackalope_illumina_hap_cpp", "_jackalope_pacbio_ref_cpp",
                "_jackalope_pacbio_hap_cpp"]


def have_glue():
    return os.path.exists(os.path.join(HERE, "_ref", "libjlp_glue.so"))


_glue = None


def glue_lib():
    global _glue
    if _glue is None:
        lib = C.CDLL(os.path.join(HERE, "_ref", "libjlp_glue.so"))
        lib.jglue_genome_new.restype = C.c_void_p
        lib.jglue_genome_new.argtypes = [C.c_uint64, C.POINTER(C.c_char_p), u64p, C.POINTER(C.c_char_p)]
        lib.jglue_genome_free.argtypes = [C.c_void_p]
        lib.jglue_hapset_new.restype = C.c_void_p
        lib.jglue_hapset_new.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p)]
        lib.jglue_hapset_free.argtypes = [C.c_void_p]
        lib.jglue_add_edits.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, u8p, u64p, u64p, u64p, C.c_char_p]
        lib.jglue_hap_chrom_size.restype = C.c_uint64
        lib.jglue_hap_chrom_size.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        lib.jglue_set_r_seed.argtypes = [C.c_uint64]
        lib.jglue_seed_after.restype = C.c_uint64
        lib.jglue_seed_after.argtypes = [C.c_uint64]
        prof = [C.c_uint64, u32p, f64p, u8p, C.c_double, C.c_double, u32p, f64p, u8p, C.c_double, C.c_double]
        lib.jglue_illumina_ref.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_uint64, C.c_double,
                                           C.c_uint64, C.c_uint64, C.c_double, C.c_double, C.c_uint64, C.c_uint64] + prof + \
            [C.c_char_p, C.c_char_p, C.c_uint64]
        lib.jglue_illumina_hap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_uint64,
                                           C.c_double, C.c_uint64, C.c_uint64, f64p, C.c_double, C.c_double, C.c_uint64,
                                           C.c_uint64] + prof + [C.POINTER(C.c_char_p), C.c_char_p, C.c_uint64]
        lib.jglue_pacbio_ref.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_double] * 5 + \
            [C.c_uint64, f64p, f64p, f64p, f64p] + [C.c_double] * 4 + [C.c_char_p, C.c_uint64]
        _glue = lib
    return _glue


class GlueGenome:
    """A jackalope RefGenome living inside libjlp_glue.so (what R holds behind the ref_genome XPtr)."""

    def __init__(self, names, seqs):
        self.lib = glue_lib()
        self.seqs = [bytes(s) for s in seqs]
        lens = np.array([len(s) for s in self.seqs], dtype=np.uint64)
        self.h = self.lib.jglue_genome_new(len(self.seqs), _strs(self.seqs), _ptr(lens, u64p), _strs(list(names)))

    def __del__(self):
        try:
            self.lib.jglue_genome_free(self.h)
        except Exception:
            pass


def edits_arrays(edits):
    """[(kind, pos, payload)] -> (kind u8[], pos u64[], size u64[], pay_off u64[], payload bytes)"""
    n = len(edits)
    kind, pos, size, off = np.zeros(n, np.uint8), np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    pay = bytearray()
    for i, (k, p, x) in enumerate(edits):
        pos[i] = p
        if k == "del":
            kind[i], size[i] = 2, x
        else:
            kind[i] = 0 if k == "sub" else 1
            off[i], size[i] = len(pay), len(x)
            pay += x
    return kind, pos, size, off, bytes(pay)


class GlueHapSet:
    """A jackalope HapSet inside libjlp_glue.so, edited through the reference's own HapChrom::add_*."""

    def __init__(self, ref: GlueGenome, hap_names, edits):
        self.lib, self.ref = ref.lib, ref
        self.h = self.lib.jglue_hapset_new(ref.h, len(hap_names), _strs(list(hap_names)))
        for h, eh in enumerate(edits):
            for c, ec in enumerate(eh):
                if ec:
                    kind, pos, size, off, pay = edits_arrays(ec)
                    assert self.lib.jglue_add_edits(self.h, h, c, len(ec), _ptr(kind, u8p), _ptr(pos, u64p), _ptr(size, u64p),
                                                    _ptr(off, u64p), pay) == 0

    def __del__(self):
        try:
            self.lib.jglue_hapset_free(self.h)
        except Exception:
            pass


def glue_illumina(obj, *, paired, matepair, out_prefix, n_reads, prof1, prof2, r_seed, sep_files=False, compress=0,
                  comp_method="bgzip", prob_dup=0.02, n_threads=1, read_pool_size=1000, hap_probs=None, shape=16.0, scale=25.0,
                  frag_len_min=None, frag_len_max=2 ** 32 - 1, ins_prob=(0.00009, 0.00015), del_prob=(0.00011, 0.00023),
                  barcodes=None):
    """.Call("_jackalope_illumina_{ref,hap}_cpp", ...) through the stock wrappers and the glue.  Returns the run seed
    the glue drew from the (stub) R RNG seeded with `r_seed`; raises RuntimeError with R's error text."""
    lib = glue_lib()
    seed = lib.jglue_seed_after(r_seed)
    lib.jglue_set_r_seed(r_seed)
    err = C.create_string_buffer(1024)
    L = prof1[0]
    fmin = L if frag_len_min is None else frag_len_min
    pa = _prof_args(paired, prof1, prof2, ins_prob, del_prob)
    if isinstance(obj, GlueHapSet):
        hp = np.ascontiguousarray(hap_probs, dtype=np.float64)
        bcs = _strs(barcodes) if barcodes is not None else None
        rc = lib.jglue_illumina_hap(obj.h, int(paired), int(matepair), out_prefix.encode(), int(sep_files), compress,
                                    comp_method.encode(), n_reads, prob_dup, n_threads, read_pool_size, _ptr(hp, f64p), shape,
                                    scale, fmin, frag_len_max, *pa, bcs, err, 1024)
    else:
        rc = lib.jglue_illumina_ref(obj.h, int(paired), int(matepair), out_prefix.encode(), compress, comp_method.encode(),
                                    n_reads, prob_dup, n_threads, read_pool_size, shape, scale, fmin, frag_len_max, *pa,
                                    (barcodes[0] if barcodes else "").encode(), err, 1024)
    if rc != 0:
        raise RuntimeError(err.value.decode(errors="replace"))
    return seed
