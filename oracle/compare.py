"""TEST INFRASTRUCTURE ONLY -- run the CPU oracle on exactly the inputs a product
run uses (same seed, same group counts, same fragment table) and compare.

Used by tests/, __graft_entry__.smoke() and bench.py's checker legs; nothing
under jackalope_b200/ imports this.  Needs no GPU: the apportioning and the
fragment-length table come from the host-only entry points of the C ABI."""
import ctypes as C

import numpy as np

import jackalope_b200 as J
from jackalope_b200 import _lib
from jackalope_b200.illumina import _prepare
from oracle import harness as H

DEFAULTS = dict(frag_mean=400, frag_sd=100, matepair=False, seq_sys=None, profile1=None, profile2=None,
                ins_prob1=0.00009, del_prob1=0.00011, ins_prob2=0.00015, del_prob2=0.00023, frag_len_min=None,
                frag_len_max=None, haplotype_probs=None, barcodes=None, prob_dup=0.02, sep_files=False,
                compress=False, comp_method="bgzip", n_threads=1, read_pool_size=1000, show_progress=False,
                overwrite=True)


def frag_table(shape, scale, fmin, fmax):
    lib = _lib.lib()
    n = C.c_uint64()
    lib.jlp_frag_table(shape, scale, fmin, fmax, None, 0, C.byref(n))
    cdf = np.zeros(max(n.value, 1), dtype=np.uint64)
    assert lib.jlp_frag_table(shape, scale, fmin, fmax, cdf.ctypes.data_as(_lib.u64p), n.value, C.byref(n)) == 0
    return cdf[:n.value]


def hap_sequences(haps: J.Haplotypes):
    """Materialise every haplotype chromosome with the oracle (get_chrom_full restatement)."""
    out = []
    for h in range(haps.n_haps()):
        row = []
        for c, m in enumerate(haps.muts[h]):
            row.append(H.materialize(haps.reference.chrom(c), m.old_pos, m.new_pos, m.nuc_off, m.pool.tobytes(),
                                     m.chrom_size))
        out.append(row)
    return out


def lazy_hap_sequences(haps: J.Haplotypes):
    """(h, c) -> bytes: one haplotype chromosome materialised with the oracle on demand (cached)."""
    cache = {}

    def get(h, c):
        if (h, c) not in cache:
            m = haps.muts[h][c]
            cache[(h, c)] = H.materialize(haps.reference.chrom(c), m.old_pos, m.new_pos, m.nuc_off, m.pool.tobytes(), m.chrom_size)
        return cache[(h, c)]
    get.cache = cache
    return get


def group_counts(p, obj, is_haps):
    """Pairs per (haplotype, chromosome) of the run `p` describes (jlp_apportion)."""
    ref = obj.reference if is_haps else obj
    nc = ref.n_chroms()
    nh = obj.n_haps() if is_haps else 1
    n_ends = 2 if p.paired else 1
    sizes = np.concatenate([obj.sizes(h) for h in range(nh)]) if is_haps else ref.sizes()
    sizes = np.ascontiguousarray(sizes, dtype=np.uint64)
    counts = np.zeros(nh * nc, dtype=np.uint64)
    rc = _lib.lib().jlp_apportion(p.seed, p.n_reads // n_ends, nh, nc, p.haplotype_probs if is_haps else None,
                                  sizes.ctypes.data_as(_lib.u64p), counts.ctypes.data_as(_lib.u64p))
    assert rc == 0
    return counts


def oracle_jobs(obj, n_reads, read_length, paired, seed, **kw):
    """Pair-index ranges [(lo, hi)] of the run's jobs (one per haplotype with sep_files, else one)."""
    return oracle_run(obj, n_reads, read_length, paired, seed, _jobs_only=True, **kw)


def oracle_run(obj, n_reads, read_length, paired, seed, lo=None, hi=None, want_ledger=False, hap_seqs=None,
               only_job=None, _jobs_only=False, **kw):
    """Oracle output for the run illumina(obj, ..., seed=seed) performs.
    Returns dict(r1, r2, fallback[, plan, ledger, ledger_cnt, groups]); with sep_files the
    jobs' outputs are concatenated in haplotype order (as sink="memory" does).
    hap_seqs: materialised haplotype chromosomes [h][c], or a callable (h, c) -> bytes asked only for the groups
    the pair range [lo, hi) can touch (runs at sizes where materialising everything on the CPU is out of reach)."""
    a = dict(DEFAULTS)
    a.update(kw)
    p, keep, (prof1, prof2), is_haps, _ = _prepare(obj, "x", n_reads, read_length, paired, a["frag_mean"],
                                                   a["frag_sd"], a["matepair"], a["seq_sys"], a["profile1"],
                                                   a["profile2"], a["ins_prob1"], a["del_prob1"], a["ins_prob2"],
                                                   a["del_prob2"], a["frag_len_min"], a["frag_len_max"],
                                                   a["haplotype_probs"], a["barcodes"], a["prob_dup"], a["sep_files"],
                                                   a["compress"], a["comp_method"], a["n_threads"],
                                                   a["read_pool_size"], a["show_progress"], True, seed, None, None,
                                                   check_files=False)
    n_ends = 2 if p.paired else 1
    ref = obj.reference if is_haps else obj
    nc = ref.n_chroms()
    nh = obj.n_haps() if is_haps else 1
    counts = group_counts(p, obj, is_haps)
    if _jobs_only:
        off = np.concatenate(([0], np.cumsum(counts))).astype(np.uint64)
        if is_haps and p.sep_files:
            return [(int(off[h * nc]), int(off[(h + 1) * nc])) for h in range(nh)]
        return [(0, int(off[-1]))]
    off_all = np.concatenate(([0], np.cumsum(counts))).astype(np.uint64)
    pool_pairs = (p.read_pool_size + n_ends - 1) // n_ends
    if is_haps and p.sep_files:
        jobs = [(int(off_all[h * nc]), int(off_all[(h + 1) * nc])) for h in range(nh)]
    else:
        jobs = [(0, int(off_all[-1]))]
    lens = None
    if is_haps and callable(hap_seqs):
        # lazy: materialise only the (haplotype, chromosome) groups the requested pairs -- and the leaders of
        # their duplicate chains, at most pool_pairs - 1 pairs earlier in the same job -- can touch
        touched = set()
        for (jl, jh) in jobs:
            if only_job is not None and (jl, jh) != tuple(only_job):
                continue
            a_lo, a_hi = (jl if lo is None else max(jl, lo)), (jh if hi is None else min(jh, hi))
            if a_hi <= a_lo:
                continue
            first = max(jl, a_lo - min(a_lo - jl, pool_pairs - 1))
            g0 = int(np.searchsorted(off_all, first, side="right")) - 1
            g1 = int(np.searchsorted(off_all, a_hi - 1, side="right")) - 1
            touched.update(range(g0, g1 + 1))
        seqs = [hap_seqs(g // nc, g % nc) if g in touched else b"" for g in range(nh * nc)]
        lens = [obj.muts[h][c].chrom_size for h in range(nh) for c in range(nc)]
        gnames = [obj.hap_names[h] for h in range(nh) for c in range(nc)]
        cnames = [ref.names[c] for h in range(nh) for c in range(nc)]
        bcs = [p.barcodes[h].decode() for h in range(nh) for c in range(nc)]
    elif is_haps:
        hap_seqs = hap_seqs or hap_sequences(obj)
        seqs = [hap_seqs[h][c] for h in range(nh) for c in range(nc)]
        gnames = [obj.hap_names[h] for h in range(nh) for c in range(nc)]
        cnames = [ref.names[c] for h in range(nh) for c in range(nc)]
        bcs = [p.barcodes[h].decode() for h in range(nh) for c in range(nc)]
    else:
        seqs = [ref.chrom(c) for c in range(nc)]
        gnames = [ref.name] * nc
        cnames = list(ref.names)
        bcs = [p.barcodes[0].decode()] * nc
    groups = H.Groups(counts, seqs, gnames, cnames, bcs, lens=lens)
    cdf = frag_table(p.frag_len_shape, p.frag_len_scale, p.frag_len_min, p.frag_len_max)
    res = dict(r1=b"", r2=b"", groups=groups, jobs=jobs, params=p, profiles=(prof1, prof2), n_chroms=nc,
               fallback=dict.fromkeys(H.FALLBACK_KINDS, 0))
    for (jl, jh) in jobs:
        if only_job is not None and (jl, jh) != tuple(only_job):
            continue
        a_lo = jl if lo is None else max(jl, lo)
        a_hi = jh if hi is None else min(jh, hi)
        if a_hi <= a_lo:
            continue
        r = H.generate(seed=p.seed, paired=bool(p.paired), matepair=bool(p.matepair), groups=groups, prof1=prof1,
                       prof2=prof2, ins_prob=[p.ins_prob1, p.ins_prob2], del_prob=[p.del_prob1, p.del_prob2],
                       prob_dup=p.prob_dup, pool_pairs=pool_pairs, frag_cdf=cdf, frag_min=p.frag_len_min,
                       lo=a_lo, hi=a_hi, job_lo=jl, job_hi=jh, want_ledger=want_ledger, want_plan=want_ledger)
        res["r1"] += r["r1"]
        res["r2"] += r["r2"]
        for k, v in r["fallback"].items():
            res["fallback"][k] += v
        if want_ledger:
            for k in ("plan", "ledger", "ledger_cnt"):
                res.setdefault(k, []).append(r[k])
    return res


def fastq_records(b: bytes):
    lines = b.split(b"\n")
    assert lines[-1] == b""
    lines = lines[:-1]
    assert len(lines) % 4 == 0
    return [tuple(lines[i:i + 4]) for i in range(0, len(lines), 4)]


def first_diff(a: bytes, b: bytes):
    n = min(len(a), len(b))
    aa, bb = np.frombuffer(a[:n], np.uint8), np.frombuffer(b[:n], np.uint8)
    d = np.nonzero(aa != bb)[0]
    if d.size == 0:
        return None if len(a) == len(b) else n
    return int(d[0])


def explain_diff(a: bytes, b: bytes, what=("got", "want")):
    """Text describing the first difference of two FASTQ byte strings: the record (4 lines) around it from both."""
    d = first_diff(a, b)
    if d is None:
        return "identical"

    def record(x):
        lo = x.rfind(b"\n@", 0, d) + 1
        hi = lo
        for _ in range(4):
            k = x.find(b"\n", hi)
            if k < 0:
                hi = len(x)
                break
            hi = k + 1
        return lo, x[lo:hi].decode(errors="replace")

    (la, ra), (lb, rb) = record(a), record(b)
    return "first difference at byte %d (record %d of %s, offset %d in it)\n%s:\n%s%s:\n%s" % (
        d, a[:la].count(b"\n") // 4, what[0], d - la, what[0], ra, what[1], rb)
