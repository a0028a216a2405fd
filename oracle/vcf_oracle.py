"""TEST INFRASTRUCTURE ONLY -- the VCF of a set of haplotypes, written straight from the definitions of DESIGN.md
section 11 in pure Python and numpy (no CUDA, nothing shared with the library's code).

Importable from tests/ and tools/ only; nothing under jackalope_b200/ imports this.
"""
from __future__ import annotations

import numpy as np


def size_modifiers(m, ref_size):
    """size_modifier per record, derived from neighbouring records as jlp_add_haplotype does."""
    op = m.old_pos.astype(np.int64)
    np_ = m.new_pos.astype(np.int64)
    M = op.size
    sm = np.zeros(M, dtype=np.int64)
    for i in range(M):
        s = (np_[i + 1] - op[i + 1]) if i + 1 < M else (m.chrom_size - ref_size)
        sm[i] = s + op[i] - np_[i]
    return sm


def _records(m, ref_size):
    """(op, consumed length, contributed bytes, span start, span end) per record."""
    sm = size_modifiers(m, ref_size)
    pool = m.pool.tobytes()
    out = []
    for i in range(m.old_pos.size):
        op, s, no = int(m.old_pos[i]), int(sm[i]), int(m.nuc_off[i])
        clen = max(1, -s)
        b = pool[no:no + max(0, s + 1)]
        if s < 0:
            lo, hi = (op - 1, op - s) if op > 0 else (0, min(ref_size, 1 - s))
        else:
            lo, hi = op, op + clen
        out.append((op, clen, b, lo, hi))
    return out


def _allele(R, recs, s, e):
    """The allele over [s, e) of a haplotype whose records touching the line are `recs`."""
    at = {op: b for op, _, b, _, _ in recs}
    inside = set()
    for op, clen, _, _, _ in recs:
        inside.update(range(op + 1, op + clen))
    out = bytearray()
    for r in range(s, e):
        if r in at:
            out += at[r]
        elif r not in inside:
            out.append(R[r])
    return bytes(out)


def header(chrom_names, chrom_lens, sample_names, file_date):
    h = ["##fileformat=VCFv4.3", "##fileDate=%s" % file_date, "##source=jackalope_b200"]
    h += ["##contig=<ID=%s,length=%d>" % (n, l) for n, l in zip(chrom_names, chrom_lens)]
    h += ['##ALT=<ID=DEL,Description="The haplotype has no bases over this line">',
          '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
          "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + list(sample_names))]
    return ("\n".join(h) + "\n").encode()


def lines(R: bytes, chrom_name, muts_by_hap, sample_matrix):
    """(s, e, alleles by haplotype, line text) of every written line of one chromosome; muts_by_hap[h] is a
    HapChromMuts or None for a haplotype not in the sample matrix."""
    S = np.asarray(sample_matrix, dtype=np.int64)
    inc = sorted(set(S.reshape(-1).tolist()))
    spans = []                                   # haplotype-major, then record order: the ties' order
    recs = {}
    for h in inc:
        recs[h] = _records(muts_by_hap[h], len(R))
        for k, r in enumerate(recs[h]):
            spans.append((r[3], r[4], h, k))
    spans.sort(key=lambda t: t[0])              # stable
    groups, cur, cur_end = [], [], -1
    for sp in spans:
        if cur and sp[0] >= cur_end:
            groups.append(cur)
            cur, cur_end = [], -1
        cur.append(sp)
        cur_end = max(cur_end, sp[1])
    if cur:
        groups.append(cur)
    out = []
    for g in groups:
        s, e = g[0][0], max(sp[1] for sp in g)
        by_hap = {}
        for _, _, h, k in g:
            by_hap.setdefault(h, []).append(recs[h][k])
        ref = R[s:e]
        alleles = {h: (_allele(R, by_hap[h], s, e) if h in by_hap else ref) for h in inc}
        alts = []
        for h in S.reshape(-1).tolist():
            a = alleles[h]
            if a != ref and a not in alts:
                alts.append(a)
        if not alts:
            continue
        idx = {h: (0 if alleles[h] == ref else 1 + alts.index(alleles[h])) for h in inc}
        gts = ["|".join(str(idx[h]) for h in row) for row in S.tolist()]
        txt = b"\t".join([chrom_name.encode(), str(s + 1).encode(), b".", ref,
                          b",".join(a if a else b"<DEL>" for a in alts), b".", b"PASS", b".", b"GT"] +
                         [x.encode() for x in gts]) + b"\n"
        out.append((s, e, alleles, txt))
    return out


def vcf(haps, sample_matrix=None, sample_names=None, file_date="20000101"):
    """The VCF text of a jackalope_b200 Haplotypes object: sample_matrix (n_samples x ploidy haplotype indices) None
    means one haploid sample per haplotype named by the haplotype."""
    ref = haps.reference
    if sample_matrix is None:
        sample_matrix = np.arange(haps.n_haps()).reshape(-1, 1)
        sample_names = list(haps.hap_names) if sample_names is None else sample_names
    S = np.asarray(sample_matrix, dtype=np.int64)
    if sample_names is None:
        sample_names = ["sample%d" % (i + 1) for i in range(S.shape[0])]
    parts = [header(ref.names, [s.size for s in ref.seqs], sample_names, file_date)]
    for c in range(ref.n_chroms()):
        R = ref.chrom(c)
        mb = [haps.muts[h][c] for h in range(haps.n_haps())]
        parts += [t for _, _, _, t in lines(R, ref.names[c], mb, S)]
    return b"".join(parts)


def apply(vcf_text: bytes, reference, slot):
    """Per chromosome name, the sequence the VCF gives sample slot `slot` (sample i, copy k: slot i * ploidy + k):
    each written line's REF replaced by the allele its GT names (<DEL> = nothing)."""
    seqs = {n: bytearray() for n in reference.names}
    pos = {n: 0 for n in reference.names}
    ref = {n: reference.chrom(i) for i, n in enumerate(reference.names)}
    for ln in vcf_text.split(b"\n"):
        if not ln or ln.startswith(b"#"):
            continue
        f = ln.split(b"\t")
        name, p, r, alts = f[0].decode(), int(f[1]) - 1, f[3], f[4].split(b",")
        gts = [g for x in f[9:] for g in x.split(b"|")]
        a = int(gts[slot])
        allele = r if a == 0 else (b"" if alts[a - 1] == b"<DEL>" else alts[a - 1])
        assert p >= pos[name] and ref[name][p:p + len(r)] == r
        seqs[name] += ref[name][pos[name]:p] + allele
        pos[name] = p + len(r)
    for n in reference.names:
        seqs[n] += ref[n][pos[n]:]
    return {n: bytes(v) for n, v in seqs.items()}
