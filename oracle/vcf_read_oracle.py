"""TEST INFRASTRUCTURE ONLY -- haplotypes read from a VCF file, written straight from the rules of DESIGN.md section 12 in
pure Python (no CUDA, nothing shared with the library's code).

read(text, names, seqs) gives the haplotypes' names and, per (haplotype, chromosome), the records in the layout
jlp_get_haplotype_muts returns (old_pos, new_pos, nuc_off, size_modifier, pool bytes, chromosome size), plus the call's
counts; a malformed file raises VcfError with the 1-based file line and the reason.

Importable from tests/ and tools/ only; nothing under jackalope_b200/ imports this.
"""
from __future__ import annotations

import gzip

# the reasons, in the order the checks of one line are made: a line's reason is the first that fails
COLUMNS = "the number of columns differs from the #CHROM line"
CHROM = "CHROM is not a reference chromosome"
POS = "POS is not an integer >= 1"
REF_LETTERS = "REF is not letters"
REF_RANGE = "REF reaches past the end of the chromosome"
REF_DIFF = "REF differs from the reference"
ALT = "ALT is not '.' or a list of letters, '*', or symbolic or breakend alleles"
FORMAT = "FORMAT does not start with GT"
GT = "GT is not alleles separated by '|' or '/'"
PLOIDY = "GT has more than 8 alleles"
INDEX = "an allele index is above the ALT count"
CONTIG = "the lines of a chromosome are not contiguous"
ORDER = "POS decreases"
# header
NO_HEADER = "no #CHROM line before the data"
HEADER = "the #CHROM line needs 10 or more columns, FORMAT the 9th"
SAMPLE = "sample names must be unique and contain no whitespace"

MAX_PLOIDY = 8
MAX_HAPS = 1 << 16


class VcfError(Exception):
    def __init__(self, line, reason):
        super().__init__("line %d: %s" % (line, reason))
        self.line, self.reason = line, reason


def text_of(raw: bytes) -> bytes:
    """The file's text: gzip (and BGZF, a gzip file of many members) is inflated, anything else is taken as it is."""
    return gzip.decompress(raw) if raw[:2] == b"\x1f\x8b" else raw


def _letters(b):
    return len(b) > 0 and b.isalpha() and b.isascii()


def _alt(entry, info):
    """('seq', bytes) for letters and the empty <DEL>, ('ref',) for '*', ('sym',) for other symbolic / breakend alleles,
    None if malformed."""
    if _letters(entry):
        return ("seq", entry)
    if entry == b"*":
        return ("ref",)
    if entry == b"<DEL>":
        keys = {kv.split(b"=", 1)[0] for kv in info.split(b";")} if info != b"." else set()
        return ("sym",) if (b"END" in keys or b"SVLEN" in keys) else ("seq", b"")
    if len(entry) >= 3 and entry[:1] == b"<" and entry[-1:] == b">":
        return ("sym",)
    if b"[" in entry or b"]" in entry:
        return ("sym",)
    return None


def _gt(field):
    """The allele list of a sample field (None = '.'), or a reason."""
    gt = field.split(b":", 1)[0]
    out = []
    for a in gt.replace(b"/", b"|").split(b"|"):
        if a == b".":
            out.append(None)
        elif a.isdigit() and a.isascii():
            out.append(int(a))
        else:
            return GT
    if len(out) > MAX_PLOIDY:
        return PLOIDY
    return out


def encode(R: bytes, s, m, A: bytes):
    """The records of one call replacing R[s, s+m) by A: (old_pos, size_modifier, pool bytes) in old_pos order."""
    n = len(A)
    recs = []
    for i in range(min(m, n)):
        if n > m and i == m - 1:
            break
        if A[i:i + 1].upper() != R[s + i:s + i + 1].upper():
            recs.append((s + i, 0, A[i:i + 1]))
    if n > m:
        first = A[m - 1:m]
        if first.upper() == R[s + m - 1:s + m].upper():
            first = R[s + m - 1:s + m]
        recs.append((s + m - 1, n - m, first + A[m:]))
    elif m > n:
        recs.append((s + n, n - m, b""))
    return recs


def read(text: bytes, names, seqs):
    """The haplotypes of a VCF text over the reference (chromosome names, sequences as bytes)."""
    chrom_of = {n: i for i, n in enumerate(names)}
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    k = 0
    while k < len(lines) and lines[k].startswith(b"##"):
        k += 1
    if k == len(lines) or not lines[k].startswith(b"#CHROM"):
        raise VcfError(k + 1, NO_HEADER)
    head = (lines[k][:-1] if lines[k].endswith(b"\r") else lines[k]).split(b"\t")
    if len(head) < 10 or head[8] != b"FORMAT":
        raise VcfError(k + 1, HEADER)
    samples = head[9:]
    if len(set(samples)) != len(samples) or any(not s or any(ch in b" \t\r\n\v\f" for ch in s) for s in samples):
        raise VcfError(k + 1, SAMPLE)
    S = len(samples)
    if S > MAX_HAPS:
        raise VcfError(k + 1, "more than 65536 haplotypes")
    stats = dict(lines=0, samples=S, calls=0, records=0, overlaps_skipped=0, symbolic_calls=0, missing_calls=0)
    ploidy = [0] * S
    calls = {}                 # (sample, copy, chrom) -> [(s, m, allele bytes)] in file order
    seen, prev = set(), None   # chromosomes whose lines have ended; (chrom, pos) of the line before
    for li in range(k + 1, len(lines)):
        ln = lines[li][:-1] if lines[li].endswith(b"\r") else lines[li]
        no = li + 1

        def bad(reason):
            raise VcfError(no, reason)
        f = ln.split(b"\t")
        if len(f) != len(head):
            bad(COLUMNS)
        c = chrom_of.get(f[0].decode("latin-1"))
        if c is None:
            bad(CHROM)
        if not (f[1].isdigit() and f[1].isascii() and len(f[1]) <= 10 and 1 <= int(f[1]) < 1 << 32):
            bad(POS)
        s = int(f[1]) - 1
        ref = f[3]
        if not _letters(ref):
            bad(REF_LETTERS)
        m = len(ref)
        R = seqs[c]
        if s + m > len(R):
            bad(REF_RANGE)
        if ref.upper() != R[s:s + m].upper():
            bad(REF_DIFF)
        alts = [] if f[4] == b"." else [_alt(e, f[7]) for e in f[4].split(b",")]
        if any(a is None for a in alts):
            bad(ALT)
        if not (f[8] == b"GT" or f[8].startswith(b"GT:")):
            bad(FORMAT)
        gts = [_gt(x) for x in f[9:]]
        for reason in (GT, PLOIDY):
            if any(g == reason for g in gts):
                bad(reason)
        if any(a is not None and a > len(alts) for g in gts for a in g):
            bad(INDEX)
        if prev is not None and prev[0] != c:
            seen.add(prev[0])
        if c in seen:
            bad(CONTIG)
        if prev is not None and prev[0] == c and s < prev[1]:
            bad(ORDER)
        prev = (c, s)
        stats["lines"] += 1
        for si, g in enumerate(gts):
            ploidy[si] = max(ploidy[si], len(g))
            for cp, a in enumerate(g):
                if a is None:
                    stats["missing_calls"] += 1
                elif a > 0:
                    kind = alts[a - 1]
                    if kind[0] == "sym":
                        stats["symbolic_calls"] += 1
                    elif kind[0] == "seq":
                        calls.setdefault((si, cp, c), []).append((s, m, kind[1]))
    ploidy = [max(1, p) for p in ploidy]
    hap_names, slots = [], []
    for si, nm in enumerate(samples):
        for cp in range(ploidy[si]):
            hap_names.append(nm.decode("latin-1") if ploidy[si] == 1 else "%s__%d" % (nm.decode("latin-1"), cp + 1))
            slots.append((si, cp))
    if len(hap_names) > MAX_HAPS:
        raise VcfError(0, "more than 65536 haplotypes")
    stats["haplotypes"] = len(hap_names)
    recs = []
    for si, cp in slots:
        row = []
        for c, R in enumerate(seqs):
            end, out = 0, []
            for s, m, A in calls.get((si, cp, c), []):
                if s < end:
                    stats["overlaps_skipped"] += 1
                    continue
                end = s + m
                stats["calls"] += 1
                out += encode(R, s, m, A)
            row.append(_pack(out, len(R)))
            stats["records"] += len(out)
        recs.append(row)
    return hap_names, recs, stats


def _pack(out, L):
    op, npos, no, sm, pool, shift = [], [], [], [], b"", 0
    for p, d, b in out:
        op.append(p); npos.append(p + shift); no.append(len(pool)); sm.append(d)
        pool += b
        shift += d
    return dict(old_pos=op, new_pos=npos, nuc_off=no, size_modifier=sm, pool=pool, size=L + shift)


def sequence(R: bytes, rec) -> bytes:
    """A haplotype chromosome from the reference and its records (substitution, insertion and deletion records)."""
    out, at = bytearray(), 0
    for i, p in enumerate(rec["old_pos"]):
        d = rec["size_modifier"][i]
        out += R[at:p]
        no = rec["nuc_off"][i]
        if d < 0:
            at = p - d
        else:
            out += rec["pool"][no:no + d + 1]
            at = p + 1
    out += R[at:]
    assert len(out) == rec["size"]
    return bytes(out)
