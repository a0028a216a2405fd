"""create_haplotypes(ref, haps_vcf(fn)) at three shapes: where the call's time goes (host inflate, the batches' kernels,
the chromosomes' sorts and walks, the copy into the haplotypes) and the text rate, two calls per row after a warm-up.

* configs[1] (8 haplotypes, 10 x 1 Mb) and configs[3] (96 haplotypes, 20 x 25 Mb): haplotypes from create_haplotypes
  (TN93, theta = 0.001, insertions and deletions), written by write_vcf plain and BGZF;
* a wide file: 2504 diploid samples over one 60 Mb chromosome, about 1.5e6 lines of one SNP each whose allele counts
  follow the neutral frequency spectrum (P(i) ~ 1/i), generated here in numpy from a seed (plain text: most of it is
  0|0 fields).

The library is called through the C ABI, so the Python copy of the records (create_haplotypes' Haplotypes object) is
not timed.  The Python oracle's time on configs[1] (plain) is reported beside the library's.

    python tools/vcf_read_probe.py [--out profiles/r07_vcf_read_probe.json] [--reps 2] [--small]
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jackalope_b200 as J  # noqa: E402
from jackalope_b200 import _lib  # noqa: E402
from oracle import vcf_read_oracle as O  # noqa: E402


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return dict(device=name, power_limit_and_max_sm_clock=q)


def call(ctx, path, n_threads=16):
    p = _lib.VcfReadParams(path.encode(), n_threads, 0)
    st = _lib.VcfReadStats()
    t0 = time.perf_counter()
    ctx._check(ctx.lib.jlp_create_haplotypes_vcf(ctx.h, C.byref(p), C.byref(st)), "jlp_create_haplotypes_vcf")
    d = st.as_dict()
    d["wall_s"] = time.perf_counter() - t0
    d["text_GB_per_s"] = d["text_bytes"] / d["total_ms"] / 1e6
    d["file_bytes"] = os.path.getsize(path)
    return d


def rows(ctx, name, path, reps):
    call(ctx, path)                                           # warm-up
    out = dict(shape=name, file=os.path.basename(path), runs=[call(ctx, path) for _ in range(reps)])
    ctx._haps = None
    print(json.dumps(out), flush=True)
    return out


def wide_vcf(path, g, n_samples, n_lines, seed, block=4000):
    """The wide file, written block by block."""
    rng = np.random.default_rng(seed)
    ref = g.seqs[0]
    N = 2 * n_samples
    pos = np.sort(rng.choice(ref.size, size=n_lines, replace=False))
    p = 1.0 / np.arange(1, N)
    ac = rng.choice(np.arange(1, N), size=n_lines, p=p / p.sum())
    tcag = np.frombuffer(b"TCAG", dtype=np.uint8)
    nxt = np.zeros(256, dtype=np.uint8)
    nxt[tcag] = np.roll(tcag, -1)
    head = ["##fileformat=VCFv4.3", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"]
    with open(path, "wb") as f:
        f.write(("\n".join(head) + "".join("\ts%d" % i for i in range(n_samples)) + "\n").encode())
        for b0 in range(0, n_lines, block):
            b1 = min(n_lines, b0 + block)
            B = b1 - b0
            thr = (ac[b0:b1] / N * 65536).astype(np.uint32)
            alt = rng.integers(0, 65536, size=(B, N), dtype=np.uint16) < thr[:, None]
            gt = np.empty((B, n_samples, 4), dtype=np.uint8)
            gt[:, :, 0] = ord("0") + alt[:, 0::2]
            gt[:, :, 1] = ord("|")
            gt[:, :, 2] = ord("0") + alt[:, 1::2]
            gt[:, :, 3] = ord("\t")
            gt[:, -1, 3] = ord("\n")
            gt = gt.reshape(B, -1)
            parts = []
            for i in range(B):
                x = int(pos[b0 + i])
                r = int(ref[x])
                parts.append(b"%s\t%d\t.\t%c\t%c\t.\tPASS\t.\tGT\t" % (g.names[0].encode(), x + 1, r, nxt[r] if nxt[r] else ord("A")))
                parts.append(gt[i].tobytes())
            f.write(b"".join(parts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_vcf_read_probe.json"))
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--small", action="store_true", help="tiny shapes (rehearsal)")
    a = ap.parse_args()
    ctx = J.Context(0)
    res = device_info()
    res["model"] = "TN93 (alpha_1 = alpha_2 = 2, beta = 1, uniform pi); theta = 0.001; indels(0.0001) both ways"
    res["n_threads"] = 16
    res["shapes"] = []
    tmp = tempfile.mkdtemp(prefix="vcf_read_probe_")
    try:
        sub = J.sub_TN93((0.25, 0.25, 0.25, 0.25), 2.0, 2.0, 1.0)
        shapes = ([("small", 2, 100_000, 8)] if a.small else
                  [("configs[1]: 8 haplotypes, 10 x 1 Mb", 10, 1_000_000, 8),
                   ("configs[3]: 96 haplotypes, 20 x 25 Mb", 20, 25_000_000, 96)])
        for k, (name, nc, L, nh) in enumerate(shapes):
            g = J.create_genome(nc, L, seed=1, ctx=ctx)
            haps = J.create_haplotypes(g, J.haps_theta(0.001, nh), sub, ins=J.indels(1e-4), del_=J.indels(1e-4), seed=2,
                                       ctx=ctx)
            for comp in (False, True):
                pre = os.path.join(tmp, "s%d%s" % (k, "z" if comp else ""))
                J.write_vcf(haps, pre, compress=comp, ctx=ctx, file_date="20261022", overwrite=True)
                path = pre + (".vcf.gz" if comp else ".vcf")
                res["shapes"].append(rows(ctx, name + (", BGZF" if comp else ", plain"), path, a.reps))
                if k == 0 and not comp:
                    text = open(path, "rb").read()
                    t0 = time.perf_counter()
                    O.read(text, g.names, [g.chrom(c) for c in range(g.n_chroms())])
                    res["oracle_configs1_plain_s"] = time.perf_counter() - t0
                    print(json.dumps({"oracle_configs1_plain_s": res["oracle_configs1_plain_s"]}), flush=True)
                os.remove(path)
            del haps
        n_samples, L, n_lines = (50, 1_000_000, 20_000) if a.small else (2504, 60_000_000, 1_500_000)
        need = n_lines * (4 * n_samples + 40)
        if shutil.disk_usage(tmp).free < 2 * need:
            n_lines = int(shutil.disk_usage(tmp).free / 2 / (4 * n_samples + 40))
            res["wide_lines_reduced_for_disk"] = n_lines
        g = J.create_genome(1, L, seed=3, ctx=ctx)
        path = os.path.join(tmp, "wide.vcf")
        t0 = time.perf_counter()
        wide_vcf(path, g, n_samples, n_lines, seed=4)
        res["wide_generation_s"] = time.perf_counter() - t0
        res["shapes"].append(rows(ctx, "wide: %d diploid samples, 1 x %d Mb, %d lines" % (n_samples, L // 10**6, n_lines),
                                  path, a.reps))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
