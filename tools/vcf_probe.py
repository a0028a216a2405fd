"""write_vcf at two benchmark shapes: CUDA-event time of the span/line phase, the text passes and BGZF (inside
jlp_write_vcf), lines, records, text and file bytes, and the wall time of the whole Python call, plain and compressed
(level 6, the device coder), to files on tmpfs; after a warm-up call per shape and variant.  The haplotypes come from
create_haplotypes (TN93 with Gamma, haps_theta(0.001)), substitutions only and with indels(0.1 mu_bar) insertions and
deletions.  At the small shape the oracle's time (pure Python) is recorded for scale.

    python tools/vcf_probe.py [--out profiles/r05_vcf_probe.json] [--reps 2] [--dir /dev/shm] [--small]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jackalope_b200 as J  # noqa: E402
from mutate_probe import device_info  # noqa: E402


def calls(ctx, haps, d, reps, compress):
    out = []
    prefix = os.path.join(d, "vcf_probe")
    J.write_vcf(haps, prefix, compress=compress, overwrite=True, ctx=ctx)            # warm-up
    for _ in range(reps):
        t0 = time.perf_counter()
        st = J.write_vcf(haps, prefix, compress=compress, overwrite=True, ctx=ctx)
        st["wall_s"] = time.perf_counter() - t0
        st["host_ms"] = st["total_ms"] - st["span_ms"] - st["text_ms"] - st["bgzf_ms"]
        out.append(st)
    for ext in (".vcf", ".vcf.gz"):
        if os.path.exists(prefix + ext):
            os.remove(prefix + ext)
    return out


def shape(ctx, name, n_chroms, chrom_len, n_haps, reps, d, with_oracle):
    g = J.create_genome(n_chroms, chrom_len, seed=1, ctx=ctx)
    sub = J.sub_TN93((0.25, 0.25, 0.25, 0.25), 2.0, 2.0, 1.0, gamma_shape=0.5, gamma_k=5)
    info = J.haps_theta(0.001, n_haps)
    m = J.indels(0.1 * sub.mu_bar())
    res = dict(shape=name, n_chroms=n_chroms, chrom_len=chrom_len, n_haps=n_haps, theta=0.001,
               model="TN93 (alpha_1 = alpha_2 = 2, beta = 1, uniform pi), gamma_shape 0.5, gamma_k 5", variants=[])
    for label, kw in (("substitutions only", {}), ("indels(0.1 mu_bar) each", dict(ins=m, del_=m, epsilon=0.03))):
        haps = J.create_haplotypes(g, info, sub, seed=7, ctx=ctx, **kw)
        v = dict(variant=label, records=haps.stats["records"])
        for key, compress in (("plain", False), ("bgzf_level6", 6)):
            try:
                v[key] = calls(ctx, haps, d, reps, compress)
            except Exception as e:                                  # e.g. the file system is full: recorded, not fatal
                v[key] = dict(error=str(e))
        if with_oracle and not kw:
            from oracle import vcf_oracle as V
            t0 = time.perf_counter()
            V.vcf(haps)
            v["oracle_s"] = time.perf_counter() - t0
        res["variants"].append(v)
        del haps
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_vcf_probe.json"))
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir())
    ap.add_argument("--small", action="store_true", help="tiny shapes (rehearsal)")
    a = ap.parse_args()
    d = tempfile.mkdtemp(dir=a.dir)
    ctx = J.Context(0)
    res = device_info()
    res["output_dir_free_bytes"] = shutil.disk_usage(d).free
    if a.small:
        shapes = [("small", 2, 100_000, 8, 1, True)]
    else:
        shapes = [("configs[1]: 8 haplotypes, 10 x 1 Mb", 10, 1_000_000, 8, a.reps, True),
                  ("configs[3]: 96 haplotypes, 20 x 25 Mb", 20, 25_000_000, 96, a.reps, False)]
    try:
        res["shapes"] = [shape(ctx, *s[:4], reps=s[4], d=d, with_oracle=s[5]) for s in shapes]
    finally:
        ctx.close()
        shutil.rmtree(d, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
