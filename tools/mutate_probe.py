"""create_haplotypes at two benchmark shapes: kernel time per pass (CUDA events inside jlp_create_haplotypes, after a
warm-up call), records and bytes copied to the host, wall time of the call, table sizes, and the wall time of
random_haplotypes for the same shape on the same host (the input generator the benchmark used so far).  Each shape runs
substitutions only and then with insertions and deletions (ins = del_ = indels(0.1 mu_bar)); the indel rows add the
host event pass (event_ms) to the kernel passes (count_ms, scan_ms, write_ms: pass 2 and the inserted columns' walk)
and the store copy (store_ms).

    python tools/mutate_probe.py [--out profiles/r04_mutate_probe.json] [--reps 3] [--small]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jackalope_b200 as J  # noqa: E402


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return dict(device=name, power_limit_and_max_sm_clock=q)


def shape(ctx, name, n_chroms, chrom_len, n_haps, theta, reps, sub_rate):
    g = J.create_genome(n_chroms, chrom_len, seed=1, ctx=ctx)
    sub = J.sub_TN93((0.25, 0.25, 0.25, 0.25), 2.0, 2.0, 1.0, gamma_shape=0.5, gamma_k=5)
    info = J.haps_theta(theta, n_haps)
    out = [one(ctx, g, sub, info, n_haps, reps, {}), one(ctx, g, sub, info, n_haps, reps, indel_kw(sub))]
    t0 = time.perf_counter()
    rh = J.random_haplotypes(g, n_haps, sub_rate=sub_rate, indel_rate=0.0, seed=5)
    rh_wall = time.perf_counter() - t0
    rh_records = sum(m.old_pos.size for hm in rh.muts for m in hm)
    del rh
    return dict(shape=name, n_chroms=n_chroms, chrom_len=chrom_len, n_haps=n_haps, theta=theta,
                model="TN93 (alpha_1 = alpha_2 = 2, beta = 1, uniform pi), gamma_shape 0.5, gamma_k 5",
                substitutions_only=out[0], indels=dict(ins_del="indels(0.1 * mu_bar) each", **out[1]),
                random_haplotypes=dict(sub_rate=sub_rate, indel_rate=0.0, wall_s=rh_wall, records=rh_records))


def indel_kw(sub):
    m = J.indels(0.1 * sub.mu_bar())
    return dict(ins=m, del_=m, epsilon=0.03)


def one(ctx, g, sub, info, n_haps, reps, kw):
    J.create_haplotypes(g, info, sub, seed=100, ctx=ctx, **kw)              # warm-up
    runs = []
    for r in range(reps):
        t0 = time.perf_counter()
        haps = J.create_haplotypes(g, info, sub, seed=101 + r, ctx=ctx, **kw)
        wall = time.perf_counter() - t0
        st = dict(haps.stats)
        st["wall_s"] = wall
        st["records_per_hap_mean"] = st["records"] / n_haps
        runs.append(st)
        del haps
    return dict(runs=runs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_mutate_probe.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--small", action="store_true", help="tiny shapes (rehearsal)")
    a = ap.parse_args()
    ctx = J.Context(0)
    res = device_info()
    if a.small:
        shapes = [("small", 2, 100_000, 8, 0.001, 2, 0.001)]
    else:
        shapes = [("configs[1]: 8 haplotypes, 10 x 1 Mb", 10, 1_000_000, 8, 0.001, a.reps, 0.001),
                  ("configs[3]: 96 haplotypes, 20 x 25 Mb", 20, 25_000_000, 96, 0.001, a.reps, 0.001)]
    res["shapes"] = [shape(ctx, *s[:5], reps=s[5], sub_rate=s[6]) for s in shapes]
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
