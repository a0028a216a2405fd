"""create_haplotypes along gene trees at two benchmark shapes, each with one tree per chromosome and with many: parse
time, table build, the two passes (CUDA events), windows, store time and the whole call, after a warm-up call.

The trees are ms text written here from a seed: a pool of 1000 Kingman trees from mutate.kingman() (coalescent units
scaled by theta / 2), each region drawing one tree from the pool and a length from 1..1000.  A pool keeps the probe's
own set-up (Python) short; the library still parses, schedules and builds tables for every tree line.

    python tools/gtrees_probe.py [--out profiles/r06_gtrees_probe.json] [--reps 2] [--small]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jackalope_b200 as J  # noqa: E402
from jackalope_b200.mutate import HapsGtrees, Tree, kingman  # noqa: E402


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return dict(device=name, power_limit_and_max_sm_clock=q)


def ms_text(n_chroms, n_haps, trees_per_chrom, theta, seed):
    rng = np.random.default_rng(seed)
    names = [str(i + 1) for i in range(n_haps)]
    pool = []
    for _ in range(min(1000, n_chroms * trees_per_chrom)):
        t = kingman(n_haps, rng).scaled(theta / 2)
        pool.append(Tree(t.parent, t.branch_len, t.tip_node, names).newick())
    out = ["ms %d %d -T\n%d\n" % (n_haps, n_chroms, seed)]
    for _ in range(n_chroms):
        out.append("\n//\n")
        if trees_per_chrom == 1:
            out.append(pool[int(rng.integers(len(pool)))] + "\n")
            continue
        pick = rng.integers(len(pool), size=trees_per_chrom)
        lens = rng.integers(1, 1001, size=trees_per_chrom)
        out += ["[%d]%s\n" % (n, pool[k]) for n, k in zip(lens.tolist(), pick.tolist())]
    return "".join(out), names


def run(ctx, g, name, n_chroms, n_haps, trees_per_chrom, reps):
    sub = J.sub_TN93((0.25, 0.25, 0.25, 0.25), 2.0, 2.0, 1.0, gamma_shape=0.5, gamma_k=5)
    text, names = ms_text(n_chroms, n_haps, trees_per_chrom, 0.001 / sub.mu_bar(), seed=7)
    info = HapsGtrees(text, names)
    J.create_haplotypes(g, info, sub, seed=100, ctx=ctx)                    # warm-up
    runs = []
    for r in range(reps):
        t0 = time.perf_counter()
        haps = J.create_haplotypes(g, info, sub, seed=101 + r, ctx=ctx)
        st = dict(haps.stats)
        st["wall_s"] = time.perf_counter() - t0
        runs.append(st)
        del haps
    return dict(shape=name, trees_per_chrom=trees_per_chrom, text_bytes=len(text), runs=runs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_gtrees_probe.json"))
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--small", action="store_true", help="tiny shapes (rehearsal)")
    a = ap.parse_args()
    ctx = J.Context(0)
    res = device_info()
    res["model"] = "TN93 (alpha_1 = alpha_2 = 2, beta = 1, uniform pi), gamma_shape 0.5, gamma_k 5; theta = 0.001"
    shapes = ([("small", 2, 100_000, 8, (1, 10))] if a.small else
              [("configs[1]: 8 haplotypes, 10 x 1 Mb", 10, 1_000_000, 8, (1, 100)),
               ("configs[3]: 96 haplotypes, 20 x 25 Mb", 20, 25_000_000, 96, (1, 10_000))])
    res["shapes"] = []
    for name, nc, L, nh, per in shapes:
        g = J.create_genome(nc, L, seed=1, ctx=ctx)
        for k in per:
            res["shapes"].append(run(ctx, g, name, nc, nh, k, a.reps))
            print(json.dumps(res["shapes"][-1]), flush=True)
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
