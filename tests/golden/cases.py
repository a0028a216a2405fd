"""Golden cases shared by make_golden.py (which runs the unmodified reference) and the
tests that check the oracle (CPU) and the CUDA path (GPU) against the stored bytes."""
import numpy as np

import jackalope_b200 as J


def _genome_with_n(seed, n, length):
    g = J.random_genome(n, length, seed=seed)
    s = g.seqs[0].copy()
    s[100:160] = ord("N")
    s[1000] = ord("x")
    g.seqs[0] = s
    return g


def _tiny():
    return J.RefGenome(["a", "b", "c"], [J.random_genome(1, 60, seed=5).seqs[0], J.random_genome(1, 4000, seed=6).seqs[0],
                                         J.random_genome(1, 130, seed=7).seqs[0]])


def _haps(return_edits=False):
    g = J.random_genome(3, 6000, seed=8)
    return J.random_haplotypes(g, 3, sub_rate=0.02, indel_rate=0.005, seed=9, return_edits=return_edits)


# name -> (object factory, n_reads, read_length, paired, seed, kwargs)
CASES = {
    "se100_default": (lambda: _genome_with_n(1, 3, 5000), 300, 100, False, 101, {}),
    "pe100_default": (lambda: _genome_with_n(1, 3, 5000), 400, 100, True, 102, {}),
    "mp100_default": (lambda: _genome_with_n(1, 3, 5000), 400, 100, True, 103, dict(matepair=True)),
    "pe150_hs25": (lambda: _genome_with_n(2, 4, 9000), 400, 150, True, 104, dict(seq_sys="HS25")),
    "pe100_indels_dups_barcode": (lambda: _genome_with_n(4, 3, 5000), 400, 100, True, 105,
                                  dict(ins_prob1=0.02, del_prob1=0.03, ins_prob2=0.05, del_prob2=0.01, prob_dup=0.4,
                                       read_pool_size=14, barcodes=["ACGTTG"])),
    "pe100_short_fragments": (_tiny, 400, 100, True, 106,
                              dict(frag_mean=120, frag_sd=40, frag_len_min=20, ins_prob1=0.01, del_prob1=0.01)),
    "hap_pe100_pooled": (_haps, 400, 100, True, 107, dict(haplotype_probs=[1, 2, 4], barcodes=["AC", "GT", "TT"])),
    "hap_se100_sep_files": (_haps, 300, 100, False, 108, dict(sep_files=True)),
}


def load(name):
    import os
    d = np.load(os.path.join(os.path.dirname(__file__), name + ".npz"))
    return d["r1"].tobytes(), d["r2"].tobytes(), d["counts"]


def assert_oracle_reproduces(name):
    """The oracle's run of case `name` is the reference's stored FASTQ byte for byte (pairs per group included);
    returns (r1, r2) for further checks."""
    from oracle.compare import oracle_run
    make, n_reads, L, paired, seed, kw = CASES[name]
    r1, r2, counts = load(name)
    o = oracle_run(make(), n_reads, L, paired, seed, **kw)
    assert np.array_equal(o["groups"].counts, counts)
    assert o["r1"] == r1 and o["r2"] == r2
    return r1, r2
