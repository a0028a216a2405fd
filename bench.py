#!/usr/bin/env python3
"""Benchmark of the Illumina read-generation hot path (BASELINE.json metric:
Illumina PE150 read pairs/s, HS25).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload ("human_pe150_hs25", BASELINE.json configs[4] / SURVEY.md section 8d config 5):
synthetic 3.1 Gb genome (24 chromosomes with human-like length spread, uniform TCAG),
PE150, HS25 profile (HiSeq2500L150R{1,2}filter), all other illumina() arguments at the
reference's defaults.  The full job is 30x coverage = 3.1e8 pairs.  A STEP is one pass of
the hot path over one batch of 2^24 pairs of that job (--launches-per-step 16 device
launches of --batch-pairs 2^20 pairs each), so the default 20 steps generate 3.36e8 pairs
per GPU -- the size of the whole job -- and the timed region of `value` is > 0.5 s.  With
N GPUs the pair-index range is sharded contiguously over the ranks (no collective on the
data path; "weak" scaling: per-GPU work is fixed).

One JSON line is printed by rank 0 (DESIGN.md section 7 for the keys):
  value     pairs/s with the genome resident in HBM and the FASTQ left in HBM
            (jlp_illumina_device_only), timed with CUDA events on the library's compute
            stream, max over ranks;
  e2e       pairs/s through the C ABI with HOST buffers: the genome is uploaded from
            pinned host memory inside the timed region and every batch's FASTQ is copied to
            the library's pinned host buffers and handed to the caller (jlp_illumina_stream);
  roofline  the dominant kernel (k_reads: template gather + quality/error model + FASTQ
            records): algorithmic bytes per launch / its CUDA-event time, against
            MEASURED_PEAKS.json;
  bgzf      the same run with compress = 6 / 1 on the device (BGZF written by k_bgzf): kernel time, and end to
            end with only compressed bytes crossing PCIe;
  full_job  strong scaling: the whole 3.1e8-pair job sharded over the N ranks, seconds (device-resident by CUDA
            events; plain and BGZF end to end by wall clock, max over ranks);
  parity_slice  "ok" when slices of this very workload (first / chromosome-crossing / last 2048 pairs of the
            timed job) are byte-identical to the CPU oracle (outside every timed region);
  e2e_files, extra_workloads (BASELINE.json configs[0..3], haplotype materialisation inside the timed call, each
            with its own cpu_baseline through illumina_ref_cpp / illumina_hap_cpp), pacbio: rank 0, N = 1 only;
  cpu_baseline  the unmodified reference (oracle/_ref/libjlp_ref.so) or, if that is not
            built, the oracle port, on the host cores, on a bounded sample.

--impl reference times the reference's own CPU implementation (illumina_ref_cpp, all
host threads) on bounded samples of the same workload; it never loads the product library.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# GRCh38 chromosome lengths (Mb, rounded) -- only their proportions are used
HUMAN_MB = [248, 242, 198, 190, 182, 171, 159, 145, 138, 134, 135, 133, 114, 107, 102, 90, 83, 80, 59, 64, 47, 51, 156, 57]
METRIC = "illumina_pe150_hs25_read_pairs_per_sec"
UNIT = "read pairs/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload(name, genome_bases):
    """(chromosome lengths, read_length, illumina kwargs, full-job pairs)"""
    if name != "human_pe150_hs25":
        raise SystemExit("unknown workload " + name)
    w = np.array(HUMAN_MB, dtype=np.float64)
    lens = np.floor(w / w.sum() * genome_bases).astype(np.int64)
    lens[0] += genome_bases - lens.sum()
    L = 150
    full_pairs = int(genome_bases * 30 // (2 * L))
    return lens, L, dict(seq_sys="HS25"), full_pairs


def make_genome_into(buf, lens, seed):
    """Uniform TCAG bases (create_genome's default pi_tcag) written into `buf` (uint8[total])."""
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"TCAG", dtype=np.uint8)
    chunk = 1 << 26
    total = int(np.sum(lens))
    for o in range(0, total, chunk):
        n = min(chunk, total - o)
        w = rng.integers(0, 2 ** 63, size=(n + 7) // 8, dtype=np.int64).view(np.uint8)[:n]
        np.take(lut, w & 3, out=buf[o:o + n])


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, polled through NVML every ~2 ms
    (nvidia-smi -lms cannot sample a region of a few tens of milliseconds); falls back to one
    nvidia-smi query if NVML is unavailable."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
            except Exception:
                pass
            if uuid:
                try:
                    self._h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
                except Exception:
                    self._h = None
            if self._h is None:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _poll(self):
        nv = self._nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self._nv is None:
            return
        self._stop.clear()
        self._thr = threading.Thread(target=self._poll, daemon=True)
        self._thr.start()

    def stop(self):
        if self._nv is None:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
                f = [float(x) for x in o.strip().split(",")]
                return {"sm_mhz": f[0], "sm_max_mhz": f[1], "samples": 1, "reasons": [], "how": "nvidia-smi after the region"}
            except Exception:
                return None
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)
        if not self.samples:
            return None
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "samples": len(self.samples),
                "reasons": sorted(self.reasons), "how": "NVML polled every 2 ms during the timed region"}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def let_openmp_use(threads):
    """torchrun exports OMP_NUM_THREADS=1; the reference refuses n_threads > omp_get_max_threads()
    (thread_check, /root/reference/src/util.h:197-205).  Set the environment before libgomp is loaded and the
    runtime's own setting in case it already is."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    try:
        C.CDLL("libgomp.so.1").omp_set_num_threads(int(threads))
    except Exception:
        pass


# ----------------------------------------------------------------- CPU baseline ---

def tmpfs_dir(need_bytes):
    import shutil
    return "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 2 * need_bytes else None


def cpu_reference_setup(lens, seqs_view):
    """The unmodified reference's RefGenome over the same bases (oracle/_ref), or None."""
    from oracle import harness as H
    if not H.have_ref(False):
        return None
    off = np.concatenate(([0], np.cumsum(lens)))
    return H.RefGenomeH(["chrom%d" % i for i in range(len(lens))],
                        [seqs_view[off[i]:off[i + 1]].tobytes() for i in range(len(lens))])


def cpu_reference_run(obj, n_pairs, L, prof1, prof2, threads, seed, matepair=False, shape=16.0, scale=25.0, prob_dup=0.02,
                      ins=(0.00009, 0.00015), dele=(0.00011, 0.00023), hap_probs=None, sep_files=False):
    """illumina_ref_cpp / illumina_hap_cpp of the unmodified reference on `threads` host threads; returns seconds."""
    from oracle import harness as H
    shm = tmpfs_dir(n_pairs * 2 * (2 * L + 32))
    with tempfile.TemporaryDirectory(dir=shm) as d:
        if shm is None and hap_probs is None:          # no room on tmpfs: the reference writes into /dev/null instead
            for k in (1, 2):
                os.symlink("/dev/null", os.path.join(d, "r_R%d.fq" % k))
        common = dict(paired=True, matepair=matepair, out_prefix=os.path.join(d, "r"), n_reads=2 * n_pairs, prob_dup=prob_dup,
                      n_threads=threads, read_pool_size=1000, shape=shape, scale=scale, frag_len_min=L, frag_len_max=2 ** 32 - 1,
                      prof1=prof1, prof2=prof2, ins_prob=list(ins), del_prob=list(dele), r_seed=seed)
        t0 = time.perf_counter()
        if hap_probs is None:
            H.ref_illumina_ref(obj, **common)
        else:
            H.ref_illumina_hap(obj, sep_files=sep_files, hap_probs=hap_probs, **common)
        return time.perf_counter() - t0


def cpu_reference_pacbio(ref, n_reads, threads):
    """pacbio_ref_cpp (defaults of pacbio()) of the unmodified reference on `threads` host threads; returns seconds."""
    from oracle import harness as H
    from oracle.harness_pacbio import DEFAULTS as D
    lib = H.ref_lib(False)
    f64p, u64p = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
    lib.jrefpb_pacbio_ref.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_double] * 5 + \
        [f64p, u64p, C.c_uint64, C.c_uint64, f64p, f64p, f64p, f64p] + [C.c_double] * 4 + [C.c_char_p, C.c_uint64]
    arr = lambda x: np.ascontiguousarray(x, dtype=np.float64)
    cn, cs, sq, nm = arr(D["chi2_params_n"]), arr(D["chi2_params_s"]), arr(D["sqrt_params"]), arr(D["norm_params"])
    ln = D["lognorm_read_length"]
    shm = tmpfs_dir(n_reads * 20000)
    err = C.create_string_buffer(256)
    with tempfile.TemporaryDirectory(dir=shm) as d:
        if shm is None:
            os.symlink("/dev/null", os.path.join(d, "p_R1.fq"))
        t0 = time.perf_counter()
        rc = lib.jrefpb_pacbio_ref(ref.h, os.path.join(d, "p").encode(), n_reads, threads, 100, 0.0, ln[2], ln[0], ln[1], 50.0, None, None,
                                   0, 40, cn.ctypes.data_as(f64p), cs.ctypes.data_as(f64p), sq.ctypes.data_as(f64p), nm.ctypes.data_as(f64p),
                                   0.2, 0.11, 0.04, 0.01, err, 256)
        if rc != 0:
            raise RuntimeError(err.value.decode())
        return time.perf_counter() - t0


def cpu_port_run(genome, n_pairs, L, kw, seed):
    """The oracle port (1 thread) on the same workload; returns seconds."""
    from oracle.compare import oracle_run
    t0 = time.perf_counter()
    oracle_run(genome, 2 * n_pairs, L, True, seed, **kw)
    return time.perf_counter() - t0


def cpu_baseline(genome, lens, flat_bases, L, kw, prof1, prof2, target_s=12.0, pacbio_out=None):
    threads = host_threads()
    let_openmp_use(threads)
    ref = cpu_reference_setup(lens, flat_bases)
    if ref is not None:
        n0 = 20000 * threads
        t = cpu_reference_run(ref, n0, L, prof1, prof2, threads, 1)
        n1 = int(max(n0, min(1e7, n0 / t * target_s)))
        t1 = cpu_reference_run(ref, n1, L, prof1, prof2, threads, 2)
        if pacbio_out is not None:
            try:        # the PacBio generator of the unmodified reference on the same genome and threads: about 3 s
                tp = cpu_reference_pacbio(ref, 2000 * threads, threads)
                npb = int(max(2000 * threads, min(4e5, 2000 * threads / tp * 3.0)))
                tp = cpu_reference_pacbio(ref, npb, threads)
                pacbio_out["cpu_baseline"] = {"value": npb / tp, "unit": "reads/s", "cores": threads, "kind": "reference",
                                              "sample": "%d reads through pacbio_ref_cpp, n_threads=%d, %.1f s" % (npb, threads, tp)}
            except Exception as e:
                pacbio_out["cpu_baseline"] = {"error": str(e)[:200]}
        return {"value": n1 / t1, "unit": UNIT, "cores": threads, "kind": "reference",
                "sample": "%d pairs of the same workload (3.1 Gb genome, PE150 HS25) through illumina_ref_cpp, "
                          "n_threads=%d, read_pool_size=1000, output to tmpfs (or /dev/null when tmpfs is too small), %.1f s" % (n1, threads, t1)}
    n0 = 20000
    t = cpu_port_run(genome, n0, L, kw, 1)
    n1 = int(max(n0, min(2e6, n0 / t * target_s)))
    t1 = cpu_port_run(genome, n1, L, kw, 2)
    return {"value": n1 / t1, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d pairs of the same workload through the C oracle port (1 thread), %.1f s" % (n1, t1)}


# ------------------------------------------------------------ parity of the benched job ---

def parity_slices(J, ctx, genome, n_reads, L, seed, kw, n_slice=2048):
    """Slices of the job the timed legs generate -- the first, one that crosses a chromosome boundary, the last --
    from the library (shard = (k, S)) and from the CPU oracle; byte for byte.  Outside every timed region."""
    from oracle.compare import DEFAULTS, first_diff, group_counts, oracle_run
    from jackalope_b200.illumina import _prepare
    from jackalope_b200 import _lib
    n_pairs = n_reads // 2
    S = max(1, n_pairs // n_slice)
    a = dict(DEFAULTS)
    a.update(kw)
    p = _prepare(genome, "x", n_reads, L, True, a["frag_mean"], a["frag_sd"], a["matepair"], a["seq_sys"], a["profile1"], a["profile2"],
                 a["ins_prob1"], a["del_prob1"], a["ins_prob2"], a["del_prob2"], a["frag_len_min"], a["frag_len_max"],
                 a["haplotype_probs"], a["barcodes"], a["prob_dup"], a["sep_files"], a["compress"], a["comp_method"], a["n_threads"],
                 a["read_pool_size"], a["show_progress"], True, seed, None, None, check_files=False)[0]
    off = np.concatenate(([0], np.cumsum(group_counts(p, genome, False)))).astype(np.int64)

    def bounds(k):
        lo, hi = C.c_uint64(), C.c_uint64()
        assert _lib.lib().jlp_shard_range(0, n_pairs, k, S, C.byref(lo), C.byref(hi)) == 0
        return lo.value, hi.value

    b = int(off[len(off) // 2])                       # a chromosome boundary in the middle of the job
    cross = [k for k in range(max(0, b * S // n_pairs - 2), min(S, b * S // n_pairs + 3)) if bounds(k)[0] < b < bounds(k)[1]]
    picks = [0] + cross[:1] + [S - 1]
    checked = []
    for k in picks:
        r1, r2, _ = J.illumina(genome, "", n_reads, L, True, seed=seed, ctx=ctx, sink="memory", shard=(k, S), **kw)
        lo, hi = bounds(k)
        o = oracle_run(genome, n_reads, L, True, seed, lo=lo, hi=hi, **kw)
        d1, d2 = first_diff(r1, o["r1"]), first_diff(r2, o["r2"])
        if d1 is not None or d2 is not None:
            return "MISMATCH slice %d of %d: R1 byte %r, R2 byte %r" % (k, S, d1, d2), checked
        checked.append([lo, hi])
    return "ok", checked


# ------------------------------------------------------------ outputs of the timed leg ---

DUMP_BYTES_PER_END, DUMP_WINDOWS_PER_BATCH = 4 << 20, 4       # 32 MB of float32 for both ends


def dump_outputs(J, ctx, genome, st, n_reads, L, seed, kw, B, launches, step, n_steps, out_dir):
    """What the device-resident leg computed in its last step, as DIR/<name>.npy.  That leg leaves its FASTQ in HBM and
    drops it; a pair's bytes depend only on the seed and its index, so the step -- shard `step` of the `n_steps` equal
    steps of the timed job, cut into the same `launches` launches of B pairs -- is generated again through the stream
    sink (the same kernels, plus the copy out).
      r1_fastq, r2_fastq  DUMP_WINDOWS_PER_BATCH windows at seeded offsets in every batch's FASTQ, one byte per float32
      step                pairs, batches and FASTQ bytes per end of the regenerated step
      timed_call          pairs and FASTQ bytes per end of the whole timed call (its caller's results, timing aside)"""
    win = max(1, DUMP_BYTES_PER_END // (DUMP_WINDOWS_PER_BATCH * launches))
    parts, calls = ([], []), [0, 0]

    def sink(job, end, buf):
        n, w = len(buf), min(win, len(buf))
        offsets = np.random.default_rng([seed, end, calls[end]]).integers(0, n - w + 1, DUMP_WINDOWS_PER_BATCH) if w else []
        calls[end] += 1
        for o in np.sort(offsets):
            parts[end].append(buf[int(o):int(o) + w])

    ss = J.illumina(genome, "", n_reads, L, True, seed=seed, ctx=ctx, sink=sink, batch_pairs=B, shard=(step, n_steps), **kw)
    assert ss["pairs"] == B * launches and ss["batches"] == launches, ss
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"r1_fastq": np.frombuffer(b"".join(parts[0]), np.uint8).astype(np.float32),
              "r2_fastq": np.frombuffer(b"".join(parts[1]), np.uint8).astype(np.float32),
              "step": np.array([ss["pairs"], ss["batches"], ss["bytes_out"][0], ss["bytes_out"][1]], dtype=np.float64),
              "timed_call": np.array([st["pairs"], st["bytes_out"][0], st["bytes_out"][1]], dtype=np.float64)}
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    return {name: list(arr.shape) for name, arr in arrays.items()}


# -------------------------------------------------- BASELINE.json configs[0..3] (rank 0, N = 1) ---

def extra_workloads(J, ctx, seed, log):
    """The other four named shapes, each timed as ONE whole illumina() call through the C ABI with host buffers
    (genome / haplotype records uploaded and haplotypes materialised inside the timed call; FASTQ handed to the
    caller from pinned host buffers), next to the unmodified reference on all host threads."""
    from oracle import harness as H
    threads = host_threads()
    let_openmp_use(threads)
    have_ref = H.have_ref(False)
    out = {}

    def profiles(L):
        return tuple(J.flatten_profile(J.read_profile(None, "HS25", L, r)) for r in (1, 2))

    def ours(obj, n_reads, L, kw, rep_seed):
        n = [0, 0]

        def sink(job, end, buf):
            n[end] += len(buf)

        ctx._genome = ctx._haps = None                       # one call = upload + (haplotypes) materialise + generate
        t0 = time.perf_counter()
        st = J.illumina(obj, "", n_reads, L, True, seed=rep_seed, ctx=ctx, sink=sink, **kw)
        t = time.perf_counter() - t0
        assert n[0] == st["bytes_out"][0] and st["pairs"] == n_reads // 2
        return t, st

    def entry(name, config, obj, n_reads, L, kw, ref_run, sample):
        ours(obj, n_reads, L, kw, seed + 1)                            # warm-up of the same size: pinned and device buffers at their final size
        t, st = ours(obj, n_reads, L, kw, seed)
        e = {"config": config, "pairs": n_reads // 2, "e2e": {"value": n_reads / 2 / t, "unit": UNIT, "seconds": t,
             "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"]}, "device_ms": st["device_ms"],
             "note": "one illumina() call through the C ABI: H2D of the inputs, haplotype materialisation (if any) and D2H of all FASTQ inside"}
        if have_ref and ref_run is not None:
            try:
                n_ref, t_ref = ref_run()
                e["cpu_baseline"] = {"value": n_ref / t_ref, "unit": UNIT, "cores": threads, "kind": "reference",
                                     "sample": sample % dict(n=n_ref, t=t_ref, thr=threads)}
            except Exception as ex:
                e["cpu_baseline"] = {"error": str(ex)[:200]}
        out[name] = e
        log("[bench] %s: %.3g pairs/s (%.2f s)%s" % (name, e["e2e"]["value"], t,
                                                      ", reference %.3g" % e["cpu_baseline"]["value"] if "value" in e.get("cpu_baseline", {}) else ""))

    # configs[0]: 10 x 1 Mb, 1e6 reads, PE100 HS25
    g = J.random_genome(10, 1_000_000, seed=101)
    p1, p2 = profiles(100)
    ref = H.RefGenomeH(g.names, [g.chrom(c) for c in range(10)]) if have_ref else None
    entry("ref_10x1Mb_pe100", "BASELINE configs[0]: create_genome(10 x 1 Mb) -> illumina(n_reads=1e6, read_length=100, paired, HS25)",
          g, 1_000_000, 100, dict(seq_sys="HS25"),
          lambda: (500_000, cpu_reference_run(ref, 500_000, 100, p1, p2, threads, 3)),
          "the whole job (%(n)d pairs) through illumina_ref_cpp, n_threads=%(thr)d, %(t).2f s")
    # configs[1]: 8 haplotypes (1 % substitutions + 0.1 % indels per site) on 10 x 1 Mb, PE150, 10x per haplotype
    haps = J.random_haplotypes(g, 8, sub_rate=0.01, indel_rate=0.001, seed=103)
    n_pairs = 8 * (10_000_000 * 10 // 300)
    p1, p2 = profiles(150)
    hs = H.hapset_from_muts(ref, haps) if have_ref else None
    entry("haps8_10Mb_pe150", "BASELINE configs[1]: 8 haplotypes (1% subs + 0.1% indels per site) on a 10 Mb genome, PE150, frag_mean=400, "
          "10x per haplotype", haps, 2 * n_pairs, 150, dict(seq_sys="HS25", frag_mean=400),
          lambda: (n_pairs, cpu_reference_run(hs, n_pairs, 150, p1, p2, threads, 4, hap_probs=[1.0] * 8)),
          "the whole job (%(n)d pairs) through illumina_hap_cpp (get_chrom_full per thread inside), n_threads=%(thr)d, %(t).2f s")
    del hs, haps
    # configs[2]: mate-pair, 100 Mb, frag_mean 3000 (sd 500), prob_dup 0.02, ins/del x10, PE150, 10x
    g = J.random_genome(20, 5_000_000, seed=104)
    n_pairs = 100_000_000 * 10 // 300
    kw = dict(matepair=True, frag_mean=3000, frag_sd=500, prob_dup=0.02, ins_prob1=9e-4, del_prob1=1.1e-3, ins_prob2=1.5e-3,
              del_prob2=2.3e-3, seq_sys="HS25")
    ref = H.RefGenomeH(g.names, [g.chrom(c) for c in range(20)]) if have_ref else None
    entry("matepair_100Mb", "BASELINE configs[2]: mate-pair on a 100 Mb genome, frag_mean=3000 (sd 500), prob_dup=0.02, ins/del probabilities x10, "
          "PE150, 10x", g, 2 * n_pairs, 150, kw,
          lambda: (n_pairs, cpu_reference_run(ref, n_pairs, 150, p1, p2, threads, 5, matepair=True, shape=36.0, scale=3000.0 / 36.0,
                                              ins=(9e-4, 1.5e-3), dele=(1.1e-3, 2.3e-3))),
          "the whole job (%(n)d pairs) through illumina_ref_cpp, n_threads=%(thr)d, %(t).2f s")
    # configs[3]: 96 haplotypes, uneven haplotype_probs (1/rank), 500 Mb, PE150, sep_files, 10x of the genome in total
    try:
        import psutil
        if psutil.virtual_memory().available < 40e9:
            raise MemoryError("less than 40 GB of host memory available")
        from concurrent.futures import ThreadPoolExecutor
        from jackalope_b200.genome import random_mutations
        t0 = time.perf_counter()
        g = J.random_genome(20, 25_000_000, seed=105)

        def one(h):
            rng = np.random.default_rng([106, h])
            return [random_mutations(s, rng, 0.001, 0.0001, want_edits=False)[0] for s in g.seqs]

        with ThreadPoolExecutor(max_workers=min(16, threads)) as ex:
            muts = list(ex.map(one, range(96)))
        haps = J.Haplotypes(g, ["hap%d" % i for i in range(96)], muts)
        log("[bench] 96 x 500 Mb haplotype records built in %.1f s" % (time.perf_counter() - t0))
        probs = (1.0 / np.arange(1, 97)).tolist()
        n_pairs = 500_000_000 * 10 // 300
        ref_run = None
        if have_ref:
            ref = H.RefGenomeH(g.names, [g.chrom(c) for c in range(20)])
            hs2 = H.hapset_from_muts(ref, haps, which=[0, 1])
            n_ref = int(n_pairs * (probs[0] + probs[1]) / sum(probs) / 4)
            ref_run = lambda: (n_ref, cpu_reference_run(hs2, n_ref, 150, p1, p2, threads, 6, hap_probs=probs[:2], sep_files=True))
        entry("mux96_500Mb_sep", "BASELINE configs[3]: 96 haplotypes (0.1% subs + 0.01% indels per site) on a 500 Mb genome, haplotype_probs "
              "proportional to 1/rank, PE150, sep_files=TRUE, 10x of the genome over the library (1.67e7 pairs, 192 outputs); 48 Gb of "
              "haplotypes materialised in HBM inside the timed call", haps, 2 * n_pairs, 150,
              dict(seq_sys="HS25", haplotype_probs=probs, sep_files=True), ref_run,
              "BOUNDED sample: haplotypes 0-1 of the 96 (the two most frequent; every thread materialises each with get_chrom_full), "
              "%(n)d pairs, sep_files, through illumina_hap_cpp, n_threads=%(thr)d, %(t).2f s")
    except Exception as ex:
        out["mux96_500Mb_sep"] = {"error": str(ex)[:300]}
    return out


# ------------------------------------------------------------------------ main ---

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="human_pe150_hs25")
    ap.add_argument("--batch-pairs", type=int, default=1 << 20, help="pairs per device launch")
    ap.add_argument("--launches-per-step", type=int, default=16, help="device launches (batches) per step")
    ap.add_argument("--genome-bases", type=float, default=3.1e9, help="shrink for a quick functional run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip BASELINE configs[0..3], files, PacBio and the full-job legs")
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, generate the last step of the device-resident "
                    "leg again and write a fixed sample of its FASTQ to DIR/*.npy (rank 0; see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else max(a.warmup, 1)
    rank, local_rank, world = dist_env()
    if a.impl == "reference" and rank != 0:
        return 0
    # stdout carries exactly one JSON line: everything else a library prints there (NCCL's version
    # banner, ...) goes to stderr
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    lens, L, kw, full_pairs = workload(a.workload, int(a.genome_bases))
    total = int(lens.sum())
    B = a.batch_pairs
    PPS = B * a.launches_per_step                     # pairs per step
    config = {"workload": a.workload, "genome_bases": total, "n_chroms": len(lens), "read_length": L, "paired": True,
              "seq_sys": "HS25", "profiles": "HiSeq2500L150R1filter/HiSeq2500L150R2filter", "frag_mean": 400,
              "frag_sd": 100, "prob_dup": 0.02, "full_job_pairs": full_pairs, "pairs_per_step": PPS, "pairs_per_launch": B,
              "sharding": "contiguous pair-index ranges, one per GPU, no collective",
              "l2": "inputs (3.1 GB genome, random gather) and per-launch outputs (~0.66 GB) are larger than the 126 MB L2"}

    if a.impl == "reference":
        return reference_arm(a, lens, L, kw, config, real_stdout)

    from __graft_entry__ import build
    build()
    import jackalope_b200 as J

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this implementation has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs: genome in PINNED host memory (the e2e leg uploads it inside its timed region)
    t0 = time.perf_counter()
    pinned = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    flat = pinned.numpy()
    make_genome_into(flat, lens, a.seed)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    genome = J.RefGenome(["chrom%d" % i for i in range(len(lens))], [flat[off[i]:off[i + 1]] for i in range(len(lens))])
    genome.flat = lambda: (flat, off.astype(np.uint64))      # already contiguous: no copy
    log("[bench] rank %d: genome %.2f Gb built in %.1f s" % (rank, total / 1e9, time.perf_counter() - t0))

    ctx = J.Context(local_rank)
    job_reads = 2 * a.steps * PPS * world             # the job the timed legs generate, sharded over the ranks

    def run(n_steps, sink, seed, **more):
        return J.illumina(genome, "", 2 * n_steps * PPS * world, L, True, seed=seed, ctx=ctx, sink=sink,
                          batch_pairs=B, shard=(rank, world), **kw, **more)

    # ---- device-resident leg
    for i in range(a.warmup):
        run(1, "device", a.seed + 100 + i)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    t0 = time.perf_counter()
    st = run(a.steps, "device", a.seed)
    barrier()
    wall = time.perf_counter() - t0
    clk = clocks.stop() if rank == 0 else None
    assert st["pairs"] == a.steps * PPS and st["batches"] == a.steps * a.launches_per_step, st
    run_ms = max_over_ranks(st["run_ms"])
    launches = int(sum_over_ranks(st["kernel_launches"]))
    value = a.steps * PPS * world / (run_ms / 1e3)
    place_ms = st["place_ms"] / st["batches"]
    reads_ms = st["reads_ms"] / st["batches"]
    if rank == 0:
        log("[bench] device leg: %.3f ms/step = %.3f ms/launch (events), wall %.3f s, k_place %.3f ms, k_reads %.3f ms, bytes/pair %.1f"
            % (run_ms / a.steps, run_ms / st["batches"], wall, place_ms, reads_ms, sum(st["bytes_out"]) / st["pairs"]))

    # ---- end-to-end leg: genome H2D + every batch's FASTQ D2H into pinned host buffers
    e2e = None
    if not a.no_e2e:
        seen = [0, 0]

        def sink(job, end, buf):
            seen[end] += len(buf)

        run(1, sink, a.seed + 200)                 # sizes the pinned buffers
        seen[0] = seen[1] = 0
        barrier()
        t0 = time.perf_counter()
        ctx._genome = None                         # force the upload: one illumina() call = one genome H2D
        st2 = run(a.steps, sink, a.seed)
        barrier()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        assert seen[0] == st2["bytes_out"][0] and seen[1] == st2["bytes_out"][1] and st2["bytes_out"] == st["bytes_out"]
        e2e = {"value": a.steps * PPS * world / t_e2e, "unit": UNIT,
               "h2d_bytes_per_step": st2["h2d_bytes"] / a.steps, "d2h_bytes_per_step": st2["d2h_bytes"] / a.steps,
               "ms_per_step": t_e2e / a.steps * 1e3,
               "note": "wall clock around jlp_set_genome_async + jlp_illumina_stream: the chromosomes this rank's shard reads "
                       "are copied from pinned host memory inside the region, every batch's FASTQ lands in the library's "
                       "pinned host buffers"}
        if rank == 0:
            log("[bench] e2e: %.2f ms/step, %.3g pairs/s" % (e2e["ms_per_step"], e2e["value"]))

    # ---- compress = TRUE on the device (BGZF members written by k_bgzf): kernel time with the output left in HBM,
    #      and end to end with only the compressed bytes crossing PCIe; level 6 (the reference's default: literals +
    #      line-prefix matches) and level 1 (literals only)
    bgzf = None
    if not a.no_e2e:
        bgzf = {"note": "compress=<level>, comp_engine=device: k_bgzf_code + k_bgzf (+ k_bgzf_own) + scan + gather after k_reads (k_bgzf_ms_per_launch is all five); e2e hands BGZF bytes to the "
                        "caller from pinned host buffers (jlp_illumina_stream); GB/s counts FASTQ bytes read + BGZF bytes written"}
        for level in (6, 1):
            zkw = dict(compress=level, comp_engine="device")
            run(1, "device", a.seed + 400, **zkw)
            barrier()
            stz = run(a.steps, "device", a.seed, **zkw)
            barrier()
            z_ms = max_over_ranks(stz["bgzf_ms"] / stz["batches"])
            zrun_ms = max_over_ranks(stz["run_ms"])
            zseen = [0, 0]

            def zsink(job, end, buf):
                zseen[end] += len(buf)

            run(1, zsink, a.seed + 401, **zkw)
            zseen[0] = zseen[1] = 0
            barrier()
            ctx._genome = None
            t0 = time.perf_counter()
            stz2 = run(a.steps, zsink, a.seed, **zkw)
            barrier()
            t_z = max_over_ranks(time.perf_counter() - t0)
            assert stz["bytes_out"] == st["bytes_out"] and zseen[0] == stz2["z_bytes"][0] + 28, (stz, zseen)
            zin, zout = sum(stz["bytes_out"]) / stz["batches"], sum(stz["z_bytes"]) / stz["batches"]
            bgzf["level%d" % level] = {
                "device_resident": {"value": a.steps * PPS * world / (zrun_ms / 1e3), "unit": UNIT, "ms_per_step": zrun_ms / a.steps},
                "e2e": {"value": a.steps * PPS * world / t_z, "unit": UNIT, "ms_per_step": t_z / a.steps * 1e3,
                        "d2h_bytes_per_step": stz2["d2h_bytes"] / a.steps},
                "ratio": zout / zin, "k_bgzf_ms_per_launch": z_ms, "k_bgzf_GBps": (zin + zout) / (z_ms / 1e3) / 1e9}
            if rank == 0:
                log("[bench] device BGZF level %d: %.3f ms/launch, ratio %.3f, e2e %.2f ms/step = %.3g pairs/s"
                    % (level, z_ms, zout / zin, t_z / a.steps * 1e3, a.steps * PPS * world / t_z))

    # ---- strong scaling: the whole 3.1e8-pair job, sharded over the ranks
    full_job = None
    if not a.no_e2e and not a.no_extras:
        def full(sink, **more):
            return J.illumina(genome, "", 2 * full_pairs, L, True, seed=a.seed + 7, ctx=ctx, sink=sink, batch_pairs=B,
                              shard=(rank, world), **kw, **more)
        barrier()
        stf = full("device")
        barrier()
        dev_s = max_over_ranks(stf["run_ms"]) / 1e3
        nb = [0]

        def fsink(job, end, buf):
            nb[0] += len(buf)

        times = {}
        for name, more in (("e2e_plain_s", {}), ("e2e_bgzf6_s", dict(compress=6, comp_engine="device"))):
            barrier()
            ctx._genome = None
            t0 = time.perf_counter()
            full(fsink, **more)
            barrier()
            times[name] = max_over_ranks(time.perf_counter() - t0)
        full_job = {"pairs": full_pairs, "scaling": "strong", "n_gpus": world, "device_resident_s": dev_s,
                    "device_resident_pairs_per_s": full_pairs / dev_s, **times,
                    "e2e_plain_pairs_per_s": full_pairs / times["e2e_plain_s"], "e2e_bgzf6_pairs_per_s": full_pairs / times["e2e_bgzf6_s"],
                    "note": "BASELINE configs[4] as ONE job: 30x of the 3.1 Gb genome, each rank generates shard (rank, N); seconds, max over ranks; "
                            "e2e = genome H2D + all FASTQ (plain / BGZF level 6) into pinned host buffers"}
        if rank == 0:
            log("[bench] full job (%.3g pairs, %d GPU): %.2f s device-resident, %.2f s plain e2e, %.2f s BGZF e2e"
                % (full_pairs, world, dev_s, times["e2e_plain_s"], times["e2e_bgzf6_s"]))

    # ---- BASELINE configs[0..3] as whole calls (before the legs that churn tens of gigabytes of page cache: the 96-haplotype
    #      call allocates 17 GB of host memory for its records and ran 2x slower after them)
    extras = None
    if not a.no_extras and rank == 0 and world == 1:
        try:
            t0 = time.perf_counter()
            extras = extra_workloads(J, ctx, a.seed, log)
            log("[bench] extra workloads took %.1f s" % (time.perf_counter() - t0))
        except Exception as e:
            extras = {"error": str(e)[:300]}

    # ---- the same through FILES (the reference-facing default sink): tmpfs, all host threads writing
    e2e_files = None
    if not a.no_e2e and not a.no_extras and rank == 0 and world == 1 and os.path.isdir("/dev/shm"):
        import shutil
        per_launch = int(sum(st["bytes_out"]) / st["batches"] * 1.05)
        n_l = int(min(a.steps * a.launches_per_step, 16, shutil.disk_usage("/dev/shm").free // (3 * per_launch)))
        if n_l >= 1:
            d = tempfile.mkdtemp(dir="/dev/shm")
            try:
                nthr = min(host_threads(), 32)
                J.illumina(genome, os.path.join(d, "w"), 2 * B, L, True, seed=a.seed + 300, ctx=ctx, batch_pairs=B,
                           n_threads=nthr, overwrite=True, **kw)
                for f in os.listdir(d):
                    os.unlink(os.path.join(d, f))
                # two runs, the second reported: the boxes are VMs whose memory is handed over by the host page by page
                # on first touch, so the first pass over 11 GB of never-used page cache measures the hypervisor
                t_runs = []
                for rep in range(2):
                    for f in os.listdir(d):
                        os.unlink(os.path.join(d, f))
                    ctx._genome = None
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    J.illumina(genome, os.path.join(d, "r"), 2 * n_l * B, L, True, seed=a.seed, ctx=ctx, batch_pairs=B,
                               n_threads=nthr, overwrite=True, **kw)
                    t_runs.append(time.perf_counter() - t0)
                t_files = t_runs[1]
                sz = os.path.getsize(os.path.join(d, "r_R1.fq")) + os.path.getsize(os.path.join(d, "r_R2.fq"))
                e2e_files = {"value": n_l * B / t_files, "unit": UNIT, "seconds": t_files, "first_run_seconds": t_runs[0], "pairs": n_l * B,
                             "writer_threads": nthr, "bytes_written": sz, "GBps": sz / t_files / 1e9,
                             "note": "illumina(obj, out_prefix, ...) writing <prefix>_R{1,2}.fq on tmpfs; genome H2D inside; "
                                     "second of two runs (the first touches the VM's memory for the first time)"}
                for f in os.listdir(d):
                    os.unlink(os.path.join(d, f))
                # compress = TRUE (the reference's default level 6 -> the device coder)
                ctx._genome = None
                t0 = time.perf_counter()
                J.illumina(genome, os.path.join(d, "z"), 2 * n_l * B, L, True, seed=a.seed, ctx=ctx, batch_pairs=B,
                           n_threads=nthr, compress=True, overwrite=True, **kw)
                t_z = time.perf_counter() - t0
                zsz = os.path.getsize(os.path.join(d, "z_R1.fq.gz")) + os.path.getsize(os.path.join(d, "z_R2.fq.gz"))
                e2e_files["bgzip_device"] = {"value": n_l * B / t_z, "unit": UNIT, "pairs": n_l * B, "compressed_bytes": zsz,
                                             "ratio": zsz / sz, "note": "compress=TRUE, comp_method=bgzip (BGZF written by the GPU)"}
                # the same with zlib level 6 on the writer threads: 1 launch
                t0 = time.perf_counter()
                J.illumina(genome, os.path.join(d, "y"), 2 * B, L, True, seed=a.seed, ctx=ctx, batch_pairs=B,
                           n_threads=nthr, compress=True, comp_engine="host", overwrite=True, **kw)
                t_z = time.perf_counter() - t0
                zsz = os.path.getsize(os.path.join(d, "y_R1.fq.gz")) + os.path.getsize(os.path.join(d, "y_R2.fq.gz"))
                e2e_files["bgzip_host_zlib6"] = {"value": B / t_z, "unit": UNIT, "pairs": B, "compressed_bytes": zsz,
                                                 "note": "comp_engine=host: zlib level 6 on the writer threads"}
                log("[bench] files on tmpfs: %.3g pairs/s plain (%.1f GB/s), %.3g device BGZF" % (e2e_files["value"], e2e_files["GBps"],
                                                                                                   e2e_files["bgzip_device"]["value"]))
            except Exception as e:
                e2e_files = {"error": str(e)[:200]}
            finally:
                shutil.rmtree(d, ignore_errors=True)

    # ---- PacBio reads (SURVEY.md section 8f rank 3), a short device-resident run of pacbio() defaults on the same genome
    pacbio = None
    if not a.no_e2e and not a.no_extras and rank == 0 and world == 1:
        try:
            nthr = min(host_threads(), 32)
            J.pacbio(genome, "", 1 << 13, seed=a.seed, ctx=ctx, sink="device", n_threads=nthr)
            runs = []
            for rep in range(5):        # five runs, the median reported (the host preparation shares the cores with whatever else runs)
                t0 = time.perf_counter()
                stp = J.pacbio(genome, "", 1 << 18, seed=a.seed + 1 + rep, ctx=ctx, sink="device", n_threads=nthr)
                runs.append(time.perf_counter() - t0)
            t_pb = sorted(runs)[len(runs) // 2]
            pacbio = {"reads": stp["pairs"], "bases": stp["bytes_out"][0] / 2, "reads_per_s": stp["pairs"] / t_pb, "wall_s_runs": runs,
                      "kernel_ms": stp["reads_ms"], "kernel_reads_per_s": stp["pairs"] / (stp["reads_ms"] / 1e3),
                      "kernel_fastq_GBps": stp["bytes_out"][0] / (stp["reads_ms"] / 1e3) / 1e9, "host_threads": nthr,
                      "note": "pacbio() defaults, reads left on the device; reads_per_s includes the per-read host preparation"}
        except Exception as e:          # the Illumina line is the contract; never lose it to the extra leg
            pacbio = {"error": str(e)[:200]}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": run_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8", "data": "synthetic", "config": config, "clocks": clk, "e2e": e2e, "e2e_files": e2e_files, "bgzf": bgzf,
           "full_job": full_job, "pacbio": pacbio, "gpu_launches": launches}

    if rank == 0:
        peaks, which = None, "fallback"
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            which = "measured"
        except Exception:
            peaks = 6650.0
        # k_reads (fused quality/error + FASTQ): reads 2L template bases (1 B/base), writes the FASTQ records
        alg_bytes = 2 * L * B + sum(st["bytes_out"]) / st["batches"]
        achieved = alg_bytes / (reads_ms / 1e3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("k_reads")
        except Exception:
            pass
        out["roofline"] = {"bound": "hbm", "kernel": "k_reads (template gather + quality/error model + FASTQ records)", "achieved": achieved, "peak": peaks,
                           "unit": "GB/s", "frac": achieved / peaks, "traffic": traffic, "peak_source": which,
                           "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": reads_ms,
                           "share_of_step": reads_ms * st["batches"] / run_ms, "k_place_ms_per_launch": place_ms,
                           "whole_path_GBps": alg_bytes / (run_ms / st["batches"] / 1e3) / 1e9}
        # parity of exactly this job, outside the timed regions
        try:
            t0 = time.perf_counter()
            verdict, checked = parity_slices(J, ctx, genome, job_reads, L, a.seed, kw)
            out["parity_slice"] = verdict
            out["parity_slice_ranges"] = checked
            log("[bench] parity slices vs the oracle: %s (%.1f s)" % (verdict, time.perf_counter() - t0))
        except Exception as e:
            out["parity_slice"] = "error: " + str(e)[:200]
        if a.dump_outputs:
            t0 = time.perf_counter()
            out["dumped_outputs"] = dump_outputs(J, ctx, genome, st, job_reads, L, a.seed, kw, B, a.launches_per_step,
                                                 rank * a.steps + a.steps - 1, a.steps * world, a.dump_outputs)
            log("[bench] outputs of the last step written to %s (%.1f s)" % (a.dump_outputs, time.perf_counter() - t0))
        if extras is not None:
            out["extra_workloads"] = extras
        if not a.no_cpu_baseline and world == 1:
            prof1, prof2 = (J.flatten_profile(J.read_profile(None, "HS25", L, r)) for r in (1, 2))
            t0 = time.perf_counter()
            out["cpu_baseline"] = cpu_baseline(genome, lens, flat, L, kw, prof1, prof2,
                                               pacbio_out=pacbio if isinstance(pacbio, dict) and "error" not in pacbio else None)
            log("[bench] cpu baseline took %.1f s" % (time.perf_counter() - t0))
        print(json.dumps(out), file=real_stdout, flush=True)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def reference_arm(a, lens, L, kw, config, real_stdout):
    """The reference's own CPU implementation on bounded samples of the workload.  Nothing of the product is built
    or loaded here: the profile parser is plain Python, the timed step is illumina_ref_cpp of oracle/_ref."""
    threads = host_threads()
    let_openmp_use(threads)
    from jackalope_b200.profiles import flatten_profile, read_profile      # pure Python; libjlp_b200.so is not touched
    from oracle import harness as H
    try:
        H.build()                     # where /root/reference exists; on the GPU box the prebuilt oracle/_ref is used
    except Exception:
        pass
    total = int(lens.sum())
    flat = np.empty(total, dtype=np.uint8)
    make_genome_into(flat, lens, a.seed)
    prof1, prof2 = (flatten_profile(read_profile(None, "HS25", L, r)) for r in (1, 2))
    ref = cpu_reference_setup(lens, flat)
    kind = "reference" if ref is not None else "port"
    cores = threads if ref is not None else 1
    genome = None
    if ref is None:                   # oracle/_ref missing: the C port of the oracle (needs the host-only entry points of the C ABI)
        import jackalope_b200 as J
        off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
        genome = J.RefGenome(["chrom%d" % i for i in range(len(lens))], [flat[off[i]:off[i + 1]] for i in range(len(lens))])

    def step(n, seed):
        if ref is not None:
            return cpu_reference_run(ref, n, L, prof1, prof2, threads, seed)
        return cpu_port_run(genome, n, L, kw, seed)

    n = 5000 * cores
    t = step(n, 1)
    budget = min(3.0, 150.0 / max(1, a.steps + a.warmup))        # seconds per step: the whole run ends within minutes
    n = int(max(n, min(4e6, n / t * budget)))
    for i in range(max(0, a.warmup - 1)):
        step(n, 10 + i)
    t0 = time.perf_counter()
    for i in range(a.steps):
        step(n, 100 + i)
    dt = time.perf_counter() - t0
    v = a.steps * n / dt
    sample = ("each step is a bounded sample of %d pairs of the same workload (config.pairs_per_step is the product arm's batch) through %s, "
              "%d host threads, output to tmpfs (or /dev/null when tmpfs is too small)"
              % (n, "illumina_ref_cpp (unmodified reference, oracle/_ref)" if ref is not None else "the C oracle port", cores))
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
                      "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config, "sample_pairs_per_step": n,
                      "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                      "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}), file=real_stdout, flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
