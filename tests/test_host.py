"""CPU tests (no GPU): the C-ABI library loads and exports what include/jlp_b200.h
declares, the host-side model preparation matches the oracle, the R-layer mirror
(profiles, argument checks) behaves like the reference's, the oracle reproduces the
committed golden vectors, and the product refuses to run without a device."""
import ctypes as C
import gzip
import os
import re

import numpy as np
import pytest

import jackalope_b200 as J
from jackalope_b200 import _lib
from golden.cases import CASES, assert_oracle_reproduces
from oracle import harness as H
from oracle.compare import fastq_records, frag_table, oracle_run

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "jlp_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(jlp_[a-z0-9_]+)\s*\(", hdr)) - {"jlp_abort_cb", "jlp_progress_cb"}
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.lib()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert b"sm_100a" in lib.jlp_version()


def test_no_device_means_failure_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        J.Context(0)
    g = J.random_genome(1, 1000, seed=1)
    with pytest.raises(RuntimeError):
        J.illumina(g, "/tmp/never_written", 10, 100, False, seed=1, overwrite=True)
    assert not os.path.exists("/tmp/never_written_R1.fq")


def test_product_does_not_import_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "jackalope_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "jlp_oracle" not in src, f


def test_philox_known_answers():
    # Random123 kat_vectors for philox4x32-10
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    lib = _lib.lib()
    for ctr, key, want in kat:
        assert tuple(int(x) for x in H.philox(ctr, key)) == want
        c, k, o = (np.array(v, dtype=np.uint32) for v in (ctr, key, (0,) * 4))
        lib.jlp_philox4x32_10(c.ctypes.data_as(_lib.u32p), k.ctypes.data_as(_lib.u32p), o.ctypes.data_as(_lib.u32p))
        assert tuple(int(x) for x in o) == want


def test_draw_addressing_matches_oracle():
    lib, orc = _lib.lib(), H.oracle()
    rng = np.random.default_rng(1)
    for _ in range(300):
        seed, j = (int(x) for x in rng.integers(0, 2 ** 64, size=2, dtype=np.uint64))
        for which in range(4):
            assert lib.jlp_draw_pair(seed, j, which) == orc.orc_draw_pair(seed, j, which)
        end, pos = int(rng.integers(0, 2)), int(rng.integers(0, 400))
        for purpose in range(6):
            assert lib.jlp_draw_pos(seed, j, end, purpose, pos) == orc.orc_draw_pos(seed, j, end, purpose, pos)


def test_alias_build_matches_oracle():
    lib = _lib.lib()
    rng = np.random.default_rng(2)
    cases = [np.array([1.0]), np.array([0.5, 0.5]), np.array([1, 0, 0, 3.0]), np.array([0.1] * 10)]
    cases += [rng.random(n) ** 3 for n in (2, 3, 7, 8, 22, 40)]
    flat = J.flatten_profile(J.read_profile(None, "HS25", 150, 1))
    off = 0
    for n in flat[1][:60]:
        cases.append(flat[2][off:off + n])
        off += int(n)
    for p in cases:
        p = np.ascontiguousarray(p, dtype=np.float64)
        P, A = np.zeros(p.size), np.zeros(p.size, dtype=np.uint64)
        assert lib.jlp_alias_build(p.ctypes.data_as(_lib.f64p), p.size, P.ctypes.data_as(_lib.f64p), A.ctypes.data_as(_lib.u64p)) == 0
        P0, A0 = H.alias_build(p)
        assert np.array_equal(P, P0) and np.array_equal(A, A0)
        # the table encodes the distribution: sum over slots of the mass routed to k
        mass = np.zeros(p.size)
        for i in range(p.size):
            mass[i] += P[i] / p.size
            mass[int(A[i])] += (1 - P[i]) / p.size
        assert np.allclose(mass, p / p.sum(), atol=1e-12)


def test_thresholds_against_the_literal_expressions():
    lib, orc = _lib.lib(), H.oracle()
    for p in (0.0, 1.0, 0.5, 0.02, 9e-5, 2e-4, 10 ** -4.1, 10 ** -0.2, 0.9999999, 1e-300, 1 / 3):
        for kind, expr, truth in ((1, 1, 1), (2, 2, 0), (3, 3, 1)):
            thr, al = C.c_uint64(), C.c_int()
            assert lib.jlp_threshold(kind, p, C.byref(thr), C.byref(al)) == 0
            if al.value:
                assert orc.orc_unif_expr(expr, 2 ** 64 - 1, p, 0) == truth
                continue
            if thr.value > 0:
                assert orc.orc_unif_expr(expr, thr.value - 1, p, 0) == truth
            assert orc.orc_unif_expr(expr, thr.value, p, 0) == 1 - truth


def test_integer_restatements_against_the_literal_expressions():
    lib, orc = _lib.lib(), H.oracle()
    rng = np.random.default_rng(5)
    xs = [0, 1, 2 ** 63 - 1, 2 ** 63, 2 ** 64 - 2, 2 ** 64 - 1] + [int(x) for x in rng.integers(0, 2 ** 64, size=5000, dtype=np.uint64)]
    for n in (3, 4, 8, 10, 22, 999901, 2 ** 32 - 1):
        for k in range(1, min(n, 12)):
            b = -(-(k << 64) // n)
            xs += [b - 2, b - 1, b]
    for x in xs:
        x &= 2 ** 64 - 1
        for n in (3, 4, 8, 10, 22, 999901):
            assert lib.jlp_unif_expr(0, x, 0.0, n) == orc.orc_unif_expr(0, x, 0.0, n)
            assert lib.jlp_unif_expr(5, x, 0.0, n) == orc.orc_unif_expr(5, x, 0.0, n)
        assert lib.jlp_unif_expr(4, x, 0.0, 0) == orc.orc_unif_expr(4, x, 0.0, 0)


def test_frag_table_is_the_clamped_floor_gamma_distribution():
    from scipy import stats
    shape, scale, fmin, fmax = 16.0, 25.0, 100, 2 ** 32 - 1
    cdf = frag_table(shape, scale, fmin, fmax).astype(np.float64) / 2.0 ** 64
    assert np.all(np.diff(cdf) >= 0) and cdf.size > 1000
    lens = fmin + np.arange(cdf.size)
    want = stats.gamma.cdf(lens + 1, a=shape, scale=scale)       # P(floor(G) <= len) = P(G < len + 1)
    assert np.max(np.abs(cdf - want)) < 1e-12
    # clamped above: every draw lands at or below frag_max
    assert frag_table(shape, scale, 100, 100).size == 0
    c2 = frag_table(shape, scale, 100, 300)
    assert c2.size == 200 and np.array_equal(c2, frag_table(shape, scale, fmin, fmax)[:200])


def test_reads_per_group_and_apportioning():
    lib = _lib.lib()
    probs = np.array([1.0, 3.0, 0.0, 6.0])
    out = np.zeros(4, dtype=np.uint64)
    tot = np.zeros(4)
    for seed in range(200):
        assert lib.jlp_reads_per_group(100000, probs.ctypes.data_as(_lib.f64p), 4, seed, out.ctypes.data_as(_lib.u64p)) == 0
        assert out.sum() == 100000 and out[2] == 0
        tot += out
    assert np.allclose(tot / tot.sum(), probs / probs.sum(), atol=2e-3)
    # two-level split used by haplotype runs; deterministic in the seed
    sizes = np.array([[1000, 3000], [2000, 2000], [500, 500]], dtype=np.uint64)
    hp = np.array([1.0, 0.0, 2.0])
    a, b = np.zeros(6, dtype=np.uint64), np.zeros(6, dtype=np.uint64)
    for o in (a, b):
        assert lib.jlp_apportion(7, 90000, 3, 2, hp.ctypes.data_as(_lib.f64p), sizes.ctypes.data_as(_lib.u64p), o.ctypes.data_as(_lib.u64p)) == 0
    assert np.array_equal(a, b) and a.sum() == 90000 and a[2] == a[3] == 0
    assert abs(int(a[0]) + int(a[1]) - 30000) < 1500 and abs(int(a[1]) - 3 * int(a[0])) < 3000
    if H.have_ref():
        # same distribution as the reference's reads_per_group (src/hts.h:58-103)
        ref_tot = np.zeros(4)
        for seed in range(200):
            H.ref_lib().jref_set_r_seed(seed + 1)
            H.ref_lib().jref_reads_per_group(100000, probs.ctypes.data_as(_lib.f64p), 4, out.ctypes.data_as(_lib.u64p))
            assert out.sum() == 100000
            ref_tot += out
        assert np.allclose(ref_tot / ref_tot.sum(), tot / tot.sum(), atol=3e-3)


def test_shard_ranges_partition_a_job():
    lib = _lib.lib()
    for lo, hi, S in ((0, 10, 3), (5, 5, 2), (7, 1000003, 8), (0, 3, 8)):
        prev = lo
        for i in range(S):
            a, b = C.c_uint64(), C.c_uint64()
            assert lib.jlp_shard_range(lo, hi, i, S, C.byref(a), C.byref(b)) == 0
            assert a.value == prev and b.value >= a.value and b.value - a.value in ((hi - lo) // S, (hi - lo) // S + 1)
            prev = b.value
        assert prev == hi
    a, b = C.c_uint64(), C.c_uint64()
    assert lib.jlp_shard_range(0, 10, 3, 3, C.byref(a), C.byref(b)) != 0


def test_deflate_members_are_valid_gzip_and_bgzf():
    import gzip
    import struct
    lib = _lib.lib()
    rng = np.random.default_rng(9)
    data = b"".join(b"@REF-chrom%d-%d-F/1\n%s\n+\n%s\n" % (i % 7, i * 31, bytes(rng.choice(np.frombuffer(b"TCAG", np.uint8), 100)),
                                                             bytes(rng.integers(35, 74, 100, dtype=np.uint8))) for i in range(3000))
    for bg in (0, 1):
        for level in (1, 6, 9):
            n = C.c_uint64()
            buf = C.create_string_buffer(len(data) + 65536)
            assert lib.jlp_deflate(bg, level, data, len(data), buf, len(buf), C.byref(n)) == 0
            z = buf.raw[:n.value]
            assert gzip.decompress(z) == data and len(z) < len(data)
            if bg:
                p, sizes = 0, []
                while p < len(z):
                    assert z[p:p + 4] == b"\x1f\x8b\x08\x04" and z[p + 12:p + 14] == b"BC"
                    b = struct.unpack_from("<H", z, p + 16)[0] + 1
                    sizes.append(struct.unpack_from("<I", z, p + b - 4)[0])
                    p += b
                assert p == len(z) and sizes[-1] == 0 and max(sizes) <= 0xff00 and sum(sizes) == len(data)
    n = C.c_uint64()
    assert lib.jlp_deflate(1, 6, b"", 0, None, 0, C.byref(n)) == 0 and n.value == 28     # an empty file is just the EOF block
    assert lib.jlp_deflate(1, 11, data, len(data), None, 0, C.byref(n)) != 0


# ------------------------------------------------------------- R-layer mirror ---

def test_builtin_profiles_are_the_reference_files():
    if not os.path.isdir(REF):
        pytest.skip("/root/reference absent")
    import glob
    files = sorted(glob.glob(os.path.join(REF, "inst", "art_profiles", "*.txt.gz")))
    assert len(files) == 27
    from jackalope_b200.profiles import _parse_text_profile
    for f in files[::4]:
        name = os.path.basename(f)[:-len(".txt.gz")]
        a = J.read_profile("builtin:" + name, None, 36, 1)
        b = J.format_profile(_parse_text_profile(f), 36)
        for nt in range(4):
            for pos in range(36):
                assert np.array_equal(a["quals"][nt][pos], b["quals"][nt][pos])
                assert np.array_equal(a["qual_probs"][nt][pos], b["qual_probs"][nt][pos])


def test_profile_selection_rules():
    assert J.seq_sys_by_read_length(36) == "GA1" and J.seq_sys_by_read_length(100) == "HS20"
    assert J.seq_sys_by_read_length(150) == "HS25" and J.seq_sys_by_read_length(250) == "MSv1"
    with pytest.raises(J.JackalopeError):
        J.seq_sys_by_read_length(251)
    assert J.find_profile_file("HS25", 100, 1) == "builtin:HiSeq2500L125R1"
    assert J.find_profile_file("HiSeq 2500", 150, 2) == "builtin:HiSeq2500L150R2filter"
    assert J.find_profile_file("HS25", 126, 1) == "builtin:HiSeq2500L150R1filter"
    with pytest.raises(J.JackalopeError, match="platform name"):
        J.find_profile_file("nope", 100, 1)
    with pytest.raises(J.JackalopeError, match="read length"):
        J.find_profile_file("HS25", 151, 1)
    with pytest.raises(J.JackalopeError, match="read number 1"):
        J.find_profile_file("MinS", 50, 2)
    p = J.read_profile(None, "HS25", 100, 1)
    assert len(p["quals"]) == 4 and all(len(x) == 100 for x in p["quals"])
    assert all(abs(pr.sum() - 1) < 1e-12 for nt in p["qual_probs"] for pr in nt)
    with pytest.raises(J.JackalopeError, match="never provide both"):
        J.read_profile("x.txt", "HS25", 100, 1)


def test_custom_profile_file_parsing(tmp_path):
    # the error-free profile of tests/testthat/test-sequencer.R:82-87
    path = str(tmp_path / "prof.txt")
    with open(path, "w") as fh:
        for nt in "ACGT":
            for pos in range(100):
                fh.write("%s\t%d\t255\n%s\t%d\t1000000\n" % (nt, pos, nt, pos))
        fh.write("N\t0\t2\nN\t0\t10\n.\t0\t1\n")
    L, nq, probs, quals = J.flatten_profile(J.read_profile(path, None, 100, 1))
    assert L == 100 and np.all(nq == 1) and np.all(probs == 1) and np.all(quals == 255)
    gz = str(tmp_path / "prof.txt.gz")
    with gzip.open(gz, "wt") as fh:
        fh.write(open(path).read())
    assert np.array_equal(J.flatten_profile(J.read_profile(gz, None, 60, 1))[3], quals[:240])
    bad = str(tmp_path / "bad.txt")
    with open(bad, "w") as fh:
        fh.write("T\t1\t30\nT\t1\t5\n")
    with pytest.raises(J.JackalopeError, match="Minimum profile position"):
        J.read_profile(bad, None, 1, 1)
    with pytest.raises(J.JackalopeError, match="Maximum profile position"):
        J.read_profile(path, None, 101, 1)


def test_check_illumina_args_rejects_what_the_reference_rejects():
    g = J.random_genome(2, 500, seed=1)
    haps = J.random_haplotypes(g, 2, seed=2)
    from oracle.compare import DEFAULTS

    def call(obj=g, n_reads=10, read_length=100, paired=True, **kw):
        a = dict(DEFAULTS)
        a.pop("overwrite")
        a.update(kw)
        J.check_illumina_args(obj, n_reads, read_length, paired, **a)

    call()
    call(haps, haplotype_probs=[1, 2], barcodes=["AC", "GT"])
    for bad in (dict(obj="x"), dict(n_reads=0), dict(read_length=1.5), dict(paired="yes"), dict(frag_mean=0),
                dict(frag_sd=-1), dict(ins_prob1=1.5), dict(prob_dup=-0.1), dict(seq_sys=5), dict(frag_len_min=0),
                dict(haplotype_probs=[1, 2]), dict(obj=haps, haplotype_probs=[1]), dict(obj=haps, haplotype_probs=[0, 0]),
                dict(barcodes=["AC", "GT"]), dict(obj=haps, barcodes=["AC"]), dict(barcodes=["ACN"]),
                dict(profile1="a"), dict(paired=False, profile2="b"), dict(compress=10), dict(comp_method="xz"),
                dict(n_threads=0), dict(read_pool_size=0), dict(sep_files=1)):
        with pytest.raises(J.JackalopeError):
            call(**bad)


def test_params_struct_matches_the_header():
    """The ctypes mirrors of jlp_illumina_params / jlp_run_stats have the fields of include/jlp_b200.h, in order
    (comp_engine and the device-BGZF statistics included), and comp_engine is validated before anything runs."""
    import re
    hdr = open(os.path.join(ROOT, "include", "jlp_b200.h")).read()

    def fields(struct):
        body = hdr[hdr.index("typedef struct " + struct):hdr.index("} " + struct + ";")]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        out = []
        for decl in body.split("{", 1)[1].split(";"):
            names = re.findall(r"([A-Za-z_][A-Za-z_0-9]*)\s*(?:\[[0-9]+\])?\s*(?:,|$)", decl.strip())
            out += [n for n in names if n]
        return out

    assert fields("jlp_illumina_params") == [f[0] for f in _lib.Params._fields_]
    assert fields("jlp_run_stats") == [f[0] for f in _lib.RunStats._fields_]
    assert fields("jlp_pacbio_params") == [f[0] for f in _lib.PacbioParams._fields_]
    g = J.random_genome(1, 500, seed=1)
    with pytest.raises(J.JackalopeError, match="comp_engine"):
        J.illumina(g, "", 10, 100, True, seed=1, sink="memory", comp_engine="gpu")


# ------------------------------------------------------------- golden vectors ---

@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_reproduces_golden(name):
    _, n_reads, _, paired, _, _ = CASES[name]
    r1, r2 = assert_oracle_reproduces(name)
    recs = fastq_records(r1)
    assert len(recs) == n_reads // (2 if paired else 1)
    assert all(r[0].startswith(b"@") and r[2] == b"+" and len(r[1]) == len(r[3]) for r in recs)


def test_oracle_pair_geometry_known_answers():
    """tests/testthat/test-sequencer.R:81-161 on the oracle: C25 N150 T25, fragment 200,
    quality-255 profile (mismatch probability 10^-25.5), no indels."""
    chrom = b"C" * 25 + b"N" * 150 + b"T" * 25
    g = J.RefGenome(["chrom0"], [chrom])
    L = 100
    nq = np.ones(4 * L, dtype=np.uint32)
    flat = (L, nq, np.ones(4 * L), np.full(4 * L, 255, dtype=np.uint8))
    groups = H.Groups([500], [chrom], ["REF"], ["chrom0"], [""])
    for matepair, want in ((False, {b"C" * 25 + b"N" * 75, b"A" * 25 + b"N" * 75}),
                           (True, {b"N" * 75 + b"T" * 25, b"N" * 75 + b"G" * 25})):
        r = H.generate(seed=3, paired=True, matepair=matepair, groups=groups, prof1=flat, prof2=flat,
                       ins_prob=[0, 0], del_prob=[0, 0], prob_dup=0.02, pool_pairs=500,
                       frag_cdf=np.zeros(0, dtype=np.uint64), frag_min=200)
        for fq in (r["r1"], r["r2"]):
            recs = fastq_records(fq)
            assert {x[1] for x in recs} == want
            assert all(x[0].split(b"-")[2] in (b"0", b"100") for x in recs)
    assert g.n_chroms() == 1


def test_rcpp_glue_type_checks_against_the_reference_headers():
    """integration/hts_illumina_b200.cpp and hts_pacbio_b200.cpp cannot be built without R, but they must at least compile
    (syntax only) against jackalope's own ref_classes.h / hap_classes.h with the stub Rcpp headers."""
    import shutil
    import subprocess
    if not os.path.isdir(REF) or shutil.which("g++") is None:
        pytest.skip("/root/reference or g++ absent")
    for glue in ("hts_illumina_b200.cpp", "hts_pacbio_b200.cpp"):
        r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-w", "-I" + os.path.join(ROOT, "oracle", "stubs"),
                            "-I" + os.path.join(REF, "inst", "include"), "-I" + os.path.join(REF, "src"),
                            "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "integration"),
                            os.path.join(ROOT, "integration", glue)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[:2000]


def test_rcpp_glue_links_against_the_stock_wrappers():
    """oracle/_ref/libjlp_glue.so = integration/*.cpp + the generated wrappers of /root/reference/src/RcppExports.cpp
    :109-243 (extracted at build time) + libjlp_b200.so under -Wl,-z,defs: the four exports resolve against the
    prototypes the stock wrappers declare (a by-value `barcodes`, as in round 1, is an undefined symbol here).
    No compute call: the GPU tests (tests/test_gpu_glue.py) go through it."""
    import subprocess
    if not os.path.isdir(REF):
        pytest.skip("/root/reference absent")
    assert H.have_glue(), "oracle/Makefile did not build _ref/libjlp_glue.so"
    so = os.path.join(ROOT, "oracle", "_ref", "libjlp_glue.so")
    syms = subprocess.run(["nm", "-D", "--defined-only", so], capture_output=True, text=True, check=True).stdout
    for s in H.GLUE_SYMBOLS:
        assert (" T " + s) in syms, s
    for export in ("illumina_ref_cpp", "illumina_hap_cpp", "pacbio_ref_cpp", "pacbio_hap_cpp"):
        assert any(("_Z%d%s" % (len(export), export)) in line for line in syms.splitlines()), export
    undef = subprocess.run(["nm", "-D", "--undefined-only", so], capture_output=True, text=True, check=True).stdout
    assert "jlp_illumina_ref" in undef and "jlp_pacbio" in undef            # bound to libjlp_b200.so, not restated
    # the wrappers in the build are the reference's, verbatim
    ext = open(os.path.join(ROOT, "oracle", "_ref", "rcpp_exports_extract.cpp")).read()
    stock = open(os.path.join(REF, "src", "RcppExports.cpp")).read()
    body = ext[ext.index("// illumina_ref_cpp"):]
    assert body in stock and "const std::vector<std::string>& barcodes);" in body


def test_oracle_lazy_haplotype_groups_match_the_full_materialisation():
    """oracle_run with a callable hap_seqs materialises only the groups a pair range can touch (used by the
    full-size GPU parity tests); the bytes must equal the run that materialises everything."""
    from common import hap_sequences, lazy_hap_sequences, oracle_jobs
    g = J.random_genome(4, 6_000, seed=71)
    haps = J.random_haplotypes(g, 5, sub_rate=0.01, indel_rate=0.003, seed=72)
    kw = dict(haplotype_probs=[1, 2, 3, 4, 5], sep_files=True, prob_dup=0.4, read_pool_size=20, seq_sys="HS25")
    full = hap_sequences(haps)
    lazy = lazy_hap_sequences(haps)
    jobs = oracle_jobs(haps, 4000, 100, True, 5, **kw)
    assert len(jobs) == 5
    jl, jh = jobs[3]
    for lo, hi in ((jl, jl + 40), (jl + (jh - jl) // 2, jl + (jh - jl) // 2 + 60), (jh - 30, jh)):
        a = oracle_run(haps, 4000, 100, True, 5, lo=lo, hi=hi, hap_seqs=full, only_job=(jl, jh), **kw)
        b = oracle_run(haps, 4000, 100, True, 5, lo=lo, hi=hi, hap_seqs=lazy, only_job=(jl, jh), **kw)
        assert a["r1"] == b["r1"] and a["r2"] == b["r2"] and len(a["r1"]) > 0
    assert 0 < len(lazy.cache) < 20 and all(h == 3 for h, _ in lazy.cache)


def test_integer_thresholds_equal_the_x87_search():
    """The comparison thresholds are computed in integer arithmetic (no x87 needed: SURVEY.md App. A.2); kinds 11-13 of
    jlp_threshold evaluate the reference's own long-double expressions at candidate draws (x86-64).  Equal on random
    probabilities of every magnitude and on doubles that sit exactly on, just below and just above a draw boundary."""
    import math
    import random
    lib = _lib.lib()

    def thr(kind, p):
        t, a = C.c_uint64(), C.c_int()
        assert lib.jlp_threshold(kind, p, C.byref(t), C.byref(a)) == 0
        return t.value, a.value

    rnd = random.Random(5)
    ps = [0.0, 1.0, 0.5, 1e-25, 2.0 ** -64, 3 * 2.0 ** -64, 1 - 2.0 ** -53, 0.02, 0.00009, 0.0002, 10 ** -2.55, 1.5, -0.5, 2.0 ** -70, 5e-324]
    for _ in range(400):
        ps.append(min(1.0, rnd.random() * 2 ** rnd.choice([rnd.uniform(-70, 0), rnd.uniform(-12, 0), 0])))
    for _ in range(150):
        v = rnd.getrandbits(rnd.randint(1, 64)) / 2 ** 64
        ps += [v, math.nextafter(v, 0), math.nextafter(v, 2)]
    for p in ps:
        for kind in (1, 2, 3):
            assert thr(kind, p) == thr(kind + 10, p), (kind, p)
