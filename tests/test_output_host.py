"""The output path without a GPU: jackalope_b200/csrc/jlp_output.cpp (the writer threads, mapped and pwrite files, zlib
on the writer threads, memory and stream sinks, truncation on errors) driven by tests/output_driver.cpp with seeded
batches, as the Illumina and PacBio drivers feed it."""
import gzip
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "jackalope_b200", "csrc")
SIZES = [9437201, 300000, 0, 8355845, 1, 4194304]        # kSizes of the driver
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("output") / "output_driver")
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-I", CSRC, os.path.join(HERE, "output_driver.cpp"),
           os.path.join(CSRC, "jlp_output.cpp"), os.path.join(CSRC, "jlp_deflate.cpp"), "-o", exe, "-lz"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def run(driver, case, d):
    res = subprocess.run([driver, case, str(d)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return res.stdout.split()


def read(d, name):
    return (d / name).read_bytes()


@pytest.mark.parametrize("case", ["plain1", "plain4"])
def test_plain_files_are_the_concatenated_batches(driver, tmp_path, case):
    """one writer thread: pwrite slices; four: the reservation task and copies into mappings"""
    assert run(driver, case, tmp_path) == ["mapped=%d" % (case == "plain4")]
    for e in (1, 2):
        assert read(tmp_path, "out_R%d.fq" % e) == read(tmp_path, "expect_R%d.fq" % e) == read(tmp_path, "plain_R%d.fq" % e)


@pytest.mark.parametrize("case", ["bgzf", "gzip"])
def test_zlib_files_equal_members_over_whole_batches(driver, tmp_path, case):
    run(driver, case, tmp_path)
    for e in (1, 2):
        z = read(tmp_path, "out_R%d.fq" % e)
        assert z == read(tmp_path, "expect_R%d.fq" % e)
        assert gzip.decompress(z) == read(tmp_path, "plain_R%d.fq" % e)
        assert z.endswith(EOF_BLOCK) == (case == "bgzf")


def test_memory_sink_counts_overflow_and_writes_nothing_past_cap(driver, tmp_path):
    n, cap = map(int, run(driver, "memory", tmp_path))
    want = read(tmp_path, "expect_R1.fq")
    assert n == len(want) == sum(SIZES) + len(EOF_BLOCK)
    mem = read(tmp_path, "out_R1.fq")
    fit = SIZES[0] + SIZES[1]                            # batches are copied whole or not at all
    assert mem[:fit] == want[:fit]
    assert mem[fit:] == b"x" * (len(mem) - fit)


def test_stream_sink_calls_back_in_order(driver, tmp_path):
    calls = run(driver, "stream", tmp_path)
    want = []
    for job, n_batches in ((0, len(SIZES)), (1, 2)):
        for s in SIZES[:n_batches]:
            want += ["%d:0:%d" % (job, s), "%d:1:%d" % (job, s >> 1)]
        want += ["%d:0:28" % job, "%d:1:28" % job]       # the device coder's stream ends with the EOF block
    assert calls == want
    for e in (0, 1):
        plain = read(tmp_path, "plain_R%d.fq" % (e + 1))
        assert read(tmp_path, "stream_0_%d" % e) == plain + EOF_BLOCK
        assert read(tmp_path, "stream_1_%d" % e) == plain[:(SIZES[0] >> e) + (SIZES[1] >> e)] + EOF_BLOCK


def test_shared_presized_file_at_base_offset(driver, tmp_path):
    """a file sized by the caller keeps its size and its bytes outside [base, base + n); no EOF block"""
    run(driver, "shared", tmp_path)
    assert read(tmp_path, "out_R1.fq") == read(tmp_path, "expect_R1.fq")


@pytest.mark.parametrize("case", ["abandon1", "abandon4"])
def test_abandon_truncates_to_the_settled_batches(driver, tmp_path, case):
    """the unsettled batch is written (pwrite) or copied into the extended, mapped file before abandon() cuts it off"""
    assert run(driver, case, tmp_path) == ["mapped=%d" % (case == "abandon4")]
    assert read(tmp_path, "out_R1.fq") == read(tmp_path, "expect_R1.fq")
