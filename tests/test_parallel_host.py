"""jlp::parallel_for (jackalope_b200/csrc/jlp_host.h), the loop that spreads the library's host work over a few threads,
driven by tests/parallel_driver.cpp without a GPU: every item runs once, the lowest failing item's exception comes back
with its type after all items ran, and one thread means the calling thread alone."""
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "jackalope_b200", "csrc")


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("parallel") / "parallel_driver")
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-I", CSRC, os.path.join(HERE, "parallel_driver.cpp"),
           "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def run(driver, *args):
    res = subprocess.run([driver] + [str(a) for a in args], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr          # a std::terminate would abort with a signal
    return dict(kv.split("=", 1) for kv in res.stdout.split())


@pytest.mark.parametrize("n,nt", [(0, 4), (1, 4), (3, 8), (2000, 4)])
def test_every_item_runs_exactly_once(driver, n, nt):
    r = run(driver, "count", n, nt)
    assert int(r["runs"]) == n
    assert int(r["threads"]) <= max(min(n, nt), 1)
    if n >= 1000:
        assert int(r["threads"]) > 1


@pytest.mark.parametrize("nt", [1, 4])
def test_lowest_failing_item_is_rethrown_with_its_type_after_all_items_ran(driver, nt):
    """item 3 (std::invalid_argument) fails after item 7 (std::out_of_range) on several threads"""
    r = run(driver, "throws", 20, nt)
    assert r == {"caught": "invalid_argument", "what": "three", "ran": "20"}


def test_one_thread_is_the_calling_thread(driver):
    assert run(driver, "serial", 50) == {"caller_only": "1"}
