"""Command-line behaviour of `mmseq -pool` that needs no GPU: the usage text lists the flag, and -pool without
-chains 2 or more exits 1 with a message before any file is written."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")


@pytest.fixture(scope="module", autouse=True)
def _built():
    if not os.path.exists(BIN):
        env = dict(os.environ); env.pop("CXX", None); env.pop("CC", None)
        subprocess.check_call(["make", "-C", ROOT, "lib", "cli"], env=env, stdout=subprocess.DEVNULL)


def run(*args):
    return subprocess.run([BIN, *args], capture_output=True, text=True, timeout=60)


def test_usage_lists_pool():
    r = run("-help")
    assert r.returncode == 1
    line = [x for x in r.stderr.splitlines() if x.strip().startswith("-pool")]
    assert len(line) == 1 and "(B200 build)" in line[0] and "-chains" in line[0]


@pytest.mark.parametrize("extra", [[], ["-chains", "1"]])
def test_pool_needs_two_chains(tmp_path, extra):
    r = run(*extra, "-pool", str(tmp_path / "missing.hits"), str(tmp_path / "out"))
    assert r.returncode == 1
    assert "Error: -pool needs -chains 2 or more." in r.stderr
    assert not os.listdir(tmp_path)


def test_pool_takes_no_value(tmp_path):
    """-pool is a flag: the word after it is the next option or argument"""
    r = run("-pool", "-chains", "0", str(tmp_path / "missing.hits"), str(tmp_path / "out"))
    assert r.returncode == 1 and "Error: -chains must be in 1..8." in r.stderr
