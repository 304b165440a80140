"""Command-line behaviour of `mmseq -chains` that needs no GPU: the usage text lists the flag, and a count outside
1..8 or not a number exits 1 with a message."""
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


def test_usage_lists_chains():
    r = run("-help")
    assert r.returncode == 1
    line = [x for x in r.stderr.splitlines() if x.strip().startswith("-chains")]
    assert len(line) == 1 and "(B200 build)" in line[0] and "1..8" in line[0]
    for name in (".convergence", ".identical.convergence", ".gene.convergence"):
        assert name in line[0]


@pytest.mark.parametrize("value", ["0", "9", "x", "-1"])
def test_chains_out_of_range_exits_1(tmp_path, value):
    r = run("-chains", value, str(tmp_path / "missing.hits"), str(tmp_path / "out"))
    assert r.returncode == 1
    assert "Error: -chains must be in 1..8." in r.stderr
    assert not os.listdir(tmp_path)


def test_chains_needs_a_value():
    r = run("-chains")
    assert r.returncode == 1 and "Error: option -chains needs a value." in r.stderr
