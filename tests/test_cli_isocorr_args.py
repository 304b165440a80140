"""Command-line behaviour of `mmseq -isocorr` that needs no GPU: the usage text lists the flag with its file name, and
the flag leaves the help and the argument-error messages and their exit code as they are."""
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
    return subprocess.run([BIN, *args], capture_output=True, text=True, timeout=120)


def test_usage_lists_isocorr():
    r = run("-help")
    assert r.returncode == 1
    line = [x for x in r.stderr.splitlines() if x.strip().startswith("-isocorr")]
    assert line == ["  -isocorr           (B200 build) also write the posterior correlation, P(first > second) and shared fragments "
                    "of every isoform pair within a gene (*.isocorr)"]


def test_isocorr_keeps_help_and_error_messages():
    for flag in ("-h", "-help", "--help"):
        base, r = run(flag), run("-isocorr", flag)
        assert r.returncode == base.returncode == 1 and r.stderr == base.stderr and r.stdout == base.stdout
    for args in ([], ["a"], ["-gibbs_iter", "1000", "-gibbs_ss", "7", "a", "b"], ["-bogus", "a", "b"], ["-pool", "a", "b"],
                 ["-chains", "9", "a", "b"]):
        base, r = run(*args), run("-isocorr", *args)
        assert r.returncode == base.returncode == 1 and r.stderr == base.stderr, args
    r = run("a", "b", "-isocorr")  # options come first: a trailing flag is a positional argument too many
    assert r.returncode == 1 and "Error: mandatory arguments missing." in r.stderr
    r = run("-isocorr", "-allelic", "-tpm", "-counts", "/nonexistent.hits", "out")
    base = run("-allelic", "-tpm", "-counts", "/nonexistent.hits", "out")
    assert r.returncode == base.returncode == 1 and r.stderr == base.stderr
