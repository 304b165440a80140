"""Command-line behaviour of `mmseq -allelic` that needs no GPU: the usage text lists the flag with its two file names;
the flag leaves the help and the argument-error messages and their exit code as they are; a hits file without a pair
STEM_A / STEM_B in one gene is refused before any device work, and transcripts named *_A / *_B without a partner in
their gene are counted on one stderr line."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
NO_PAIR = "Error: -allelic found no pair of transcripts STEM_A / STEM_B in one gene."


@pytest.fixture(scope="module", autouse=True)
def _built():
    if not os.path.exists(BIN):
        env = dict(os.environ); env.pop("CXX", None); env.pop("CC", None)
        subprocess.check_call(["make", "-C", ROOT, "lib", "cli"], env=env, stdout=subprocess.DEVNULL)


def run(*args):
    return subprocess.run([BIN, *args], capture_output=True, text=True, timeout=120)


def _hits(path, transcripts, genes, records):
    with open(path, "w") as f:
        for t in transcripts:
            f.write(f"@TranscriptMetaData\t{t}\t1000\t1200\n")
        for g, mem in genes.items():
            f.write(f"@GeneIsoforms\t{g}\t" + "\t".join(mem) + "\n")
        for r, hits in enumerate(records):
            f.write(f">r{r}\n" + "".join(h + "\n" for h in hits))
    return str(path)


def test_usage_lists_allelic():
    r = run("-help")
    assert r.returncode == 1
    line = [x for x in r.stderr.splitlines() if x.strip().startswith("-allelic")]
    assert line == ["  -allelic           (B200 build) also write the posterior and EM allelic fraction of every haplotype pair "
                    "STEM_A / STEM_B and gene (*.allelic, *.gene.allelic)"]


def test_allelic_keeps_help_and_error_messages():
    for flag in ("-h", "-help", "--help"):
        base, r = run(flag), run("-allelic", flag)
        assert r.returncode == base.returncode == 1 and r.stderr == base.stderr and r.stdout == base.stdout
    for args in ([], ["a"], ["-gibbs_iter", "1000", "-gibbs_ss", "7", "a", "b"], ["-bogus", "a", "b"], ["-pool", "a", "b"],
                 ["-chains", "9", "a", "b"]):
        base, r = run(*args), run("-allelic", *args)
        assert r.returncode == base.returncode == 1 and r.stderr == base.stderr, args
    r = run("a", "b", "-allelic")  # options come first: a trailing flag is a positional argument too many
    assert r.returncode == 1 and "Error: mandatory arguments missing." in r.stderr
    r = run("-allelic", "-tpm", "-counts", "/nonexistent.hits", "out")
    base = run("-tpm", "-counts", "/nonexistent.hits", "out")
    assert r.returncode == base.returncode == 1 and r.stderr == base.stderr


@pytest.mark.parametrize("case", ["no_haplotypes", "partner_missing", "partner_in_another_gene"])
def test_no_pair_is_refused_before_any_device_work(tmp_path, case):
    tr = {"no_haplotypes": ["t1", "t2"], "partner_missing": ["x_A", "t2"], "partner_in_another_gene": ["x_A", "x_B"]}[case]
    genes = {"g1": [tr[0]], "g2": [tr[1]]} if case == "partner_in_another_gene" else {"g1": tr}
    path = _hits(tmp_path / "h.hits", tr, genes, [[tr[0]], [tr[0], tr[1]]])
    r = run("-allelic", "-notraces", path, str(tmp_path / "out"))
    assert r.returncode == 1 and r.stderr == NO_PAIR + "\n" and r.stdout == ""
    assert os.listdir(tmp_path) == ["h.hits"]                             # nothing written


def test_transcripts_without_partner_are_noted(tmp_path):
    tr = ["x_A", "x_B", "y_A", "z_B", "w_A", "iso"]
    path = _hits(tmp_path / "h.hits", tr, {"g1": ["x_A", "x_B", "y_A", "iso"], "g2": ["z_B", "w_A"]}, [["x_A"], ["x_B", "iso"]])
    r = run("-allelic", "-notraces", "-gibbs_iter", "1024", path, str(tmp_path / "out"))
    notes = [x for x in r.stderr.splitlines() if x.startswith("Note: -allelic")]
    assert notes == ["Note: -allelic: 3 transcripts named *_A / *_B have no partner in their gene."]
    assert r.stderr.startswith(notes[0] + "\n")                            # before any device work
