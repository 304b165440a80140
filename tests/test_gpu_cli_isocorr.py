"""`mmseq -isocorr` on small samples: the .isocorr file matches the numpy reference (tests/isocorr_reference.py) cell by
cell on the chains rebuilt through the C ABI, for text, binary and schema-2 files and with -chains 4 -pool; every other
file, and stdout apart from the one name in the list of output files, is byte-identical with and without the flag;
-chains 4 without -pool gives chain 1's file; batch mode equals single runs and two GPUs agree with one; a gene of more
than 64 observed isoforms; a sample without a gene of two observed isoforms gets the two header lines.  Known answer:
two isoforms sharing one class of K fragments, beside singletons, have the closed-form stationary correlation."""
import math
import os
import subprocess

import numpy as np
import pytest

from mmseq_b200 import synth
from tests import exact_reference as xref
from tests import isocorr_reference as iref
from tests.test_gpu_cli_tpm import _abi, _csr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
HEAD = ["gene_id", "transcript_1", "transcript_2", "shared_fragments", "corr_mu", "corr_log_mu", "prob_1_gt_2"]


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    return r


def _rows(path, N=None):
    lines = open(path).read().split("\n")
    assert lines[-1] == "" and lines[1] == "\t".join(HEAD)
    if N is not None:
        assert lines[0] == "# Mapped fragments: %d" % N
    return [ln.split("\t") for ln in lines[2:-1]]


def _write(tmp, fmt, s=None):
    s = s or synth.Synth(77, 300, 6000)
    path = str(tmp / f"h.{fmt}.hits")
    if fmt == "text":
        synth.write_hits_text(s, path)
    elif fmt == "binary":
        synth.write_hits_binary(s, path)
    else:
        w = np.random.default_rng(5).uniform(0.2, 1.0, len(s.frag_tid)).astype(np.float32)
        synth.write_hits_binary(s, path, weights=w)
    return path


def _close(cell, want):
    if math.isnan(want):
        return cell == "NA"
    return cell != "NA" and abs(float(cell) - want) <= 1e-5 * abs(want) + 1e-9


def _check_file(base, h, mu, weighted=False):
    gptr, mem = _csr(h, h.gene_ptr, h.gene_members)
    g, a, b, ma, mb, _ = iref.pairs(gptr, mem)
    rows = _rows(base + ".isocorr", h.N)
    assert len(rows) == len(g)
    ref = iref.summaries(mu, gptr, mem)
    shared = iref.shared(h.row_ptr, h.col, None if weighted else h.k, gptr, mem)
    names = [h.names[h.col2hdr[c]] for c in range(h.n)]
    for p, cells in enumerate(rows):
        assert cells[:4] == [h.gene_names[g[p]], names[ma[p]], names[mb[p]], str(shared[p])], (p, cells)
        for c, k in zip(cells[4:], ("corr_mu", "corr_log_mu", "prob_1_gt_2")):
            assert _close(c, float(ref[k][p])), (p, k, cells, ref[k][p])
    return rows


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("isocorr")
    path = _write(tmp, "binary")
    out = dict(path=path)
    for name, args in (("plain", ["-counts", "-tpm", "-chains", "4"]), ("iso", ["-counts", "-tpm", "-chains", "4", "-isocorr"]),
                       ("c1", ["-isocorr", "-notraces"]), ("pool", ["-chains", "4", "-pool", "-isocorr", "-notraces"])):
        d = tmp / name
        d.mkdir()
        out[name] = str(d / "out")
        r = _run(args + ARGS, path, out[name])
        out[name + "_stdout"] = r.stdout
    return out


def test_isocorr_changes_no_other_file(runs):
    da, db = os.path.dirname(runs["plain"]), os.path.dirname(runs["iso"])
    files = sorted(os.listdir(da))
    assert sorted(os.listdir(db)) == sorted(files + ["out.isocorr"])
    for f in files:
        assert open(os.path.join(da, f), "rb").read() == open(os.path.join(db, f), "rb").read(), f
    after = f"  {runs['plain']}.gene.tpm\n"
    want = runs["plain_stdout"].replace(after, after + f"  {runs['plain']}.isocorr\n", 1).replace(runs["plain"], runs["iso"])
    assert runs["iso_stdout"] == want


def test_file_matches_the_reference_binary_and_chains(runs):
    h, _, mu = _abi(runs["path"], 4)
    rows = _check_file(runs["c1"], h, mu[:1])
    assert len(rows) > 50 and sum(int(r[3]) > 0 for r in rows) > 10
    _check_file(runs["pool"], h, mu)
    assert open(runs["iso"] + ".isocorr", "rb").read() == open(runs["c1"] + ".isocorr", "rb").read()   # -chains 4: chain 1's


@pytest.mark.parametrize("fmt", ["text", "schema2"])
def test_file_matches_the_reference_text_and_schema2(tmp_path, fmt):
    path = _write(tmp_path, fmt)
    _run(["-isocorr", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    h, _, mu = _abi(path, 1)
    _check_file(str(tmp_path / "out"), h, mu, weighted=fmt == "schema2")


def test_batch_and_two_gpus_equal_single_runs(tmp_path):
    paths = [_write(tmp_path, "text"), _write(tmp_path, "binary"), _write(tmp_path, "schema2")]
    args = ["-isocorr", "-notraces", "-chains", "2", "-pool"] + ARGS
    bases = []
    for i, p in enumerate(paths):
        _run(args, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN] + args + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    for i in range(len(paths)):
        assert open(bases[i] + ".isocorr", "rb").read() == open(str(tmp_path / f"single{i}") + ".isocorr", "rb").read(), i
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    for i, p in enumerate(paths[1:], 1):
        _run(["-isocorr", "-notraces", "-gpus", "2"] + ARGS, p, str(tmp_path / f"g2_{i}"))
        _run(["-isocorr", "-notraces"] + ARGS, p, str(tmp_path / f"g1_{i}"))
        assert open(str(tmp_path / f"g2_{i}.isocorr"), "rb").read() == open(str(tmp_path / f"g1_{i}.isocorr"), "rb").read(), i


def _hits(path, transcripts, genes, records):
    with open(path, "w") as f:
        for t in transcripts:
            f.write(f"@TranscriptMetaData\t{t}\t1000\t1200\n")
        for g, mem in genes.items():
            f.write(f"@GeneIsoforms\t{g}\t" + "\t".join(mem) + "\n")
        for r, hits in enumerate(records):
            f.write(f">r{r}\n" + "".join(h + "\n" for h in hits))
    return str(path)


def test_gene_of_more_than_64_isoforms(tmp_path):
    rng = np.random.default_rng(9)
    tr = [f"big{i}" for i in range(70)] + ["s0", "s1", "lone"]
    records = [sorted(set(rng.choice(70, int(rng.integers(1, 6))).tolist())) for _ in range(3000)]
    records = [[tr[i] for i in r] for r in records] + [["s0", "s1"]] * 5 + [["lone"]]
    path = _hits(tmp_path / "h.hits", tr, {"gb": tr[:70], "gs": ["s0", "s1"], "gl": ["lone"]}, records)
    _run(["-isocorr", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    h, _, mu = _abi(path, 1)
    rows = _check_file(str(tmp_path / "out"), h, mu)
    assert len(rows) == 70 * 69 // 2 + 1 and rows[-1][:4] == ["gs", "s0", "s1", "5"]


def test_no_gene_of_two_observed_isoforms_gives_the_header(tmp_path):
    tr = ["a", "b", "c"]
    path = _hits(tmp_path / "h.hits", tr, {"g1": ["a", "b"], "g2": ["c"]}, [["a"], ["a", "c"], ["c"]])   # b has no hits
    r = _run(["-isocorr", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    assert open(str(tmp_path / "out.isocorr")).read() == "# Mapped fragments: 3\n" + "\t".join(HEAD) + "\n"
    assert f"  {tmp_path}/out.isocorr\n" in r.stdout


def test_shared_class_known_answer(tmp_path):
    """Transcripts t0, t1 share one class of K fragments and have u0, u1 singletons; t2, t3 have singletons only.  The
    Gamma step draws mu_j ~ Gamma(a_j, r_j), a_j = alpha + u_j + x_j, x_1 = K - x_0, so at stationarity
    corr(mu_0, mu_1) = -Var(x_0) / sqrt((E a_0 + Var x_0)(E a_1 + Var x_0)) with the exact pmf of x_0 (SharedClass).
    4 chains of 1024 draws thinned by 16 (S = 4096); the Monte-Carlo tolerance 4 (1 - rho^2) / sqrt(ESS) uses the
    smallest bulk ESS of the two transcripts' mu in .convergence.  The independent pair is within 4 / sqrt(ESS) of 0."""
    K, u0, u1, alpha = 40, 10, 3, 0.1
    tr = ["t0", "t1", "t2", "t3"]
    records = [["t0", "t1"]] * K + [["t0"]] * u0 + [["t1"]] * u1 + [["t2"]] * 20 + [["t3"]] * 25
    path = _hits(tmp_path / "h.hits", tr, {"g": ["t0", "t1"], "h": ["t2", "t3"]}, records)
    _run(["-isocorr", "-notraces", "-chains", "4", "-pool", "-seed", "7"], path, str(tmp_path / "out"))
    rows = {(r[1], r[2]): r for r in _rows(str(tmp_path / "out.isocorr"))}
    conv = [ln.split("\t") for ln in open(str(tmp_path / "out.convergence")).read().split("\n")[1:] if ln]
    head = open(str(tmp_path / "out.convergence")).read().split("\n")[1].split("\t")
    col = head.index("ess_bulk")
    ess = {c[0]: float(c[col]) for c in conv[1:]}
    N = len(records)
    length = 1000.0 * N / 1e9                                           # scaled effective length, equal for all
    sc = xref.SharedClass(K, [u0, u1], [length, length], alpha, 0.1)
    p = sc.pmf(0)
    x = np.arange(K + 1)
    ex = (p * x).sum()
    vx = (p * x * x).sum() - ex * ex
    rho = -vx / math.sqrt((alpha + u0 + ex + vx) * (alpha + u1 + K - ex + vx))
    r01 = rows[("t0", "t1")]
    assert r01[3] == str(K)
    e01 = min(ess["t0"], ess["t1"])
    assert e01 > 500, ess
    assert abs(float(r01[4]) - rho) <= 4 * (1 - rho * rho) / math.sqrt(e01), (r01, rho, e01)
    r23 = rows[("t2", "t3")]
    assert r23[3] == "0"
    assert abs(float(r23[4])) <= 4 / math.sqrt(min(ess["t2"], ess["t3"])), r23
