"""The `mmseq` host program on weighted (schema 2) hits files: fragment f picks transcript t with probability
proportional to mu_t * w_ft.  Every output cell against the CPU oracle's weighted route, .k / .M and the
debug files against the unweighted file with the same records, and the multi-GPU and batch paths."""
import os
import subprocess

import numpy as np
import pytest

from mmseq_b200 import hostlib, synth
from oracle import tables
from tests import weighted_oracle
from tests.test_loader_weighted import _with_repeats

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "2048", "-seed", "99", "-percentiles", "5,50,95"]
BAD = ("NA", "-inf", "inf", "nan", "-nan")


def _sample(repeats=True):
    """Identical sets (observed, mixed, hit-less), hit-less transcripts, single-isoform genes and (repeats) records that
    repeat a transcript."""
    s = synth.Synth(77, 150, 4000, weights=True)
    s = _with_repeats(s) if repeats else s
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    unobs = [t for t in range(s.T) if h.hdr2col[t] < 0]
    obs = [t for t in range(s.T) if h.hdr2col[t] >= 0]
    assert len(unobs) >= 4, "the case needs transcripts without hits"
    return s, [obs[:2], [obs[5], unobs[0], obs[9]], unobs[1:3]]


def _write(tmp_path, name, weights="sample", repeats=True):
    """The sample as schema 2 (weights: "sample", an array, or None for schema 1)."""
    s, ident = _sample(repeats)
    path = str(tmp_path / f"{name}.hits")
    synth.write_hits_binary(s, path, identical=ident, weights=s.frag_w if isinstance(weights, str) else weights)
    return s, path


def _run(args, path, base, ok=True):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=600)
    if ok:
        assert r.returncode == 0, r.stderr
    return r


def _compare_table(got_path, want_rows):
    got = tables.read_table(got_path)
    assert len(got) == len(want_rows), (len(got), len(want_rows))
    bad = []
    for r, (a, b) in enumerate(zip(got, want_rows)):
        assert len(a) == len(b), (r, a, b)
        bad += [(r, c, x, y) for c, (x, y) in enumerate(zip(a, b)) if not tables.cells_match(x, y)]
    assert not bad, bad[:10]


def _em_iters(stderr):
    return int(stderr.split("EM: ")[1].split(" ")[0])


def _log_mu_within_mcse(a, b):
    """Column log_mu of two .mmseq tables within 6 combined Monte-Carlo standard errors; returns the rows compared."""
    ra, rb = tables.read_table(a)[2:], tables.read_table(b)[2:]
    assert [x[0] for x in ra] == [y[0] for y in rb]
    n = 0
    for x, y in zip(ra, rb):
        if x[1] not in BAD and y[1] not in BAD and x[12] == "1":
            se = np.hypot(float(x[3]), float(y[3]))
            assert abs(float(x[1]) - float(y[1])) <= 6.0 * se + 1e-9, (x[0], x[1], y[1], se)
            n += 1
    return n


def test_weighted_cli_matches_oracle(tmp_path):
    path = _write(tmp_path, "w2")[1]
    one = _write(tmp_path, "w1", None)[1]
    base, base1 = str(tmp_path / "out"), str(tmp_path / "one")
    r = _run(ARGS, path, base)
    assert "Running mmseq with parameters:" in r.stdout and "Output files:" in r.stdout
    assert "fragment allocations/s" in r.stderr
    _run(ARGS + ["-notraces"], one, base1)
    want = weighted_oracle.run(path, gibbs_iter=2048, seed=99, percentiles=(5.0, 50.0, 95.0))
    assert f"Found {want['n']} transcripts in {want['m']} transcript combinations." in r.stdout
    assert open(base + ".k").read().split("\n")[:-1] == want["k"]
    assert open(base + ".M").read().split("\n")[:-1] == want["M"]
    for ext in (".k", ".M"):                                          # the weights do not appear in .k / .M
        assert open(base + ext, "rb").read() == open(base1 + ext, "rb").read(), ext
    _compare_table(base + ".mmseq", want["mmseq"])
    _compare_table(base + ".identical.mmseq", want["identical"])
    _compare_table(base + ".gene.mmseq", want["gene"])
    rows = tables.read_table(base + ".mmseq")[2:]
    assert any(rw[10] == "-nan" and rw[9] == "inf" for rw in rows)   # single-isoform genes
    assert any(rw[11] == "NA" and rw[12] == "0" for rw in rows)       # hit-less transcripts
    ids, tr = tables.read_trace_gz(base + ".trace_gibbs.gz")
    assert ids == want["names_by_col"] and tr.shape == want["trace"].shape
    assert np.allclose(tr, want["trace"], rtol=2e-5, atol=1e-300)
    ids, ptr = tables.read_trace_gz(base + ".prop.trace_gibbs.gz")
    assert ids == want["names_by_col"] and np.allclose(ptr, want["prop_trace"], rtol=2e-5, atol=1e-300)
    ids, gtr = tables.read_trace_gz(base + ".gene.trace_gibbs.gz")
    keep = [g for g, nm in enumerate(want["gene_names"]) if np.isfinite(np.log(want["gene_trace"][g, 0]))]
    assert ids == [want["gene_names"][g] for g in keep] and np.allclose(gtr, want["gene_trace"][keep], rtol=2e-5)
    ids, itr = tables.read_trace_gz(base + ".identical.trace_gibbs.gz")
    keep = [s for s in range(len(want["identical_ids"])) if want["ident_trace"][s, 0] > 0]
    assert ids == [want["identical_ids"][s] for s in keep] and np.allclose(itr, want["ident_trace"][keep], rtol=2e-5)


def test_unit_weights_agree_with_the_unweighted_file(tmp_path):
    """Every weight 1.0: the model is the unweighted one.  Only the Philox streams differ (one counter per fragment
    row instead of per set), so deterministic columns are equal and log_mu agrees within Monte-Carlo error.  (No record
    repeats a transcript here: a repeat adds its weight, so unit weights would count it twice.)"""
    path = _write(tmp_path, "u2", np.ones_like(_sample(False)[0].frag_w), repeats=False)[1]
    one = _write(tmp_path, "u1", None, repeats=False)[1]
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    ra = _run(ARGS + ["-notraces"], path, a)
    rb = _run(ARGS + ["-notraces"], one, b)
    for ext in (".k", ".M"):
        assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), ext
    assert _em_iters(ra.stderr) == _em_iters(rb.stderr)
    ta, tb = tables.read_table(a + ".mmseq"), tables.read_table(b + ".mmseq")
    assert ta[:2] == tb[:2]
    for x, y in zip(ta[2:], tb[2:]):
        assert [x[i] for i in (0, 5, 6, 7, 12, 13)] == [y[i] for i in (0, 5, 6, 7, 12, 13)], (x, y)
        if x[11] == "NA":
            assert y[11] == "NA"
        else:
            assert abs(float(x[11]) - float(y[11])) <= 1e-6 * abs(float(y[11])) + 1e-12, (x[0], x[11], y[11])
    assert _log_mu_within_mcse(a + ".mmseq", b + ".mmseq") > 50
    for ext, cols in ((".identical.mmseq", (0, 5, 6, 7, 8, 9)), (".gene.mmseq", (0, 7, 8, 9))):
        ga, gb = tables.read_table(a + ext)[2:], tables.read_table(b + ext)[2:]
        assert [[x[i] for i in cols] for x in ga] == [[y[i] for i in cols] for y in gb], ext


def test_weighted_debug_files(tmp_path):
    path = _write(tmp_path, "d2")[1]
    one = _write(tmp_path, "d1", None)[1]
    base, base1 = str(tmp_path / "dbg"), str(tmp_path / "dbg1")
    _run(["-debug", "-notraces", "-gibbs_iter", "1024", "-max_em_iter", "7"], path, base)
    _run(["-debug", "-notraces", "-gibbs_iter", "1024", "-max_em_iter", "7"], one, base1)
    for ext in (".trace_em.gz", ".sharedcounts", ".Mt-nodups", ".doublehits", ".dupIDs"):
        assert os.path.exists(base + ext), ext
    ids, em = tables.read_trace_gz(base + ".trace_em.gz")
    assert em.shape[1] == 7
    for ext in (".sharedcounts", ".Mt-nodups", ".doublehits", ".dupIDs"):   # written from the sets, as for schema 1
        assert open(base + ext).read() == open(base1 + ext).read(), ext
    assert any(int(v) > 0 for v in open(base + ".doublehits").read().split())
    sc = [ln.split("\t") for ln in open(base + ".sharedcounts").read().split("\n") if ln]
    uh = {rw[0]: int(rw[7]) for rw in tables.read_table(base + ".mmseq")[2:]}
    assert len(sc) == len(uh) and all(int(rw[1]) == uh[rw[0]] for rw in sc)   # bin 0 == unique_hits column


def test_weighted_two_gpu_flag_matches_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    path = _write(tmp_path, "g")[1]
    for g in (1, 2):
        _run(["-gpus", str(g), "-notraces", "-gibbs_iter", "1024"], path, str(tmp_path / f"g{g}"))
    a, b = str(tmp_path / "g1"), str(tmp_path / "g2")
    for ext in (".k", ".M"):
        assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), ext
    ta, tb = tables.read_table(a + ".mmseq"), tables.read_table(b + ".mmseq")
    assert ta[:2] == tb[:2]
    assert all(x[0] == y[0] and x[7] == y[7] for x, y in zip(ta[2:], tb[2:]))
    assert _log_mu_within_mcse(a + ".mmseq", b + ".mmseq") > 50


def test_batch_mixes_weighted_and_unweighted_samples(tmp_path):
    import torch
    ngpu = torch.cuda.device_count()
    paths, singles = [], []
    for i in range(4):
        s = synth.Synth(300 + i, 120 + 10 * i, 3000 + 500 * i, weights=True)
        p = str(tmp_path / f"b{i}.hits")
        synth.write_hits_binary(s, p, weights=s.frag_w if i % 2 else None)
        paths.append(p)
        base = str(tmp_path / f"single{i}")
        _run(["-notraces", "-gibbs_iter", "1024", "-seed", "5"], p, base)
        singles.append(base)
    listing = str(tmp_path / "batch.txt")
    with open(listing, "w") as f:
        for i, p in enumerate(paths):
            f.write(f"{p} {tmp_path / ('batch%d' % i)}\n")
    r = subprocess.run([BIN, "-notraces", "-gibbs_iter", "1024", "-seed", "5", "-gpus", str(ngpu), "-per_gpu", "3", "-batch", listing],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert "Batch done: 4 samples" in r.stdout
    for i, base in enumerate(singles):
        for ext in (".mmseq", ".identical.mmseq", ".gene.mmseq", ".k", ".M"):
            assert open(base + ext).read() == open(str(tmp_path / f"batch{i}") + ext).read(), (i, ext)
    assert "fragment allocations/s" in open(str(tmp_path / "batch1") + ".log").read()
    assert "hit-class allocations/s" in open(str(tmp_path / "batch0") + ".log").read()


def test_all_zero_and_negative_weights_are_refused(tmp_path):
    s, _ = _sample()
    w = s.frag_w.copy()
    w[s.frag_ptr[17]:s.frag_ptr[18]] = 0.0
    path = _write(tmp_path, "z", w)[1]
    base = str(tmp_path / "z")
    r = _run([], path, base, ok=False)
    assert r.returncode == 1
    assert f'Error: fragment record 18 of "{path}" has per-hit weights that are all zero' in r.stderr
    assert not any(os.path.exists(base + ext) for ext in (".mmseq", ".k", ".M", ".gene.mmseq"))
    w = s.frag_w.copy()
    w[5] = -0.5
    path = _write(tmp_path, "n", w)[1]
    r = _run([], path, str(tmp_path / "n"), ok=False)
    assert r.returncode == 1 and "Error: per-hit weights must be finite and non-negative." in r.stderr
    assert not os.path.exists(str(tmp_path / "n") + ".mmseq")
