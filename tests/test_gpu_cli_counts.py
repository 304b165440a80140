"""`mmseq -counts`: the .counts, .identical.counts and .gene.counts files on the GPU — ids and order as the .mmseq
tables, values as the C ABI gives them for the same chain, sums to N, batch mode, two GPUs, and no change to any other
file."""
import math
import os
import subprocess

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests.test_gpu_cli import _make_hits
from tests.test_gpu_cli_weighted import _write as _write_weighted

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
EXTS = (".counts", ".identical.counts", ".gene.counts")
TABLES = (".mmseq", ".identical.mmseq", ".gene.mmseq")


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


def _read_counts(path):
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    return lines[0], lines[1], [ln.split("\t") for ln in lines[2:-1]]


def _ids(table):
    return [ln.split("\t")[0] for ln in open(table).read().split("\n")[2:-1]]


def _check_layout(base, N):
    for ext, table in zip(EXTS, TABLES):
        head, cols, rows = _read_counts(base + ext)
        assert head == f"# Mapped fragments: {N}"
        assert cols == "feature_id\tposterior_mean_count\tposterior_sd_count\tem_count"
        assert [r[0] for r in rows] == _ids(base + table), ext
        assert all(len(r) == 4 for r in rows)
        v = np.array([[float(x) for x in r[1:]] for r in rows])
        assert (v >= 0).all()
        if ext != ".identical.counts":                                   # every fragment: on transcripts and on genes
            assert abs(v[:, 0].sum() - N) <= 1e-5 * N and abs(v[:, 2].sum() - N) <= 1e-5 * N, ext


def _abi_counts(path):
    """The host program's chain through the C ABI: load, initial mu, EM, expected counts, count moments over the
    whole chain.  Returns {ext: {feature_id: (mean, sd, em)}} for the features with hits."""
    h = hostlib.load_hits(path)
    ident_of = np.full(h.n, -1, np.int32)
    for s in range(h.I):
        for t in h.ident_members[h.ident_ptr[s]:h.ident_ptr[s + 1]]:
            if h.hdr2col[t] >= 0:
                ident_of[h.hdr2col[t]] = s
    gene_of = h.gene_of[h.col2hdr].astype(np.int32)
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.init_mu()
        H.em(1000, 0.1)
        e = H.expected_counts()
        H.count_moments_begin(ident_of, h.I, gene_of, h.G)
        H.gibbs(99, 0, 1024, stride=1, trace_len=1024)
        mom = [H.count_moments(w) for w in range(3)]

    def stats(w, r):
        S, s, lo, hi = mom[w]
        x, q = int(s[r]), (int(hi[r]) << 64) | int(lo[r])
        return x / S, math.sqrt(float(S * q - x * x) / (float(S) * float(S - 1)))
    out = {".counts": {}, ".identical.counts": {}, ".gene.counts": {}}
    for t in range(h.n):
        out[".counts"][h.names[h.col2hdr[t]]] = stats(0, t) + (e[t],)
    for g in range(h.G):
        mem = [h.hdr2col[t] for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]] if h.hdr2col[t] >= 0]
        out[".gene.counts"][h.gene_names[g]] = stats(2, g) + (sum(e[c] for c in mem),)
    out[".identical.counts"] = [stats(1, s) + (sum(e[ident_of == s]),) for s in range(h.I)]
    return out


@pytest.mark.parametrize("fmt", ["text", "binary"])
def test_counts_files_match_the_abi(tmp_path, fmt):
    path = _make_hits(tmp_path, fmt)
    base = str(tmp_path / "out")
    r = _run(["-counts"] + ARGS, path, base)
    for ext in EXTS:
        assert base + ext in r.stdout                                   # listed under "Output files"
    N = hostlib.load_hits(path).N
    _check_layout(base, N)
    want = _abi_counts(path)
    for ext in (".counts", ".gene.counts"):
        _, _, rows = _read_counts(base + ext)
        for fid, m, sd, em in rows:
            if fid in want[ext]:
                wm, wsd, wem = want[ext][fid]
                assert m == "%g" % wm and sd == "%g" % wsd, (ext, fid, m, sd, wm, wsd)
                assert abs(float(em) - wem) <= 5e-6 * abs(wem), (ext, fid, em, wem)
            else:
                assert (m, sd, em) == ("0", "0", "0"), (ext, fid)
    _, _, rows = _read_counts(base + ".identical.counts")
    for (fid, m, sd, em), (wm, wsd, wem) in zip(rows, want[".identical.counts"]):
        assert m == "%g" % wm and sd == "%g" % wsd and abs(float(em) - wem) <= 5e-6 * abs(wem) + 1e-300, fid
    assert any(r[1:] == ["0", "0", "0"] for r in rows)                    # the set without hits


def test_weighted_counts_files(tmp_path):
    s, path = _write_weighted(tmp_path, "w")
    base = str(tmp_path / "out")
    _run(["-counts"] + ARGS, path, base)
    _check_layout(base, s.N)


def test_counts_leaves_every_other_file_unchanged(tmp_path):
    path = _make_hits(tmp_path, "binary")
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    _run(ARGS, path, str(a / "out"))
    _run(["-counts"] + ARGS, path, str(b / "out"))
    files = sorted(os.listdir(a))
    assert sorted(os.listdir(b)) == sorted(files + ["out" + e for e in EXTS])
    for f in files:
        assert open(a / f, "rb").read() == open(b / f, "rb").read(), f


def test_counts_batch_equals_single_runs(tmp_path):
    paths, bases = [], []
    for i in range(3):
        s = synth.Synth(300 + i, 120 + 10 * i, 3000 + 500 * i, weights=(i == 1))
        p = str(tmp_path / f"s{i}.hits")
        synth.write_hits_binary(s, p, weights=s.frag_w if i == 1 else None)
        paths.append(p)
        _run(["-counts", "-notraces"] + ARGS, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN, "-counts", "-notraces"] + ARGS + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    for i in range(3):
        for ext in EXTS:
            assert open(bases[i] + ext, "rb").read() == open(str(tmp_path / f"single{i}") + ext, "rb").read(), (i, ext)


def test_counts_two_gpus_against_one(tmp_path):
    """EM counts within the printed precision; posterior means within Monte-Carlo error (the two runs' EM results
    differ in the last bits, fp64 all-reduce order, so their chains differ)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    path = _make_hits(tmp_path, "binary")
    res = []
    for g in (1, 2):
        base = str(tmp_path / f"g{g}")
        _run(["-counts", "-notraces", "-gpus", str(g)] + ARGS, path, base)
        res.append({ext: _read_counts(base + ext)[2] for ext in EXTS})
    for ext in EXTS:
        a = np.array([[float(x) for x in r[1:]] for r in res[0][ext]])
        b = np.array([[float(x) for x in r[1:]] for r in res[1][ext]])
        assert [r[0] for r in res[0][ext]] == [r[0] for r in res[1][ext]]
        assert np.all(np.abs(a[:, 2] - b[:, 2]) <= 1e-5 * np.abs(a[:, 2])), ext
        tol = 6.0 * np.maximum(a[:, 1], b[:, 1]) * math.sqrt(2 * 50 / 1024) + 1e-9
        assert np.all(np.abs(a[:, 0] - b[:, 0]) <= tol), ext
