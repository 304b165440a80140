"""`mmseq -chains`: the existing files stay byte-identical, the .convergence files match the numpy reference applied
to the same chains rerun through the C ABI, transcripts with an exact posterior converge, batch mode and schema-2 files,
and two GPUs against one."""
import math
import os
import subprocess
import time

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests import chain_reference as ref
from tests.test_gpu_cli import _make_hits
from tests.test_gpu_cli_weighted import _write as _write_weighted

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
EXTS = (".convergence", ".identical.convergence", ".gene.convergence")
TABLES = (".mmseq", ".identical.mmseq", ".gene.mmseq")
HEADER = "feature_id\tlog_mu\tsd\trhat\tess_bulk\tess_tail"


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_cli_chains: {time.time() - t0:.1f} s wall")


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


def _rows(path):
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    return lines[0], lines[1], [ln.split("\t") for ln in lines[2:-1]]


def _table(path):
    """feature_id -> (log_mu, sd, observed) cells of a .mmseq table"""
    lines = open(path).read().split("\n")[1:-1]
    head = lines[0].split("\t")
    obs = head.index("observed")
    return [(c[0], c[1], c[2], c[obs]) for c in (ln.split("\t") for ln in lines[1:])]


@pytest.mark.parametrize("counts", [False, True])
def test_chains_leave_every_existing_file_unchanged(tmp_path, counts):
    path = _make_hits(tmp_path, "binary")
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    extra = ["-counts"] if counts else []
    _run(extra + ARGS, path, str(a / "out"))
    r = _run(extra + ["-chains", "4"] + ARGS, path, str(b / "out"))
    files = sorted(os.listdir(a))
    assert sorted(os.listdir(b)) == sorted(files + ["out" + e for e in EXTS])
    for f in files:
        assert open(a / f, "rb").read() == open(b / f, "rb").read(), f
    assert "  chains:        4" in r.stdout
    assert sum(ln.startswith("Convergence of the ") for ln in r.stderr.splitlines()) == 3


def _abi_chains(path, nchains, seed=99, L=1024):
    """The host program's chains through the C ABI: EM once, every chain from the EM estimate with its own seed, groups
    with each chain's own prior draws.  Returns {ext: (rows fp64[5, R] of the reference, margins)} per table."""
    h = hostlib.load_hits(path)
    ipt, gpt = [0], [0]
    imem, gmem = [], []
    for s in range(h.I):
        imem += [h.hdr2col[t] for t in h.ident_members[h.ident_ptr[s]:h.ident_ptr[s + 1]] if h.hdr2col[t] >= 0]
        ipt.append(len(imem))
    unobs = [t for t in range(h.T) if h.hdr2col[t] < 0]
    slot = {t: u for u, t in enumerate(unobs)}
    for g in range(h.G):
        gmem += [h.hdr2col[t] for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]] if h.hdr2col[t] >= 0]
        gpt.append(len(gmem))
    rate = 0.1 + h.efflen[unobs] * h.N / 1e9
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.init_mu()
        H.em(1000, 0.1)
        mu = H.get_mu()
    traces = [[], [], []]
    for c in range(nchains):
        sd = capi.chain_seed(seed, c)
        simu = capi.prior_draws(np.array(unobs, np.int64), rate, 0.1, sd, L) if unobs else np.zeros((0, L))
        extra = np.zeros((h.G, L))
        for g in range(h.G):
            for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]]:
                if h.hdr2col[t] < 0:
                    extra[g] += simu[slot[t]]
        with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
            H.set_mu(mu)
            H.gibbs(sd, 0, 1024, stride=1024 // L, trace_len=L)
            H.set_groups(capi.MMQ_GROUP_IDENTICAL, ipt, imem)
            H.set_groups(capi.MMQ_GROUP_GENE, gpt, gmem, extra)
            traces[0].append(H.get_trace())
            traces[1].append(H.get_group_trace(1))
            traces[2].append(H.get_group_trace(2))
    out = {}
    for ext, tr in zip(EXTS, traces):
        d, margin = ref.diagnose_rows(np.stack(tr))
        out[ext] = (np.stack([d[k] for k in ref.OUTPUTS]), margin)
    return h, out


def _close(cell, want, rel=2e-5):
    if math.isnan(want):
        return cell == "NA"
    if math.isinf(want):
        return float(cell) == want
    return abs(float(cell) - want) <= rel * abs(want) + 1e-300


def test_convergence_files_match_the_reference(tmp_path):
    path = _make_hits(tmp_path, "binary")
    base = str(tmp_path / "out")
    r = _run(["-chains", "4", "-notraces"] + ARGS, path, base)
    for ext in EXTS:
        assert base + ext in r.stdout                                   # listed under "Output files"
    h, want = _abi_chains(path, 4)
    for ext, table in zip(EXTS, TABLES):
        head, cols, rows = _rows(base + ext)
        assert head == f"# Mapped fragments: {h.N}" and cols == HEADER
        tab = _table(base + table)
        assert [x[0] for x in rows] == [t[0] for t in tab], ext
        vals, margin = want[ext]
        for i, (cells, (fid, log_mu, sd, observed)) in enumerate(zip(rows, tab)):
            assert len(cells) == 6
            if observed == "0":
                assert cells[1:] == [log_mu, sd, "NA", "NA", "NA"], (ext, fid)
                continue
            q = h.hdr2col[i] if ext == ".convergence" else i               # transcript rows are in header order
            got = [cells[3], cells[4], cells[5], cells[1], cells[2]]      # rhat, ess_bulk, ess_tail, log_mean, log_sd
            for k, (cell, wv) in enumerate(zip(got, vals[:, q])):
                if k in (1, 2) and margin[q] < 1e-9:
                    continue
                assert _close(cell, wv), (ext, fid, ref.OUTPUTS[k], cell, wv)


def test_unique_fragment_transcripts_converge(tmp_path):
    """A transcript all of whose fragments hit it alone has an exact Gamma posterior, drawn afresh every sweep: its
    chains agree and its draws are independent."""
    s = synth.Synth(78, 400, 3000)
    path = str(tmp_path / "u.hits")
    synth.write_hits_binary(s, path)
    base = str(tmp_path / "out")
    _run(["-chains", "4", "-notraces"] + ARGS, path, base)
    h = hostlib.load_hits(path)
    d = np.diff(h.row_ptr)
    multi = set(h.col[np.repeat(d > 1, d)].tolist())
    unique = {h.names[h.col2hdr[t]] for t in range(h.n) if t not in multi}
    assert len(unique) >= 5, len(unique)
    S = 4 * 1024
    seen = 0
    for fid, _, _, rhat, ess_bulk, _ in _rows(base + ".convergence")[2]:
        if fid in unique:
            seen += 1
            assert abs(float(rhat) - 1) <= 0.01 and float(ess_bulk) >= 0.5 * S, (fid, rhat, ess_bulk)
    assert seen == len(unique)


def test_batch_and_schema2_with_chains_equal_single_runs(tmp_path):
    paths, bases = [], []
    for i in range(2):
        s = synth.Synth(300 + i, 120 + 10 * i, 3000 + 500 * i)
        p = str(tmp_path / f"s{i}.hits")
        synth.write_hits_binary(s, p)
        paths.append(p)
    _, wp = _write_weighted(tmp_path, "w")
    paths.append(wp)
    for i, p in enumerate(paths):
        _run(["-chains", "2", "-notraces"] + ARGS, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN, "-chains", "2", "-notraces"] + ARGS + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    for i in range(len(paths)):
        for ext in TABLES + EXTS + (".k", ".M"):
            assert open(bases[i] + ext, "rb").read() == open(str(tmp_path / f"single{i}") + ext, "rb").read(), (i, ext)
    _, _, rows = _rows(str(tmp_path / "single2.convergence"))             # the schema-2 sample
    assert sum(x[3] != "NA" for x in rows) > 0


def test_chains_on_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    path = _make_hits(tmp_path, "binary")
    for g in (1, 2):
        _run(["-chains", "2", "-gpus", str(g)] + ARGS, path, str(tmp_path / f"g{g}"))
    for f in sorted(os.listdir(tmp_path)):
        if f.startswith("g1."):
            assert open(tmp_path / f, "rb").read() == open(tmp_path / ("g2." + f[3:]), "rb").read(), f
