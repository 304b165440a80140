"""`mmseq -tpm`: the three .tpm files match the numpy reference (tests/tpm_reference.py) on the same chain rebuilt through
the C ABI, for text, binary and schema-2 files, and with -chains 4 -pool on the four chains; posterior_mean_tpm sums to
1e6 over transcripts and over genes; every other file is byte-identical with and without -tpm (also under
-counts -chains 4); -chains 4 without -pool gives the single-chain files; batch mode equals single runs and two GPUs
agree with one; on singleton classes of equal length the TPM draws are Dirichlet and the columns match its moments."""
import math
import os
import subprocess
import time

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib
from tests import tpm_reference as tref
from tests.test_gpu_cli import _make_hits
from tests.test_gpu_cli_weighted import _write as _write_weighted

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
TPM = (".tpm", ".identical.tpm", ".gene.tpm")
TABLES = (".mmseq", ".identical.mmseq", ".gene.mmseq")
PCTS = (5, 25, 50, 75, 95)
L = 1024


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_cli_tpm: {time.time() - t0:.1f} s wall")


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


def _table(path):
    """(header lines, {feature_id: cells}, ids in file order) of a table"""
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    rows = [ln.split("\t") for ln in lines[2:-1]]
    return lines[:2], {c[0]: c for c in rows}, [c[0] for c in rows]


def _close(cell, want, rel=2e-5):
    got = [float(v) for v in cell.split(",")]
    want = np.atleast_1d(np.asarray(want, np.float64))
    return len(got) == len(want) and all(g == w or abs(g - w) <= rel * abs(w) for g, w in zip(got, want))


def _abi(path, nchains, seed=99):
    """the host program's chains through the C ABI: EM once, chain c from the EM estimate with mmq_chain_seed(seed, c);
    a schema-2 file one row per fragment, by length, with its weights, as the host program loads it"""
    h = hostlib.load_hits(path, hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
    weighted = h.schema == 2
    if not weighted:
        h = hostlib.load_hits(path, hostlib.LAYOUT_COLLAPSED)
    k, w = (None, h.w) if weighted else (h.k, None)
    with capi.Handle(h.row_ptr, h.col, k, h.len, weight=w) as H:
        H.init_mu()
        H.em(1000, 0.1)
        mu_em = H.get_mu()
    mu = []
    for c in range(nchains):
        with capi.Handle(h.row_ptr, h.col, k, h.len, weight=w) as H:
            H.set_mu(mu_em)
            H.gibbs(capi.chain_seed(seed, c), 0, 1024, stride=1, trace_len=L)
            mu.append(H.get_trace())
    return h, mu_em, np.stack(mu)


def _csr(h, ptr, members):
    """a header-index CSR -> (group_ptr, observed members in column indices, in CSR order)"""
    gp, gm = [0], []
    for g in range(len(ptr) - 1):
        gm += [int(h.hdr2col[t]) for t in members[ptr[g]:ptr[g + 1]] if h.hdr2col[t] >= 0]
        gp.append(len(gm))
    return np.array(gp, np.int64), np.array(gm, np.int32)


def _check_files(base, h, mu_em, mu):
    """the three files of `base` against the reference on the chains mu (C, n, L)"""
    C = mu.shape[0]
    totals = np.stack([tref.totals_tiled(mu[c]) for c in range(C)])
    idx = tref.pct_index(PCTS, C * L)
    head = ["# Mapped fragments: %d" % h.N,
            "feature_id\tposterior_mean_tpm\tposterior_sd_tpm\tem_tpm\tpercentiles_tpm5,25,50,75,95"]
    _, mm, mm_ids = _table(base + ".mmseq")
    _, im, im_ids = _table(base + ".identical.mmseq")
    _, gm, gm_ids = _table(base + ".gene.mmseq")
    ident = _csr(h, h.ident_ptr, h.ident_members)
    genes = _csr(h, h.gene_ptr, h.gene_members)
    for ext, csr, ids in ((".tpm", None, mm_ids), (".identical.tpm", ident, im_ids), (".gene.tpm", genes, gm_ids)):
        lines, tab, order = _table(base + ext)
        assert lines == head and order == ids, ext
        ref = tref.features(mu, totals, *(csr or (None, None)), idx)
        for r, fid in enumerate(order):
            cells = tab[fid]
            if ext == ".tpm":
                q = h.hdr2col[h.names.index(fid)]
                mem = [q] if q >= 0 else []
            else:
                q = r
                mem = csr[1][csr[0][r]:csr[0][r + 1]].tolist()
            if not mem:
                assert cells[1:] == ["0", "0", "0", ",".join(["0"] * len(PCTS))], (ext, fid)
                continue
            assert _close(cells[1], ref["mean"][q]) and _close(cells[2], ref["sd"][q]), (ext, fid, cells, ref["mean"][q])
            assert _close(cells[3], tref.em_tpm(mu_em, mem)), (ext, fid, cells[3])
            assert _close(cells[4], ref["pct"][q]), (ext, fid, cells[4])
    for ext in (".tpm", ".gene.tpm"):
        total = math.fsum(float(c[1]) for c in _table(base + ext)[1].values())
        assert abs(total - 1e6) <= 1e-5 * 1e6, (ext, total)


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("tpm")
    path = _make_hits(tmp, "binary")
    out = dict(path=path)
    for name, args in (("plain", ["-counts"]), ("tpm", ["-counts", "-tpm"]), ("c4", ["-counts", "-chains", "4"]),
                       ("c4tpm", ["-counts", "-chains", "4", "-tpm"]), ("pool", ["-chains", "4", "-pool", "-tpm", "-notraces"])):
        d = tmp / name
        d.mkdir()
        out[name] = str(d / "out")
        out[name + "_stdout"] = _run(args + ARGS, path, out[name]).stdout
    return out


def test_tpm_changes_no_other_file(runs):
    for a, b in (("plain", "tpm"), ("c4", "c4tpm")):
        da, db = os.path.dirname(runs[a]), os.path.dirname(runs[b])
        files = sorted(os.listdir(da))
        assert sorted(os.listdir(db)) == sorted(files + ["out" + e for e in TPM])
        for f in files:
            assert open(os.path.join(da, f), "rb").read() == open(os.path.join(db, f), "rb").read(), (b, f)
        extra = "".join(f"  {runs[b]}{e}\n" for e in TPM)
        want = runs[a + "_stdout"].replace(f"  {runs[a]}.gene.counts\n", f"  {runs[a]}.gene.counts\n" + extra).replace(runs[a], runs[b])
        assert runs[b + "_stdout"] == want


def test_files_match_the_reference_binary_and_chains(runs):
    h, mu_em, mu = _abi(runs["path"], 4)
    _check_files(runs["tpm"], h, mu_em, mu[:1])
    _check_files(runs["pool"], h, mu_em, mu)
    for e in TPM:                                                        # -chains 4 without -pool: chain 1's files
        assert open(runs["c4tpm"] + e, "rb").read() == open(runs["tpm"] + e, "rb").read(), e


@pytest.mark.parametrize("fmt", ["text", "schema2"])
def test_files_match_the_reference_text_and_schema2(tmp_path, fmt):
    path = _make_hits(tmp_path, "text") if fmt == "text" else _write_weighted(tmp_path, "w")[1]
    _run(["-tpm", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    h, mu_em, mu = _abi(path, 1)
    _check_files(str(tmp_path / "out"), h, mu_em, mu)


def test_batch_and_two_gpus_equal_single_runs(tmp_path):
    paths = [_make_hits(tmp_path, "text"), _make_hits(tmp_path, "binary"), _write_weighted(tmp_path, "w")[1]]
    args = ["-tpm", "-notraces", "-chains", "2", "-pool"] + ARGS
    bases = []
    for i, p in enumerate(paths):
        _run(args, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN] + args + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    for i in range(len(paths)):
        for ext in TPM:
            assert open(bases[i] + ext, "rb").read() == open(str(tmp_path / f"single{i}") + ext, "rb").read(), (i, ext)
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    for i, p in enumerate(paths[1:], 1):
        _run(["-tpm", "-notraces", "-gpus", "2"] + ARGS, p, str(tmp_path / f"g2_{i}"))
        _run(["-tpm", "-notraces"] + ARGS, p, str(tmp_path / f"g1_{i}"))
        for ext in TPM:
            _, a, ia = _table(str(tmp_path / f"g2_{i}") + ext)
            _, b, ib = _table(str(tmp_path / f"g1_{i}") + ext)
            assert ia == ib
            for fid in ia:                                               # EM's sums may round apart in the last bits
                assert a[fid][:3] + a[fid][4:] == b[fid][:3] + b[fid][4:], (ext, fid)
                assert _close(a[fid][3], float(b[fid][3]), 1e-5), (ext, fid)


def test_singleton_classes_give_dirichlet_draws(tmp_path):
    """Every fragment hits one transcript and all effective lengths are equal: each sweep draws mu_t ~ Gamma(alpha + k_t,
    beta + l) independently, so every recorded draw of mu / sum mu is an independent Dirichlet(alpha + k) draw over the
    observed transcripts.  posterior_mean_tpm lies within 4.5 standard errors of 1e6 a_t / A (a = alpha + k, A = sum a),
    posterior_sd_tpm within 4.5 of its own standard errors of the Dirichlet sd, and em_tpm is 1e6 k_t / N."""
    rng = np.random.default_rng(12)
    T = 60
    k = rng.integers(1, 300, T)
    k[[3, 17, 40]] = 0                                                   # hit-less: 0 in every column
    path = str(tmp_path / "single.hits")
    with open(path, "w") as f:
        for t in range(T):
            f.write(f"@TranscriptMetaData\tt{t}\t1000\t1200\n")
        for g in range(T // 2):
            f.write(f"@GeneIsoforms\tg{g}\tt{2 * g}\tt{2 * g + 1}\n")
        r = 0
        for t in range(T):
            for _ in range(k[t]):
                f.write(f">r{r}\nt{t}\n")
                r += 1
    _run(["-tpm", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    _, tab, _ = _table(str(tmp_path / "out.tpm"))
    a = 0.1 + k[k > 0]
    A = a.sum()
    N = k.sum()
    S = L
    for t in range(T):
        cells = tab[f"t{t}"]
        if k[t] == 0:
            assert cells[1:4] == ["0", "0", "0"]
            continue
        at = 0.1 + k[t]
        mean, sd = 1e6 * at / A, 1e6 * math.sqrt(at * (A - at) / (A * A * (A + 1)))
        assert abs(float(cells[1]) - mean) <= 4.5 * sd / math.sqrt(S), (t, cells[1], mean)
        # sd of a sample sd: sd sqrt((kurtosis excess + 2) / (4 S)); the excess of a Beta(at, A - at) marginal is near
        # the Gamma(at)'s 6 / at for small at
        assert abs(float(cells[2]) - sd) <= 4.5 * sd * math.sqrt((6.0 / at + 2.0) / (4 * S)), (t, cells[2], sd)
        em = 1e6 * k[t] / N
        assert float(cells[3]) == float("%g" % em) or abs(float(cells[3]) - em) <= 5e-6 * em, (t, cells[3], em)
