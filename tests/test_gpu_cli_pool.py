"""`mmseq -chains 4 -pool`: every file but the three tables (and the .counts files under -counts) stays byte-identical
to the run without -pool; the tables' deterministic columns stay, their stochastic columns match the numpy reference on
the same four chains rerun through the C ABI; pooled log_mu and sd equal the .convergence files'; transcripts with an
exact posterior land within 4 pooled mcse of its mean; the pooled mcse falls as 1/sqrt(C); the pooled counts are the
exact sums of the chains' moments; batch mode, text and schema-2 files and two GPUs give the tables of single runs."""
import math
import os
import subprocess
import time

import numpy as np
import pytest
from scipy.special import digamma

from mmseq_b200 import capi, hostlib, synth
from tests import pool_reference as pref
from tests.test_gpu_cli import _make_hits
from tests.test_gpu_cli_weighted import _write as _write_weighted

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
TABLES = (".mmseq", ".identical.mmseq", ".gene.mmseq")
COUNTS = (".counts", ".identical.counts", ".gene.counts")
C4, L = 4, 1024
PCTS = (5, 25, 50, 75, 95)


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_cli_pool: {time.time() - t0:.1f} s wall")


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


def _table(path):
    """(column names, {feature_id: cells}) of a table"""
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    head = lines[1].split("\t")
    return head, {c[0]: c for c in (ln.split("\t") for ln in lines[2:-1])}


def _num(cell):
    return [float(v) for v in cell.split(",")]


def _close(cell, want, rel=2e-5):
    got = _num(cell)
    want = np.atleast_1d(np.asarray(want, np.float64))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        if math.isnan(w):
            if not math.isnan(g):
                return False
        elif math.isinf(w):
            if g != w:
                return False
        elif not abs(g - w) <= rel * abs(w) + 1e-300:
            return False
    return True


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """the sample run with -chains 4 -counts, with and without -pool, and the four chains rebuilt through the C ABI"""
    tmp = tmp_path_factory.mktemp("pool")
    path = _make_hits(tmp, "binary")
    a, b = tmp / "a", tmp / "b"
    a.mkdir(); b.mkdir()
    _run(["-counts", "-chains", "4"] + ARGS, path, str(a / "out"))
    r = _run(["-counts", "-chains", "4", "-pool"] + ARGS, path, str(b / "out"))
    return dict(path=path, plain=str(a / "out"), pool=str(b / "out"), stdout=r.stdout, abi=_abi_chains(path, C4))


def _abi_chains(path, nchains, seed=99):
    """the host program's chains through the C ABI: EM once, every chain from the EM estimate with its own seed, groups
    with each chain's own prior draws, count moments over every sweep"""
    h = hostlib.load_hits(path)
    ipt, gpt, imem, gmem = [0], [0], [], []
    ident_of = np.full(h.n, -1, np.int32)
    for s in range(h.I):
        mem = [h.hdr2col[t] for t in h.ident_members[h.ident_ptr[s]:h.ident_ptr[s + 1]] if h.hdr2col[t] >= 0]
        imem += mem
        ipt.append(len(imem))
        ident_of[mem] = s
    unobs = [t for t in range(h.T) if h.hdr2col[t] < 0]
    slot = {t: u for u, t in enumerate(unobs)}
    for g in range(h.G):
        gmem += [h.hdr2col[t] for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]] if h.hdr2col[t] >= 0]
        gpt.append(len(gmem))
    gene_of = np.array([h.gene_of[h.col2hdr[t]] for t in range(h.n)], np.int32)
    rate = 0.1 + h.efflen[unobs] * h.N / 1e9
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.init_mu()
        H.em(1000, 0.1)
        mu = H.get_mu()
    out = dict(h=h, slot=slot, mu=[], ident=[], gene=[], simu=[], moments=[[], [], []])
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
            H.count_moments_begin(ident_of, h.I, gene_of, h.G)
            H.gibbs(sd, 0, 1024, stride=1024 // L, trace_len=L)
            H.set_groups(capi.MMQ_GROUP_IDENTICAL, ipt, imem)
            H.set_groups(capi.MMQ_GROUP_GENE, gpt, gmem, extra)
            out["mu"].append(H.get_trace())
            out["ident"].append(H.get_group_trace(1))
            out["gene"].append(H.get_group_trace(2))
            for w in range(3):
                out["moments"][w].append(H.count_moments(w))
        out["simu"].append(simu)
    for k in ("mu", "ident", "gene", "simu"):
        out[k] = np.stack(out[k])
    return out


def test_pool_changes_only_the_tables_and_counts(runs):
    a, b = os.path.dirname(runs["plain"]), os.path.dirname(runs["pool"])
    files = sorted(os.listdir(a))
    assert sorted(os.listdir(b)) == files
    for f in files:
        if any(f == "out" + e for e in TABLES + COUNTS):
            continue
        assert open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read(), f
    assert "  chains:        4\n  pooled:        yes" in runs["stdout"]


def test_tables_match_the_reference(runs):
    A, h = runs["abi"], runs["abi"]["h"]
    S = C4 * L
    idx = pref.pct_index(PCTS, S)
    gene_of_col = np.array([h.gene_of[h.col2hdr[t]] for t in range(h.n)])
    size = np.diff(h.gene_ptr)
    checked = 0
    for ext, chains in zip(TABLES, (A["mu"], A["ident"], A["gene"])):
        head, plain = _table(runs["plain"] + ext)
        head2, pool = _table(runs["pool"] + ext)
        assert head == head2 and list(plain) == list(pool), ext
        col = {c: i for i, c in enumerate(head)}
        det = [c for c in ("effective_length", "true_length", "unique_hits", "log_mu_em", "observed", "ntranscripts") if c in col]
        if ext == ".gene.mmseq":
            det.remove("effective_length")                               # the weights are the pooled means
        rows = {name: i for i, name in enumerate(h.names)} if ext == ".mmseq" else None
        for r, (fid, cells) in enumerate(pool.items()):
            old = plain[fid]
            for c in det:
                assert cells[col[c]] == old[col[c]], (ext, fid, c)
            pcol = [i for i, c in enumerate(head) if c.startswith("percentiles")]
            if cells[col["observed"]] == "0":
                if ext != ".mmseq":                                      # unobserved sets and genes: unchanged
                    assert cells == old, (ext, fid)
                    continue
                t = rows[fid]
                assert cells[1:5] == old[1:5]                            # closed forms
                g = h.gene_of[t]
                w = pref.pooled_props(A["simu"][:, A["slot"][t], :], A["gene"][:, g, :], size[g] > 1, idx)
                assert _close(cells[pcol[0]], pref.percentiles(A["simu"][:, A["slot"][t], :], idx)), (fid, "pct")
            else:
                q = h.hdr2col[rows[fid]] if ext == ".mmseq" else r
                lm, sd, ess, margin = pref.pooled_log(chains[:, q, :])
                mcse, iact = pref.mcse_iact(sd, ess, S)
                for c, v in (("log_mu", lm), ("sd", sd), ("mcse", mcse), ("iact", iact)):
                    if c in ("mcse", "iact") and margin < 1e-9:                # an ESS branch decided by the last bits
                        continue
                    assert _close(cells[col[c]], v), (ext, fid, c, cells[col[c]], v)
                assert _close(cells[pcol[0]], pref.percentiles(chains[:, q, :], idx)), (ext, fid, "pct")
                checked += 1
                if ext != ".mmseq":
                    continue
                g = gene_of_col[q]
                w = pref.pooled_props(chains[:, q, :], A["gene"][:, g, :], size[g] > 1, idx)
            for c, k in (("mean_proportion", "mean"), ("mean_probit_proportion", "mean_probit")):
                assert _close(cells[col[c]], w[k]), (fid, c, cells[col[c]], w[k])
            # sd_probit: sqrt(sum z^2 - (sum z)^2 / S) cancels when the probits hardly vary (proportions clamped at
            # 1 - 1e-9); there both sides are rounding noise of about 1e-7, or NaN when the noise is negative
            got, want = float(cells[col["sd_probit_proportion"]]), w["sd_probit"]
            if size[g] == 1:
                assert math.isnan(got) and math.isnan(want), fid
            else:
                assert (math.isnan(got) or got < 1e-6) and (math.isnan(want) or want < 1e-6) or \
                    _close(cells[col["sd_probit_proportion"]], want), (fid, got, want)
            assert _close(cells[pcol[1]], w["pct"]), (fid, "pct_prop")
    assert checked > 100
    # gene effective_length: the expression-weighted length over the pooled means
    _, pool_t = _table(runs["pool"] + ".mmseq")
    _, pool_g = _table(runs["pool"] + ".gene.mmseq")
    for g in range(h.G):
        name = h.gene_names[g]
        if pool_g[name][9] != "1":
            continue
        num = den = 0.0
        for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]]:
            m = math.exp(float(pool_t[h.names[t]][1])) if h.hdr2col[t] >= 0 else \
                math.exp(digamma(0.1) - math.log(0.1 + h.efflen[t] * h.N / 1e9))
            num += h.efflen[t] * m
            den += m
        assert _close(pool_g[name][5], num / den, 1e-4), name


def test_pooled_log_mu_and_sd_equal_the_convergence_files(runs):
    for ext, conv in zip(TABLES, (".convergence", ".identical.convergence", ".gene.convergence")):
        _, tab = _table(runs["pool"] + ext)
        _, cv = _table(runs["pool"] + conv)
        n = 0
        for fid, cells in tab.items():
            obs = cells[12] if ext == ".mmseq" else cells[8] if ext == ".identical.mmseq" else cells[9]
            if obs == "1":
                assert cells[1:3] == cv[fid][1:3], (ext, fid)
                n += 1
        assert n > 0, ext


def test_pooled_counts_are_the_exact_sums_of_the_chains(runs):
    A, h = runs["abi"], runs["abi"]["h"]
    for w, ext in enumerate(COUNTS):
        S, tot, sq = pref.add_count_moments(A["moments"][w])
        assert S == C4 * 1024
        mean, sd = pref.count_columns(S, tot, sq)
        _, plain = _table(runs["plain"] + ext)
        _, pool = _table(runs["pool"] + ext)
        for r, (fid, cells) in enumerate(pool.items()):
            assert cells[3] == plain[fid][3], (ext, fid)                  # em_count
            q = h.hdr2col[r] if w == 0 else r
            if q < 0:
                assert cells[1:] == ["0", "0", "0"]
                continue
            assert float(cells[1]) == float("%g" % mean[q]) and float(cells[2]) == float("%g" % sd[q]), (ext, fid)


def test_exact_posterior_transcripts_and_the_mcse_ratio(tmp_path):
    """A transcript all of whose fragments hit it alone has the Gamma(alpha + k, beta + l) posterior, drawn afresh each
    sweep: E log mu = digamma(alpha + k) - log(beta + l).  The pooled log_mu lies within 4 pooled mcse of it.  Over all
    observed transcripts the median of pooled mcse over the chain-1 mcse of the run without -pool is 1/sqrt(C) for
    well-mixed chains (the error of a mean of C times as many draws); the two estimators differ (Geyer's sequence on all
    chains, Sokal's adaptive window on one), and the median of a few hundred ratios scatters by a few per cent, so the
    band is 0.8 / sqrt(C) .. 1.25 / sqrt(C)."""
    s = synth.Synth(78, 400, 3000)
    path = str(tmp_path / "u.hits")
    synth.write_hits_binary(s, path)
    _run(["-chains", "4", "-pool", "-notraces"] + ARGS, path, str(tmp_path / "pool"))
    _run(["-chains", "4", "-notraces"] + ARGS, path, str(tmp_path / "one"))
    h = hostlib.load_hits(path)
    d = np.diff(h.row_ptr)
    multi = set(h.col[np.repeat(d > 1, d)].tolist())
    k = np.zeros(h.n)
    np.add.at(k, h.col[np.repeat(d == 1, d)], h.k[d == 1])
    head, pool = _table(str(tmp_path / "pool.mmseq"))
    _, one = _table(str(tmp_path / "one.mmseq"))
    inside = total = 0
    for t in range(h.n):
        if t in multi:
            continue
        cells = pool[h.names[h.col2hdr[t]]]
        want = digamma(0.1 + k[t]) - math.log(0.1 + h.len[t])
        total += 1
        inside += abs(float(cells[1]) - want) <= 4 * float(cells[3])
    assert total >= 5 and inside >= 0.999 * total, (inside, total)
    ratio = [float(c[3]) / float(one[f][3]) for f, c in pool.items() if c[12] == "1" and float(one[f][3]) > 0]
    ratio = [v for v in ratio if math.isfinite(v)]
    assert len(ratio) > 100
    med = float(np.median(ratio))
    assert 0.8 / math.sqrt(C4) <= med <= 1.25 / math.sqrt(C4), med


def test_batch_text_schema2_and_two_gpus_equal_single_runs(tmp_path):
    paths = [_make_hits(tmp_path, "text")]
    s = synth.Synth(301, 130, 3500)
    paths.append(str(tmp_path / "s1.hits"))
    synth.write_hits_binary(s, paths[-1])
    paths.append(_write_weighted(tmp_path, "w")[1])
    args = ["-chains", "2", "-pool", "-notraces", "-counts"] + ARGS
    bases = []
    for i, p in enumerate(paths):
        _run(args, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN] + args + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    for i in range(len(paths)):
        for ext in TABLES + COUNTS:
            assert open(bases[i] + ext, "rb").read() == open(str(tmp_path / f"single{i}") + ext, "rb").read(), (i, ext)
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(args[:-len(ARGS)] + ["-gpus", "2"] + ARGS, paths[1], str(tmp_path / "g2"))
    for ext in TABLES + COUNTS:
        assert open(str(tmp_path / "g2") + ext, "rb").read() == open(str(tmp_path / "single1") + ext, "rb").read(), ext
