"""`mmseq -allelic` on a small haplotype synth in which some pairs have a hit-less _B copy: .allelic and .gene.allelic
match the numpy reference (tests/allelic_reference.py) on the chains rebuilt through the C ABI, with the hit-less copies'
prior draws from capi.prior_draws, for text, binary and schema-2 files and with -chains 4 -pool; every other file and
stdout (apart from the two names in the list of output files) are byte-identical with and without -allelic; batch mode
equals single runs and two GPUs agree with one.  Analytic anchor: a pair with only A-only and B-only singleton records
and equal lengths draws phi ~ Beta(alpha + k_A, alpha + k_B) independently.  Recovery: the generator's 0.6 / 0.4 split."""
import math
import os
import subprocess
import time

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests import allelic_reference as aref
from tests.test_gpu_cli_tpm import _abi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
ARGS = ["-gibbs_iter", "1024", "-seed", "99"]
ALLELIC = (".allelic", ".gene.allelic")
PCTS = (5, 25, 50, 75, 95)
HEAD = ("feature_id\tpairs\ta_only_fragments\tb_only_fragments\tem_fraction_a\tposterior_mean_fraction_a\tposterior_sd_fraction_a"
        "\tprob_a_gt_b\tpercentiles_fraction_a5,25,50,75,95")
L = 1024


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_cli_allelic: {time.time() - t0:.1f} s wall")


def _run(args, path, base):
    r = subprocess.run([BIN] + args + [path, base], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    return r


def _table(path):
    lines = open(path).read().split("\n")
    assert lines[-1] == ""
    rows = [ln.split("\t") for ln in lines[2:-1]]
    return lines[:2], {c[0]: c for c in rows}, [c[0] for c in rows]


def _haplo_synth(T=300, N=6000, seed=88):
    """a haplotype synth; every fifth pair loses its _B copy (its hits move to _A), so that copy is hit-less"""
    s = synth.Synth(seed, T, N, haplo=True)
    ptr, tid = [0], []
    for r in range(s.N):
        hits = []
        for t in s.frag_tid[s.frag_ptr[r]:s.frag_ptr[r + 1]]:
            t = int(t)
            if t % 2 == 1 and (t // 2) % 5 == 0:
                t -= 1
            if t not in hits:
                hits.append(t)
        tid += hits
        ptr.append(len(tid))
    s.frag_ptr = np.array(ptr, np.int64)
    s.frag_tid = np.array(tid, np.int32)
    return s


def _write(tmp, fmt, s=None):
    s = s or _haplo_synth()
    path = str(tmp / f"h.{fmt}.hits")
    if fmt == "text":
        synth.write_hits_text(s, path)
    elif fmt == "binary":
        synth.write_hits_binary(s, path)
    else:
        w = np.random.default_rng(5).uniform(0.2, 1.0, len(s.frag_tid)).astype(np.float32)
        synth.write_hits_binary(s, path, weights=w)
    return path


def _close(cell, want, rel=2e-5):
    if isinstance(want, float) and math.isnan(want):
        return cell == "NA"
    return cell != "NA" and (float(cell) == want or abs(float(cell) - want) <= rel * abs(want) + 1e-300)


def _reference(h, mu_em, mu, seed=99):
    """(pairs, genes): per level (ids, csr, unit_of, side, npairs) and the reference dicts on the chains mu (C, n, L)"""
    C = mu.shape[0]
    a, b, stems, _ = aref.find_pairs(h.names, h.gene_of)
    col = [int(c) for c in h.hdr2col]
    prior_hdr = [t for t in range(h.T) if col[t] < 0 and (t in set(a) or t in set(b))]
    ids = {t: (col[t] if col[t] >= 0 else h.n + prior_hdr.index(t)) for t in a + b}
    rate = 0.1 + h.efflen[prior_hdr] * h.N / 1e9
    priors = np.stack([capi.prior_draws(prior_hdr, rate, 0.1, capi.chain_seed(seed, c), L) for c in range(C)]) if prior_hdr else None
    idx = aref.pct_index(PCTS, C * L)
    out = []
    for units, names in (([[p] for p in range(len(a))], stems), (aref.gene_units(a, h.gene_of, h.G), h.gene_names)):
        csr = aref.csr(units, [ids[t] for t in a], [ids[t] for t in b])
        unit_of = np.full(h.n, -1, np.int32)
        side = np.zeros(h.n, np.uint8)
        for u, ps in enumerate(units):
            for p in ps:
                for sd, t in ((0, a[p]), (1, b[p])):
                    if col[t] >= 0:
                        unit_of[col[t]], side[col[t]] = u, sd
        out.append(dict(ids=list(names), csr=csr, units=units, unit_of=unit_of, side=side,
                        ref=aref.units(mu, priors, *csr, idx)))
    return out


def _check_files(base, h, mu_em, mu, weighted=False):
    levels = _reference(h, mu_em, mu)
    k = None if weighted else h.k
    for ext, lv in zip(ALLELIC, levels):
        lines, tab, order = _table(base + ext)
        assert lines == ["# Mapped fragments: %d" % h.N, HEAD] and order == lv["ids"], ext
        a_ptr, a_mem, b_ptr, b_mem = lv["csr"]
        a_only, b_only = aref.allele_only(h.row_ptr, h.col, k, lv["unit_of"], lv["side"], len(order))
        ref = lv["ref"]
        for u, fid in enumerate(order):
            cells = tab[fid]
            am, bm = a_mem[a_ptr[u]:a_ptr[u + 1]], b_mem[b_ptr[u]:b_ptr[u + 1]]
            obs = any(m < h.n for m in list(am) + list(bm))
            assert cells[1:4] == [str(len(lv["units"][u])), str(a_only[u]), str(b_only[u])], (ext, fid, cells)
            nan = math.nan
            want = [aref.em_fraction(mu_em, am, bm) if obs else nan] + [ref[q][u] if obs else nan for q in ("mean", "sd", "prob_a")]
            for c, w in zip(cells[4:8], want):
                assert _close(c, float(w)), (ext, fid, cells, want)
            pct = cells[8].split(",")
            assert len(pct) == len(PCTS) and all(_close(c, float(w) if obs else nan) for c, w in zip(pct, ref["pct"][u])), (ext, fid, cells)
    return levels


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("allelic")
    path = _write(tmp, "binary")
    out = dict(path=path)
    for name, args in (("plain", ["-counts", "-tpm"]), ("allelic", ["-counts", "-tpm", "-allelic"]), ("c4", ["-chains", "4"]),
                       ("c4al", ["-chains", "4", "-allelic"]), ("pool", ["-chains", "4", "-pool", "-allelic", "-notraces"])):
        d = tmp / name
        d.mkdir()
        out[name] = str(d / "out")
        r = _run(args + ARGS, path, out[name])
        out[name + "_stdout"], out[name + "_stderr"] = r.stdout, r.stderr
    return out


def test_allelic_changes_no_other_file(runs):
    for a, b, after in (("plain", "allelic", ".gene.tpm"), ("c4", "c4al", ".gene.mmseq")):
        da, db = os.path.dirname(runs[a]), os.path.dirname(runs[b])
        files = sorted(os.listdir(da))
        assert sorted(os.listdir(db)) == sorted(files + ["out" + e for e in ALLELIC])
        for f in files:
            assert open(os.path.join(da, f), "rb").read() == open(os.path.join(db, f), "rb").read(), (b, f)
        extra = "".join(f"  {runs[b]}{e}\n" for e in ALLELIC)
        want = runs[a + "_stdout"].replace(f"  {runs[a]}{after}\n", f"  {runs[a]}{after}\n" + extra, 1).replace(runs[a], runs[b])
        assert runs[b + "_stdout"] == want
        assert "Note: -allelic" not in runs[b + "_stderr"]


def test_files_match_the_reference_binary_and_chains(runs):
    h, mu_em, mu = _abi(runs["path"], 4)
    levels = _check_files(runs["allelic"], h, mu_em, mu[:1])
    _check_files(runs["pool"], h, mu_em, mu)
    pairs = levels[0]
    a_ptr, a_mem, b_ptr, b_mem = pairs["csr"]
    hitless_b = [u for u in range(len(pairs["ids"])) if b_mem[u] >= h.n and a_mem[u] < h.n]
    assert len(hitless_b) >= 5                                           # the case covers prior rows on one side
    for e in ALLELIC:                                                    # -chains 4 without -pool: chain 1's files
        assert open(runs["c4al"] + e, "rb").read() == open(runs["allelic"] + e, "rb").read(), e


@pytest.mark.parametrize("fmt", ["text", "schema2"])
def test_files_match_the_reference_text_and_schema2(tmp_path, fmt):
    path = _write(tmp_path, fmt)
    _run(["-allelic", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    h, mu_em, mu = _abi(path, 1)
    _check_files(str(tmp_path / "out"), h, mu_em, mu, weighted=fmt == "schema2")


def test_batch_and_two_gpus_equal_single_runs(tmp_path):
    paths = [_write(tmp_path, "text"), _write(tmp_path, "binary"), _write(tmp_path, "schema2")]
    args = ["-allelic", "-notraces", "-chains", "2", "-pool"] + ARGS
    bases = []
    for i, p in enumerate(paths):
        _run(args, p, str(tmp_path / f"single{i}"))
        bases.append(str(tmp_path / f"batch{i}"))
    listing = str(tmp_path / "batch.txt")
    open(listing, "w").write("".join(f"{p} {b}\n" for p, b in zip(paths, bases)))
    r = subprocess.run([BIN] + args + ["-per_gpu", "2", "-batch", listing], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    for i in range(len(paths)):
        for ext in ALLELIC:
            assert open(bases[i] + ext, "rb").read() == open(str(tmp_path / f"single{i}") + ext, "rb").read(), (i, ext)
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    for i, p in enumerate(paths[1:], 1):
        _run(["-allelic", "-notraces", "-gpus", "2"] + ARGS, p, str(tmp_path / f"g2_{i}"))
        _run(["-allelic", "-notraces"] + ARGS, p, str(tmp_path / f"g1_{i}"))
        for ext in ALLELIC:
            _, a, ia = _table(str(tmp_path / f"g2_{i}") + ext)
            _, b, ib = _table(str(tmp_path / f"g1_{i}") + ext)
            assert ia == ib
            for fid in ia:                                               # EM's sums may round apart in the last bits
                assert a[fid][:4] + a[fid][5:] == b[fid][:4] + b[fid][5:], (ext, fid)
                assert a[fid][4] == b[fid][4] or _close(a[fid][4], float(b[fid][4]), 1e-5), (ext, fid)


def test_singleton_records_give_beta_fractions(tmp_path):
    """Each pair's records hit one copy only and every effective length is equal: each sweep draws mu_A ~ Gamma(alpha +
    k_A, beta + l) and mu_B ~ Gamma(alpha + k_B, beta + l) independently (a copy without records: its prior draw, the
    same law with k = 0), so the 1024 recorded fractions are independent Beta(alpha + k_A, alpha + k_B) draws.  The mean,
    prob_a_gt_b and the percentiles lie within 4 Monte-Carlo standard errors of the Beta values."""
    stats = pytest.importorskip("scipy.stats")
    k = {"p0": (30, 10), "p1": (5, 5), "p2": (0, 12), "p3": (200, 170)}
    path = str(tmp_path / "pairs.hits")
    with open(path, "w") as f:
        for p in k:
            for c in "AB":
                f.write(f"@TranscriptMetaData\t{p}_{c}\t1000\t1200\n")
        f.write("@TranscriptMetaData\tsolo\t1000\t1200\n@TranscriptMetaData\tw_A\t1000\t1200\n")
        for g, p in enumerate(k):
            f.write(f"@GeneIsoforms\tg{g}\t{p}_A\t{p}_B\n")
        f.write("@GeneIsoforms\tgs\tsolo\n@GeneIsoforms\tgw\tw_A\n")
        r = 0
        for p, (ka, kb) in k.items():
            for c, kc in (("A", ka), ("B", kb)):
                for _ in range(kc):
                    f.write(f">r{r}\n{p}_{c}\n")
                    r += 1
        f.write(f">r{r}\nsolo\n>r{r + 1}\nw_A\n")
    res = _run(["-allelic", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    assert "Note: -allelic: 1 transcripts named *_A / *_B have no partner in their gene." in res.stderr
    _, tab, order = _table(str(tmp_path / "out.allelic"))
    _, gtab, gorder = _table(str(tmp_path / "out.gene.allelic"))
    assert order == list(k) and gorder == ["g0", "g1", "g2", "g3", "gs", "gw"]
    for g in ("gs", "gw"):
        assert gtab[g][1:] == ["0", "0", "0"] + ["NA"] * 4 + [",".join(["NA"] * len(PCTS))]
    S, alpha = L, 0.1
    for g, (p, (ka, kb)) in enumerate(k.items()):
        cells = tab[p]
        assert gtab[f"g{g}"][2:] == cells[2:] and gtab[f"g{g}"][1] == "1"
        assert cells[1:4] == ["1", str(ka), str(kb)]
        assert _close(cells[4], ka / (ka + kb), 1e-3) if ka else cells[4] == "0"
        beta = stats.beta(alpha + ka, alpha + kb)
        assert abs(float(cells[5]) - beta.mean()) <= 4 * beta.std() / math.sqrt(S), (p, cells[5], beta.mean())
        pa = beta.sf(0.5)
        assert abs(float(cells[7]) - pa) <= 4 * math.sqrt(pa * (1 - pa) / S) + 1.0 / S, (p, cells[7], pa)
        for c, q in zip(cells[8].split(","), PCTS):                     # the sorted draw at index round(q (S - 1)):
            band = 4 * math.sqrt(q / 100 * (1 - q / 100) / S) + 1.0 / S   # its Beta cdf within 4 binomial SE of q
            lo, hi = beta.ppf(max(0.0, q / 100 - band)), beta.ppf(min(1.0, q / 100 + band))
            assert lo * (1 - 1e-5) <= float(c) <= hi * (1 + 1e-5), (p, q, c, beta.ppf(q / 100))


def test_recovery_of_the_generators_split(tmp_path):
    """The generator gives copy A 0.6 of the pair's mu.  A fragment drawn from a pair hits its own copy alone with
    probability 0.1, so a pair expected to draw at least 1000 fragments of its own has at least about 100 of its own
    fragments that tell the copies apart; over those pairs the median posterior_mean_fraction_a is within 0.03 of 0.6.
    The pairs are chosen by the generator's truth, not by the a_only + b_only columns: the generator also gives a pair
    hits from the other isoforms of its gene and from other genes, on copy A or B at random whatever the pair's own split
    (in this sample the median pair with a_only + b_only >= 100 draws under 4 % of those fragments itself), and 30 % of
    the pairs have mu = 0 and no split at all."""
    s = synth.Synth(2026, 4000, 1000000, haplo=True)
    path = str(tmp_path / "big.hits")
    s.write_hits_fast(path, binary=True)
    _run(["-allelic", "-notraces"] + ARGS, path, str(tmp_path / "out"))
    _, tab, _ = _table(str(tmp_path / "out.allelic"))
    w = s.mu * s.efflen
    own = s.N * (w[0::2] + w[1::2]) / w.sum()                            # expected fragments drawn from each pair
    cells = [tab[s.transcript_name(2 * p)[:-2]][5] for p in np.flatnonzero(own >= 1000)]
    assert len(cells) >= 50 and "NA" not in cells, len(cells)
    med = float(np.median([float(c) for c in cells]))
    assert abs(med - 0.6) <= 0.03, (med, len(vals))
