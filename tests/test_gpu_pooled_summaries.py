"""mmq_pooled_summaries_dev and mmq_pooled_summaries against the numpy reference (tests/pool_reference.py): every
(chains, trace length) shape the C ABI accepts at the edges and in the middle, with enough rows that every CTA of the
grid-capped loop takes several; mixed rows (iid, AR(1), shifted and scaled chains, log-normal, ties, zeros, constant,
NaN, +inf); percentiles bit for bit, the same bits under repetition, row permutation, another grid, the handle form and
a second GPU; arguments outside the limits."""
import ctypes
import math
import multiprocessing
import os
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from mmseq_b200 import capi
from tests import pool_reference as pref
from tests.test_gpu_chain_diagnostics import KINDS, _chains, _problem, grid_rows, mixed

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = [(C, L) for C in (2, 3, 4, 8) for L in (8, 64, 1024, 2048) if C * L <= 8192]
PCTS = (0, 2.5, 5, 25, 50, 75, 95, 97.5, 100)
_POOL = []


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    for ex in _POOL:
        ex.shutdown()
    print(f"\ntest_gpu_pooled_summaries: {time.time() - t0:.1f} s wall")


def run_dev(x, mode=0, idx=None):
    C, rows, L = x.shape
    idx = pref.pct_index(PCTS, C * L) if idx is None else np.asarray(idx, np.int32)
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    d_idx = torch.from_numpy(idx).cuda()
    out = torch.full((3 * rows,), 12345.0, dtype=torch.float64, device="cuda")
    pct = torch.empty(rows * len(idx), dtype=torch.float64, device="cuda")
    capi.pooled_summaries_dev([t.data_ptr() for t in chains], rows, L, mode, len(idx), d_idx.data_ptr(), out.data_ptr(),
                              pct.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(3, rows), pct.cpu().numpy().reshape(rows, len(idx))


def reference(x, idx):
    """pool_reference over the rows of x, split over host processes (spawned: this process runs CUDA threads)"""
    workers = max(1, min(16, os.cpu_count() or 1))
    if not _POOL:
        _POOL.append(ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")))
    parts = [p for p in np.array_split(np.arange(x.shape[1]), workers * 4) if len(p)]
    res = list(_POOL[0].map(pref.pooled_rows, [x[:, p, :] for p in parts], [idx] * len(parts)))
    return {k: np.concatenate([r[k] for r in res]) for k in res[0]}


def same_bits_or_both_nan(a, b):
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


def close(g, w, rel, skip=None):
    skip = np.zeros(g.shape, bool) if skip is None else skip
    assert np.array_equal(np.isnan(g) | skip, np.isnan(w) | skip)
    with np.errstate(invalid="ignore"):
        ok = np.isnan(w) | (g == w) | (np.abs(g - w) <= rel * np.abs(w) + 1e-13) | skip
    bad = np.flatnonzero(~ok)
    assert not len(bad), (bad[:5], g[bad[:5]], w[bad[:5]])


@pytest.mark.parametrize("C,L", CASES)
def test_against_reference(C, L):
    rng = np.random.default_rng(2000 * C + L)
    rows = grid_rows()
    x = mixed(rng, C, L, rows)
    idx = pref.pct_index(PCTS, C * L)
    out, pct = run_dev(x, 0, idx)
    want = reference(x, idx)
    assert same_bits_or_both_nan(pct, want["pct"])
    close(out[0], want["log_mean"], 1e-13)
    close(out[1], want["sd"], 1e-13)
    exempt = want["margin"] < 1e-9
    assert exempt.sum() <= max(1, int(0.001 * rows)), exempt.sum()
    close(out[2], want["ess_mean"], 1e-9, exempt)
    kinds = np.arange(rows) % len(KINDS)
    for k in ("nan", "inf", "constant"):
        assert np.isnan(out[2, kinds == KINDS.index(k)]).all(), k
    zero = (x == 0).any(axis=(0, 2))                                     # a zero draw: log x = -inf
    assert zero.any() and np.isnan(out[2, zero]).all() and (out[0, zero] == -np.inf).all()
    assert np.isnan(out[:2, kinds == KINDS.index("nan")]).all()
    if L >= 1024:                                                        # iid draws: ESS near S
        iid = out[2, kinds == KINDS.index("iid")]
        assert (iid > 0.7 * C * L).all() and (iid < 1.4 * C * L).all()


@pytest.mark.parametrize("C,L", [(2, 8), (3, 64), (4, 1024), (8, 1024)])
def test_proportion_mode_against_reference(C, L):
    rng = np.random.default_rng(77 * C + L)
    rows = grid_rows()
    x = rng.beta(0.5, 2.0, (C, rows, L))
    x[:, 1::9, :] = np.round(x[:, 1::9, :], 1)                           # ties
    x[:, 2::9, :] = 1.0                                                  # one isoform
    x[0, 3::9, 5] = math.nan                                             # a gene trace of 0: 0 / 0
    idx = pref.pct_index(PCTS, C * L)
    out, pct = run_dev(x, 1, idx)
    want = np.array([np.sum(x[:, r, :]) / (C * L) for r in range(rows)])
    close(out[0], want, 1e-13)
    assert (out[1:] == 12345.0).all()                                    # q = 1, 2 are left unwritten
    assert same_bits_or_both_nan(pct, np.stack([pref.percentiles(x[:, r, :], idx) for r in range(rows)]))


def test_bits_repeat_row_order_and_grid():
    rng = np.random.default_rng(7)
    C, L = 4, 1024
    rows = grid_rows()
    x = mixed(rng, C, L, rows)
    a, pa = run_dev(x)
    b, pb = run_dev(x)
    assert a.tobytes() == b.tobytes() and pa.tobytes() == pb.tobytes()
    perm = rng.permutation(rows)
    c, pc = run_dev(x[:, perm, :])
    assert a[:, perm].tobytes() == c.tobytes() and pa[perm].tobytes() == pc.tobytes()
    d, pd = run_dev(x[:, :17, :])                                        # another grid: 17 CTAs
    assert a[:, :17].tobytes() == d.tobytes() and pa[:17].tobytes() == pd.tobytes()


def test_log_statistics_equal_the_chain_diagnostics_bits():
    rng = np.random.default_rng(11)
    C, L = 3, 1024
    rows = grid_rows()
    x = mixed(rng, C, L, rows)
    out, _ = run_dev(x)
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    diag = torch.empty(5 * rows, dtype=torch.float64, device="cuda")
    capi.chain_diagnostics_dev([t.data_ptr() for t in chains], rows, L, diag.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    diag = diag.cpu().numpy().reshape(5, rows)
    assert same_bits_or_both_nan(out[0], diag[3]) and same_bits_or_both_nan(out[1], diag[4])


def test_arguments_outside_the_limits():
    lib = capi.lib()
    buf = torch.zeros(8 * 8192, dtype=torch.float64, device="cuda")
    out = torch.zeros(3 * 8, dtype=torch.float64, device="cuda")
    pct = torch.zeros(8 * 2, dtype=torch.float64, device="cuda")
    idx = torch.zeros(2, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(C, L, rows=8, mode=0, npct=2, null_at=-1, out_ptr=out.data_ptr(), pct_ptr=pct.data_ptr(), idx_ptr=idx.data_ptr()):
        ptrs = [buf.data_ptr()] * max(C, 1)
        if null_at >= 0:
            ptrs[null_at] = None
        arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        return lib.mmq_pooled_summaries_dev(arr, C, rows, L, mode, npct, idx_ptr, out_ptr, pct_ptr, stream)
    assert call(2, 8) == 0 and call(2, 8, mode=1) == 0
    for C, L in [(1, 1024), (9, 512), (0, 64), (2, 4), (2, 12), (2, 4096), (8, 2048), (5, 2048), (3, 100)]:
        assert call(C, L) == 1, (C, L)
    assert call(2, 64, rows=-1) == 1
    assert call(2, 64, mode=2) == 1 and call(2, 64, mode=-1) == 1
    assert call(2, 64, npct=-1) == 1
    assert call(2, 64, null_at=1) == 1
    assert call(2, 64, out_ptr=None) == 1
    assert call(2, 64, pct_ptr=None) == 1 and call(2, 64, idx_ptr=None) == 1
    assert call(2, 64, npct=0, pct_ptr=None, idx_ptr=None) == 0
    assert call(2, 64, rows=0, out_ptr=None) == 0
    torch.cuda.synchronize()


def _handle_results(hs, h, L):
    idx = pref.pct_index(PCTS, len(hs) * L)
    gene_of = np.repeat(np.arange((h.n + 2) // 3, dtype=np.int32), 3)[:h.n]     # _chains' genes: runs of three
    multi = np.array([np.sum(gene_of == g) > 1 for g in gene_of], np.uint8)
    res = [capi.pooled_summaries(hs, w, idx) for w in (0, 1, 2)]
    res.append(capi.pooled_summaries(hs, 3, idx, gene_of, multi))
    return idx, gene_of, multi, res


def test_handle_form_equals_dev_form_and_the_reference():
    h = _problem()
    hs = _chains(h, [0, 0, 0, 0])
    try:
        L = 64
        idx, gene_of, multi, res = _handle_results(hs, h, L)
        for which in (0, 1, 2):
            tr = np.stack([H.get_trace() if which == 0 else H.get_group_trace(which) for H in hs])
            out, pct = run_dev(tr, 0, idx)
            got = res[which]
            for q, k in enumerate(capi.POOL_OUTPUTS):
                assert got[k].tobytes() == out[q].tobytes(), (which, k)
            assert got["pct"].tobytes() == pct.tobytes()
        mu = np.stack([H.get_trace() for H in hs])
        gene = np.stack([H.get_group_trace(2) for H in hs])
        got = res[3]
        props = np.stack([mu[c] / gene[c][gene_of] for c in range(len(hs))])
        out, pct = run_dev(props, 1, idx)
        assert got["mean"].tobytes() == out[0].tobytes() and got["pct"].tobytes() == pct.tobytes()
        assert np.isnan(got["sd"]).all() and np.isnan(got["ess_mean"]).all()
        # the probit sums: each chain's k_prop sums, added in chain order
        per = [H.prop_summaries(gene_of, multi) for H in hs]
        s1, s2 = per[0]["sum_probit"].copy(), per[0]["sumsq_probit"].copy()
        for p in per[1:]:
            s1 += p["sum_probit"]
            s2 += p["sumsq_probit"]
        assert got["sum_probit"].tobytes() == s1.tobytes() and got["sumsq_probit"].tobytes() == s2.tobytes()
        for t in range(h.n):
            w = pref.pooled_props(mu[:, t, :], gene[:, gene_of[t], :], bool(multi[t]), idx)
            S = len(hs) * L
            assert math.isclose(got["mean"][t], w["mean"], rel_tol=1e-13)
            if multi[t]:
                assert math.isclose(got["sum_probit"][t] / S, w["mean_probit"], rel_tol=1e-9, abs_tol=1e-12)
            else:
                assert got["sum_probit"][t] == math.inf
        with pytest.raises(capi.MmqError):
            capi.pooled_summaries(hs[:1], 0)
        with pytest.raises(capi.MmqError):
            capi.pooled_summaries(hs, 0, [len(hs) * L])                  # percentile index outside [0, S)
        with pytest.raises(capi.MmqError):
            capi.pooled_summaries(hs, 3, idx)                              # proportions need gene_of / multi_iso
    finally:
        for H in hs:
            H.close()


def test_chains_on_two_devices_equal_one_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    h = _problem()
    res = []
    for devices in ([0, 0], [0, 1]):
        hs = _chains(h, devices)
        try:
            res.append(_handle_results(hs, h, 64)[3])
        finally:
            for H in hs:
                H.close()
    for a, b in zip(*res):
        for k in a:
            assert a[k].tobytes() == b[k].tobytes(), k


def test_concurrent_calls_of_other_shapes_and_modes():
    """The host threads of a -batch run call the kernel at once with other modes and shapes (and the diagnostics kernel
    with other sizes): every call succeeds and gives the bits of the same call alone."""
    import threading
    rng = np.random.default_rng(21)
    rows = 64
    cases = [(mixed(rng, 4, 1024, rows), 0), (rng.beta(0.5, 2.0, (2, rows, 8)), 1), (mixed(rng, 8, 1024, rows), 0),
             (rng.beta(0.5, 2.0, (3, rows, 64)), 1)]
    alone = [run_dev(x, m) for x, m in cases]
    diag_x = mixed(rng, 2, 64, rows)
    errors = []

    def worker(k):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for it in range(12):
                    x, m = cases[(k + it) % len(cases)]
                    out, pct = run_dev(x, m)
                    want = alone[(k + it) % len(cases)]
                    assert out.tobytes() == want[0].tobytes() and pct.tobytes() == want[1].tobytes()
                    if it % 3 == 0:
                        chains = [torch.from_numpy(np.ascontiguousarray(diag_x[c])).cuda() for c in range(2)]
                        d = torch.empty(5 * rows, dtype=torch.float64, device="cuda")
                        capi.chain_diagnostics_dev([t.data_ptr() for t in chains], rows, 64, d.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream)
                        torch.cuda.synchronize()
        except Exception as e:                                           # reported by the main thread
            errors.append(repr(e))
    th = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors[:3]
