"""mmq_draw_totals_dev, mmq_tpm_summaries_dev and mmq_tpm_summaries against the numpy reference (tests/tpm_reference.py):
the totals within 1e-12 of the exact sum and equal to the tile-order sum bit for bit, at single rows, ragged tile edges
and 200,000 rows; the summaries over the kernel's own totals at every (chains, trace length) shape accepted at the
edges, with enough features that every CTA of the grid-capped loop takes several and groups of 0, 1 and 30 members:
percentiles bit for bit, mean and sd within 1e-12 of the mean TPM; the same bits under repetition, alone or among
others, under row permutation, through the handle form, on a second GPU and from concurrent host threads; arguments
outside the limits."""
import ctypes
import threading
import time

import numpy as np
import pytest

from mmseq_b200 import capi
from tests import tpm_reference as tref
from tests.test_gpu_chain_diagnostics import _chains, _problem, grid_rows

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = [(C, L) for C in (1, 2, 4, 8) for L in (4, 8, 64, 1024, 2048) if C * L <= 8192]
PCTS = (0, 2.5, 5, 25, 50, 75, 95, 97.5, 100)


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_tpm: {time.time() - t0:.1f} s wall")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def totals_dev(tr):
    """tr: a (rows, L) fp64 tensor on the device -> fp64[L] on the host (mmq_draw_totals_dev)"""
    rows, L = tr.shape
    ws = torch.empty(max(1, capi.draw_totals_workspace_bytes(rows, L) // 8), dtype=torch.float64, device=tr.device)
    out = torch.full((L,), 12345.0, dtype=torch.float64, device=tr.device)
    capi.draw_totals_dev(tr.data_ptr(), rows, L, out.data_ptr(), ws.data_ptr(), _stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def run_dev(x, totals, gptr=None, members=None, idx=None):
    """x (C, n, L) on the host, totals (C, L) -> (out (2, rows), pct (rows, npct)) of mmq_tpm_summaries_dev"""
    C, n, L = x.shape
    idx = tref.pct_index(PCTS, C * L) if idx is None else np.asarray(idx, np.int32)
    rows = n if gptr is None else len(gptr) - 1
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    d_tot = torch.from_numpy(np.ascontiguousarray(totals, np.float64)).cuda()
    d_idx = torch.from_numpy(idx).cuda()
    d_ptr = None if gptr is None else torch.from_numpy(np.asarray(gptr, np.int64)).cuda()
    d_mem = None if gptr is None else torch.from_numpy(np.asarray(members, np.int32).reshape(-1)).cuda()
    if d_mem is not None and d_mem.numel() == 0:
        d_mem = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.full((2 * rows,), 12345.0, dtype=torch.float64, device="cuda")
    pct = torch.empty(max(1, rows * len(idx)), dtype=torch.float64, device="cuda")
    capi.tpm_summaries_dev([t.data_ptr() for t in chains], d_tot.data_ptr(), rows, L, None if d_ptr is None else d_ptr.data_ptr(),
                           None if d_mem is None else d_mem.data_ptr(), len(idx), d_idx.data_ptr(), out.data_ptr(), pct.data_ptr(), _stream())
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(2, rows), pct.cpu().numpy()[:rows * len(idx)].reshape(rows, len(idx))


def sample(rng, C, n, L):
    """log-normal draws with transcript levels spread over five orders of magnitude"""
    return np.exp(rng.normal(0.0, 1.0, (C, n, L)) + rng.normal(0.0, 3.0, (1, n, 1)))


def groups(rng, n, rows):
    """a CSR of `rows` features over the n transcripts: every 7th empty, every 7th + 1 of 30 members, the rest of one to
    five, drawn with repetition across features"""
    ptr, mem = [0], []
    for r in range(rows):
        k = 0 if r % 7 == 0 else 30 if r % 7 == 1 else int(rng.integers(1, 6))
        mem += rng.choice(n, k, replace=False).tolist()
        ptr.append(len(mem))
    return np.array(ptr, np.int64), np.array(mem, np.int32)


def same_bits_or_both_nan(a, b):
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


def check(out, pct, want):
    assert same_bits_or_both_nan(pct, want["pct"])
    scale = np.abs(want["mean"])
    for q, k in enumerate(("mean", "sd")):
        g, w = out[q], want[k]
        assert np.array_equal(np.isnan(g), np.isnan(w)), k
        ok = np.isnan(w) | (np.abs(g - w) <= 1e-12 * scale)
        bad = np.flatnonzero(~ok)
        assert not len(bad), (k, bad[:5], g[bad[:5]], w[bad[:5]])


@pytest.mark.parametrize("rows,L", [(1, 1024), (511, 64), (512, 64), (513, 1024), (1000, 8), (1025, 4), (1537, 2048), (200000, 512)])
def test_totals_within_1e_12_of_the_exact_sum(rows, L):
    if rows * L * 8 * 2 > torch.cuda.mem_get_info()[0]:
        pytest.skip("not enough free device memory")
    gen = torch.Generator(device="cuda").manual_seed(rows + L)
    tr = torch.exp(torch.randn((rows, L), dtype=torch.float64, device="cuda", generator=gen) * 2.0)
    got = totals_dev(tr)
    host = tr.cpu().numpy()
    exact = tref.totals_fsum(host)
    assert (np.abs(got - exact) <= 1e-12 * exact).all()
    assert got.tobytes() == tref.totals_tiled(host).tobytes()
    assert got.tobytes() == totals_dev(tr).tobytes()                      # repeat
    if torch.cuda.device_count() > 1:
        assert got.tobytes() == totals_dev(tr.to("cuda:1")).tobytes()    # another device
    assert (totals_dev(tr[:0]) == 0).all()                               # no rows: 0.0


@pytest.mark.parametrize("C,L", CASES)
def test_summaries_against_reference(C, L):
    rng = np.random.default_rng(100 * C + L)
    rows = grid_rows()
    n = rows + 37
    x = sample(rng, C, n, L)
    totals = np.stack([totals_dev(torch.from_numpy(x[c]).cuda()) for c in range(C)])
    for c in range(C):
        assert totals[c].tobytes() == tref.totals_tiled(x[c]).tobytes()
    idx = tref.pct_index(PCTS, C * L)
    out, pct = run_dev(x, totals, idx=idx)                               # one feature per transcript
    check(out, pct, tref.features(x, totals, None, None, idx))
    assert np.sum(out[0]) == pytest.approx(1e6, rel=1e-10)
    gptr, mem = groups(rng, n, rows)
    out, pct = run_dev(x, totals, gptr, mem, idx)
    want = tref.features(x, totals, gptr, mem, idx)
    check(out, pct, want)
    empty = np.diff(gptr) == 0
    assert (out[:, empty] == 0).all() and (pct[empty] == 0).all()


def test_non_finite_draws():
    rng = np.random.default_rng(9)
    C, L, n = 2, 64, 400
    x = sample(rng, C, n, L)
    x[0, 5, 3] = np.inf                                                  # that slot's total is inf: 0 elsewhere, NaN here
    x[1, 9, 7] = np.nan                                                  # that slot's total is NaN: NaN everywhere
    totals = np.stack([totals_dev(torch.from_numpy(x[c]).cuda()) for c in range(C)])
    assert np.isinf(totals[0, 3]) and np.isnan(totals[1, 7])
    idx = np.append(tref.pct_index(PCTS, C * L), [-1, C * L])           # indices outside [0, S) give NaN
    out, pct = run_dev(x, totals, idx=idx)
    check(out, pct, tref.features(x, totals, None, None, idx))
    assert np.isnan(out).all() and np.isnan(pct[:, -3:]).all()


def test_bits_alone_among_others_and_permuted():
    rng = np.random.default_rng(10)
    C, L = 4, 1024
    rows = grid_rows()
    n = rows
    x = sample(rng, C, n, L)
    totals = np.stack([tref.totals_tiled(x[c]) for c in range(C)])
    gptr, mem = groups(rng, n, rows)
    a, pa = run_dev(x, totals, gptr, mem)
    b, pb = run_dev(x, totals, gptr, mem)
    assert a.tobytes() == b.tobytes() and pa.tobytes() == pb.tobytes()
    perm = rng.permutation(rows)
    pptr = np.concatenate([[0], np.cumsum(np.diff(gptr)[perm])])
    pmem = np.concatenate([mem[gptr[r]:gptr[r + 1]] for r in perm])
    c, pc = run_dev(x, totals, pptr, pmem)
    assert a[:, perm].tobytes() == c.tobytes() and pa[perm].tobytes() == pc.tobytes()
    for r in (1, 2, rows - 1):                                           # one feature alone: one CTA
        d, pd = run_dev(x, totals, np.array([0, gptr[r + 1] - gptr[r]]), mem[gptr[r]:gptr[r + 1]])
        assert a[:, r:r + 1].tobytes() == d.tobytes() and pa[r:r + 1].tobytes() == pd.tobytes()


def _csr(h):
    """the identical pairs and genes of three of tests/test_gpu_chain_diagnostics._chains"""
    n = h.n
    return ((np.arange(0, n - n % 2 + 1, 2, dtype=np.int64), np.arange(n - n % 2, dtype=np.int32)),
            (np.append(np.arange(0, n, 3, dtype=np.int64), n), np.arange(n, dtype=np.int32)))


def _handle_results(hs, L):
    idx = tref.pct_index(PCTS, len(hs) * L)
    return [capi.tpm_summaries(hs, w, idx) for w in (0, 1, 2)]


@pytest.mark.parametrize("nchains,L", [(1, 4), (1, 64), (4, 64)])
def test_handle_form_equals_dev_form(nchains, L):
    h = _problem()
    hs = _chains(h, [0] * nchains, L=L)
    try:
        res = _handle_results(hs, L)
        tr = np.stack([H.get_trace() for H in hs])
        totals = np.stack([totals_dev(torch.from_numpy(tr[c]).cuda()) for c in range(nchains)])
        idx = tref.pct_index(PCTS, nchains * L)
        for which, csr in zip((0, 1, 2), (None,) + _csr(h)):
            got = res[which]
            assert got["totals"].tobytes() == totals.tobytes()
            out, pct = run_dev(tr, totals, *(csr or (None, None)), idx=idx)
            assert got["mean"].tobytes() == out[0].tobytes() and got["sd"].tobytes() == out[1].tobytes(), which
            assert got["pct"].tobytes() == pct.tobytes(), which
            if which != 1:                                               # the identical pairs leave out an odd last transcript
                assert np.sum(got["mean"]) == pytest.approx(1e6, rel=1e-10)
        with pytest.raises(capi.MmqError):
            capi.tpm_summaries(hs, 0, [nchains * L])                      # percentile index outside [0, S)
        with pytest.raises(capi.MmqError):
            capi.tpm_summaries(hs, 0, [-1])
        with pytest.raises(capi.MmqError):
            capi.tpm_summaries(hs, 3)
    finally:
        for H in hs:
            H.close()


def test_handles_that_differ_are_rejected():
    h = _problem()
    a = _chains(h, [0], L=64)
    b = _chains(h, [0], L=32)
    try:
        with pytest.raises(capi.MmqError):
            capi.tpm_summaries(a + b, 0)
        lib = capi.lib()
        arr = (ctypes.c_void_p * 9)(*([a[0]._h] * 9))
        assert lib.mmq_tpm_summaries(arr, 9, 0, 0, None, None, None, None, None) == 1
        assert lib.mmq_tpm_summaries(arr, 0, 0, 0, None, None, None, None, None) == 1
        assert lib.mmq_tpm_summaries(arr, 1, 0, 0, None, None, None, None, None) == 0
    finally:
        for H in a + b:
            H.close()


def test_chains_on_two_devices_equal_one_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    h = _problem()
    res = []
    for devices in ([0, 0], [0, 1]):
        hs = _chains(h, devices)
        try:
            res.append(_handle_results(hs, 64))
        finally:
            for H in hs:
                H.close()
    for a, b in zip(*res):
        for k in a:
            assert a[k].tobytes() == b[k].tobytes(), k


def test_arguments_outside_the_limits():
    lib = capi.lib()
    buf = torch.zeros(8 * 8192, dtype=torch.float64, device="cuda")
    tot = torch.ones(8192, dtype=torch.float64, device="cuda")
    out = torch.zeros(2 * 8, dtype=torch.float64, device="cuda")
    pct = torch.zeros(8 * 2, dtype=torch.float64, device="cuda")
    idx = torch.zeros(2, dtype=torch.int32, device="cuda")
    gp = torch.zeros(9, dtype=torch.int64, device="cuda")
    mem = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = _stream()

    def call(C, L, rows=8, npct=2, null_at=-1, tot_ptr=tot.data_ptr(), gptr=None, members=None, out_ptr=out.data_ptr(),
             pct_ptr=pct.data_ptr(), idx_ptr=idx.data_ptr()):
        ptrs = [buf.data_ptr()] * max(C, 1)
        if null_at >= 0:
            ptrs[null_at] = None
        arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        return lib.mmq_tpm_summaries_dev(arr, tot_ptr, C, rows, L, gptr, members, npct, idx_ptr, out_ptr, pct_ptr, stream)
    assert call(1, 4) == 0 and call(8, 1024) == 0 and call(4, 2048) == 0
    assert call(2, 64, gptr=gp.data_ptr(), members=mem.data_ptr()) == 0
    for C, L in [(0, 64), (9, 512), (1, 2), (1, 12), (1, 4096), (8, 2048), (5, 2048), (3, 100)]:
        assert call(C, L) == 1, (C, L)
    assert call(2, 64, rows=-1) == 1 and call(2, 64, npct=-1) == 1 and call(2, 64, null_at=1) == 1
    assert call(2, 64, gptr=gp.data_ptr()) == 1 and call(2, 64, members=mem.data_ptr()) == 1
    assert call(2, 64, tot_ptr=None) == 1 and call(2, 64, out_ptr=None) == 1
    assert call(2, 64, pct_ptr=None) == 1 and call(2, 64, idx_ptr=None) == 1
    assert call(2, 64, npct=0, pct_ptr=None, idx_ptr=None) == 0
    assert call(2, 64, rows=0, out_ptr=None, tot_ptr=None) == 0
    ws = torch.zeros(1024, dtype=torch.float64, device="cuda")
    assert capi.draw_totals_workspace_bytes(513, 64) == 8 * 2 * 64 and capi.draw_totals_workspace_bytes(0, 64) == 0
    assert capi.draw_totals_workspace_bytes(-1, 64) == 0 and capi.draw_totals_workspace_bytes(8, 12) == 0
    for rows, L, t, w in [(8, 2, buf, ws), (8, 4096, buf, ws), (8, 12, buf, ws), (-1, 64, buf, ws), (8, 64, None, ws), (8, 64, buf, None)]:
        rc = lib.mmq_draw_totals_dev(None if t is None else t.data_ptr(), rows, L, out.data_ptr(), None if w is None else w.data_ptr(), stream)
        assert rc == 1, (rows, L)
    assert lib.mmq_draw_totals_dev(buf.data_ptr(), 8, 64, None, ws.data_ptr(), stream) == 1
    assert lib.mmq_draw_totals_dev(None, 0, 64, tot.data_ptr(), None, stream) == 0
    torch.cuda.synchronize()


def test_concurrent_calls_of_other_shapes():
    """Host threads (as the samples of a -batch run) call the kernels at once with other shapes and with and without
    groups, beside the pooled-summaries kernel: every call succeeds and gives the bits of the same call made alone."""
    rng = np.random.default_rng(21)
    cases = []
    for C, L in ((1, 4), (8, 1024), (2, 64), (4, 2048)):
        n = 300
        x = sample(rng, C, n, L)
        totals = np.stack([tref.totals_tiled(x[c]) for c in range(C)])
        gptr, mem = groups(rng, n, 200) if C % 2 == 0 else (None, None)
        cases.append((x, totals, gptr, mem))
    alone = [run_dev(*cs) for cs in cases]
    tot_alone = [totals_dev(torch.from_numpy(cs[0][0]).cuda()) for cs in cases]
    pool_x = np.exp(rng.normal(0.0, 1.0, (4, 64, 1024)))
    errors = []

    def worker(k):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for it in range(10):
                    i = (k + it) % len(cases)
                    out, pct = run_dev(*cases[i])
                    assert out.tobytes() == alone[i][0].tobytes() and pct.tobytes() == alone[i][1].tobytes()
                    assert totals_dev(torch.from_numpy(cases[i][0][0]).cuda()).tobytes() == tot_alone[i].tobytes()
                    if it % 3 == 0:
                        chains = [torch.from_numpy(pool_x[c]).cuda() for c in range(4)]
                        o = torch.empty(3 * 64, dtype=torch.float64, device="cuda")
                        capi.pooled_summaries_dev([t.data_ptr() for t in chains], 64, 1024, 0, 0, None, o.data_ptr(), None, _stream())
                        torch.cuda.synchronize()
        except Exception as e:                                           # reported by the main thread
            errors.append(repr(e))
    th = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors[:3]
