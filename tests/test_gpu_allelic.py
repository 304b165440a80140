"""mmq_allelic_summaries_dev, mmq_allelic_summaries and mmq_allele_only_counts against the numpy reference
(tests/allelic_reference.py).  The summaries at every (chains, trace length) shape accepted at the edges, with enough
units that every CTA of the grid-capped loop takes several, units of 0, 1 and many members per side, members among the
trace rows and the prior rows, ties a = b, and a + b = 0: percentiles and prob_a_gt_b bit for bit, mean and sd within
1e-13 relative; the same bits under repetition, row permutation, alone, through the handle form, on a second GPU and
from concurrent host threads; arguments outside the limits.  The allele-only counts equal a brute-force count over the
records for collapsed and per-fragment layouts, on one shard and split into two."""
import ctypes
import threading
import time

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests import allelic_reference as aref
from tests.test_gpu_chain_diagnostics import _chains, _problem, grid_rows

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = [(C, L) for C in (1, 2, 4, 8) for L in (4, 8, 64, 1024, 2048) if C * L <= 8192]
PCTS = (0, 2.5, 5, 25, 50, 75, 95, 97.5, 100)


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntest_gpu_allelic: {time.time() - t0:.1f} s wall")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev(a, dtype):
    a = np.asarray(a, dtype).reshape(-1)
    return torch.from_numpy(a if a.size else np.zeros(1, dtype)).cuda()


def run_dev(x, priors, csr, idx=None):
    """x (C, n, L), priors (C, nprior, L) or None, csr (a_ptr, a_mem, b_ptr, b_mem) -> (out (3, rows), pct (rows, npct))"""
    C, n, L = x.shape
    idx = aref.pct_index(PCTS, C * L) if idx is None else np.asarray(idx, np.int32)
    a_ptr, a_mem, b_ptr, b_mem = csr
    rows = len(a_ptr) - 1
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    nprior = 0 if priors is None else priors.shape[1]
    pri = None if priors is None else [torch.from_numpy(np.ascontiguousarray(priors[c])).cuda() for c in range(C)]
    d = [_dev(a_ptr, np.int64), _dev(a_mem, np.int32), _dev(b_ptr, np.int64), _dev(b_mem, np.int32), _dev(idx, np.int32)]
    out = torch.full((3 * rows,), 12345.0, dtype=torch.float64, device="cuda")
    pct = torch.full((max(1, rows * len(idx)),), 12345.0, dtype=torch.float64, device="cuda")
    capi.allelic_summaries_dev([t.data_ptr() for t in chains], None if pri is None else [t.data_ptr() for t in pri], n, nprior, rows, L,
                               *[t.data_ptr() for t in d[:4]], len(idx), d[4].data_ptr(), out.data_ptr(), pct.data_ptr(), _stream())
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(3, rows), pct.cpu().numpy()[:rows * len(idx)].reshape(rows, len(idx))


def sample(rng, C, n, L):
    """log-normal draws over five orders of magnitude; row 0 all zeros, row 1 a copy of row 2 (exact ties)"""
    x = np.exp(rng.normal(0.0, 1.0, (C, n, L)) + rng.normal(0.0, 3.0, (1, n, 1)))
    x[:, 0] = 0.0
    x[:, 1] = x[:, 2]
    return x


def units(rng, n, nprior, rows):
    """rows units over ids [0, n + nprior): by r % 9 an empty A side, an empty B side, one member each, 12 against 20,
    A = B (ties), prior rows only, the zero row on both sides (a + b = 0), the rest one to four members of any kind"""
    A, B = [], []
    ids = n + nprior
    for r in range(rows):
        k = r % 9
        if k == 0:
            a, b = [], [int(rng.integers(ids))]
        elif k == 1:
            a, b = [int(rng.integers(ids))], []
        elif k == 2:
            a, b = [int(rng.integers(n))], [int(rng.integers(n))]
        elif k == 3:
            a, b = rng.choice(ids, 12, replace=False).tolist(), rng.choice(ids, 20, replace=False).tolist()
        elif k == 4:
            a = [1] if r % 2 else [2, 7]
            b = [2] if r % 2 else [7, 2]
        elif k == 5 and nprior:
            a, b = [n + int(rng.integers(nprior))], [n + int(rng.integers(nprior))]
        elif k == 6:
            a, b = [0], [0]
        else:
            a, b = rng.choice(ids, int(rng.integers(1, 5))).tolist(), rng.choice(ids, int(rng.integers(1, 5))).tolist()
        A.append(a)
        B.append(b)
    ptr = lambda u: np.concatenate([[0], np.cumsum([len(v) for v in u])]).astype(np.int64)
    mem = lambda u: np.array([m for v in u for m in v], np.int32)
    return ptr(A), mem(A), ptr(B), mem(B)


def same_bits_or_both_nan(a, b):
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


def check(out, pct, want):
    assert same_bits_or_both_nan(pct, want["pct"])
    assert same_bits_or_both_nan(out[2], want["prob_a"])
    for q, k in enumerate(("mean", "sd")):
        g, w = out[q], want[k]
        assert np.array_equal(np.isnan(g), np.isnan(w)), k
        ok = np.isnan(w) | (np.abs(g - w) <= 1e-13 * np.abs(w))
        bad = np.flatnonzero(~ok)
        assert not len(bad), (k, bad[:5], g[bad[:5]], w[bad[:5]])


@pytest.mark.parametrize("C,L", CASES)
def test_summaries_against_reference(C, L):
    rng = np.random.default_rng(100 * C + L)
    rows = grid_rows()
    n, nprior = 300, 40
    x = sample(rng, C, n, L)
    priors = rng.gamma(0.1, 1.0, (C, nprior, L))
    csr = units(rng, n, nprior, rows)
    idx = np.append(aref.pct_index(PCTS, C * L), [-1, C * L])            # indices outside [0, S) give NaN
    out, pct = run_dev(x, priors, csr, idx)
    want = aref.units(x, priors, *csr, idx)
    check(out, pct, want)
    kind = np.arange(rows) % 9
    assert np.isnan(out[:, kind == 6]).all()                             # a + b = 0
    fin = np.isfinite(out[0])
    assert (out[0, fin & (kind == 0)] == 0.0).all() and (out[0, fin & (kind == 1)] == 1.0).all()   # one side empty
    ties = kind == 4
    assert (out[0, ties] == 0.5).all() and (out[1, ties] == 0.0).all() and (out[2, ties] == 0.5).all()
    assert np.isfinite(out[:, kind == 3]).all()
    out0, _ = run_dev(x, None, units(np.random.default_rng(1), n, 0, 40), idx)      # no prior rows
    check(out0, _, aref.units(x, None, *units(np.random.default_rng(1), n, 0, 40), idx))


def test_bits_repeated_alone_and_permuted():
    rng = np.random.default_rng(10)
    C, L, n, nprior = 4, 1024, 200, 30
    rows = grid_rows()
    x = sample(rng, C, n, L)
    priors = rng.gamma(0.1, 1.0, (C, nprior, L))
    a_ptr, a_mem, b_ptr, b_mem = units(rng, n, nprior, rows)
    a, pa = run_dev(x, priors, (a_ptr, a_mem, b_ptr, b_mem))
    b, pb = run_dev(x, priors, (a_ptr, a_mem, b_ptr, b_mem))
    assert a.tobytes() == b.tobytes() and pa.tobytes() == pb.tobytes()
    perm = rng.permutation(rows)

    def permute(ptr, mem):
        return (np.concatenate([[0], np.cumsum(np.diff(ptr)[perm])]).astype(np.int64),
                np.concatenate([mem[ptr[r]:ptr[r + 1]] for r in perm]).astype(np.int32))
    c, pc = run_dev(x, priors, (*permute(a_ptr, a_mem), *permute(b_ptr, b_mem)))
    assert same_bits_or_both_nan(a[:, perm], c) and same_bits_or_both_nan(pa[perm], pc)
    for r in (2, 3, rows - 1):                                           # one unit alone: one CTA
        one = (np.array([0, a_ptr[r + 1] - a_ptr[r]]), a_mem[a_ptr[r]:a_ptr[r + 1]], np.array([0, b_ptr[r + 1] - b_ptr[r]]),
               b_mem[b_ptr[r]:b_ptr[r + 1]])
        d, pd = run_dev(x, priors, one)
        assert same_bits_or_both_nan(a[:, r:r + 1], d) and same_bits_or_both_nan(pa[r:r + 1], pd)


@pytest.mark.parametrize("nchains,L", [(1, 4), (1, 64), (4, 64)])
def test_handle_form_equals_dev_form(nchains, L):
    h = _problem()
    hs = _chains(h, [0] * nchains, L=L)
    try:
        rng = np.random.default_rng(nchains + L)
        nprior = 7
        priors = rng.gamma(0.1, 1.0, (nchains, nprior, L))
        csr = units(rng, h.n, nprior, 300)
        idx = aref.pct_index(PCTS, nchains * L)
        got = capi.allelic_summaries(hs, *csr, priors=list(priors), pct_idx=idx)
        tr = np.stack([H.get_trace() for H in hs])
        out, pct = run_dev(tr, priors, csr, idx)
        for q, k in enumerate(("mean", "sd", "prob_a")):
            assert same_bits_or_both_nan(got[k], out[q]), k
        assert same_bits_or_both_nan(got["pct"], pct)
        check(out, pct, aref.units(tr, priors, *csr, idx))
        a_ptr, a_mem, b_ptr, b_mem = csr
        for bad in (dict(pct_idx=[nchains * L]), dict(pct_idx=[-1])):
            with pytest.raises(capi.MmqError):
                capi.allelic_summaries(hs, *csr, priors=list(priors), **bad)
        with pytest.raises(capi.MmqError):                                # a member past the prior rows
            capi.allelic_summaries(hs, a_ptr, np.where(np.arange(len(a_mem)) == 3, h.n + nprior, a_mem), b_ptr, b_mem, priors=list(priors))
        with pytest.raises(capi.MmqError):                                # prior ids without prior rows
            capi.allelic_summaries(hs, *csr)
        with pytest.raises(capi.MmqError):                                # a decreasing CSR
            capi.allelic_summaries(hs, np.array([0, 2, 1]), a_mem[:2], np.array([0, 1, 1]), b_mem[:1], priors=list(priors))
    finally:
        for H in hs:
            H.close()


def test_chains_on_two_devices_equal_one_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    h = _problem()
    rng = np.random.default_rng(4)
    priors = list(rng.gamma(0.1, 1.0, (2, 5, 64)))
    csr = units(rng, h.n, 5, 100)
    res = []
    for devices in ([0, 0], [0, 1]):
        hs = _chains(h, devices)
        try:
            res.append(capi.allelic_summaries(hs, *csr, priors=priors, pct_idx=aref.pct_index(PCTS, 128)))
        finally:
            for H in hs:
                H.close()
    for k in res[0]:
        assert same_bits_or_both_nan(res[0][k], res[1][k]), k


def test_arguments_outside_the_limits():
    lib = capi.lib()
    buf = torch.zeros(8 * 8192, dtype=torch.float64, device="cuda")
    out = torch.zeros(3 * 8, dtype=torch.float64, device="cuda")
    pct = torch.zeros(8 * 2, dtype=torch.float64, device="cuda")
    idx = torch.zeros(2, dtype=torch.int32, device="cuda")
    ptr = torch.zeros(9, dtype=torch.int64, device="cuda")
    mem = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = _stream()

    def call(C, L, rows=8, npct=2, nprior=0, null_chain=-1, prior=None, ptrs=(ptr, mem, ptr, mem), null_csr=-1, out_ptr=out.data_ptr(),
             pct_ptr=pct.data_ptr(), idx_ptr=idx.data_ptr()):
        ch = [buf.data_ptr()] * max(C, 1)
        if null_chain >= 0:
            ch[null_chain] = None
        arr = (ctypes.c_void_p * len(ch))(*ch)
        pri = None if prior is None else (ctypes.c_void_p * len(prior))(*prior)
        p = [t.data_ptr() for t in ptrs]
        if null_csr >= 0:
            p[null_csr] = None
        return lib.mmq_allelic_summaries_dev(arr, pri, C, 1, nprior, rows, L, *p, npct, idx_ptr, out_ptr, pct_ptr, stream)
    assert call(1, 4) == 0 and call(8, 1024) == 0 and call(4, 2048) == 0
    assert call(2, 64, nprior=3, prior=[buf.data_ptr()] * 2) == 0
    for C, L in [(0, 64), (9, 512), (1, 2), (1, 12), (1, 4096), (8, 2048), (5, 2048), (3, 100)]:
        assert call(C, L) == 1, (C, L)
    assert call(2, 64, rows=-1) == 1 and call(2, 64, npct=-1) == 1 and call(2, 64, null_chain=1) == 1
    assert call(2, 64, nprior=3) == 1 and call(2, 64, nprior=3, prior=[buf.data_ptr(), None]) == 1 and call(2, 64, nprior=-1) == 1
    for q in range(4):
        assert call(2, 64, null_csr=q) == 1, q
    assert call(2, 64, out_ptr=None) == 1 and call(2, 64, pct_ptr=None) == 1 and call(2, 64, idx_ptr=None) == 1
    assert call(2, 64, npct=0, pct_ptr=None, idx_ptr=None) == 0
    assert call(2, 64, rows=0, out_ptr=None, null_csr=0) == 0
    torch.cuda.synchronize()
    h = _problem()
    hs = _chains(h, [0], L=64)
    try:
        arr = (ctypes.c_void_p * 9)(*([hs[0]._h] * 9))
        z = np.zeros(2, np.int64)
        assert lib.mmq_allelic_summaries(arr, 9, None, 0, 0, None, None, None, None, 0, None, None, None, None, None) == 1
        assert lib.mmq_allelic_summaries(arr, 0, None, 0, 0, None, None, None, None, 0, None, None, None, None, None) == 1
        assert lib.mmq_allelic_summaries(arr, 1, None, 0, 0, None, None, None, None, 0, None, None, None, None, None) == 0
        assert lib.mmq_allelic_summaries(arr, 1, None, 3, 1, z.ctypes.data, None, z.ctypes.data, None, 0, None, None, None, None, None) == 1
        H = hs[0]
        unit_of = np.full(h.n, -1, np.int32)
        side = np.zeros(h.n, np.uint8)
        for bad_unit, bad_side in ((5, 0), (-2, 0), (0, 2)):
            u, s = unit_of.copy(), side.copy()
            u[3], s[3] = bad_unit, bad_side
            with pytest.raises(capi.MmqError):
                H.allele_only_counts(u, s, 5)
        assert [v.tolist() for v in H.allele_only_counts(unit_of, side, 0)] == [[], []]
    finally:
        for H in hs:
            H.close()


def test_concurrent_calls_of_other_shapes():
    """Host threads (as the samples of a -batch run) call the kernel at once with other shapes, beside the TPM kernel:
    every call succeeds and gives the bits of the same call made alone."""
    rng = np.random.default_rng(21)
    cases = []
    for C, L in ((1, 4), (8, 1024), (2, 64), (4, 2048)):
        n = 300
        x = sample(rng, C, n, L)
        priors = rng.gamma(0.1, 1.0, (C, 9, L)) if C % 2 == 0 else None
        cases.append((x, priors, units(rng, n, 0 if priors is None else 9, 200)))
    alone = [run_dev(*cs) for cs in cases]
    tpm_x = np.exp(rng.normal(0.0, 1.0, (4, 64, 1024)))
    errors = []

    def worker(k):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for it in range(10):
                    i = (k + it) % len(cases)
                    out, pct = run_dev(*cases[i])
                    assert out.tobytes() == alone[i][0].tobytes() and pct.tobytes() == alone[i][1].tobytes()
                    if it % 3 == 0:
                        chains = [torch.from_numpy(tpm_x[c]).cuda() for c in range(4)]
                        tot = torch.ones(4 * 1024, dtype=torch.float64, device="cuda")
                        o = torch.empty(2 * 64, dtype=torch.float64, device="cuda")
                        capi.tpm_summaries_dev([t.data_ptr() for t in chains], tot.data_ptr(), 64, 1024, None, None, 0, None, o.data_ptr(), None,
                                               _stream())
                        torch.cuda.synchronize()
        except Exception as e:                                           # reported by the main thread
            errors.append(repr(e))
    th = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors[:3]


# ------------------------------------------------------------------ allele-only fragments

def _haplo(layout):
    s = synth.Synth(31, 400, 20000, haplo=True)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=layout)
    rng = np.random.default_rng(3)
    # pairs: copies 2p, 2p + 1 of the header; units of the gene level: the pairs' gene; a few transcripts in no unit
    pair_of = np.full(h.n, -1, np.int32)
    gene_unit = np.full(h.n, -1, np.int32)
    side = np.zeros(h.n, np.uint8)
    for t in range(s.T):
        c = h.hdr2col[t]
        if c >= 0 and rng.random() > 0.05:
            pair_of[c], gene_unit[c], side[c] = t // 2, s.gene_of[t], t % 2
    return s, h, ((pair_of, s.T // 2), (gene_unit, s.G)), side


@pytest.mark.parametrize("layout", ["collapsed", "per_fragment"])
def test_allele_only_counts_equal_brute_force(layout):
    lay = hostlib.LAYOUT_COLLAPSED if layout == "collapsed" else hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH
    s, h, levels, side = _haplo(lay)
    k = h.k if layout == "collapsed" else None
    cut = h.m // 3
    for unit_of, nunits in levels:
        want = aref.allele_only(h.row_ptr, h.col, k, unit_of, side, nunits)
        assert want[0].sum() > 0 and want[1].sum() > 0
        # the records, fragment by fragment: the same counts from the generator's hit lists
        col_of = np.asarray(h.hdr2col)
        frag = aref.allele_only(s.frag_ptr, col_of[s.frag_tid], None, unit_of, side, nunits)
        assert (frag[0] == want[0]).all() and (frag[1] == want[1]).all()
        with capi.Handle(h.row_ptr, h.col, k, h.len) as H:
            got = H.allele_only_counts(unit_of, side, nunits)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
        # two shards without a communicator: each counts its own rows, and the two add up to the whole
        parts = []
        for a, b in ((0, cut), (cut, h.m)):
            rp = h.row_ptr[a:b + 1] - h.row_ptr[a]
            with capi.Handle(rp, h.col[h.row_ptr[a]:h.row_ptr[b]], None if k is None else k[a:b], h.len, class_id_base=a) as H:
                parts.append(H.allele_only_counts(unit_of, side, nunits))
        assert ((parts[0][0] + parts[1][0]) == want[0]).all() and ((parts[0][1] + parts[1][1]) == want[1]).all()


def test_allele_only_counts_all_reduced_over_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from tests.test_gpu_counts import _on_threads
    s, h, levels, side = _haplo(hostlib.LAYOUT_COLLAPSED)
    cut = [0, h.m // 3, h.m]
    hs = []
    for r in range(2):
        a, b = cut[r], cut[r + 1]
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        hs.append(capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], h.k[a:b], h.len, class_id_base=a, device=r))
    try:
        uid = capi.comm_id()
        _on_threads(lambda r: hs[r].comm_init(uid, r, 2), 2)
        for unit_of, nunits in levels:
            want = aref.allele_only(h.row_ptr, h.col, h.k, unit_of, side, nunits)
            for got in _on_threads(lambda r: hs[r].allele_only_counts(unit_of, side, nunits), 2):
                assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
    finally:
        for H in hs:
            H.close()
