"""mmq_isocorr_summaries_dev, mmq_isocorr_summaries and mmq_pair_shared_counts against the numpy reference
(tests/isocorr_reference.py).  Genes of 1, 2, 3, 31-33, 63-65 and 300 members (tiles split, several items per gene)
beside enough small genes that every CTA of the grid-capped loop takes several items; planted positive, negative and
no correlation; rows with NaN, +-inf, zeros, negative and constant values.  Correlations within 1e-10, prob_1_gt_2 bit
for bit; the same bits on a repeat and with the genes permuted; the handle form equal to the dev form and, at L = 1024,
within the stated bound of the tensor-core covariance (mmq_handle_trace_cov, nsplit 3); arguments outside the limits.
The shared fragments equal the reference for collapsed and per-fragment layouts, on one shard and split into two."""
import ctypes

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests import isocorr_reference as iref
from tests.test_gpu_chain_diagnostics import _chains, _problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = [(1, 4), (1, 1024), (1, 2048), (4, 4), (4, 1024), (4, 2048), (8, 4), (8, 1024)]
BIG = [1, 2, 3, 31, 32, 33, 63, 64, 65, 300]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev(a, dtype):
    a = np.asarray(a, dtype).reshape(-1)
    return torch.from_numpy(a if a.size else np.zeros(1, dtype)).cuda()


def run_dev(x, gptr, mem):
    """x (C, n, L) -> out (3, npairs)"""
    C, n, L = x.shape
    gptr = np.asarray(gptr, np.int64)
    *_, base = iref.pairs(gptr, mem)
    npairs = int(sum(int(k) * (int(k) - 1) // 2 for k in np.diff(gptr)))
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    d = [_dev(gptr, np.int64), _dev(mem, np.int32), _dev(base, np.int64)]
    ngenes, nmem = len(gptr) - 1, int(gptr[-1])
    ws = torch.empty(max(1, capi.isocorr_workspace_bytes(ngenes, nmem)), dtype=torch.uint8, device="cuda")
    out = torch.full((max(1, 3 * npairs),), 12345.0, dtype=torch.float64, device="cuda")
    capi.isocorr_summaries_dev([t.data_ptr() for t in chains], ngenes, nmem, L, *[t.data_ptr() for t in d], npairs, out.data_ptr(),
                               ws.data_ptr(), _stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()[:3 * npairs].reshape(3, npairs)


def grid_items():
    return 3 * 2 * torch.cuda.get_device_properties(0).multi_processor_count + 5


def case(rng, C, L, sizes):
    """gene CSR over a permutation of the rows, and draws: per gene a shared factor that members load on with weight
    +0.9, -0.9 or 0 (by member), log-normal levels; a few special rows"""
    n = int(sum(sizes)) + 7                                              # 7 rows in no gene
    perm = rng.permutation(n)[:int(sum(sizes))].astype(np.int32)
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    x = np.exp(rng.normal(0.0, 1.0, (1, n, 1)) + 0.3 * rng.standard_normal((C, n, L)))
    for g in range(len(sizes)):
        mem = perm[gptr[g]:gptr[g + 1]]
        z = rng.standard_normal((C, 1, L))
        w = np.array([0.9, -0.9, 0.0])[np.arange(len(mem)) % 3][None, :, None]
        x[:, mem] *= np.exp(w * z)
    if len(perm) > 12:
        x[:, perm[0], 3 % L] = np.nan
        x[:, perm[1], 1] = np.inf
        x[:, perm[2], 2] = -np.inf
        x[:, perm[3], 0] = 0.0
        x[:, perm[4]] = 3.0                                              # constant: sum of squares exactly 0
        x[:, perm[5], 1] = -2.0
        x[:, perm[7]] = x[:, perm[6]]                                    # exact copy: ties, correlation 1
    return x, gptr, perm


def check(out, want):
    for q, k in enumerate(("corr_mu", "corr_log_mu", "prob_1_gt_2")):
        g, w = out[q], want[k]
        assert np.array_equal(np.isnan(g), np.isnan(w)), (k, np.flatnonzero(np.isnan(g) != np.isnan(w))[:5])
        if k == "prob_1_gt_2":
            assert g[~np.isnan(g)].tobytes() == w[~np.isnan(w)].tobytes()
        else:
            err = np.abs(g - w)[~np.isnan(w)]
            assert err.max(initial=0) <= 1e-10, (k, err.max())


def sizes_for(rng, L):
    small = rng.integers(1, 6, grid_items()).tolist()
    return BIG + small if L <= 1024 else [2, 3, 33, 65, 300] + small[:400]


@pytest.mark.parametrize("C,L", CASES)
def test_summaries_against_reference(C, L):
    rng = np.random.default_rng(10 * C + L)
    x, gptr, mem = case(rng, C, L, sizes_for(rng, L))
    out = run_dev(x, gptr, mem)
    want = iref.summaries(x, gptr, mem)
    check(out, want)
    g, a, b, ma, mb, _ = iref.pairs(gptr, mem)
    fin = np.isfinite(out[0])
    if L >= 1024:                                                        # the planted signs come through
        wa, wb = a % 3, b % 3
        assert np.median(out[0, fin & (wa == 0) & (wb == 1)]) < -0.3
        assert np.median(out[0, fin & (wa == 0) & (wb == 0)]) > 0.3
        assert abs(np.median(out[0, fin & ((wa == 2) | (wb == 2))])) < 0.1
    cp = (ma == mem[6]) & (mb == mem[7]) | (ma == mem[7]) & (mb == mem[6])
    assert (np.abs(out[0, cp] - 1.0) < 1e-12).all() and (out[2, cp] == 0.5).all()


def test_bits_repeated_and_genes_permuted():
    rng = np.random.default_rng(7)
    C, L = 4, 1024
    sizes = BIG + rng.integers(1, 6, grid_items()).tolist()
    x, gptr, mem = case(rng, C, L, sizes)
    a = run_dev(x, gptr, mem)
    b = run_dev(x, gptr, mem)
    assert a.tobytes() == b.tobytes()
    perm = rng.permutation(len(sizes))
    gptr2 = np.concatenate([[0], np.cumsum(np.diff(gptr)[perm])]).astype(np.int64)
    mem2 = np.concatenate([mem[gptr[g]:gptr[g + 1]] for g in perm]).astype(np.int32)
    c = run_dev(x, gptr2, mem2)
    *_, base = iref.pairs(gptr, mem)
    order = np.concatenate([np.arange(base[g], base[g] + np.diff(gptr)[g] * (np.diff(gptr)[g] - 1) // 2) for g in perm]).astype(np.int64)
    assert a[:, order].tobytes() == c.tobytes()
    one = np.flatnonzero(np.diff(gptr) == 300)[0]                        # one gene alone
    d = run_dev(x, gptr[[0]].tolist() + [300], mem[gptr[one]:gptr[one + 1]])
    sel = np.arange(base[one], base[one] + 300 * 299 // 2)
    assert a[:, sel].tobytes() == d.tobytes()


def _gene_groups(n, sizes):
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    assert gptr[-1] <= n
    return gptr, np.random.default_rng(5).permutation(n)[:gptr[-1]].astype(np.int32)


@pytest.mark.parametrize("nchains,L", [(1, 4), (1, 1024), (4, 64)])
def test_handle_form_equals_dev_form(nchains, L):
    h = _problem()
    hs = _chains(h, [0] * nchains, L=L)
    try:
        gptr, mem = _gene_groups(h.n, [1, 2, 3, 33, 70, 0, 4])
        for H in hs:
            H.set_groups(capi.MMQ_GROUP_GENE, gptr, mem)
        npairs = sum(k * (k - 1) // 2 for k in np.diff(gptr))
        got = capi.isocorr_summaries(hs, npairs)
        tr = np.stack([H.get_trace() for H in hs])
        out = run_dev(tr, gptr, mem)
        for q, k in enumerate(("corr_mu", "corr_log_mu", "prob_1_gt_2")):
            assert got[k].tobytes() == out[q].tobytes(), k
        check(out, iref.summaries(tr, gptr, mem))
        assert np.isfinite(out).mean() > 0.9
        for bad in (npairs - 1, npairs + 1):
            with pytest.raises(capi.MmqError):
                capi.isocorr_summaries(hs, bad)
        if nchains == 1 and L == 1024:
            # the independent cross-check: the tensor-core covariance of one gene's members (nsplit 3, stated bound at
            # L = 1024 1.6e-5 in correlation units)
            g = 4
            feats = mem[gptr[g]:gptr[g + 1]]
            R = hs[0].trace_cov(feats, nsplit=3)
            d = np.sqrt(np.diag(R))
            corr = R / d[:, None] / d[None, :]
            *_, base = iref.pairs(gptr, mem)
            k = len(feats)
            a, b = np.triu_indices(k, 1)
            mine = got["corr_mu"][base[g] + np.arange(k * (k - 1) // 2)]
            assert np.abs(mine - corr[a, b]).max() < 1.6e-5
    finally:
        for H in hs:
            H.close()


def test_arguments_outside_the_limits():
    lib = capi.lib()
    buf = torch.zeros(8 * 8192, dtype=torch.float64, device="cuda")
    out = torch.zeros(3, dtype=torch.float64, device="cuda")
    ws = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    gp = _dev([0, 2], np.int64)
    mem = _dev([0, 1], np.int32)
    pb = _dev([0], np.int64)
    stream = _stream()

    def call(C, L, ngenes=1, nmem=2, npairs=1, null_chain=-1, null=-1):
        ch = [buf.data_ptr()] * max(C, 1)
        if null_chain >= 0:
            ch[null_chain] = None
        arr = (ctypes.c_void_p * len(ch))(*ch)
        p = [gp.data_ptr(), mem.data_ptr(), pb.data_ptr(), out.data_ptr(), ws.data_ptr()]
        if null >= 0:
            p[null] = None
        return lib.mmq_isocorr_summaries_dev(arr, C, ngenes, nmem, L, p[0], p[1], p[2], npairs, p[3], p[4], stream)
    assert call(1, 4) == 0 and call(8, 1024) == 0 and call(4, 2048) == 0
    for C, L in [(0, 64), (9, 512), (1, 2), (1, 12), (1, 4096), (8, 2048), (5, 2048), (3, 100)]:
        assert call(C, L) == 1, (C, L)
    assert call(2, 64, ngenes=-1) == 1 and call(2, 64, nmem=-1) == 1 and call(2, 64, npairs=-1) == 1 and call(2, 64, null_chain=1) == 1
    for q in range(5):
        assert call(2, 64, null=q) == 1, q
    assert call(2, 64, npairs=0, null=0) == 0
    torch.cuda.synchronize()
    assert capi.isocorr_workspace_bytes(3, 10) == 40 * 10 + 8 * 4 and capi.isocorr_workspace_bytes(-1, 3) == 0
    h = _problem()
    hs = _chains(h, [0], L=64)
    try:
        arr = (ctypes.c_void_p * 9)(*([hs[0]._h] * 9))
        assert lib.mmq_isocorr_summaries(arr, 9, 0, None, None, None) == 1
        assert lib.mmq_isocorr_summaries(arr, 0, 0, None, None, None) == 1
        assert lib.mmq_isocorr_summaries(arr, 1, -1, None, None, None) == 1
        H = hs[0]
        gptr, mem_ = _gene_groups(h.n, [3, 1, 4])
        H.set_groups(capi.MMQ_GROUP_GENE, gptr, mem_)
        gene_of, local_of = iref.gene_local(gptr, mem_, h.n)
        base = np.array([0, 3, 3], np.int64)
        assert H.pair_shared_counts(gene_of, local_of, base, 9).shape == (9,)
        for gi, li, b, npairs in ((3, 0, base, 9), (-2, 0, base, 9), (0, 3, base, 9), (0, -1, base, 9), (0, 0, np.array([1, 3, 3]), 9),
                                  (0, 0, np.array([0, 3, 2]), 9), (0, 0, base, 8), (0, 0, np.array([0, 2, 3]), 9), (0, 0, base, 10)):
            g2, l2 = gene_of.copy(), local_of.copy()
            g2[mem_[0]], l2[mem_[0]] = gi, li
            with pytest.raises(capi.MmqError):
                H.pair_shared_counts(g2, l2, b, npairs)
        with pytest.raises(capi.MmqError):                               # pairs without genes
            H.pair_shared_counts(np.full(h.n, -1, np.int32), np.full(h.n, -1, np.int32), np.zeros(0, np.int64), 1)
        assert H.pair_shared_counts(np.full(h.n, -1, np.int32), np.full(h.n, -1, np.int32), np.zeros(0, np.int64), 0).shape == (0,)
    finally:
        for H in hs:
            H.close()


# ------------------------------------------------------------------ shared fragments

def _genes_of(h, s):
    """every generator gene's observed isoforms in header order, as the host program builds them"""
    gptr, mem = [0], []
    for g in range(s.G):
        for t in range(int(s.gene_ptr[g]), int(s.gene_ptr[g + 1])):
            if h.hdr2col[t] >= 0:
                mem.append(int(h.hdr2col[t]))
        gptr.append(len(mem))
    return np.array(gptr, np.int64), np.array(mem, np.int32)


@pytest.mark.parametrize("layout", ["collapsed", "per_fragment"])
def test_shared_counts_equal_reference(layout):
    lay = hostlib.LAYOUT_COLLAPSED if layout == "collapsed" else hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH
    s = synth.Synth(31, 400, 20000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=lay)
    k = h.k if layout == "collapsed" else None
    gptr, mem = _genes_of(h, s)
    gene_of, local_of = iref.gene_local(gptr, mem, h.n)
    *_, base = iref.pairs(gptr, mem)
    npairs = int(sum(int(d) * (int(d) - 1) // 2 for d in np.diff(gptr)))
    want = iref.shared(h.row_ptr, h.col, k, gptr, mem)
    col_of = np.asarray(h.hdr2col)
    assert (iref.shared(s.frag_ptr, col_of[s.frag_tid], None, gptr, mem) == want).all()     # record by record
    assert want.sum() > 0 and (want == 0).any()
    with capi.Handle(h.row_ptr, h.col, k, h.len) as H:
        got = H.pair_shared_counts(gene_of, local_of, base, npairs)
    assert (got == want).all()
    cut = h.m // 3
    parts = []
    for a, b in ((0, cut), (cut, h.m)):
        rp = h.row_ptr[a:b + 1] - h.row_ptr[a]
        with capi.Handle(rp, h.col[h.row_ptr[a]:h.row_ptr[b]], None if k is None else k[a:b], h.len, class_id_base=a) as H:
            parts.append(H.pair_shared_counts(gene_of, local_of, base, npairs))
    assert ((parts[0] + parts[1]) == want).all()


def test_shared_counts_all_reduced_over_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from tests.test_gpu_counts import _on_threads
    s = synth.Synth(31, 400, 20000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    gptr, mem = _genes_of(h, s)
    gene_of, local_of = iref.gene_local(gptr, mem, h.n)
    *_, base = iref.pairs(gptr, mem)
    npairs = int(sum(int(d) * (int(d) - 1) // 2 for d in np.diff(gptr)))
    want = iref.shared(h.row_ptr, h.col, h.k, gptr, mem)
    cut = [0, h.m // 3, h.m]
    hs = []
    for r in range(2):
        a, b = cut[r], cut[r + 1]
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        hs.append(capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], h.k[a:b], h.len, class_id_base=a, device=r))
    try:
        uid = capi.comm_id()
        _on_threads(lambda r: hs[r].comm_init(uid, r, 2), 2)
        for got in _on_threads(lambda r: hs[r].pair_shared_counts(gene_of, local_of, base, npairs), 2):
            assert (got == want).all()
    finally:
        for H in hs:
            H.close()
