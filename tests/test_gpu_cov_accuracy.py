"""The covariance kernel (mmq_cov.cu: k_cov_prep + k_cov_gemm2, mmcollapse's row f3) against exact correlations, at every
trace length and size the C ABI accepts, on the inputs where a split-bf16 / fp32-accumulation product goes wrong.

Reference: the same fp64 input, centred in two passes in numpy (exact_cov in tests/collapse_case.py; the means by
math.fsum where they are many orders above the spread).  The centring is exact (Sterbenz) and the fp64 dot products are
good to ~1e-13 in correlation units at L = 65536: seven or more orders below every bound asserted here.

Metric: corr_err, |R_gpu - R_ref| / (sd_i sd_j), against cov_bound(nsplit, L) = COV_A[nsplit] + COV_B L, the contract
include/mmq.h states.  Each case also records the signed mean error sign(r) (r_gpu - r) over the pairs with |r| > 0.9
(negative: towards zero, what a truncating accumulation does); it is reported, not asserted.  The module prints the
table of both and its wall time at the end."""
import math
import time

import numpy as np
import pytest

from mmseq_b200 import capi
from tests.collapse_case import corr_err, cov_bound, exact_cov, make_gene_problem, make_traces, mean_corrs_rows

pytestmark = pytest.mark.gpu

LENGTHS = [64, 128, 1024, 2048, 4096, 16384, 65536]   # 64 .. cov_check's 65536
C_SMALL = 300                                           # one full and one ragged 256-wide tile a side
EPS = 2.0 ** -52
_TABLE = []


@pytest.fixture(scope="module", autouse=True)
def _report(pytestconfig):
    t0 = time.perf_counter()
    yield
    lines = [f"covariance accuracy (correlation units), {time.perf_counter() - t0:.1f} s",
             f"{'family':<16}{'L':>7}{'C':>7}{'nsplit':>7}{'max err':>11}{'bound':>11}{'bias |r|>0.9':>14}"]
    for fam, L, C, ns, e, b, bias in _TABLE:
        lines.append(f"{fam:<16}{L:>7}{C:>7}{ns:>7}{e:>11.2e}{b:>11.2e}{bias:>14.2e}")
    cap = pytestconfig.pluginmanager.getplugin("capturemanager")
    with cap.global_and_fixture_disabled():
        print("\n" + "\n".join(lines))


def _check(fam, R, ref, L, nsplit, extra=0.0):
    """Exact symmetry, the exact variance on the diagonal, the bound; records the row of the table."""
    C = R.shape[0]
    d = np.sqrt(np.diag(ref))
    d = np.where(d > 0, d, 1.0)
    err = (R - ref) / (d[:, None] * d[None, :])
    r = ref / (d[:, None] * d[None, :])
    hi = (np.abs(r) > 0.9) & ~np.eye(C, dtype=bool)
    bias = float(np.mean(np.sign(r[hi]) * err[hi])) if hi.any() else float("nan")
    e = float(np.max(np.abs(err)))
    b = cov_bound(nsplit, L) + extra
    _TABLE.append((fam, L, C, nsplit, e, b, bias))
    assert np.array_equal(R, R.T), (fam, L, nsplit, "not exactly symmetric")
    assert e < b, (fam, L, nsplit, e, b)
    return e


def _diag_exact(R, ref, rtol=1e-12):
    assert np.allclose(np.diag(R), np.diag(ref), rtol=rtol, atol=0.0), "the diagonal is the fp64 variance"


def _background(L, C, rng):
    """Traces of positive levels around 1 with blocks of anti-correlated members (the shape of make_traces)."""
    M = make_traces(L, C, seed=int(rng.integers(1 << 30)))
    return M / np.exp2(np.round(np.log2(M.mean(axis=0))))     # power-of-two rescale: the same correlations, exactly


def _walsh(L, k):
    """(-1)^popcount(s & k): mean exactly 0 and mutually orthogonal for 0 < k < 64 over any multiple of 64 samples."""
    s = np.arange(L)
    return np.where(np.array([bin(v).count("1") for v in (s & k)]) % 2 == 0, 1.0, -1.0)


def constructed_pairs(L, seed=0):
    """r = +1 and -1 exactly, 1 - |r| = 1e-2 / 1e-4 / 1e-6 (both signs), and exactly orthogonal Walsh columns, spread over
    both tile rows including the ragged last tile, on a background of realistic traces."""
    rng = np.random.default_rng(seed)
    C = C_SMALL
    M = _background(L, C, rng)
    x = M[:, 0].copy()
    M[:, C - 1] = x                    # r = +1, pair in the ragged tile
    M[:, 257] = -x                     # r = -1: the centred column is exactly the negated one
    xc = x - x.mean()
    cols = iter([(1, 2), (3, 200), (100, 290), (40, 41), (130, 270), (5, 299 - 4)])
    for delta in (1e-2, 1e-4, 1e-6):
        for sign in (1.0, -1.0):
            a, b = next(cols)
            w = rng.standard_normal(L)
            w -= w.mean()
            w -= (w @ xc) / (xc @ xc) * xc
            th = math.acos(1.0 - delta)
            M[:, a] = 3.0 + xc / np.linalg.norm(xc)
            M[:, b] = 5.0 + sign * (math.cos(th) * xc / np.linalg.norm(xc) + math.sin(th) * w / np.linalg.norm(w))
    for c, k in zip((10, 11, 150, 271, 272, 273), (1, 2, 3, 5, 33, 63)):
        M[:, c] = 3.0 + 0.5 * _walsh(L, k)   # values and mean exact; all pairwise products sum to exactly 0
    return M


def spikes(L, seed=0):
    """Features whose variance sits almost all in one draw, |z| ~ 1 there (the bf16 split of values near 1), in groups
    that share the draw: pairs with r -> +-1.  Draw 0 is the worst case of a truncating accumulation (the partial sum
    is ~r from the first MMA step on), draws L / 2 and L - 1 the others."""
    rng = np.random.default_rng(seed)
    C = C_SMALL
    M = _background(L, C, rng)
    slots = [0, 0, L // 2, L - 1, int(rng.integers(L)), 0]
    c = 0
    for slot in slots:
        for _ in range(40):
            x = 1.0 + 1e-3 * rng.standard_normal(L)
            x[slot] += rng.choice([-1.0, 1.0]) * rng.uniform(0.5, 2.0)
            M[:, c] = x
            c += 1
    return M


def offsets(L, kappa, seed=0):
    """mean / sd = kappa: make_traces' correlation structure, standardised, at levels spread over eight orders."""
    rng = np.random.default_rng(seed)
    G = make_traces(L, C_SMALL, seed=seed + 1)
    G = (G - G.mean(axis=0)) / G.std(axis=0)
    s = np.exp(rng.normal(0.0, 4.0, C_SMALL))
    return s * (kappa + G)


@pytest.mark.parametrize("L", LENGTHS)
def test_constructed_pairs(L):
    M = constructed_pairs(L, seed=L)
    ref = exact_cov(M)
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        _diag_exact(R, ref)
        _check("pairs", R, ref, L, nsplit)
        for c, k in ((10, 11), (11, 150), (150, 271), (272, 273)):
            assert abs(R[c, k]) / math.sqrt(R[c, c] * R[k, k]) < cov_bound(nsplit, L)   # orthogonal stays orthogonal


@pytest.mark.parametrize("L", LENGTHS)
def test_spikes(L):
    M = spikes(L, seed=L + 1)
    ref = exact_cov(M)
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        _diag_exact(R, ref)
        _check("spikes", R, ref, L, nsplit)


@pytest.mark.parametrize("kappa", [1e4, 1e8])
@pytest.mark.parametrize("L", LENGTHS)
def test_large_offsets(L, kappa):
    """The centring is exact on both sides (Sterbenz); what differs is the mean itself: the kernel's block sum is off by
    up to ~L eps kappa sd, which moves a covariance by that squared.  So the tolerance is the bound plus 2 (L eps kappa)^2
    (4e-6 at kappa = 1e8, L = 65536; nothing at kappa = 1e4), and the diagonal is the exact variance to 1e-12 plus the
    same term."""
    M = offsets(L, kappa, seed=L + 2)
    ref = exact_cov(M, fsum_mean=True)
    cond = 2.0 * (L * EPS * kappa) ** 2
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        _diag_exact(R, ref, rtol=1e-12 + cond)
        _check(f"offset {kappa:.0e}", R, ref, L, nsplit, extra=cond)


@pytest.mark.parametrize("L", LENGTHS)
def test_levels_1e_150_to_1e150(L):
    """Features scaled by 2^k, k spread over -498..498 (1e-150 .. 1e150): in correlation units the result is that of the
    unscaled traces (z, and so every tensor-core product, are the same; the fp64 rescaling r sd_i sd_j neither overflows
    nor underflows), to 1e-13 — and within the bound of the exact reference."""
    rng = np.random.default_rng(L + 3)
    base = _background(L, C_SMALL, rng)
    k = rng.permutation(np.linspace(-498, 498, C_SMALL).astype(np.int64))
    M = np.ldexp(base, k[None, :])
    ref = exact_cov(M)
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        assert np.all(np.isfinite(R))
        _diag_exact(R, ref)
        _check("levels 1e+-150", R, ref, L, nsplit)
        R0 = capi.trace_cov(base, nsplit=nsplit)
        d0 = np.sqrt(np.diag(R0))
        back = np.ldexp(R, -(k[:, None] + k[None, :]))
        assert np.max(np.abs(back - R0) / (d0[:, None] * d0[None, :])) < 1e-13


@pytest.fixture(scope="module")
def chain_traces():
    """Posterior traces of a gene-structured problem: EM, then Gibbs with stride 1 (slow trends, isoforms of one gene
    anti-correlated), 4200 transcripts in any order.  Both chains start from the EM estimate."""
    row_ptr, col, k, length, _, _, _ = make_gene_problem()
    feats = np.random.default_rng(3).permutation(len(length))[:4200].astype(np.int32)
    out = {}
    with capi.Handle(row_ptr, col, k, length) as H:
        H.init_mu()
        H.em(50, 0.1)
        mu_em = H.get_mu()
        for L in (1024, 2048):
            H.set_mu(mu_em)
            H.gibbs(7, 0, L, stride=1, trace_len=L)
            out[L] = (H.get_trace()[feats].T.copy(), [H.trace_cov(feats, nsplit=s) for s in (1, 2, 3)])
    return out


@pytest.mark.parametrize("L", [1024, 2048])
def test_chain_traces(chain_traces, L):
    M, Rs = chain_traces[L]
    ref = exact_cov(M)
    for nsplit, R in zip((1, 2, 3), Rs):
        _diag_exact(R, ref)
        e = _check("chain", R, ref, L, nsplit)
        if L == 1024 and nsplit == 2:
            assert e < 3e-5, e                  # what mmcollapse and bench.py run


def test_overflowing_feature_is_zeroed():
    """A feature whose centred sum of squares overflows (values ~1e160) gets a zero row and column, the diagonal included
    (include/mmq.h); every other entry is the covariance of the remaining features."""
    L = 1024
    M = make_traces(L, C_SMALL, seed=11)
    M[:, 7] = 1e160 * (1.0 + 0.5 * np.random.default_rng(12).standard_normal(L))
    keep = np.array([c for c in range(C_SMALL) if c != 7])
    ref = exact_cov(M[:, keep])
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        assert np.all(R[7, :] == 0) and np.all(R[:, 7] == 0)
        assert corr_err(R[np.ix_(keep, keep)], ref) < cov_bound(nsplit, L)


def _free_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


def test_large_C_64bit_output_offsets():
    """C = 47104 (C^2 > 2^31: the epilogue's R + gi + C gj needs 64 bits) at L = 64 on device pointers, R = 17.8 GB left
    on the device.  Sampled rows — the first and the last 256-row tile and 256 rows between — against the exact
    reference over all C columns (so every tile column, the last one included), and the same entries read from the
    mirrored columns: exactly equal."""
    import torch
    L, C = 64, 47104
    need = C * C * 8 + 2 * C * L * 8 + capi.trace_cov_workspace_bytes(L, C, 3) + (2 << 30)
    if _free_bytes() < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {_free_bytes() / 2**30:.1f} free")
    rng = np.random.default_rng(47)
    M = make_traces(L, C, seed=47)
    for a, b in ((5, C - 3), (C // 2, C - 200), (C - 256, 100)):
        M[:, b] = M[:, a]                      # duplicates between far tiles
    X = M - M.mean(axis=0)
    sd = np.sqrt((X * X).sum(axis=0) / (L - 1))
    rows = np.concatenate([np.arange(256), np.sort(rng.choice(np.arange(256, C - 256), 256, replace=False)),
                           np.arange(C - 256, C)])
    ref = (X[:, rows].T @ X) / (L - 1)
    dev = torch.device("cuda:0")
    Md = torch.from_numpy(np.ascontiguousarray(M.T)).to(dev)
    Rd = torch.empty((C, C), dtype=torch.float64, device=dev)
    rows_d = torch.from_numpy(rows).to(dev)
    try:
        for nsplit in (1, 2, 3):
            ws = torch.empty(capi.trace_cov_workspace_bytes(L, C, nsplit), dtype=torch.uint8, device=dev)
            Rd.fill_(float("nan"))
            st = torch.cuda.current_stream(dev)
            capi.trace_cov_dev(Md.data_ptr(), L, C, nsplit, Rd.data_ptr(), ws.data_ptr(), st.cuda_stream)
            Rr = Rd.index_select(0, rows_d).cpu().numpy()           # rows of the row-major tensor = columns of R
            Rc = Rd.index_select(1, rows_d).cpu().numpy().T
            del ws
            assert np.array_equal(Rr, Rc), "not exactly symmetric"
            assert np.allclose(Rr[np.arange(len(rows)), rows], sd[rows] ** 2, rtol=1e-12, atol=0.0)
            err = np.abs(Rr - ref) / (sd[rows][:, None] * sd[None, :])
            e = float(np.max(err))
            _TABLE.append(("large C", L, C, nsplit, e, cov_bound(nsplit, L), float("nan")))
            assert e < cov_bound(nsplit, L), (nsplit, e)
    finally:
        del Rd, Md
        torch.cuda.empty_cache()


def test_large_mean_corrs_64bit_slice_offsets():
    """mean_corrs_dev over ns = 9 slices of C = 16384 (ns C^2 = 2.4e9 > 2^31: k_mean_corrs' R + s C C needs 64 bits),
    the rows ts — first, middle and last, so the reads reach the end of the last slice — against mean_corrs_numpy's
    definition on the same slices."""
    import torch
    C, ns, L = 16384, 9, 64
    assert ns * C * C > 2 ** 31
    need = (ns + 2) * C * C * 8 + (2 << 30)
    if _free_bytes() < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {_free_bytes() / 2**30:.1f} free")
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(9)
    Rd = torch.empty((ns, C, C), dtype=torch.float64, device=dev)
    ws = torch.empty(capi.trace_cov_workspace_bytes(L, C, 2), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    try:
        for s in range(ns):
            Md = torch.from_numpy(np.ascontiguousarray(make_traces(L, C, seed=900 + s).T)).to(dev)
            capi.trace_cov_dev(Md.data_ptr(), L, C, 2, Rd[s].data_ptr(), ws.data_ptr(), st.cuda_stream)
            st.synchronize()
        S = (rng.random((C, ns)) < 0.8).astype(np.uint8)
        S[C - 1, :] = 1
        S[1, :] = 0
        Sd = torch.from_numpy(np.ascontiguousarray(S.T)).to(dev)       # C x ns column-major
        ts = np.array([0, 1, 4097, C // 2, C - 2, C - 1], np.int32)
        tsd = torch.from_numpy(ts).to(dev)
        idx = torch.from_numpy(ts.astype(np.int64)).to(dev)
        Rt = Rd.index_select(1, idx).cpu().numpy()
        D = torch.diagonal(Rd, dim1=1, dim2=2).cpu().numpy()
        for pen in (0.0, 0.5):
            Vd = torch.zeros((C, C), dtype=torch.float64, device=dev)
            Wd = torch.zeros((C, C), dtype=torch.float64, device=dev)
            capi.mean_corrs_dev(Rd.data_ptr(), Sd.data_ptr(), C, ns, tsd.data_ptr(), len(ts), pen, Vd.data_ptr(), Wd.data_ptr(),
                                st.cuda_stream)
            st.synchronize()
            Vo, Wo = mean_corrs_rows(Rt, D, S, ts, pen)
            for V, W in ((Vd.index_select(0, idx), Wd.index_select(0, idx)), (Vd.index_select(1, idx).T, Wd.index_select(1, idx).T)):
                V, W = V.cpu().numpy(), W.cpu().numpy()
                assert np.allclose(V, Vo, rtol=1e-12, atol=1e-14 + 1e-7 * pen, equal_nan=True)
                assert np.allclose(W, Wo, rtol=1e-9, atol=1e-7, equal_nan=True)
            del Vd, Wd
    finally:
        del Rd, ws
        torch.cuda.empty_cache()

