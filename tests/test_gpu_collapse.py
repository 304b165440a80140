"""mmcollapse's covariance step on the GPU (SURVEY.md section 8, row f3; src/mmcollapse.cpp:483-561) against the oracle,
through the C ABI.  Tolerances, in correlation units (|cov_gpu - cov_oracle| / (sd_i sd_j)): the tensor-core products are
split bf16 (nsplit terms per value, fp32 accumulation) and held to cov_bound(nsplit, L) = A + 1.5e-8 L, A = 6e-3 / 1.2e-5 /
2e-7 for nsplit = 1 / 2 / 3 (include/mmq.h; tests/test_gpu_cov_accuracy.py asserts it at every accepted L); everything
else (means, variances = the diagonal, the scaling back to covariance, mean_corrs) is fp64: 1e-12."""
import numpy as np
import pytest

from mmseq_b200 import capi
from oracle import oracle as orc
from tests.collapse_case import corr_err, cov_bound, make_gene_problem, make_traces

pytestmark = pytest.mark.gpu


def _pair_tiles(C, sms):
    """k_cov_gemm2's work (mmq_cov.cu:467-468): T (T + 1) / 2 upper-triangle tiles of 256 x 256, T = ceil(C / 256), swept
    by min(tiles, sms / 2) CTA pairs."""
    T = -(-C // 256)
    return T * (T + 1) // 2, sms // 2


# C = 5197: 21 tiles a side (the last one ragged), 231 tiles, more than 3 x 74 CTA pairs on 148 SMs: every pair takes three
# or more tiles, so each reuses TMEM accumulator 0 at least twice and the mbarrier phases wrap.  L = 64, 192 and 1024: one,
# three and sixteen MMA iterations per tile (nsplit 1) against the 4-stage ring.
@pytest.mark.parametrize("L,C", [(64, 1), (64, 5), (1024, 37), (1024, 128), (1024, 129), (1024, 300), (512, 1000), (2048, 257),
                                 (64, 5197), (192, 5197), (1024, 5197)])
def test_cov_matches_oracle(L, C):
    import torch
    if C > 5000:
        tiles, pairs = _pair_tiles(C, torch.cuda.get_device_properties(0).multi_processor_count)
        assert tiles > 3 * pairs, (tiles, pairs)
    M = make_traces(L, C, seed=L + C)
    ref = orc.trace_cov(M)
    for nsplit in (1, 2, 3):
        R = capi.trace_cov(M, nsplit=nsplit)
        assert np.array_equal(R, R.T), "not exactly symmetric"
        assert np.allclose(np.diag(R), np.diag(ref), rtol=1e-12, atol=0.0), "diagonal is the fp64 variance"
        e = corr_err(R, ref)
        assert e < cov_bound(nsplit, L), (nsplit, e)
    if C > 8:
        d = np.sqrt(np.diag(R))
        assert abs(R[0, C - 1] / (d[0] * d[C - 1]) - 1.0) < cov_bound(3, L)     # duplicated feature


def test_cov_full_size_tile_grid():
    """Several tiles per side incl. a ragged last tile; every tile of the upper triangle and its mirror written."""
    L, C = 1024, 5 * 128 + 77
    M = make_traces(L, C, seed=99)
    ref = orc.trace_cov(M)
    R = capi.trace_cov(M, nsplit=2)
    assert np.array_equal(R, R.T)
    assert corr_err(R, ref) < cov_bound(2, L)
    r_gpu = R / np.sqrt(np.outer(np.diag(R), np.diag(R)))
    r_ref = ref / np.sqrt(np.outer(np.diag(ref), np.diag(ref)))
    assert np.sqrt(np.mean((r_gpu - r_ref) ** 2)) < 2e-6                 # typical error far below the bound


def test_cov_non_finite_and_constant_features():
    M = make_traces(256, 140, seed=4)
    M[17, 3] = np.nan
    M[5, 130] = np.inf
    M[:, 77] = 2.5
    ref = orc.trace_cov(M)
    R = capi.trace_cov(M, nsplit=2)
    for c in (3, 130, 77):
        assert np.all(R[c, :] == 0) and np.all(R[:, c] == 0)
    assert np.all(np.isfinite(R)) and corr_err(R, ref) < cov_bound(2, 256)


def test_cov_rejects_bad_arguments():
    with pytest.raises(capi.MmqError):
        capi.trace_cov(np.ones((100, 4)))          # L not a multiple of 64
    with pytest.raises(capi.MmqError):
        capi.trace_cov(np.ones((128, 4)), nsplit=4)


def test_cov_device_pointers_and_stream():
    import torch
    L, C = 1024, 384
    M = make_traces(L, C, seed=8)
    dev = torch.device("cuda:0")
    Md = torch.from_numpy(np.ascontiguousarray(M.T)).to(dev)            # [C][L]: column c of M contiguous
    Rd = torch.empty((C, C), dtype=torch.float64, device=dev)
    ws = torch.empty(capi.trace_cov_workspace_bytes(L, C, 2), dtype=torch.uint8, device=dev)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        capi.trace_cov_dev(Md.data_ptr(), L, C, 2, Rd.data_ptr(), ws.data_ptr(), st.cuda_stream)
    st.synchronize()
    R = Rd.cpu().numpy()
    assert np.array_equal(R, capi.trace_cov(M, nsplit=2))


def test_cov_from_a_handles_trace(small_problem):
    p = small_problem
    H = capi.Handle(p.row_ptr, p.col, p.k, p.len)
    H.init_mu()
    H.em(50, 0.1)
    L = 256
    H.gibbs(7, 0, L * 4, stride=4, trace_len=L)
    tr = H.get_trace()                                                   # [n][L]
    feats = np.arange(0, p.n, 2, dtype=np.int32)[::-1].copy()            # any order, any subset
    R = H.trace_cov(feats, nsplit=3)
    ref = orc.trace_cov(tr[feats].T)
    assert corr_err(R, ref) < cov_bound(3, L)
    assert np.array_equal(R, capi.trace_cov(tr[feats].T, nsplit=3))
    H.close()


def test_cov_from_a_handles_trace_many_tiles():
    """The gather path (features picked from the handle's trace on the device) with more tiles than CTA pairs."""
    import torch
    row_ptr, col, k, length, _, _, _ = make_gene_problem()
    C, L = 4200, 1024
    tiles, pairs = _pair_tiles(C, torch.cuda.get_device_properties(0).multi_processor_count)
    assert tiles > 2 * pairs, (tiles, pairs)
    feats = np.random.default_rng(3).permutation(len(length))[:C].astype(np.int32)
    with capi.Handle(row_ptr, col, k, length) as H:
        H.init_mu()
        H.em(50, 0.1)
        H.gibbs(7, 0, L, stride=1, trace_len=L)
        tr = H.get_trace()
        R = H.trace_cov(feats, nsplit=3)
    assert np.array_equal(R, capi.trace_cov(tr[feats].T, nsplit=3))     # the gather path is the host-matrix path
    ref = orc.trace_cov(tr[feats].T)
    assert np.array_equal(R, R.T)
    assert np.allclose(np.diag(R), np.diag(ref), rtol=1e-12, atol=0.0)
    assert corr_err(R, ref) < cov_bound(3, L)


def _check_mean_corrs(ns, C):
    rng = np.random.default_rng(7)
    R = np.stack([capi.trace_cov(make_traces(256, C, seed=20 + s), nsplit=2) for s in range(ns)])
    S = (rng.random((C, ns)) < 0.8).astype(np.uint8)
    S[1, :] = 0
    S[2, :] = 0
    S[2, 1] = 1
    ts = np.arange(C)
    for pen in (0.0, 0.5):
        V, W = capi.mean_corrs(R, S, ts, pen)
        Vo, Wo = orc.mean_corrs(R, S, ts, pen)
        # the sd is a difference of two nearly equal terms when the correlations agree over the samples: sqrt(1e-16) = 1e-8
        assert np.allclose(V, Vo, rtol=1e-12, atol=1e-14 + 1e-7 * pen, equal_nan=True)
        assert np.allclose(W, Wo, rtol=1e-9, atol=1e-7, equal_nan=True)
    V0, W0 = capi.mean_corrs(R, S, ts)
    V1, W1 = capi.mean_corrs(R, S, [4, 9], 0.0, V0.copy() + 1.0, W0.copy())
    Vo, Wo = orc.mean_corrs(R, S, [4, 9], 0.0, V0.copy() + 1.0, W0.copy())
    assert np.allclose(V1, Vo, rtol=1e-12, atol=1e-14, equal_nan=True)


def test_mean_corrs_matches_oracle():
    _check_mean_corrs(6, 150)


def test_mean_corrs_many_pairs_matches_oracle():
    """C = 1600: C^2 = 2.56 M (row, column) pairs, more than twice what one pass of k_mean_corrs covers: min(pairs / 256,
    148 * 32) CTAs of 256 threads (mmq_cov.cu:587)."""
    C = 1600
    assert C * C > 2 * 148 * 32 * 256
    _check_mean_corrs(4, C)
