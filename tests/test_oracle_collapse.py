"""The oracle's restatement of mmcollapse's covariance step (SURVEY.md section 8, row f3) against independent numpy
implementations: orc_cov vs numpy.cov (src/mmcollapse.cpp:553-558), orc_mean_corrs vs a literal numpy transcription of
src/mmcollapse.cpp:483-511.  CPU only."""
import numpy as np

from oracle import oracle as orc
from tests.collapse_case import exact_cov, make_traces, mean_corrs_numpy, mean_corrs_rows


def test_cov_matches_numpy_cov():
    M = make_traces(1024, 61, seed=3)
    R = orc.trace_cov(M)
    ref = np.cov(M, rowvar=False)
    d = np.sqrt(np.diag(ref))
    assert np.max(np.abs(R - ref) / (d[:, None] * d[None, :])) < 1e-13      # in correlation units (sums of 1024 products cancel)
    assert np.array_equal(R, R.T)


def test_cov_non_finite_entries_become_zero():
    M = make_traces(256, 9, seed=4)
    M[17, 3] = np.nan
    M[5, 6] = np.inf
    R = orc.trace_cov(M)
    assert np.all(R[3, :] == 0) and np.all(R[:, 3] == 0) and np.all(R[6, :] == 0) and np.all(R[:, 6] == 0)
    keep = [0, 1, 2, 4, 5, 7, 8]
    ref = np.cov(M[:, keep], rowvar=False)
    d = np.sqrt(np.diag(ref))
    assert np.max(np.abs(R[np.ix_(keep, keep)] - ref) / (d[:, None] * d[None, :])) < 1e-13


def test_constant_feature_has_zero_covariance():
    M = make_traces(128, 5, seed=5)
    M[:, 2] = 3.25
    R = orc.trace_cov(M)
    assert np.all(R[2, :] == 0) and np.all(R[:, 2] == 0)


def test_mean_corrs_matches_the_literal_transcription():
    rng = np.random.default_rng(7)
    ns, C = 5, 23
    R = np.stack([orc.trace_cov(make_traces(256, C, seed=10 + s)) for s in range(ns)])
    S = (rng.random((C, ns)) < 0.8).astype(np.uint8)
    S[0, :] = 1
    S[1, :] = 0                      # never observed: every mean is 0/0
    S[2, :] = 0
    S[2, 1] = 1                      # observed once: sd is not finite -> 0
    ts = np.arange(C)
    for pen in (0.0, 0.7):
        V, W = orc.mean_corrs(R, S, ts, pen)
        Vn, Wn = mean_corrs_numpy(R, S, ts, pen)
        assert np.allclose(V, Vn, rtol=1e-12, atol=1e-15, equal_nan=True)
        assert np.allclose(W, Wn, rtol=1e-12, atol=1e-15, equal_nan=True)
        assert np.isnan(V[1, 5]) and W[1, 5] == 0.0
    # a refresh of two rows only touches their rows and columns (src/mmcollapse.cpp:771)
    V0, W0 = orc.mean_corrs(R, S, ts, 0.0)
    R2 = R.copy()
    R2[:, 4, :] *= 1.5
    R2[:, :, 4] *= 1.5
    V1, W1 = orc.mean_corrs(R2, S, [4, 9], 0.0, V0.copy(), W0.copy())
    mask = np.ones((C, C), bool)
    mask[[4, 9], :] = False
    mask[:, [4, 9]] = False
    assert np.array_equal(V1[mask], V0[mask], equal_nan=True)


def test_single_sample_has_zero_sd():
    R = orc.trace_cov(make_traces(128, 6, seed=2))[None]
    V, W = orc.mean_corrs(R, np.ones((6, 1), np.uint8), np.arange(6))
    d = np.sqrt(np.diag(R[0]))
    assert np.allclose(V, R[0] / d[:, None] / d[None, :], rtol=1e-13) and np.all(W == 0)


def test_exact_cov_matches_the_oracle():
    """exact_cov, the reference of tests/test_gpu_cov_accuracy.py, is cov() with non-finite entries 0; its fsum means agree
    with numpy's where the mean is 1e8 times the spread."""
    M = make_traces(1024, 61, seed=3)
    M[3, 5] = np.nan
    R = exact_cov(M)
    ref = orc.trace_cov(M)
    d = np.sqrt(np.diag(ref))
    d = np.where(d > 0, d, 1.0)
    assert np.max(np.abs(R - ref) / (d[:, None] * d[None, :])) < 1e-13
    assert np.all(R[5, :] == 0) and np.all(R[:, 5] == 0)
    G = M[:, :4] - M[:, :4].mean(axis=0)
    Rb = exact_cov(G + 1e8 * G.std(axis=0), fsum_mean=True)
    d = np.sqrt(np.diag(Rb))
    assert np.max(np.abs(Rb - exact_cov(G)) / (d[:, None] * d[None, :])) < 1e-9


def test_mean_corrs_rows_matches_the_literal_transcription():
    rng = np.random.default_rng(8)
    ns, C = 4, 19
    R = np.stack([orc.trace_cov(make_traces(256, C, seed=30 + s)) for s in range(ns)])
    S = (rng.random((C, ns)) < 0.7).astype(np.uint8)
    S[1, :] = 0
    S[2, :] = 0
    S[2, 3] = 1
    ts = np.array([0, 1, 2, 7, C - 1])
    D = np.stack([np.diag(R[s]) for s in range(ns)])
    for pen in (0.0, 0.5):
        V, W = mean_corrs_numpy(R, S, ts, pen)
        Vr, Wr = mean_corrs_rows(R[:, ts, :], D, S, ts, pen)
        assert np.allclose(Vr, V[ts], rtol=1e-13, atol=1e-15, equal_nan=True)
        assert np.allclose(Wr, W[ts], rtol=1e-12, atol=1e-15, equal_nan=True)
