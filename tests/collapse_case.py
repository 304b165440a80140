"""Shared inputs of the mmcollapse-covariance tests: trace matrices shaped like the posterior traces of collapse candidates
(raw-scale mu: log-normal levels over several orders of magnitude, blocks of anti-correlated features as unidentifiable
transcripts produce, a few exactly duplicated and a few tiny-variance columns), a literal numpy transcription of
src/mmcollapse.cpp:483-511, an exact fp64 covariance and the covariance kernel's error bound."""
import math

import numpy as np

# k_cov_gemm2's error bound in correlation units, |cov_gpu - cov_exact| / (sd_i sd_j), for nsplit bf16 terms per value
# and trace length L; include/mmq.h states the same.  COV_A[nsplit] is the bf16 split: each term keeps 8 significant bits
# of what the previous ones left.  COV_B * L is the fp32 accumulation in TMEM, which truncates towards zero: the error is
# a bias towards r = 0 that grows linearly with L (L / 16 MMA steps per split product).  Fitted on one B200 (1000 W) to
# the largest error of tests/test_gpu_cov_accuracy.py at each (nsplit, L), L = 64 .. 65536, and to 2.0e-5 measured on chain
# traces at nsplit = 3, L = 2048: at least 1.5x that error everywhere (nsplit = 1 at L = 1024: 4.0e-3 on chain traces;
# nsplit = 2 at L = 1024: 1.66e-5 on chain traces, L = 64: 7.5e-6 at C = 47104; at L = 65536 about 3.4e-4, 2.9x).
COV_A = {1: 6e-3, 2: 1.2e-5, 3: 2e-7}
COV_B = 1.5e-8


def cov_bound(nsplit, L):
    return COV_A[nsplit] + COV_B * L


def corr_err(R, ref):
    """max |R - ref| / (sd_i sd_j), sd from the reference's diagonal (1 where it is 0)."""
    d = np.sqrt(np.diag(ref))
    d = np.where(d > 0, d, 1.0)
    return np.max(np.abs(R - ref) / (d[:, None] * d[None, :]))


def exact_cov(M, fsum_mean=False):
    """Two-pass centred fp64 covariance of the L x C matrix M (column = feature), non-finite entries -> 0 as
    src/mmcollapse.cpp:556-558.  The centring of x against an fp64 mean is exact wherever |x - mean| <= |mean| (Sterbenz),
    so what is left is the fp64 dot products: ~1e-13 relative to sd_i sd_j at L = 65536.  fsum_mean: the means by
    math.fsum (correctly rounded), for columns whose mean is many orders above their spread."""
    M = np.asarray(M, np.float64)
    L = M.shape[0]
    if fsum_mean:
        mean = np.array([math.fsum(M[:, c]) / L for c in range(M.shape[1])])
    else:
        mean = M.mean(axis=0)
    X = M - mean
    with np.errstate(all="ignore"):
        R = (X.T @ X) / max(L - 1, 1)
    R[~np.isfinite(R)] = 0.0
    return R


def mean_corrs_rows(Rt, D, S, ts, sdpenalty=0.0):
    """mean_corrs_numpy for the rows ts only, vectorised: Rt[s, i, v] = R[s, ts[i], v], D[s, v] = R[s, v, v].  Returns the
    rows V[ts, :], W[ts, :]."""
    ns = Rt.shape[0]
    ts = np.asarray(ts)
    with np.errstate(all="ignore"):
        r = Rt / np.sqrt(D[:, ts])[:, :, None]
        r = r / np.sqrt(D)[:, None, :]
        u = (S[ts, :].T.astype(np.int64)[:, :, None] * S.T.astype(np.int64)[:, None, :]).astype(np.float64)
        r = np.where(u == 0, 0.0, r)
        n = u.sum(axis=0)
        mean = (u * r).sum(axis=0) / n
        if ns > 1:
            sd = np.sqrt((n / (n - 1.0)) * ((u * r * r).sum(axis=0) / n - mean * mean))
            sd = np.where(np.isfinite(sd), sd, 0.0)
        else:
            sd = np.zeros_like(mean)
    return mean + sdpenalty * sd, sd


def make_traces(L, C, seed=0, blocks=True):
    rng = np.random.default_rng(seed)
    level = np.exp(rng.normal(0.0, 3.0, C))
    M = np.empty((L, C))
    c = 0
    while c < C:
        g = int(min(C - c, rng.integers(1, 6))) if blocks else 1
        total = np.exp(rng.normal(0.0, 0.15, L))             # the well-identified sum of the block
        w = rng.dirichlet(np.ones(g) * 2.0, size=L)          # how the sum splits: anti-correlated members
        for j in range(g):
            M[:, c + j] = level[c] * total * w[:, j] * np.exp(rng.normal(0, 0.05, L))
        c += g
    if C > 8:
        M[:, C - 1] = M[:, 0]                                 # duplicate feature: correlation exactly 1
        M[:, C - 2] = 1e-9 * (1.0 + 1e-3 * rng.standard_normal(L))   # tiny level
    return M


def mean_corrs_numpy(R, S, ts, sdpenalty=0.0):
    """src/mmcollapse.cpp:483-511, loop for loop."""
    ns, C, _ = R.shape
    V = np.zeros((C, C))
    W = np.zeros((C, C))
    with np.errstate(all="ignore"):
        for t in ts:
            for v in range(C):
                r = R[:, t, v].copy()
                r = r / np.sqrt(R[:, t, t])
                r = r / np.sqrt(R[:, v, v])
                u = (S[t, :].astype(np.int64) * S[v, :].astype(np.int64)).astype(np.float64)
                r[u == 0] = 0.0
                n = u.sum()
                mean = np.dot(u, r) / n
                if ns > 1:
                    sd = np.sqrt((n / (n - 1.0)) * (np.dot(u, r * r) / n - mean * mean))
                    if not np.isfinite(sd):
                        sd = 0.0
                else:
                    sd = 0.0
                V[t, v] = V[v, t] = mean + sdpenalty * sd
                W[t, v] = W[v, t] = sd
    return V, W


def make_gene_problem(n=12000, G=5000, n_ident=5000, m=30000, seed=0):
    """A hand-built collapsed problem with a gene structure: n transcripts in G non-empty genes (1..~6 isoforms), m
    classes of 1..6 members drawn among neighbouring isoforms, counts k in 1..49, and n_ident disjoint identical-transcript
    sets of two.  Returns (row_ptr, col, k, len, gene_of, ident_ptr, ident_members)."""
    rng = np.random.default_rng(seed)
    gene_of = np.concatenate([np.arange(G), rng.integers(0, G, n - G)])
    rng.shuffle(gene_of)
    by_gene = np.argsort(gene_of, kind="stable").astype(np.int32)     # isoforms of a gene are neighbours here
    d = rng.integers(1, 7, m)
    start = rng.integers(0, n - 6, m)
    pos = np.repeat(start, d) + (np.arange(int(d.sum())) - np.repeat(np.cumsum(d) - d, d))
    row = np.repeat(np.arange(m), d)
    col = by_gene[pos]
    o = np.lexsort((col, row))                                          # members ascending within a class
    col = col[o]
    row_ptr = np.concatenate([[0], np.cumsum(d)]).astype(np.int64)
    k = rng.integers(1, 50, m).astype(np.int32)
    length = rng.uniform(1e-6, 1e-2, n)
    ident_mem = rng.permutation(n)[:2 * n_ident].astype(np.int32)
    ident_ptr = np.arange(0, 2 * n_ident + 1, 2, dtype=np.int64)
    return row_ptr, col, k, length, gene_of.astype(np.int32), ident_ptr, ident_mem
