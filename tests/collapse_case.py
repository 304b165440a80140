"""Shared inputs of the mmcollapse-covariance tests: trace matrices shaped like the posterior traces of collapse candidates
(raw-scale mu: log-normal levels over several orders of magnitude, blocks of anti-correlated features as unidentifiable
transcripts produce, a few exactly duplicated and a few tiny-variance columns) and a literal numpy transcription of
src/mmcollapse.cpp:483-511."""
import numpy as np


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
