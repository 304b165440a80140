"""The definitions of include/mmq.h's isoform pairs (mmseq -isocorr), restated in numpy.

Pairs: for every gene, its observed members m_0 .. m_{k-1} in CSR order; every (a, b) with a < b, a-major; genes in
order.  Draws: x[c, i, s], chain c's draw of trace row i at slot s; a pair's values come from the same (c, s).  Per pair:
the two-pass correlation of x and of log x over all S = C L draws (centred on the pooled mean, clamped to [-1, 1]) and
P(x_i > x_j) with ties counting one half.  Shared fragments: the sum of k_r over the hit classes r holding both members."""
import numpy as np


def pairs(gene_ptr, members):
    """(gene, a, b, member_a, member_b) int64 arrays of every pair in pair order, and pair_base int64[ngenes]"""
    gene_ptr = np.asarray(gene_ptr, np.int64)
    members = np.asarray(members, np.int64)
    g_, a_, b_, base = [], [], [], []
    for g in range(len(gene_ptr) - 1):
        base.append(len(g_))
        k = int(gene_ptr[g + 1] - gene_ptr[g])
        for a in range(k):
            for b in range(a + 1, k):
                g_.append(g); a_.append(a); b_.append(b)
    g_, a_, b_ = (np.array(v, np.int64) for v in (g_, a_, b_))
    q0 = gene_ptr[g_] if len(g_) else np.zeros(0, np.int64)
    return g_, a_, b_, members[q0 + a_] if len(g_) else g_, members[q0 + b_] if len(g_) else g_, np.array(base, np.int64)


def pair_index(pair_base, g, a, b, k):
    return pair_base[g] + a * (2 * k - a - 1) // 2 + (b - a - 1)


def gene_local(gene_ptr, members, n):
    """gene_of / local_of int32[n] of mmq_pair_shared_counts: -1 unless the row is a member of a gene of two or more"""
    gene_of = np.full(n, -1, np.int32)
    local_of = np.full(n, -1, np.int32)
    for g in range(len(gene_ptr) - 1):
        mem = members[gene_ptr[g]:gene_ptr[g + 1]]
        if len(mem) >= 2:
            gene_of[mem] = g
            local_of[mem] = np.arange(len(mem))
    return gene_of, local_of


def _corr(u, v):
    """two-pass correlation of the rows of u and v (pairs, S); NaN when a value is not finite or a sum of squares is 0"""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        du = u - u.mean(axis=1, keepdims=True)
        dv = v - v.mean(axis=1, keepdims=True)
        suu, svv, suv = (du * du).sum(1), (dv * dv).sum(1), (du * dv).sum(1)
        c = suv / np.sqrt(suu * svv)
    bad = ~np.isfinite(u).all(1) | ~np.isfinite(v).all(1) | (suu == 0) | (svv == 0)
    c = np.clip(c, -1.0, 1.0)
    c[bad] = np.nan
    return c


def summaries(x, gene_ptr, members):
    """x (C, n, L) -> dict(corr_mu, corr_log_mu, prob_1_gt_2: fp64[npairs])"""
    x = np.asarray(x, np.float64)
    C, n, L = x.shape
    _, _, _, ma, mb, _ = pairs(gene_ptr, members)
    flat = np.transpose(x, (1, 0, 2)).reshape(n, C * L)                  # row i: chain 0's L draws, then chain 1's, ...
    u, v = flat[ma], flat[mb]
    with np.errstate(invalid="ignore", divide="ignore"):
        lu, lv = np.log(u), np.log(v)
    lu[~(np.isfinite(u) & (u > 0))] = np.nan
    lv[~(np.isfinite(v) & (v > 0))] = np.nan
    prob = ((u > v).sum(1) + 0.5 * (u == v).sum(1)) / (C * L)
    out = dict(corr_mu=_corr(u, v), corr_log_mu=_corr(lu, lv), prob_1_gt_2=prob.astype(np.float64))
    anynan = np.isnan(u).any(1) | np.isnan(v).any(1)
    for k in out:
        out[k][anynan] = np.nan
    return out


def shared(row_ptr, col, k, gene_ptr, members):
    """shared fragments int64[npairs]: per hit class (k None: 1 per row) every two positions that are members of one
    gene, added at that pair"""
    gene_ptr = np.asarray(gene_ptr, np.int64)
    n = int(max(np.max(col, initial=-1), np.max(members, initial=-1))) + 1
    gene_of, local_of = gene_local(gene_ptr, np.asarray(members, np.int64), n)
    _, _, _, _, _, base = pairs(gene_ptr, members)
    npairs = int(sum(int(d) * (int(d) - 1) // 2 for d in np.diff(gene_ptr)))
    out = np.zeros(npairs, np.int64)
    for r in range(len(row_ptr) - 1):
        w = 1 if k is None else int(k[r])
        row = [int(t) for t in col[row_ptr[r]:row_ptr[r + 1]]]
        for i in range(len(row)):
            for j in range(i + 1, len(row)):
                t, u = row[i], row[j]
                g = gene_of[t]
                if g < 0 or gene_of[u] != g or local_of[t] == local_of[u]:
                    continue
                a, b = sorted((int(local_of[t]), int(local_of[u])))
                kk = int(gene_ptr[g + 1] - gene_ptr[g])
                out[pair_index(base, g, a, b, kk)] += w
    return out
