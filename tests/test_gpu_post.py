"""Device post-processing (mmq_summarize, mmq_prop_summaries, mmq_unique_hits_sets,
mmq_sokal_batch) against the reference's own sokal golden vectors and the numpy oracle."""
import os

import numpy as np
import pytest
from scipy import special

from mmseq_b200 import capi
from oracle import oracle as orc
from tests.collapse_case import make_gene_problem

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "sokal_golden.npz")


def test_sokal_kernel_matches_reference_golden():
    g = np.load(GOLD)
    meta = g["meta"]
    for i in range(int(g["nseries"])):
        x = g[f"x{i}"]
        var, tau, win, st = capi.sokal_batch(x[None, :])
        erc, evar, etau, em = meta[i]
        assert st[0] == int(erc) and win[0] == int(em), (i, win[0], em)
        assert np.isclose(var[0], evar, rtol=1e-10, atol=1e-300)
        assert (np.isnan(tau[0]) and np.isnan(etau)) or np.isclose(tau[0], etau, rtol=1e-9, atol=1e-12)
    for n, code in ((3, 200), (6, 201), (1000, 201)):
        assert capi.sokal_batch(np.zeros((2, n)))[3].tolist() == [code, code]


def test_sokal_batch_many_rows_vs_oracle():
    """Every row, with more rows than one pass of the grid: mmq_sokal_batch runs k_row_sokal on min(rows, 148 * 8) CTAs,
    one row per CTA and pass (mmq_post.cu:272)."""
    rows = 4000
    assert rows > 3 * 148 * 8
    rng = np.random.default_rng(2)
    x = np.cumsum(rng.standard_normal((rows, 1024)), axis=1) * 0.02 + rng.standard_normal((rows, 1024))
    var, tau, win, st = capi.sokal_batch(x)
    for r in range(rows):
        rc, v, t, m = orc.sokal(x[r])
        assert st[r] == rc == 0 and win[r] == m, r
        assert np.isclose(var[r], v, rtol=1e-10) and np.isclose(tau[r], t, rtol=1e-9), r


def _check_summaries_groups_props_uh(row_ptr, col, k, length, gene_of_col, G, ident_ptr, ident_mem, L, stride):
    """Group traces, per-row summaries of transcripts, identical sets and genes, proportions and uh() of one handle against
    the numpy/oracle restatements.  Genes are over observed columns, with an "extra" (prior-simulated) term for gene 3."""
    n = len(length)
    P = orc.Problem(row_ptr, col, k, length)
    mu0, _, _ = P.init_mu()
    order = np.argsort(gene_of_col, kind="stable")
    gptr = np.concatenate([[0], np.cumsum(np.bincount(gene_of_col, minlength=G))])
    members = order.astype(np.int32)
    rng = np.random.default_rng(4)
    extra = np.zeros((G, L)); extra[3] = rng.gamma(0.1, 5.0, L)
    with capi.Handle(row_ptr, col, k, length) as H:
        H.set_mu(mu0)
        H.gibbs(1234, 0, L * stride, stride=stride, trace_len=L)
        tr = H.get_trace()
        H.set_groups(capi.MMQ_GROUP_GENE, gptr, members, extra)
        H.set_groups(capi.MMQ_GROUP_IDENTICAL, ident_ptr, ident_mem)
        pct_idx = [int(round(p / 100.0 * (L - 1))) for p in (5, 25, 50, 75, 95)]
        S0 = H.summarize(0, pct_idx)
        S1 = H.summarize(1, pct_idx)
        S2 = H.summarize(2, pct_idx)
        gt = H.get_group_trace(2)
        it = H.get_group_trace(1)
        multi = (np.diff(gptr)[gene_of_col] > 1).astype(np.uint8)
        PR = H.prop_summaries(gene_of_col, multi, pct_idx, want_trace=True)
        set_of = gene_of_col.astype(np.int32)
        uh = H.unique_hits_sets(set_of, G)
    # group traces
    gt_o = np.zeros((G, L)); np.add.at(gt_o, gene_of_col, tr); gt_o += extra
    assert np.allclose(gt, gt_o, rtol=1e-13)
    it_o = np.zeros((len(ident_ptr) - 1, L)); np.add.at(it_o, np.repeat(np.arange(len(ident_ptr) - 1), np.diff(ident_ptr)), tr[ident_mem])
    assert np.allclose(it, it_o, rtol=1e-14)
    # per-row summaries vs the numpy/oracle restatement
    for S, trace in ((S0, tr), (S1, it), (S2, gt)):
        O = orc.summaries_transcripts(trace)
        # genes without any observed member have an all-zero trace: log -> -inf, var/tau -> nan on both sides
        with np.errstate(invalid="ignore"):
            assert np.allclose(S["log_mean"], O["log_mu"], rtol=1e-12, atol=1e-12, equal_nan=True)
        assert np.array_equal(S["win"], O["win"])
        assert np.allclose(S["var"], O["var"], rtol=1e-9, equal_nan=True)
        assert np.allclose(S["tau"], O["iact"], rtol=1e-8, atol=1e-10, equal_nan=True)
        assert np.array_equal(S["pct"], O["pct"])                  # order statistics: exact
    # proportions
    prop = tr / gt[gene_of_col]
    assert np.allclose(PR["prop_trace"], prop, rtol=1e-15)
    assert np.allclose(PR["mean_prop"], prop.mean(axis=1), rtol=1e-12)
    z = special.ndtri(np.clip(prop, 1e-9, 1 - 1e-9))
    m = multi.astype(bool)
    assert np.allclose(PR["sum_probit"][m], z[m].sum(axis=1), rtol=1e-9, atol=1e-7)
    assert np.allclose(PR["sumsq_probit"][m], (z[m] ** 2).sum(axis=1), rtol=1e-9)
    assert np.all(np.isinf(PR["sum_probit"][~m]))                  # single-isoform genes: +inf (src/mmseq.cpp:1252)
    assert np.array_equal(PR["pct"], np.sort(prop, axis=1)[:, pct_idx])
    # uh(): literal restatement of src/uh.cpp on the same sets
    uh_o = orc.uh_literal(row_ptr, col, k, gptr, members)
    assert np.array_equal(uh, uh_o)


def test_summaries_groups_props_uh(small_problem, small_synth):
    h, s = small_problem, small_synth
    _check_summaries_groups_props_uh(h.row_ptr, h.col, h.k, h.len, s.gene_of[h.col2hdr], s.G,
                                     np.array([0, 2, 5]), np.array([0, 1, 4, 5, 6], np.int32), L=256, stride=2)


@pytest.mark.parametrize("L", [4, 2048])
def test_summaries_groups_props_uh_many_rows(L):
    """The checks of test_summaries_groups_props_uh with more transcripts, genes and identical sets than one pass of each
    grid covers, at the shortest and the longest trace mmq_summarize accepts (4 and MMQ_MAX_ROW_LEN = 2048)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    row_ptr, col, k, length, gene_of, ident_ptr, ident_mem = make_gene_problem()
    n, G, I = len(length), int(gene_of.max()) + 1, len(ident_ptr) - 1
    assert min(n, G, I) > 4 * 148 * 8        # k_row_sokal, k_row_percentiles (mmq_post.cu:272,283): min(rows, 148 * 8) CTAs
    assert n > 4 * sms * 8                   # k_prop (mmq_post.cu:386): min(n, sms * 8) CTAs, one transcript per CTA pass
    assert min(G, I) > 2 * sms * 16          # k_group_trace (mmq_post.cu:248): min(groups, sms * 16) CTAs
    _check_summaries_groups_props_uh(row_ptr, col, k, length, gene_of, G, ident_ptr, ident_mem, L=L, stride=2 if L == 4 else 1)


def test_prior_draws_bit_exact_and_distributed():
    """mmq_prior_draws (src/mmseq.cpp:971-978 on the device) equals the CPU replay bit for bit
    and follows Gamma(alpha, rate)."""
    from scipy import stats
    ids = np.array([3, 17, 123456], np.int64)
    ls = np.array([1e-3, 5.0, 2e-5])
    alpha, beta = 0.1, 0.1
    got = capi.prior_draws(ids, beta + ls, alpha, 1234, 1024)
    want = orc.prior_replay(ids, ls, alpha, beta, 1234, 1024)
    assert np.array_equal(got, want)
    big = capi.prior_draws(np.arange(64, dtype=np.int64), np.full(64, 2.5), 0.7, 99, 1024).ravel()
    assert stats.kstest(big, "gamma", args=(0.7, 0, 1 / 2.5)).pvalue > 1e-4
