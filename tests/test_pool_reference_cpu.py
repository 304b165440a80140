"""The numpy definitions of the pooled summaries (tests/pool_reference.py) on analytic anchors: iid and AR(1) chains,
the percentile rule, constant, zero and NaN rows, the single-isoform probit columns and the exact sum of count moments."""
import math

import numpy as np
import pytest

from tests import pool_reference as pref


def ar1(rng, C, L, phi):
    x = np.empty((C, L))
    x[:, 0] = rng.standard_normal(C)
    e = rng.standard_normal((C, L)) * math.sqrt(1 - phi * phi)
    for s in range(1, L):
        x[:, s] = phi * x[:, s - 1] + e[:, s]
    return x


@pytest.mark.parametrize("C", [2, 4, 8])
def test_iid_chains_give_ess_near_S(C):
    rng = np.random.default_rng(C)
    L = 1024
    x = np.exp(rng.standard_normal((C, L)))
    lm, sd, ess, _ = pref.pooled_log(x)
    S = C * L
    assert abs(lm - np.log(x).mean()) < 1e-12 and abs(sd - np.log(x).std(ddof=1)) < 1e-12
    assert 0.8 * S < ess < 1.25 * S, ess
    mcse, iact = pref.mcse_iact(sd, ess, S)
    assert mcse == pytest.approx(sd / math.sqrt(ess)) and iact == pytest.approx(S / ess)


@pytest.mark.parametrize("phi", [0.5, 0.9])
def test_ar1_chains_give_ess_near_the_ar1_value(phi):
    rng = np.random.default_rng(int(phi * 10))
    C, L = 4, 2048
    x = np.exp(ar1(rng, C, L, phi))
    _, _, ess, _ = pref.pooled_log(x)
    want = C * L * (1 - phi) / (1 + phi)
    assert 0.7 * want < ess < 1.4 * want, (ess, want)


def test_percentiles_are_the_sorted_concatenation_at_the_rounded_indices():
    rng = np.random.default_rng(3)
    C, L = 3, 64
    x = rng.gamma(0.5, size=(C, L))
    idx = pref.pct_index([5, 25, 50, 75, 95], C * L)
    assert list(idx) == [round(p / 100 * (C * L - 1) + 1e-9) for p in (5, 25, 50, 75, 95)]
    assert np.array_equal(pref.percentiles(x, idx), np.sort(np.concatenate(list(x)))[idx])
    # half-way cases round away from zero, as C's round()
    assert list(pref.pct_index([50], 4)) == [2] and list(pref.pct_index([50], 2)) == [1]


def test_constant_zero_and_nan_rows():
    C, L = 2, 64
    lm, sd, ess, _ = pref.pooled_log(np.full((C, L), 0.7))
    assert lm == pytest.approx(math.log(0.7)) and sd < 1e-12 and math.isnan(ess)
    assert all(math.isnan(v) for v in pref.mcse_iact(sd, ess, C * L))
    z = np.random.default_rng(1).gamma(1.0, size=(C, L))
    z[1, 5] = 0.0
    lm, sd, ess, _ = pref.pooled_log(z)
    assert lm == -math.inf and math.isnan(sd) and math.isnan(ess)
    q = z.copy()
    q[0, 3] = math.nan
    assert all(math.isnan(v) for v in pref.pooled_log(q)[:3])
    # a NaN draw sorts last in the percentiles
    p = pref.percentiles(q, [0, C * L - 1])
    assert p[0] == 0.0 and math.isnan(p[1])


def test_proportions_pool_each_chain_over_its_own_gene():
    rng = np.random.default_rng(9)
    C, L = 3, 32
    mu = rng.gamma(2.0, size=(C, L))
    other = rng.gamma(2.0, size=(C, L))
    gene = mu + other
    idx = pref.pct_index([5, 50, 95], C * L)
    r = pref.pooled_props(mu, gene, True, idx)
    p = mu / gene
    from scipy.special import ndtri
    z = ndtri(np.clip(p, 1e-9, 1 - 1e-9))
    S = C * L
    assert r["mean"] == pytest.approx(p.mean(), rel=1e-14)
    assert r["mean_probit"] == pytest.approx(z.mean(), rel=1e-12)
    assert r["sd_probit"] == pytest.approx(z.std(ddof=1), rel=1e-10)
    assert np.array_equal(r["pct"], np.sort(p.ravel())[idx])
    # a gene of one isoform: probits are +inf, so the mean is inf and the sd inf - inf = NaN
    one = pref.pooled_props(mu, mu, False, idx)
    assert one["mean_probit"] == math.inf and math.isnan(one["sd_probit"])
    assert one["mean"] == 1.0 and S == 96


def test_count_moments_add_exactly_across_the_128_bit_carry():
    lo_near = np.array([2**64 - 5, 7], np.uint64)
    a = (100, np.array([10, 20], np.uint64), lo_near, np.array([0, 1], np.uint64))
    b = (100, np.array([30, 40], np.uint64), np.array([9, 2**64 - 1], np.uint64), np.array([2, 0], np.uint64))
    S, tot, sq = pref.add_count_moments([a, b])
    assert S == 200 and tot == [40, 60]
    assert sq == [(2**64 - 5) + 9 + (2 << 64), 7 + (2**64 - 1) + (1 << 64)]
    mean, sd = pref.count_columns(S, tot, sq)
    assert mean == [0.2, 0.3] and all(v > 0 for v in sd)
