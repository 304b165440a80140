"""The numpy definitions of transcripts per million (tests/tpm_reference.py) on anchors: the three-transcript hand
example, TPM summing to 1e6 over transcripts and over genes in every draw, empty groups, non-finite draws, the totals'
tile order against the exact sum, one chain against several and the percentile indices."""
import math

import numpy as np
import pytest

from tests import tpm_reference as tref


def test_hand_example():
    """SURVEY.md section 4: three transcripts of equal effective length 1000, classes {A}:10, {A,B}:5, {B,C}:3, N = 18,
    mu0 = (12.5, 4, 1.5) / 1.8e-5.  With equal lengths TPM is the share of the fragments: (12.5, 4, 1.5) / 18 * 1e6."""
    mu0 = np.array([12.5, 4.0, 1.5]) / 1.8e-5
    chains = np.repeat(mu0[None, :, None], 4, axis=2)                    # one chain of four equal draws
    totals = tref.totals_tiled(chains[0])[None, :]
    want = np.array([12.5, 4.0, 1.5]) / 18 * 1e6
    for t in range(3):
        mean, sd, pct = tref.summaries(tref.tpm_draws(chains, totals, [t]), tref.pct_index((5, 50, 95), 4))
        assert mean == pytest.approx(want[t], rel=1e-15) and sd == 0.0 and (pct == mean).all()
        assert tref.em_tpm(mu0, [t]) == pytest.approx(want[t], rel=1e-15)
    mean, _, _ = tref.summaries(tref.tpm_draws(chains, totals, [0, 1]), [0])   # a gene {A, B}
    assert mean == pytest.approx(16.5 / 18 * 1e6, rel=1e-15)
    assert tref.em_tpm(mu0, [0, 1, 2]) == pytest.approx(1e6, rel=1e-15)


def _sample(rng, C, n, L):
    return np.exp(rng.normal(0.0, 2.0, (C, n, L)) + rng.normal(0.0, 3.0, (1, n, 1)))


def test_every_draw_sums_to_a_million_over_transcripts_and_over_genes():
    rng = np.random.default_rng(3)
    C, n, L = 2, 700, 16
    x = _sample(rng, C, n, L)
    totals = np.stack([tref.totals_tiled(x[c]) for c in range(C)])
    per_t = np.stack([tref.tpm_draws(x, totals, [t]) for t in range(n)])
    assert np.allclose(per_t.sum(axis=0), 1e6, rtol=1e-12, atol=0)
    genes = np.array_split(rng.permutation(n), 90)                       # a partition of the transcripts
    per_g = np.stack([tref.tpm_draws(x, totals, g) for g in genes])
    assert np.allclose(per_g.sum(axis=0), per_t.sum(axis=0), rtol=1e-12, atol=0)
    em = rng.gamma(2.0, 1.0, n)
    assert math.fsum(tref.em_tpm(em, [t]) for t in range(n)) == pytest.approx(1e6, rel=1e-12)
    assert math.fsum(tref.em_tpm(em, g) for g in genes) == pytest.approx(1e6, rel=1e-12)


def test_empty_groups_give_zero():
    rng = np.random.default_rng(4)
    x = _sample(rng, 3, 20, 8)
    totals = np.stack([tref.totals_tiled(x[c]) for c in range(3)])
    d = tref.tpm_draws(x, totals, [])
    assert (d == 0).all() and not np.signbit(d).any()
    mean, sd, pct = tref.summaries(d, tref.pct_index((5, 50, 95), 24))
    assert mean == 0.0 and sd == 0.0 and (pct == 0).all()
    assert tref.em_tpm(np.ones(20), []) == 0.0
    out = tref.features(x, totals, [0, 0, 2, 2], [4, 7], [0, 23])
    assert (out["mean"][[0, 2]] == 0).all() and out["mean"][1] > 0


@pytest.mark.parametrize("bad", [math.nan, math.inf])
def test_non_finite_draws_give_nan_mean_and_sd_and_sort_last(bad):
    rng = np.random.default_rng(5)
    x = _sample(rng, 2, 10, 8)
    x[1, 3, 5] = bad
    totals = np.stack([tref.totals_tiled(x[c]) for c in range(2)])
    idx = np.arange(16)
    mean, sd, pct = tref.summaries(tref.tpm_draws(x, totals, [3]), idx)
    assert math.isnan(mean) and math.isnan(sd)
    assert np.isnan(pct[-1]) and np.isfinite(pct[:-1]).all() and (np.diff(pct[:-1]) >= 0).all()
    # the total of that draw is not finite either: another transcript's draw there is NaN / NaN or finite / inf = 0
    other = tref.tpm_draws(x, totals, [4])
    if math.isnan(bad):
        assert math.isnan(tref.summaries(other, idx)[0])
    else:
        assert other[1, 5] == 0.0 and math.isfinite(tref.summaries(other, idx)[0])
    assert (np.isnan(tref.summaries(x[:1, :1, :] * math.nan, [0, 99])[2])).all()   # NaN draws; an index outside [0, S)


@pytest.mark.parametrize("n", [1, 511, 512, 513, 1025, 5000])
def test_tiled_totals_within_1e_12_of_the_exact_sum(n):
    rng = np.random.default_rng(n)
    tr = _sample(rng, 1, n, 8)[0]
    exact, tiled = tref.totals_fsum(tr), tref.totals_tiled(tr)
    assert (np.abs(tiled - exact) <= 1e-12 * exact).all()
    if n <= tref.TILE:                                                   # one tile: the plain sequential sum
        seq = np.zeros(8)
        for t in range(n):
            seq = seq + tr[t]
        assert tiled.tobytes() == seq.tobytes()


def test_one_chain_against_several():
    """C chains each over its own totals are the draws of one chain of C L slots over the concatenated totals"""
    rng = np.random.default_rng(6)
    C, n, L = 4, 30, 8
    x = _sample(rng, C, n, L)
    totals = np.stack([tref.totals_tiled(x[c]) for c in range(C)])
    one = np.concatenate(list(x), axis=1)[None]                          # (1, n, C L)
    idx = tref.pct_index((5, 25, 50, 75, 95), C * L)
    for mem in ([2], [0, 5, 9]):
        a = tref.summaries(tref.tpm_draws(x, totals, mem), idx)
        b = tref.summaries(tref.tpm_draws(one, totals.reshape(1, -1), mem), idx)
        assert a[0] == b[0] and a[1] == b[1] and a[2].tobytes() == b[2].tobytes()
    # chain 0 alone is the single-chain run
    a = tref.summaries(tref.tpm_draws(x[:1], totals[:1], [2]), tref.pct_index((50,), L))
    assert a[0] == pytest.approx(np.mean(x[0, 2] / totals[0] * 1e6), rel=1e-14)


def test_percentile_indices():
    P = (5, 25, 50, 75, 95)
    assert tref.pct_index(P, 4).tolist() == [0, 1, 2, 2, 3]
    assert tref.pct_index(P, 1024).tolist() == [51, 256, 512, 767, 972]
    assert tref.pct_index(P, 8192).tolist() == [410, 2048, 4096, 6143, 7781]
    assert tref.pct_index((0, 100), 8192).tolist() == [0, 8191]
