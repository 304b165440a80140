"""The numpy reference of `mmseq -allelic` (tests/allelic_reference.py): the pairing rules, the symmetry of A and B, and on
independent Gamma draws of the two copies the Beta law of the fraction."""
import math

import numpy as np
import pytest

from tests import allelic_reference as aref

scipy_stats = pytest.importorskip("scipy.stats")


def test_pairs_need_both_copies_in_one_gene():
    names = ["x_A", "x_B", "lone_A", "far_A", "iso", "far_B", "y_B", "y_A", "z_A", "z_B", "w_B", "_A", "_B"]
    gene_of = [0, 0, 0, 0, 0, 1, 1, 1, 2, 2, 2, 3, 3]
    a, b, stems, lonely = aref.find_pairs(names, gene_of)
    # pairs in the header order of the _A copy; far_A / far_B sit in two genes; lone_A and w_B have no partner
    assert stems == ["x", "y", "z", ""] and a == [0, 7, 8, 11] and b == [1, 6, 9, 12]
    assert lonely == 4                                                    # lone_A, far_A, far_B, w_B


def test_gene_with_several_pairs_and_unpaired_isoforms():
    names = ["g0_iso", "p_A", "p_B", "q_A", "solo_A", "q_B", "r_A", "r_B", "h_iso"]
    gene_of = [0, 0, 0, 0, 0, 0, 1, 1, 2]
    a, b, stems, lonely = aref.find_pairs(names, gene_of)
    assert stems == ["p", "q", "r"] and lonely == 1
    units = aref.gene_units(a, gene_of, 3)
    assert units == [[0, 1], [2], []]
    a_ptr, a_mem, b_ptr, b_mem = aref.csr(units, a, b)
    assert a_ptr.tolist() == [0, 2, 3, 3] and a_mem.tolist() == [1, 3, 6]
    assert b_ptr.tolist() == [0, 2, 3, 3] and b_mem.tolist() == [2, 5, 7]


def _case(rng, C=2, n=40, L=256, nprior=5):
    chains = np.exp(rng.normal(0.0, 2.0, (C, n, L)))
    priors = rng.gamma(0.1, 1.0, (C, nprior, L))
    units = []
    for r in range(30):
        ka, kb = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        units.append((rng.choice(n + nprior, ka, replace=False), rng.choice(n + nprior, kb, replace=False)))
    a_ptr = np.concatenate([[0], np.cumsum([len(u[0]) for u in units])])
    b_ptr = np.concatenate([[0], np.cumsum([len(u[1]) for u in units])])
    a_mem = np.concatenate([u[0] for u in units]).astype(np.int32)
    b_mem = np.concatenate([u[1] for u in units]).astype(np.int32)
    return chains, priors, a_ptr, a_mem, b_ptr, b_mem


def test_swapping_sides_mirrors_every_column():
    rng = np.random.default_rng(1)
    chains, priors, a_ptr, a_mem, b_ptr, b_mem = _case(rng)
    S = chains.shape[0] * chains.shape[2]
    idx = aref.pct_index((0, 5, 25, 75, 95, 100), S)                    # indices that mirror: q and S - 1 - q
    assert (idx == S - 1 - idx[::-1]).all()
    fwd = aref.units(chains, priors, a_ptr, a_mem, b_ptr, b_mem, idx)
    rev = aref.units(chains, priors, b_ptr, b_mem, a_ptr, a_mem, idx)
    for r in range(len(a_ptr) - 1):
        _, _, phi = aref.fraction(chains, priors, a_mem[a_ptr[r]:a_ptr[r + 1]], b_mem[b_ptr[r]:b_ptr[r + 1]])
        _, _, psi = aref.fraction(chains, priors, b_mem[b_ptr[r]:b_ptr[r + 1]], a_mem[a_ptr[r]:a_ptr[r + 1]])
        # a / (a + b) + b / (b + a) = 1 within one ulp of 1 (three roundings), summed exactly
        err = [abs(math.fsum((float(x), float(y), -1.0))) for x, y in zip(phi.ravel(), psi.ravel())]
        assert max(err) <= np.spacing(1.0)
    assert np.allclose(fwd["mean"], 1.0 - rev["mean"], rtol=0, atol=1e-14)
    assert np.allclose(fwd["sd"], rev["sd"], rtol=1e-12, atol=0)
    assert (fwd["prob_a"] == 1.0 - rev["prob_a"]).all()
    assert np.allclose(fwd["pct"], 1.0 - rev["pct"][:, ::-1], rtol=0, atol=1e-15)
    # allele-only fragments: the two columns swap
    row_ptr = np.array([0, 2, 3, 5, 6, 8])
    col = np.array([0, 1, 1, 2, 3, 3, 0, 2])
    k = np.array([5, 7, 11, 13, 17])
    unit_of = np.array([0, 0, 1, 1])
    side = np.array([0, 1, 0, 1], np.uint8)
    a, b = aref.allele_only(row_ptr, col, k, unit_of, side, 2)
    assert a.tolist() == [17, 17] and b.tolist() == [7, 13]              # rows 0 and 2 hold both sides of their unit
    b2, a2 = aref.allele_only(row_ptr, col, k, unit_of, 1 - side, 2)
    assert (a == a2).all() and (b == b2).all()
    a1, b1 = aref.allele_only(row_ptr, col, None, unit_of, side, 2)       # one per row when there are no counts
    assert a1.tolist() == [1, 1] and b1.tolist() == [1, 1]


def test_non_finite_fraction_is_nan_everywhere():
    a = np.array([[1.0, 0.0, 2.0, 1.0]])
    b = np.array([[1.0, 0.0, 1.0, 3.0]])
    with np.errstate(invalid="ignore"):
        phi = a / (a + b)
    mean, sd, prob, pct = aref.summaries(a, b, phi, [0, 2])
    assert math.isnan(mean) and math.isnan(sd) and math.isnan(prob) and np.isnan(pct).all()
    a[0, 1] = 3.0
    mean, sd, prob, pct = aref.summaries(a, b, a / (a + b), [0, 1, 2, 3])
    assert prob == (2 + 0.5) / 4 and pct.tolist() == sorted((a / (a + b)).ravel().tolist())
    assert aref.em_fraction([0.0, 0.0], [0, 5], [1]) != aref.em_fraction([0.0, 0.0], [0, 5], [1])   # NaN
    assert aref.em_fraction([2.0, 6.0], [0, 5], [1]) == 0.25             # id 5 >= n: a hit-less copy counts 0


@pytest.mark.parametrize("ka,kb", [(0, 0), (3, 1), (40, 25)])
def test_independent_gamma_draws_give_a_beta_fraction(ka, kb):
    """x_A ~ Gamma(alpha + k_A, r), x_B ~ Gamma(alpha + k_B, r) independent: x_A / (x_A + x_B) ~ Beta(alpha + k_A,
    alpha + k_B); P(a > b) is that Beta's mass above one half."""
    rng = np.random.default_rng(100 + ka)
    alpha, rate, L = 0.1, 3.7, 8192
    chains = np.stack([rng.gamma(alpha + ka, 1.0 / rate, L), rng.gamma(alpha + kb, 1.0 / rate, L)])[None]
    a, b, phi = aref.fraction(chains, None, [0], [1])
    beta = scipy_stats.beta(alpha + ka, alpha + kb)
    assert scipy_stats.kstest(phi.ravel(), beta.cdf).pvalue > 1e-3
    idx = aref.pct_index((50,), L)
    mean, sd, prob, pct = aref.summaries(a, b, phi, idx)
    assert abs(mean - beta.mean()) <= 4 * beta.std() / math.sqrt(L)
    p = beta.sf(0.5)
    assert abs(prob - p) <= 4 * math.sqrt(p * (1 - p) / L) + 1e-12
