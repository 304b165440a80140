"""The numpy reference of the several-chain diagnostics (tests/chain_reference.py) on analytic anchors, and the chain
seeds restated in Python against the library's mmq_chain_seed.  No GPU needed."""
import ctypes
import math
import os

import numpy as np
import pytest
from scipy.signal import lfilter

from tests import chain_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ar1(rng, shape, phi):
    """stationary AR(1) with unit marginal variance along the last axis"""
    e = rng.standard_normal(shape) * math.sqrt(1 - phi * phi)
    e[..., 0] = rng.standard_normal(shape[:-1])
    return lfilter([1.0], [1.0, -phi], e, axis=-1)


def test_iid_normal_rhat_one_and_ess_equal_to_draws():
    rng = np.random.default_rng(1)
    C, L, rows = 4, 1024, 2000
    out, _ = ref.diagnose_rows(rng.standard_normal((C, rows, L)))
    assert abs(out["rhat"].mean() - 1.0) < 0.003
    assert 0.95 < out["ess_bulk"].mean() / (C * L) < 1.05
    assert 0.9 < out["ess_tail"].mean() / (C * L) < 1.1
    assert np.isnan(out["log_mean"]).sum() == rows                      # half the draws are negative: log is NaN


def test_ar1_bulk_ess_matches_the_integrated_autocorrelation():
    rng = np.random.default_rng(2)
    C, L, rows, phi = 4, 1024, 200, 0.9
    out, _ = ref.diagnose_rows(ar1(rng, (C, rows, L), phi))
    want = (1 - phi) / (1 + phi)
    assert abs(out["ess_bulk"].mean() / (C * L) / want - 1) < 0.1


def test_one_chain_shifted_by_one_sd_is_caught():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((4, 300, 1024))
    x[2] += 1.0
    out, _ = ref.diagnose_rows(x)
    assert (out["rhat"] > 1.05).all(), out["rhat"].min()


def test_one_chain_scaled_is_caught_by_the_folded_term():
    rng = np.random.default_rng(4)
    x = rng.standard_normal((4, 300, 1024))
    x[1] *= 3.0
    out, _ = ref.diagnose_rows(x)
    assert (out["rhat"] > 1.05).all(), out["rhat"].min()
    unfolded = np.array([ref.rhat(ref.split(ref.rank_normalise(x[:, r].ravel()).reshape(4, 1024))) for r in range(300)])
    assert (unfolded < 1.01).all(), unfolded.max()


def test_constant_ties_zeros_and_non_finite_rows():
    rng = np.random.default_rng(5)
    d, _ = ref.diagnose(np.full((3, 64), 2.5))
    assert math.isnan(d["rhat"]) and math.isnan(d["ess_bulk"]) and math.isnan(d["ess_tail"])
    assert abs(d["log_mean"] - math.log(2.5)) < 1e-15 and d["log_sd"] < 1e-15
    ties = rng.choice([0.5, 1.0, 2.0], size=(4, 256))
    d, _ = ref.diagnose(ties)
    assert 0.9 < d["rhat"] < 1.1 and 0.5 * 1024 < d["ess_bulk"] < 2 * 1024
    assert math.isnan(d["ess_tail"])                                     # q95 is the top level: every draw is <= q95
    z = rng.gamma(0.5, size=(2, 128))
    z[0, :7] = 0.0
    d, _ = ref.diagnose(z)
    assert d["log_mean"] == -math.inf and math.isnan(d["log_sd"]) and math.isfinite(d["rhat"]) and math.isfinite(d["ess_bulk"])
    for bad in (math.nan, math.inf, -math.inf):
        x = rng.gamma(2.0, size=(2, 64))
        x[1, 5] = bad
        d, _ = ref.diagnose(x)
        assert all(math.isnan(d[k]) for k in ref.OUTPUTS)


def test_tail_indicator_without_variance_gives_nan():
    x = np.ones((2, 64))
    x[0, 0] = 2.0                                                        # q05 = q95 = 1: every draw but one is <= both
    d, _ = ref.diagnose(x)
    assert not math.isnan(d["ess_tail"])                                 # one draw above q95: the indicator varies
    x = np.ones((2, 64))
    x[:, :32] = 0.5                                                      # q95 = 1: all draws are <= q95
    d, _ = ref.diagnose(x)
    assert math.isnan(d["ess_tail"])


def test_chain_seeds_restated():
    assert ref.chain_seeds(1234, 1) == [1234]
    seeds = np.random.default_rng(6).integers(0, 2 ** 32, 10000)
    for s in seeds:
        got = ref.chain_seeds(int(s), ref.CHAINS_MAX)
        assert got[0] == s and len(set(got)) == ref.CHAINS_MAX


def test_chain_seeds_match_the_library():
    path = os.path.join(ROOT, "mmseq_b200", "libmmseq_b200.so")
    if not os.path.exists(path):
        import __graft_entry__ as g
        g.build()
    lib = ctypes.CDLL(path)
    lib.mmq_chain_seed.restype = ctypes.c_uint32
    lib.mmq_chain_seed.argtypes = [ctypes.c_uint32, ctypes.c_int]
    for s in [0, 1, 99, 1234, 2 ** 32 - 1] + list(np.random.default_rng(7).integers(0, 2 ** 32, 200)):
        want = ref.chain_seeds(int(s), ref.CHAINS_MAX)
        assert [lib.mmq_chain_seed(int(s), c) for c in range(ref.CHAINS_MAX)] == want
        assert lib.mmq_chain_seed(int(s), ref.CHAINS_MAX) == s and lib.mmq_chain_seed(int(s), -1) == s
