"""The shared samplers (include/mmq_sampler.h, compiled into the CPU replay) against exact distributions: one allocation
step at fixed mu on every path of mmq_alloc_row, per-fragment rows with weights, one Gamma step, and the composed
chain against the exact stationary posterior (tests/exact_reference.py).  The GPU kernels must reproduce this replay
bit for bit (tests/test_gpu_parity.py and others), so a wrong distribution here is a wrong distribution there; the
kernels are checked against the same references in tests/test_gpu_exact_distribution.py.  CPU only, smaller sample
sizes than the GPU file."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import exact_reference as E

SEED = 20261020


# ------------------------------------------------------------------ one allocation step

def _class_cases():
    """(d, k): every path of mmq_alloc_row and both sides of every routing boundary of the class plan."""
    cases = [(2, 1), (5, 1), (64, 1)]                                       # one categorical (CAT stream)
    cases += [(5, k) for k in (2, 63, 64, 65, 128, 129)]                   # categorical draws across 64-draw groups
    cases += [(12, k) for k in (16, 17, 32, 33, 352)]                      # ... and 16-draw slots (d > 8)
    for d in (2, 3, 5, 7, 9, 13, 16):                                       # categorical at the limit, chain above
        cases += [(d, E.cat_limit(d)), (d, E.cat_limit(d) + 1)]
    cases += [(7, 5000), (13, 100000), (3, 2000)]                           # chain with BTRS nodes; (3, 2000): BINV too
    cases += [(17, 512), (17, 513), (64, 513), (65, 300), (200, 300)]      # general path
    return sorted(set(cases))


@pytest.mark.parametrize("pattern", ["equal", "spread", "zero"])
@pytest.mark.parametrize("d,k", _class_cases())
def test_alloc_row_is_exact_multinomial(d, k, pattern):
    """mmq_alloc_row (through orc_draw_alloc: class ids 0..N-1, sweep 0) against Multinomial(k; p)."""
    mu = E.mu_pattern(d, pattern)
    N = 20000 if d * min(k, E.cat_limit(d)) <= 4096 else 6000
    X = orc.draw_alloc(SEED + d, N, mu, k)
    E.assert_multinomial(X, k, E.member_probs(mu), f"d={d} k={k} {pattern}")


def test_alloc_row_singletons_and_empty_classes():
    assert (orc.draw_alloc(SEED, 100, np.array([3.0]), 17) == 17).all()
    for d in (1, 2, 7, 65):
        assert (orc.draw_alloc(SEED, 100, np.ones(d), 0) == 0).all()


@pytest.mark.parametrize("d,k", [(5, 64), (13, 385), (65, 100)])
def test_class_plan_replay_is_exact_multinomial(d, k):
    """The class plan's CPU replay (mmq_cls_replay_host: the draws and sums of k_alloc_cls / k_alloc_chain / the
    general kernel) on R replicas of one class, S sweeps: routing statistics and the multinomial."""
    R, S = 2000, 4
    mu1 = E.mu_pattern(d, "spread")
    row_ptr, col, kk, mu = E.replicated_class(R, d, k, mu1)
    P = orc.Problem(row_ptr, col, kk, np.ones(R * d))
    X = []
    for s in range(S):
        c, st = P.cls_plan_replay(mu, SEED, s)
        x, c_r, _ = P.sweep_replay(mu, SEED, s, do_gamma=False)
        assert np.array_equal(c, c_r)
        X.append(c.reshape(R, d))
    assert st["in_use"] == 1
    piece = "small_classes" if k <= E.cat_limit(d) and d <= 64 else "chain_classes" if d <= 16 else "rest_classes"
    assert st[piece] == R, st
    E.assert_multinomial(np.concatenate(X), k, E.member_probs(mu1), f"class plan d={d} k={k}")


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("d,G", [(2, 8), (3, 1), (6, 4), (9, 3), (13, 2), (40, 5)])
def test_grouped_rows_are_sums_of_categoricals(d, G, weighted):
    """Per-fragment rows (k = NULL) through sweep_replay: groups of G identical neighbouring rows, unweighted or with
    per-row weights (some exactly 0), class-id base 3.  The group's counts are a sum of independent categoricals."""
    rng = np.random.default_rng(SEED + 97 * d + G)
    R, S = 3000, 4
    W = E.row_weights(rng, R, G, d) if weighted else None
    mu1 = E.mu_pattern(d, "spread")
    row_ptr, col, w, mu, Pr = E.grouped_rows(R, G, d, mu1, W)
    P = orc.Problem(row_ptr, col, None, np.ones(R * d), weight=w)
    X = np.concatenate([P.sweep_replay(mu, SEED, s, class_id_base=3, do_gamma=False)[1].reshape(R, d) for s in range(S)])
    E.assert_categorical_sum(X, Pr, f"d={d} G={G} weighted={weighted}")


# ------------------------------------------------------------------ one Gamma step

GAMMA_COUNTS = [0, 1, 3, 1000, 1000000, 500000000]


@pytest.mark.parametrize("c", GAMMA_COUNTS)
def test_gamma_step_collapsed_is_exact(c):
    """Singleton classes of c fragments (c = 0: the shape alpha < 1 boost path), lengths spread over 10^4: the Gamma
    step of sweep_replay, by PIT and mean."""
    n = 100000
    l = np.exp(np.random.default_rng(c % 1000 + 1).uniform(np.log(1e-3), np.log(10.0), n))
    row_ptr = np.arange(n + 1, dtype=np.int64)
    P = orc.Problem(row_ptr, np.arange(n, dtype=np.int32), np.full(n, c, np.int32), l)
    _, counts, mu = P.sweep_replay(np.ones(n), SEED, 5)
    assert (counts == c).all()
    E.assert_gamma_step(mu, counts, l, P.alpha, P.beta, f"collapsed c={c}")


@pytest.mark.parametrize("c", [0, 1, 3, 10])
def test_gamma_step_per_fragment_is_exact(c):
    """The same with c one-member rows per transcript (k = NULL)."""
    n = 100000
    l = np.exp(np.random.default_rng(c + 7).uniform(np.log(1e-3), np.log(10.0), n))
    row_ptr = np.arange(n * c + 1, dtype=np.int64)
    P = orc.Problem(row_ptr, np.repeat(np.arange(n, dtype=np.int32), c), None, l)
    _, counts, mu = P.sweep_replay(np.ones(n), SEED, 6)
    assert (counts == c).all()
    E.assert_gamma_step(mu, counts, l, P.alpha, P.beta, f"per-fragment c={c}")


@pytest.mark.parametrize("a", [0.1, 0.55, 0.999, 1.1, 3.1, 1000.1])
def test_draw_gamma_is_exact(a):
    x = orc.draw_gamma(SEED, 100000, a, 2.5)
    E.assert_gamma_step(x, np.full(len(x), a - 0.1), np.full(len(x), 2.4), 0.1, 0.1, f"draw_gamma a={a}")


# ------------------------------------------------------------------ the chain against the exact posterior

@pytest.mark.parametrize("name", list(E.posterior_components()))
def test_gibbs_replay_matches_exact_posterior(name):
    """R replicas of one component from exact stationary draws, 48 sweeps of gibbs_replay with a trace: per member the
    time-averages of log mu and of 1{mu <= q} at the exact quartiles."""
    kind, spec = E.posterior_components()[name]
    R, S = 300, 48
    post = E.posterior_of(kind, spec)
    row_ptr, col, k, w, l = E.posterior_problem(kind, spec, R)
    P = orc.Problem(row_ptr, col, k, l, weight=w, alpha=E.POSTERIOR_ALPHA, beta=E.POSTERIOR_BETA)
    mu0 = post.sample_mu(np.random.default_rng(SEED), R).reshape(-1)
    _, trace = P.gibbs_replay(mu0, SEED, 0, S, 1, S)
    z, where = E.posterior_z(post, trace, R)
    assert abs(z) <= E.Z_MAX, f"{name}: worst z = {z:.2f} ({where})"
