"""The sampler kernels against exact distributions (tests/exact_reference.py), through the C ABI.

The parity tests compare every kernel with the CPU replay bit for bit; both compile include/mmq_sampler.h, so those
tests cannot see a distribution that is wrong on both sides.  Here each kernel path is checked against the exact law of
what it samples:
  * one allocation step at fixed mu: R replicas of one class (or of a group of one-fragment rows) over members of its
    own, S sweeps: per-member mean and variance, pairwise covariance, binomial marginals, the joint pmf when small;
    members with p = 0 never receive a fragment.  Each case asserts that it reached the kernel it is meant for
    (cls_stats for collapsed shards, the run structure of the by-length layout for per-fragment ones).
  * one Gamma step: PIT values of mu' given known counts, KS per shape stratum, and the mean.
  * the composed chain (CUDA graph, trace) from an exact stationary start against the exact stationary posterior.
At least 10^5 draws per statistic.  Seeds are fixed; runs are deterministic."""
import functools
import time

import numpy as np
import pytest

from mmseq_b200 import capi
from tests import exact_reference as E

pytestmark = pytest.mark.gpu

SEED = 20261021
S_SWEEPS = 16
MMQ_SEG_MAX = 96        # mmq_seg.cu: a per-fragment shard with more runs of equal class size takes the ragged kernel


@pytest.fixture(scope="module", autouse=True)
def _report_wall_time(request):
    t0 = time.perf_counter()
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    if tr is not None:
        tr.write_line(f"\n{__name__}: {time.perf_counter() - t0:.1f} s wall time")


def _sweep_counts(H, mu, R, d, flags, S=S_SWEEPS):
    """S sweeps at fixed mu: the counts of every sweep, (S R, d)."""
    out = []
    for s in range(S):
        H.set_mu(mu)
        _, c, _ = H.sweep_debug(SEED, 1000 + s, flags, want_x=False)
        out.append(c.reshape(R, d))
    return np.concatenate(out)


# ------------------------------------------------------------------ collapsed: the class plan

def _piece(d, k):
    """The piece of the class plan (mmq_cls_plan.h) that allocates a class of k fragments over d members."""
    if d == 1 or k == 0:
        return "none"
    if d <= 64 and k <= E.cat_limit(d):
        return "small"
    return "chain" if d <= 16 else "rest"


def _collapsed_cases():
    """(d, k, piece of the class plan it must reach)."""
    cases = [(2, 0), (1, 5)]                                                # nothing random: empty classes, singletons
    cases += [(d, 1) for d in (2, 3, 8, 9, 33, 64)]                         # k_alloc_cls1
    cases += [(d, k) for d in (2, 5, 8) for k in (2, 32)]                   # k_alloc_cls<LO>
    cases += [(8, k) for k in (63, 64, 65, 128, 129)]                       # LO, across 64-draw slots
    cases += [(12, k) for k in (16, 17, 32, 33)]                            # k_alloc_cls<HI>, across 16-draw slots
    cases += [(9, 256), (40, 512), (64, 512)]
    for d in (2, 3, 5, 7, 9, 13, 16):                                       # categorical at the limit, chain above
        cases += [(d, E.cat_limit(d)), (d, E.cat_limit(d) + 1)]
    cases += [(3, 2000), (7, 5000), (13, 100000)]                           # BINV and BTRS nodes
    cases += [(17, 512), (17, 513), (64, 513), (65, 300), (200, 300)]       # above 16 and 64 members: the general kernel
    return [(d, k, _piece(d, k)) for d, k in cases]


def _assert_routing(st, R, d, k, piece):
    """cls_stats of R classes of (d, k) built by the default (device) plan builder, whose small-set count is in slots
    (mmq_cls.cu: a class takes ceil(k / draws per slot) of them: 64 draws per slot up to 8 members, 16 above)."""
    assert st["in_use"] == 1, st
    slots = (-(-k // (64 if d <= 8 else 16))) if piece == "small" else 0
    want = dict(small_classes=R * slots, chain_classes=R if piece == "chain" else 0, rest_classes=R if piece == "rest" else 0)
    assert {key: st[key] for key in want} == want, (d, k, st)
    assert st["class_slots"] == 32 * (-(-R * slots // 32)), (d, k, st)       # 32-slot chunks


@pytest.mark.parametrize("pattern", ["equal", "spread", "zero"])
@pytest.mark.parametrize("d,k,piece", _collapsed_cases())
def test_class_plan_allocation_is_exact(d, k, piece, pattern):
    if d == 1 and pattern != "equal":
        pytest.skip("one member: no pattern")
    R = 8192 if d <= 64 else 6400
    mu1 = np.ones(1) if d == 1 else E.mu_pattern(d, pattern)
    row_ptr, col, kk, mu = E.replicated_class(R, d, k, mu1)
    with capi.Handle(row_ptr, col, kk, np.ones(R * d)) as H:
        _assert_routing(H.cls_stats(), R, d, k, piece)
        X = _sweep_counts(H, mu, R, d, capi.MMQ_GIBBS_DEFAULT)
    E.assert_multinomial(X, k, E.member_probs(mu1), f"d={d} k={k} {pattern}")


@pytest.mark.parametrize("flags", [capi.MMQ_GIBBS_GENERIC_KERNEL, capi.MMQ_GIBBS_TRANSPOSED])
@pytest.mark.parametrize("d,k", [(2, 1), (5, 65), (12, 33), (7, E.cat_limit(7)), (7, E.cat_limit(7) + 1), (13, 100000),
                                 (65, 300)])
def test_general_and_transposed_allocation_is_exact(d, k, flags):
    """The same shards through the general kernel and the transposed kernel (k_alloc with X, then k_count_reduce)."""
    R = 8192
    mu1 = E.mu_pattern(d, "zero")
    row_ptr, col, kk, mu = E.replicated_class(R, d, k, mu1)
    with capi.Handle(row_ptr, col, kk, np.ones(R * d)) as H:
        X = _sweep_counts(H, mu, R, d, flags)
    E.assert_multinomial(X, k, E.member_probs(mu1), f"d={d} k={k} flags={flags}")


# ------------------------------------------------------------------ per fragment: the by-length layout

PF_SIZES = [2, 3, 4, 5, 6, 7, 9, 12, 13, 40]  # k_alloc_seg4: registers (2..6), staged pairs (7..12), global (13, 40)
PF_GROUPS = 8
PF_REPLICAS = 6400                             # per (class size, group size): 10^5 draws per statistic in 16 sweeps


@functools.lru_cache(maxsize=None)
def _pf_shard(weighted):
    """One by-length shard: for every class size D of PF_SIZES, PF_REPLICAS groups of G identical neighbouring rows for
    each G in 1..8, over D members of their own; weights exp(N(0, 1/2)) with 1 in 8 exactly 0.  Singleton rows (some
    transcripts get fragments no other transcript explains) come first, as in the loader's layout."""
    rng = np.random.default_rng(SEED + int(weighted))
    rows_ptr, cols, ws, mus, blocks = [np.zeros(1, np.int64)], [], [], [], []
    n = 0
    n_single = 5000
    cols.append(np.arange(n_single, dtype=np.int32)); mus.append(np.ones(n_single))
    if weighted:
        ws.append(np.ones(n_single, np.float32))
    rows_ptr.append(np.arange(1, n_single + 1, dtype=np.int64))
    n = n_single
    nnz = n_single
    for D in PF_SIZES:
        mu1 = E.mu_pattern(D, "spread")
        for G in range(1, PF_GROUPS + 1):
            R = PF_REPLICAS
            W = E.row_weights(rng, R, G, D) if weighted else None
            rp, col, w, mu, P = E.grouped_rows(R, G, D, mu1, W)
            cols.append(col + n); mus.append(mu)
            if weighted:
                ws.append(w)
            rows_ptr.append(rp[1:] + nnz)
            blocks.append((D, G, n, R, P))
            n += R * D
            nnz += int(rp[-1])
    row_ptr = np.concatenate(rows_ptr)
    return row_ptr, np.concatenate(cols), (np.concatenate(ws) if weighted else None), np.concatenate(mus), n, blocks


@pytest.mark.parametrize("flags", [capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_RAGGED_KERNEL, capi.MMQ_GIBBS_GENERIC_KERNEL,
                                   capi.MMQ_GIBBS_TRANSPOSED])
@pytest.mark.parametrize("weighted", [False, True])
def test_per_fragment_allocation_is_exact(weighted, flags):
    """k_alloc_seg4 (default), k_alloc_cat (ragged), the general and the transposed kernel on the by-length layout,
    class-id base 3 (not a multiple of 4: the segment kernel pads each run with dummy rows)."""
    row_ptr, col, w, mu, n, blocks = _pf_shard(weighted)
    d = np.diff(row_ptr)
    assert (np.diff(d) >= 0).all() and np.count_nonzero(np.bincount(d)) <= MMQ_SEG_MAX    # the by-length layout
    with capi.Handle(row_ptr, col, None, np.ones(n), weight=w, class_id_base=3) as H:
        counts = []
        for s in range(S_SWEEPS):
            H.set_mu(mu)
            _, c, _ = H.sweep_debug(SEED, 2000 + s, flags, want_x=False)
            counts.append(c)
    C = np.stack(counts)
    assert (C[:, :5000] == 1).all()                                        # singleton rows
    worst = 0.0
    for D, G, off, R, P in blocks:
        X = C[:, off:off + R * D].reshape(S_SWEEPS * R, D)
        z = E.assert_categorical_sum(X, P, f"D={D} G={G} weighted={weighted} flags={flags}")
        worst = max(worst, abs(z))
    print(f"per-fragment weighted={weighted} flags={flags}: worst |z| = {worst:.2f}")


# ------------------------------------------------------------------ one Gamma step

GAMMA_N = 100000


def _lengths(c):
    return np.exp(np.random.default_rng(c % 1000 + 11).uniform(np.log(1e-3), np.log(10.0), GAMMA_N))


def test_gamma_step_collapsed_is_exact():
    """Singleton classes of c fragments per stratum (c = 0: the shape alpha < 1 boost path), lengths spread over 10^4.
    Three consecutive sweeps: the counts restart from the singleton base each sweep (seg_base), so each sweep's count
    must be exactly c; the PIT values of the three sweeps are pooled per stratum."""
    cs = [0, 1, 3, 1000, 1000000, 500000000]
    n = GAMMA_N * len(cs)
    l = np.concatenate([_lengths(c) for c in cs])
    k = np.repeat(np.array(cs, np.int32), GAMMA_N)
    with capi.Handle(np.arange(n + 1, dtype=np.int64), np.arange(n, dtype=np.int32), k, l) as H:
        H.set_mu(np.ones(n))
        mus = []
        for s in range(3):
            _, c, mu = H.sweep_debug(SEED, 7 + s, capi.MMQ_GIBBS_DEFAULT, want_x=False)
            assert np.array_equal(c, k), s
            mus.append(mu)
    for i, c in enumerate(cs):
        sl = slice(i * GAMMA_N, (i + 1) * GAMMA_N)
        E.assert_gamma_step(np.concatenate([m[sl] for m in mus]), np.full(3 * GAMMA_N, c), np.tile(l[sl], 3), 0.1, 0.1,
                            f"collapsed c={c}")


def test_gamma_step_per_fragment_is_exact():
    """The same per fragment: c one-member rows per transcript (the counts restart from the singleton base)."""
    cs = [0, 1, 3, 10]
    n = GAMMA_N * len(cs)
    l = np.concatenate([_lengths(c) for c in cs])
    cnt = np.repeat(np.array(cs), GAMMA_N)
    col = np.repeat(np.arange(n, dtype=np.int32), cnt)
    with capi.Handle(np.arange(len(col) + 1, dtype=np.int64), col, None, l) as H:
        H.set_mu(np.ones(n))
        mus = []
        for s in range(3):
            _, c, mu = H.sweep_debug(SEED, 17 + s, capi.MMQ_GIBBS_DEFAULT, want_x=False)
            assert np.array_equal(c, cnt), s
            mus.append(mu)
    for i, c in enumerate(cs):
        sl = slice(i * GAMMA_N, (i + 1) * GAMMA_N)
        E.assert_gamma_step(np.concatenate([m[sl] for m in mus]), np.full(3 * GAMMA_N, c), np.tile(l[sl], 3), 0.1, 0.1,
                            f"per-fragment c={c}")


# ------------------------------------------------------------------ the chain against the exact posterior

@pytest.mark.parametrize("name", list(E.posterior_components()))
def test_gibbs_chain_matches_exact_posterior(name):
    """R replicas of one component in one handle, each from an exact stationary draw of mu; 64 sweeps through the CUDA
    graph with stride 1 and a trace (slot = sweep number).  Per member the replica time-averages of log mu and of
    1{mu <= q} at the exact quartiles."""
    kind, spec = E.posterior_components()[name]
    R, S = 4000, 64
    post = E.posterior_of(kind, spec)
    row_ptr, col, k, w, l = E.posterior_problem(kind, spec, R)
    mu0 = post.sample_mu(np.random.default_rng(SEED), R).reshape(-1)
    with capi.Handle(row_ptr, col, k, l, alpha=E.POSTERIOR_ALPHA, beta=E.POSTERIOR_BETA, weight=w) as H:
        if k is None:                                                   # the by-length layout: k_alloc_seg4
            assert (np.diff(np.diff(row_ptr)) >= 0).all()
        elif kind == "rows":                                            # R G classes of one fragment: k_alloc_cls1
            _assert_routing(H.cls_stats(), R * spec["G"], 2, 1, "small")
        else:                                                           # singleton classes are in no piece
            _assert_routing(H.cls_stats(), R, spec["d"], spec["k"], _piece(spec["d"], spec["k"]))
        H.set_mu(mu0)
        H.gibbs(SEED, 0, S, stride=1, trace_len=S)
        trace = H.get_trace()
    z, where = E.posterior_z(post, trace, R)
    assert abs(z) <= E.Z_MAX, f"{name}: worst z = {z:.2f} ({where})"
