"""Parity of the CUDA path (through the C ABI) against the CPU oracle.
  (a) allocations X, counts and the Gamma draws: BIT-EXACT with the shared Philox stream
  (b) EM: relative 1e-6 (north_star), same iteration count
  (c) posterior mean / sd of log mu vs the GSL-style reference-like chain: within Monte-Carlo error
"""
import numpy as np
import pytest

from mmseq_b200 import capi, hostlib
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

SEED = 1234


def _handle(h, **kw):
    return capi.Handle(h.row_ptr, h.col, h.k, h.len, weight=h.w, **kw)


def _oracle(h, **kw):
    return orc.Problem(h.row_ptr, h.col, h.k, h.len, weight=h.w, **kw)


def test_init_mu_and_unique_hits(small_problem):
    h = small_problem
    mu_o, uh_o, _ = _oracle(h).init_mu()
    with _handle(h) as H:
        uh = H.init_mu()
        mu = H.get_mu()
    assert np.array_equal(uh, uh_o)
    assert np.allclose(mu, mu_o, rtol=1e-12)


def test_loglik_and_em_match_oracle(small_problem):
    h = small_problem
    P = _oracle(h)
    mu0, _, _ = P.init_mu()
    mu_o, it_o, ll_o, llr_o = P.em(mu0, 1000, 0.1)
    with _handle(h) as H:
        H.init_mu()
        assert np.isclose(H.loglik(), P.loglik(mu0), rtol=1e-12)
        it, ll, llr = H.em(1000, 0.1)
        mu = H.get_mu()
    assert it == it_o
    assert np.max(np.abs(mu / mu_o - 1)) <= 1e-6          # north_star (b)
    assert np.isclose(ll, ll_o, rtol=1e-10) and abs(llr - llr_o) < 1e-6 * abs(ll_o)
    assert np.isclose((mu * h.len).sum(), h.N, rtol=1e-10)  # EM mass conservation


@pytest.mark.parametrize("layout", ["collapsed", "per_fragment"])
def test_sweep_bit_exact_vs_cpu_replay(small_problem, small_problem_pf, layout):
    h = small_problem if layout == "collapsed" else small_problem_pf
    P = _oracle(h)
    mu, _, _ = P.init_mu()
    with _handle(h) as H:
        H.set_mu(mu)
        for sweep in range(4):
            x_o, c_o, mu_o = P.sweep_replay(mu, SEED, sweep)
            x, c, mu_g = H.sweep_debug(SEED, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o), f"X differs at sweep {sweep}"
            assert np.array_equal(c, c_o)
            assert c.sum() == h.N                                   # per-sweep conservation
            kk = h.k if h.k is not None else np.ones(h.m, np.int32)
            assert np.array_equal(np.add.reduceat(x, h.row_ptr[:-1]), kk)   # per-class conservation
            assert np.array_equal(mu_g, mu_o), "Gamma draws not bit-exact"
            mu = mu_o
        # the fused (reduction) path produces the same integers and the same chain
        H.set_mu(mu)
        _, c_f, mu_f = H.sweep_debug(SEED, 4, capi.MMQ_GIBBS_DEFAULT)
        _, c_o, mu_o = P.sweep_replay(mu, SEED, 4)
        assert np.array_equal(c_f, c_o) and np.array_equal(mu_f, mu_o)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("cid_base", [0, 7])
def test_categorical_fast_path_edges(weighted, cid_base):
    """k == 1 kernel: ragged tail (m % 64 != 0), rows longer than the warp slab, singletons,
    class-id base that is not a multiple of 4 (Philox quads straddle lanes), zero and tiny mu — against the CPU replay and
    against the general kernel."""
    rng = np.random.default_rng(5)
    n = 4000
    lens = np.concatenate([rng.integers(1, 9, 700), [1, 1, 900, 2, 1500, 3], rng.integers(1, 40, 331)])
    rows = [np.sort(rng.choice(n, size=int(d), replace=False)) for d in lens]
    row_ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate(rows).astype(np.int32)
    assert (len(lens) % 64) != 0
    w = np.exp(0.5 * rng.standard_normal(len(col))).astype(np.float32) if weighted else None
    l = rng.uniform(1e-6, 1e-2, n)
    mu = rng.gamma(0.3, 100.0, n)
    mu[:40] = 1e-300
    mu[40:60] = 0.0
    P = orc.Problem(row_ptr, col, None, l, weight=w)
    with capi.Handle(row_ptr, col, None, l, weight=w, class_id_base=cid_base) as H:
        for sweep in range(3):
            _, c_o, mu_o = P.sweep_replay(mu, 77, sweep, class_id_base=cid_base)
            assert c_o.sum() == len(lens)
            for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_GENERIC_KERNEL, capi.MMQ_GIBBS_TRANSPOSED):
                H.set_mu(mu)
                _, c, mu_g = H.sweep_debug(77, sweep, flags, want_x=False)
                assert np.array_equal(c, c_o), (sweep, flags)
                assert np.array_equal(mu_g, mu_o)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("cid_base", [0, 5, 2, 7])
def test_by_length_layout_kernels_match_replay(small_synth, weighted, cid_base):
    """The loader's by-length layout: runs of equal class size, singletons skipped, no row
    pointers read — same integers and the same chain as the CPU replay and as the other kernels."""
    s = small_synth
    w = None
    if weighted:
        w = np.exp(0.5 * np.random.default_rng(8).standard_normal(len(s.frag_tid))).astype(np.float32)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=w, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
    d = np.diff(h.row_ptr)
    assert (np.diff(d) >= 0).all() and d[0] == 1 and d.max() > 8          # singletons first, long rows last
    P = orc.Problem(h.row_ptr, h.col, None, h.len, weight=h.w)
    mu, _, _ = P.init_mu()
    with capi.Handle(h.row_ptr, h.col, None, h.len, weight=h.w, class_id_base=cid_base) as H:
        for sweep in range(3):
            _, c_o, mu_o = P.sweep_replay(mu, SEED, sweep, class_id_base=cid_base)
            for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_RAGGED_KERNEL, capi.MMQ_GIBBS_GENERIC_KERNEL, capi.MMQ_GIBBS_TRANSPOSED,
                          capi.MMQ_GIBBS_DEFAULT):
                H.set_mu(mu)
                _, c, mu_g = H.sweep_debug(SEED, sweep, flags, want_x=False)
                assert np.array_equal(c, c_o), (sweep, flags)
                assert c.sum() == h.m and np.array_equal(mu_g, mu_o)
            mu = mu_o
        # a multi-sweep run on the default (segment) path reproduces the replayed chain
        H.set_mu(mu)
        H.gibbs(SEED, 3, 29, stride=4, trace_len=8)
        mu_end, tr_o = P.gibbs_replay(mu, SEED, 3, 29, 4, 8) if cid_base == 0 else (None, None)
        if cid_base == 0:
            assert np.array_equal(H.get_mu(), mu_end) and np.array_equal(H.get_trace()[:, 1:], tr_o[:, 1:])


def test_zero_weights_never_chosen(small_synth):
    """Weights of exactly 0 are legal (a hit that cannot have produced the fragment): such a member is never chosen, by
    the segment kernel (the default for this layout) and by every other kernel."""
    s = small_synth
    rng = np.random.default_rng(12)
    w = np.exp(0.5 * rng.standard_normal(len(s.frag_tid))).astype(np.float32)
    w[rng.random(len(w)) < 0.2] = 0.0
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=w, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
    P = orc.Problem(h.row_ptr, h.col, None, h.len, weight=h.w)
    mu = np.random.default_rng(1).gamma(0.5, 10.0, h.n)
    with capi.Handle(h.row_ptr, h.col, None, h.len, weight=h.w) as H:
        for sweep in range(2):
            _, c_o, mu_o = P.sweep_replay(mu, SEED, sweep)
            for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_RAGGED_KERNEL, capi.MMQ_GIBBS_GENERIC_KERNEL, capi.MMQ_GIBBS_TRANSPOSED):
                H.set_mu(mu)
                _, c, mu_g = H.sweep_debug(SEED, sweep, flags, want_x=False)
                assert np.array_equal(c, c_o) and np.array_equal(mu_g, mu_o), (sweep, flags)


def test_weighted_rows_bit_exact(small_synth):
    s = small_synth
    rng = np.random.default_rng(3)
    w = np.exp(0.5 * rng.standard_normal(len(s.frag_tid))).astype(np.float32)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=w, layout=hostlib.LAYOUT_PER_FRAGMENT)
    assert h.w is not None
    P = _oracle(h)
    mu, _, _ = P.init_mu()
    with _handle(h) as H:
        H.set_mu(mu)
        for sweep in range(2):
            x_o, c_o, mu_o = P.sweep_replay(mu, SEED, sweep)
            x, c, mu_g = H.sweep_debug(SEED, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o) and np.array_equal(c, c_o) and np.array_equal(mu_g, mu_o)
            mu = mu_o
        mu_o2, it_o, ll_o, _ = P.em(P.init_mu()[0], 50, 0.1)
        H.init_mu()
        it, ll, _ = H.em(50, 0.1)
        assert it == it_o and np.max(np.abs(H.get_mu() / mu_o2 - 1)) <= 1e-6


def test_trace_bit_exact_over_many_sweeps(small_problem):
    h = small_problem
    P = _oracle(h)
    mu0, _, _ = P.init_mu()
    mu_o, tr_o = P.gibbs_replay(mu0, SEED, 0, 64, 4, 16)
    for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_TRANSPOSED):
        with _handle(h) as H:
            H.set_mu(mu0)
            H.gibbs(SEED, 0, 40, stride=4, trace_len=16, flags=flags)
            H.gibbs(SEED, 40, 24, stride=4, trace_len=16, flags=flags)   # restartable from (seed, sweep)
            tr = H.get_trace()
            assert np.array_equal(tr, tr_o)
            assert np.array_equal(H.get_mu(), mu_o)


@pytest.mark.parametrize("layout", ["collapsed", "by_length"])
def test_cuda_graph_replay_equals_plain_launches(small_synth, layout):
    """Long runs are replayed from one CUDA graph of 16 sweeps whose sweep counter lives on the
    device; the chain must equal the plain-launch chain and the CPU replay, also when the run is
    split into unaligned pieces and when the stride does not divide the graph length."""
    s = small_synth
    lay = hostlib.LAYOUT_COLLAPSED if layout == "collapsed" else hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=lay)
    P = _oracle(h)
    mu0, _, _ = P.init_mu()
    n_sw, stride, L = 150, 6, 32
    mu_o, tr_o = P.gibbs_replay(mu0, SEED, 0, n_sw, stride, L)
    with _handle(h) as H:
        H.set_mu(mu0)
        H.gibbs(SEED, 0, n_sw, stride=stride, trace_len=L, flags=capi.MMQ_GIBBS_NO_GRAPH)
        tr_plain, mu_plain = H.get_trace(), H.get_mu()
        H.set_mu(mu0)
        l0 = capi.launch_count()
        H.gibbs(SEED, 0, 100, stride=stride, trace_len=L)            # graph: 1 + 6*16 + 3
        H.gibbs(SEED, 100, 50, stride=stride, trace_len=L)           # graph reused: 1 + 3*16 + 1
        tr_g, mu_g = H.get_trace(), H.get_mu()
        assert capi.launch_count() - l0 >= 2 * n_sw
    assert np.array_equal(tr_plain, tr_o) and np.array_equal(mu_plain, mu_o)
    assert np.array_equal(tr_g, tr_o) and np.array_equal(mu_g, mu_o)


def test_ragged_and_extreme_rows():
    """Singletons, a row longer than the staging tile, huge k, tiny mu."""
    rng = np.random.default_rng(11)
    n = 5000
    rows = [[0], [1], [0, 1], list(range(2, 2 + 3000)), [7, 9], [4999]]
    rows += [sorted(rng.choice(n, size=int(d), replace=False).tolist()) for d in rng.integers(1, 40, 300)]
    k = [2_000_000_000 // 4, 1, 123456, 777, 1, 5] + rng.integers(1, 5000, 300).tolist()
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    col = np.concatenate(rows).astype(np.int32)
    l = rng.uniform(1e-6, 1e-2, n)
    mu = rng.gamma(0.3, 100.0, n)
    mu[:50] = 1e-300
    mu[2] = 0.0                                # an exact zero inside a long row
    P = orc.Problem(row_ptr, col, k, l)
    with capi.Handle(row_ptr, col, k, l) as H:
        for sweep in (0, 1, 2):
            H.set_mu(mu)
            x_o, c_o, mu_o = P.sweep_replay(mu, 99, sweep)
            x, c, mu_g = H.sweep_debug(99, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o) and np.array_equal(c, c_o) and np.array_equal(mu_g, mu_o)
            H.set_mu(mu)
            _, c_f, _ = H.sweep_debug(99, sweep, capi.MMQ_GIBBS_DEFAULT)
            assert np.array_equal(c_f, c_o)


@pytest.mark.parametrize("plan_threads", ["1", "5", "device"])
@pytest.mark.parametrize("cid_base", [0, (1 << 32) * 5 + 3])
def test_class_plan_kernel_bit_exact(monkeypatch, cid_base, plan_threads):
    """Collapsed shards (mmq_cls.cu): every regime of the plan against the CPU replay — k = 0, 1,
    2..64 (categorical draws, four per Philox block; block boundaries and the full 64-draw slot),
    k > 64 (conditional-binomial chains, one class per lane of k_alloc_chain, BINV and BTRS regimes), class sizes 1,
    2..8 and 9..16 (the two register instances), 17..64 (generic), > 64 (general kernel), all-zero and partly-zero mu
    rows, class ids above 2^32, chunks that end inside a warp; the plan built by one host thread and
    by several (MMQ_PLAN_THREADS)."""
    if plan_threads == "device":   # the default: the plan is built on the device (mmq_cls.cu: cls_plan_device)
        monkeypatch.delenv("MMQ_CLS_HOST_PLAN", raising=False)
    else:                          # the host builder of mmq_cls_plan.h (what the CPU tests replay)
        monkeypatch.setenv("MMQ_CLS_HOST_PLAN", "1")
        monkeypatch.setenv("MMQ_PLAN_THREADS", plan_threads)
    rng = np.random.default_rng(5)
    n = 4000
    sizes = np.concatenate([rng.integers(1, 17, 5000), rng.integers(17, 65, 300), rng.integers(65, 200, 20), [2] * 37, [16] * 33])
    rows = [np.sort(rng.choice(n, size=int(d), replace=False)) for d in sizes]
    rows[10] = np.array([0, 1, 2]); rows[11] = np.array([0, 1]); rows[12] = np.array([1, 2, 3, 5])
    m = len(rows)
    k = np.where(rng.random(m) < 0.5, 1, rng.integers(0, 70, m))
    big = rng.random(m) < 0.05
    k[big] = rng.integers(65, 100000, big.sum())
    k[:64] = np.arange(64) + 1                       # every k of the small set at least once
    k[100:120] = [4, 5, 8, 61, 62, 63, 64, 65, 66, 127, 128, 129, 512, 1000, 1024, 1025, 8191, 8192, 8193, 8194]
    k = k.astype(np.int32)
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate(rows).astype(np.int32)
    l = rng.uniform(1e-6, 1e-2, n)
    mu = rng.gamma(0.3, 100.0, n)
    mu[0:3] = 0.0                                    # rows 10, 11: all-zero; row 12: zeros in front
    mu[3990:] = 1e-300
    P = orc.Problem(row_ptr, col, k, l)
    with capi.Handle(row_ptr, col, k, l, class_id_base=cid_base) as H:
        st = H.cls_stats()
        assert st["in_use"] == 1 and st["small_classes"] > 4000 and st["rest_classes"] >= 20 and st["chain_classes"] > 150
        assert st["class_slots"] >= st["small_classes"] and st["chain_slots"] % 32 == 0
        for sweep in (0, 1, 7):
            H.set_mu(mu)
            x_o, c_o, mu_o = P.sweep_replay(mu, 4321, sweep, class_id_base=cid_base)
            _, c_f, mu_f = H.sweep_debug(4321, sweep, capi.MMQ_GIBBS_DEFAULT)
            assert np.array_equal(c_f, c_o) and np.array_equal(mu_f, mu_o)
            assert c_f.sum() == k.sum()
            H.set_mu(mu)                             # the X-materialising path follows the same contract
            x, c, _ = H.sweep_debug(4321, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o) and np.array_equal(c, c_o)
            H.set_mu(mu)                             # and so does the general kernel on the whole shard
            _, c_g, _ = H.sweep_debug(4321, sweep, capi.MMQ_GIBBS_GENERIC_KERNEL)
            assert np.array_equal(c_g, c_o)
        # a chain that alternates the three paths stays on the replay's trajectory (counts[] restarts
        # from the singleton base or from zero as each kernel expects)
        H.set_mu(mu)
        mu_c = mu
        for sweep, flags in enumerate([capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_GENERIC_KERNEL, capi.MMQ_GIBBS_DEFAULT,
                                       capi.MMQ_GIBBS_TRANSPOSED, capi.MMQ_GIBBS_DEFAULT]):
            _, c_o, mu_c = P.sweep_replay(mu_c, 4321, sweep, class_id_base=cid_base)
            _, c_x, mu_x = H.sweep_debug(4321, sweep, flags)
            assert np.array_equal(c_x, c_o) and np.array_equal(mu_x, mu_c)


def test_class_id_base_shards_reproduce_the_whole(small_problem):
    """Two shards on one GPU (handles are independent): summed counts == unsharded counts."""
    h = small_problem
    P = _oracle(h)
    mu, _, _ = P.init_mu()
    _, c_o, _ = P.sweep_replay(mu, SEED, 3)
    cut = h.m // 3
    parts = []
    for a, b in ((0, cut), (cut, h.m)):
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        with capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], h.k[a:b], h.len, class_id_base=a) as H:
            H.set_mu(mu)
            parts.append(H.sweep_debug(SEED, 3, capi.MMQ_GIBBS_DEFAULT)[1])
    assert np.array_equal(parts[0] + parts[1], c_o)


def test_explicit_class_ids_make_the_chain_order_independent(small_problem):
    """mmq_problem.class_id: classes handed over sorted by cost (what the host program does) give
    the counts and the chain of the canonical order, bit for bit."""
    h = small_problem
    P = _oracle(h)
    mu, _, _ = P.init_mu()
    rp, col, k, cid = hostlib.sort_classes_by_cost(h)
    assert not np.array_equal(cid, np.arange(h.m))
    with capi.Handle(rp, col, k, h.len, class_id=cid) as H:
        for sweep in range(3):
            x_o, c_o, mu_o = P.sweep_replay(mu, SEED, sweep)
            for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_TRANSPOSED):
                H.set_mu(mu)
                x, c, mu_g = H.sweep_debug(SEED, sweep, flags)
                assert np.array_equal(c, c_o) and np.array_equal(mu_g, mu_o)
                if x is not None:   # X comes back in the order the classes were handed over
                    d = np.diff(h.row_ptr)[cid]
                    starts = h.row_ptr[:-1][cid]
                    idx = np.repeat(starts - rp[:-1], d) + np.arange(int(rp[-1]))
                    assert np.array_equal(x, x_o[idx])
            mu = mu_o
        H.init_mu()
        it, ll, _ = H.em(1000, 0.1)
        mu_em, it_o, ll_o, _ = P.em(P.init_mu()[0], 1000, 0.1)
        assert it == it_o and np.max(np.abs(H.get_mu() / mu_em - 1)) <= 1e-6
    with pytest.raises(capi.MmqError):
        capi.Handle(rp, col, None, h.len, class_id=cid)      # k == 1 shards pair consecutive ids


def test_posterior_matches_reference_like_chain(small_problem):
    """north_star (c): log_mu within the stated Monte-Carlo standard error of the GSL-style
    MT19937 chain, and the sd of log mu no further from it than a second, independently
    seeded reference-like chain is."""
    h = small_problem
    P = _oracle(h)
    mu0, _, _ = P.init_mu()
    mu_em, _, _, _ = P.em(mu0, 1000, 0.1)
    L, stride = 1024, 4
    _, tr_a, _ = P.gibbs_gsl(mu_em, SEED, L * stride, stride, L, threads=1)
    _, tr_b, _ = P.gibbs_gsl(mu_em, SEED + 4321, L * stride, stride, L, threads=1)
    with _handle(h) as H:
        H.set_mu(mu_em)
        H.gibbs(SEED, 0, L * stride, stride=stride, trace_len=L)
        tr = H.get_trace()
    g = orc.summaries_transcripts(tr)
    a = orc.summaries_transcripts(tr_a)
    b = orc.summaries_transcripts(tr_b)

    def zfrac(x, y):
        z = np.abs(x["log_mu"] - y["log_mu"]) / np.sqrt(x["mcse"] ** 2 + y["mcse"] ** 2)
        return np.mean(z <= 4.0)

    def sd_spread(x, y):
        return np.mean(np.abs(np.log(x["sd"] / y["sd"])) < 0.5)

    assert zfrac(g, a) >= 0.99 and zfrac(g, b) >= 0.99
    assert zfrac(g, a) >= zfrac(b, a) - 0.01
    assert abs(np.median(g["sd"] / a["sd"]) - 1) < 0.05
    assert sd_spread(g, a) >= sd_spread(b, a) - 0.03


def test_errors_are_reported_not_fatal(small_problem):
    h = small_problem
    with _handle(h) as H:
        with pytest.raises(capi.MmqError):
            H.get_trace()                                          # no trace yet
        with pytest.raises(capi.MmqError):
            H.gibbs(SEED, 0, 4, stride=0, trace_len=8)
        with pytest.raises(capi.MmqError):
            H.tune(3, 1)                                           # not a knob
    with pytest.raises(capi.MmqError):
        capi.Handle(h.row_ptr, np.where(np.arange(h.nnz) == 5, h.n + 3, h.col), h.k, h.len)   # column out of range
    with pytest.raises(capi.MmqError):
        capi.Handle(h.row_ptr, h.col, h.k, np.where(np.arange(h.n) == 0, 0.0, h.len))          # zero length
