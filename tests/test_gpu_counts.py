"""Posterior fragment-count moments (mmq_count_moments_begin / mmq_get_count_moments) and EM expected counts
(mmq_expected_counts) on the GPU.

The accumulators are exact integers, so every check of them is exact: against Python-integer sums of the counts each
sweep returns (mmq_sweep_debug), against the CPU replay's counts, graph against plain launches, one GPU against two.
The posterior moments of a shared class are also checked against its exact stationary law (tests/exact_reference.py)."""
import threading

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from oracle import oracle as orc
from tests import exact_reference as E

pytestmark = pytest.mark.gpu

SEED = 4321


def _moments(H, which):
    """(S, sum, sumsq) with sum and sumsq as Python integers (object arrays)."""
    S, s, lo, hi = H.count_moments(which)
    sq = np.array([(int(h) << 64) | int(l) for l, h in zip(lo, hi)], dtype=object)
    return S, s.astype(object), sq


def _host_moments(C):
    """C (S, rows) per-sweep counts: exact sum and sum of squares per row."""
    C = np.asarray(C, np.int64).astype(object)
    return C.sum(axis=0), (C * C).sum(axis=0)


def _groups(n, seed, n_ident=None, n_gene=None):
    """Random identical sets (about a third of the transcripts in none) and genes (every transcript in one)."""
    rng = np.random.default_rng(seed)
    n_ident = n_ident or max(1, n // 7)
    n_gene = n_gene or max(1, n // 3)
    ident = rng.integers(0, n_ident, n).astype(np.int32)
    ident[rng.random(n) < 0.35] = -1
    gene = rng.integers(0, n_gene, n).astype(np.int32)
    return ident, n_ident, gene, n_gene


def _group_counts(C, of, ng):
    """Per-sweep group counts from per-sweep transcript counts C (S, n)."""
    G = np.zeros((C.shape[0], ng), np.int64)
    sel = of >= 0
    for s in range(C.shape[0]):
        np.add.at(G[s], of[sel], np.asarray(C[s], np.int64)[sel])
    return G


def _check_against_sweeps(H, C, ident, ni, gene, ng, N=None):
    """Accumulators of H equal the exact sums of the per-sweep counts C (S, n) and of their group sums."""
    S = C.shape[0]
    s0, sq0 = _host_moments(C)
    got = _moments(H, 0)
    assert got[0] == S and np.array_equal(got[1], s0) and np.array_equal(got[2], sq0)
    for which, of, cnt in ((1, ident, ni), (2, gene, ng)):
        Cg = _group_counts(C, of, cnt)
        gs, gsq = _host_moments(Cg)
        S_, s, sq = _moments(H, which)
        assert S_ == S and np.array_equal(s, gs) and np.array_equal(sq, gsq), which
        member_sum = np.zeros(cnt, np.int64)
        np.add.at(member_sum, of[of >= 0], got[1][of >= 0].astype(np.int64))
        assert np.array_equal(s.astype(np.int64), member_sum), which                     # a group's sum is its members' sum
    if N is not None:
        assert int(got[1].sum()) == N * S                               # every fragment is counted every sweep
    return got


def _debug_sweeps(H, S, flags, first=100):
    out = []
    for s in range(S):
        _, c, _ = H.sweep_debug(SEED, first + s, flags, want_x=False)
        out.append(c)
    return np.stack(out)


# ------------------------------------------------------------------ every allocation path against its own counts

CLASS_CASES = {"cls1": (3, 1), "lo": (5, 32), "hi": (12, 33), "chain": (7, E.cat_limit(7) + 1), "general": (65, 300)}


@pytest.mark.parametrize("flags", [capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_TRANSPOSED], ids=["plan", "transposed"])
@pytest.mark.parametrize("piece", list(CLASS_CASES))
def test_class_plan_pieces_accumulate_exact_counts(piece, flags):
    """Replicas of one class reaching one piece of the class plan (or the transposed kernel), plus singleton classes
    for every other transcript of a replica: the accumulators equal the sums of the counts mmq_sweep_debug returns."""
    d, k = CLASS_CASES[piece]
    R = 512
    row_ptr, col, kk, mu = E.replicated_class(R, d, k, E.mu_pattern(d, "spread"))
    single = np.arange(0, R * d, 2, dtype=np.int32)                     # singleton classes of 3 fragments
    row_ptr = np.concatenate([row_ptr, row_ptr[-1] + np.arange(1, len(single) + 1)])
    col = np.concatenate([col, single]); kk = np.concatenate([kk, np.full(len(single), 3, np.int32)])
    n = R * d
    ident, ni, gene, ng = _groups(n, d)
    with capi.Handle(row_ptr, col, kk, np.ones(n)) as H:
        if flags == capi.MMQ_GIBBS_DEFAULT:
            assert H.cls_stats()["in_use"] == 1
        H.set_mu(mu)
        H.count_moments_begin(ident, ni, gene, ng)
        C = _debug_sweeps(H, 6, flags)
        _check_against_sweeps(H, C, ident, ni, gene, ng, N=int(kk.sum()))


@pytest.mark.parametrize("flags", [capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_RAGGED_KERNEL, capi.MMQ_GIBBS_GENERIC_KERNEL],
                         ids=["segment", "ragged", "generic"])
@pytest.mark.parametrize("weighted", [False, True])
def test_per_fragment_shards_accumulate_exact_counts(weighted, flags):
    """Per-fragment shards (one row per fragment, the by-length layout), with and without per-hit weights, through the
    segment, ragged and generic kernels: singleton rows enter the counts through the singleton base."""
    s = synth.Synth(20260101 + 7, 300, 20000, weights=weighted)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w if weighted else None,
                             layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
    ident, ni, gene, ng = _groups(h.n, 11)
    with capi.Handle(h.row_ptr, h.col, None, h.len, weight=h.w, class_id_base=3) as H:
        H.init_mu()
        H.count_moments_begin(ident, ni, gene, ng)
        C = _debug_sweeps(H, 6, flags)
        _check_against_sweeps(H, C, ident, ni, gene, ng, N=h.m)


def test_accumulators_match_the_cpu_replay():
    """The sums formed from the CPU replay's per-sweep counts (not the GPU's) equal the accumulators."""
    s = synth.Synth(20260101, 200, 5000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    P = orc.Problem(h.row_ptr, h.col, h.k, h.len)
    mu, _, _ = P.init_mu()
    ident, ni, gene, ng = _groups(h.n, 3)
    C = []
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.set_mu(mu)
        H.count_moments_begin(ident, ni, gene, ng)
        for sweep in range(8):
            _, c_o, mu = P.sweep_replay(mu, SEED, sweep)
            C.append(c_o)
            H.sweep_debug(SEED, sweep, capi.MMQ_GIBBS_DEFAULT, want_x=False)
        _check_against_sweeps(H, np.stack(C), ident, ni, gene, ng, N=int(h.k.sum()))


# ------------------------------------------------------------------ CUDA graph, restart, the 128-bit carry

def test_graph_equals_plain_launches_and_restart():
    """64 sweeps from sweep 5 (replays start off a multiple of 16) through the CUDA graph equal plain launches and the
    sums of the per-sweep counts; begin restarts from zero, end frees the accumulators and turns accumulation off."""
    s = synth.Synth(20260101 + 2, 400, 30000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    ident, ni, gene, ng = _groups(h.n, 5)
    res = {}
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.init_mu()
        mu0 = H.get_mu()
        H.gibbs(SEED, 0, 32, stride=4, trace_len=8)                     # a graph captured without accumulation ...
        for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_NO_GRAPH):
            H.set_mu(mu0)
            H.count_moments_begin(ident, ni, gene, ng)                  # ... is not replayed with it
            H.gibbs(SEED, 5, 64, stride=4, trace_len=32, flags=flags)
            res[flags] = [_moments(H, w) for w in range(3)] + [H.get_trace()]
        H.count_moments_end()
        H.set_mu(mu0)
        bytes0 = H.device_bytes()
        H.count_moments_begin(ident, ni, gene, ng)
        C = _debug_sweeps(H, 64, capi.MMQ_GIBBS_DEFAULT, first=5)
        _check_against_sweeps(H, C, ident, ni, gene, ng, N=int(h.k.sum()))
        H.count_moments_end()
        assert H.device_bytes() == bytes0
        with pytest.raises(capi.MmqError, match="mmq_count_moments_begin first"):
            H.count_moments(0)
        H.set_mu(mu0)
        H.gibbs(SEED, 5, 64, stride=4, trace_len=32)                    # without accumulation: the same chain
        tr_off = H.get_trace()
    g, p = res[capi.MMQ_GIBBS_DEFAULT], res[capi.MMQ_GIBBS_NO_GRAPH]
    for w in range(3):
        assert g[w][0] == p[w][0] == 64 and np.array_equal(g[w][1], p[w][1]) and np.array_equal(g[w][2], p[w][2]), w
    assert np.array_equal(g[0][1], _host_moments(C)[0]) and np.array_equal(g[0][2], _host_moments(C)[1])
    assert np.array_equal(g[3], p[3]) and np.array_equal(g[3], tr_off)


def test_sum_of_squares_carries_into_the_high_word():
    """Singleton classes of 2^30 and of 7 fragments, 17 sweeps: sum c^2 = 17 * 2^60 passes 2^64.  Transcripts whose
    classes are all singletons have mean sum k and sd 0; their gene gets (2^30 + 7)^2 per sweep."""
    K = 1 << 30
    S = 17
    with capi.Handle([0, 1, 2], [0, 1], [K, 7], np.array([1.0, 2.0])) as H:
        H.set_mu(np.ones(2))
        H.count_moments_begin(None, 0, np.zeros(2, np.int32), 1)
        H.gibbs(SEED, 3, S, stride=1, trace_len=0)                      # one graph of 16 sweeps + one plain launch
        St, s, lo, hi = H.count_moments(0)
        Sg, gs, glo, ghi = H.count_moments(2)
    assert St == Sg == S
    assert [int(x) for x in s] == [S * K, S * 7]
    assert int(hi[0]) == (S * K * K) >> 64 == 1 and int(lo[0]) == (S * K * K) & (2 ** 64 - 1)
    assert int(hi[1]) == 0 and int(lo[1]) == S * 49
    assert int(gs[0]) == S * (K + 7) and (int(ghi[0]) << 64 | int(glo[0])) == S * (K + 7) ** 2
    for i in range(2):   # sd 0: S sumsq == sum^2 exactly
        assert S * ((int(hi[i]) << 64) | int(lo[i])) == int(s[i]) ** 2


def test_gene_sd_is_not_derived_from_its_isoforms():
    """Two isoforms sharing one class of 1000 fragments: each isoform's count varies, the gene's is 1000 every sweep
    (sd 0), so the gene's sum of squares is far from the sum of its isoforms'."""
    R, k, S = 256, 1000, 16
    row_ptr, col, kk, mu = E.replicated_class(R, 2, k, np.ones(2))
    gene = np.repeat(np.arange(R, dtype=np.int32), 2)
    with capi.Handle(row_ptr, col, kk, np.ones(2 * R)) as H:
        H.set_mu(mu)
        H.count_moments_begin(None, 0, gene, R)
        H.gibbs(SEED, 0, S, stride=1, trace_len=0)
        St, s, sq = _moments(H, 0)
        Sg, gs, gsq = _moments(H, 2)
    assert Sg == S and all(int(x) == S * k for x in gs) and all(int(x) == S * k * k for x in gsq)
    diff = np.array([int(g) - int(m) for g, m in zip(gsq, sq[0::2] + sq[1::2])], dtype=np.float64)   # 2 sum_s c0 c1
    assert (diff > 0).all() and diff.mean() > S * k * k / 4
    sd_t = np.sqrt([(S * int(q) - int(x) ** 2) / (S * (S - 1)) for x, q in zip(s, sq)])
    assert sd_t.mean() > 5.0


# ------------------------------------------------------------------ against the exact posterior

@pytest.mark.parametrize("name", [nm for nm, (kind, _) in E.posterior_components().items() if kind == "class"])
def test_count_moments_match_exact_posterior(name):
    """R replicas of a shared-class component from exact stationary draws, 64 sweeps through the CUDA graph: per member
    the replicas' time-averages of c = u_j + x_j and of (c - E c)^2 against the exact mean and variance."""
    kind, spec = E.posterior_components()[name]
    R, S = 4000, 64
    post = E.posterior_of(kind, spec)
    row_ptr, col, k, w, l = E.posterior_problem(kind, spec, R)
    mu0 = post.sample_mu(np.random.default_rng(SEED), R).reshape(-1)
    with capi.Handle(row_ptr, col, k, l, alpha=E.POSTERIOR_ALPHA, beta=E.POSTERIOR_BETA, weight=w) as H:
        H.set_mu(mu0)
        H.count_moments_begin()
        H.gibbs(SEED, 0, S, stride=1, trace_len=0)
        St, s, sq = _moments(H, 0)
    assert St == S
    d = post.d
    s = np.array([float(x) for x in s]).reshape(R, d)
    sq = np.array([float(x) for x in sq]).reshape(R, d)
    worst = (0.0, "none")
    for j in range(d):
        pmf = post.pmf(j)
        x = np.arange(len(pmf))
        mean = post.u[j] + pmf @ x
        var = pmf @ (x - (mean - post.u[j])) ** 2
        m_r = s[:, j] / S
        v_r = sq[:, j] / S - 2.0 * mean * m_r + mean * mean                # time-average of (c - E c)^2
        for z, what in ((E.replica_mean_z(m_r[:, None], mean)[0], "mean"), (E.replica_mean_z(v_r[:, None], var)[0], "variance")):
            if abs(z) > abs(worst[0]):
                worst = (float(z), f"{what} of member {j}")
    assert abs(worst[0]) <= E.Z_MAX, f"{name}: worst z = {worst[0]:.2f} ({worst[1]})"


# ------------------------------------------------------------------ EM expected counts

def _numpy_estep(row_ptr, col, k, w, mu):
    d = np.diff(row_ptr)
    row = np.repeat(np.arange(len(d)), d)
    p = mu[col] * (1.0 if w is None else w.astype(np.float64))
    D = np.bincount(row, weights=p, minlength=len(d))
    kk = np.ones(len(d)) if k is None else k.astype(np.float64)
    return np.bincount(col, weights=kk[row] * p / D[row], minlength=len(mu))


@pytest.mark.parametrize("weighted", [False, True])
def test_expected_counts_are_one_e_step(weighted):
    s = synth.Synth(20260101 + 3, 300, 20000, weights=weighted)
    if weighted:
        h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
        k, N = None, h.m
    else:
        h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
        k, N = h.k, int(h.k.sum())
    mu = np.random.default_rng(1).gamma(0.5, 50.0, h.n) + 1e-3
    with capi.Handle(h.row_ptr, h.col, k, h.len, weight=h.w) as H:
        H.set_mu(mu)
        e = H.expected_counts()
        assert np.array_equal(H.get_mu(), mu)
    want = _numpy_estep(h.row_ptr, h.col, k, h.w, mu)
    assert np.max(np.abs(e - want) / np.maximum(want, 1e-300)) <= 1e-12
    assert abs(e.sum() / N - 1.0) <= 1e-9


# ------------------------------------------------------------------ several GPUs

def _need_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


def _on_threads(fn, n):
    out, err = [None] * n, []

    def run(r):
        try:
            out[r] = fn(r)
        except Exception as e:          # re-raised on the test's thread
            err.append(e)
    th = [threading.Thread(target=run, args=(r,)) for r in range(n)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if err:
        raise err[0]
    return out


def _collapsed_sample():
    s = synth.Synth(20260101 + 1, 300, 20000)
    return hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)


def test_two_ranks_over_nccl_match_one_gpu():
    """Two shards with NCCL communicators (one thread per GPU): every rank accumulates the all-reduced counts, bit for
    bit what one GPU accumulates from the same mu; EM expected counts within EM's tolerance."""
    _need_two_gpus()
    h = _collapsed_sample()
    ident, ni, gene, ng = _groups(h.n, 9)
    cut = [0, h.m // 3, h.m]
    mu0 = np.random.default_rng(2).gamma(0.5, 50.0, h.n) + 1e-3
    hs = []
    for r in range(2):
        a, b = cut[r], cut[r + 1]
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        hs.append(capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], h.k[a:b], h.len, class_id_base=a, device=r))
    uid = capi.comm_id()
    _on_threads(lambda r: hs[r].comm_init(uid, r, 2), 2)

    def run(r):
        H = hs[r]
        H.set_mu(mu0)
        e = H.expected_counts()
        H.count_moments_begin(ident, ni, gene, ng)
        H.gibbs(SEED, 0, 40, stride=4, trace_len=10)
        return e, [_moments(H, w) for w in range(3)]
    out = _on_threads(run, 2)
    for H in hs:
        H.close()
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.set_mu(mu0)
        e1 = H.expected_counts()
        H.count_moments_begin(ident, ni, gene, ng)
        H.gibbs(SEED, 0, 40, stride=4, trace_len=10)
        one = [_moments(H, w) for w in range(3)]
    for e, mom in out:
        assert np.max(np.abs(e / e1 - 1.0)) <= 1e-9
        for w in range(3):
            assert mom[w][0] == one[w][0] == 40 and np.array_equal(mom[w][1], one[w][1]) and np.array_equal(mom[w][2], one[w][2]), w


@pytest.mark.parametrize("weighted", [False, True])
def test_peer_attached_shards_match_one_gpu(weighted):
    """Two handles with mmq_p2p_attach_local (the fused peer-memory Gamma kernel), per-fragment shards cut in two, with
    and without weights: the same accumulators as one GPU, bit for bit.  Under the reduce-scatter exchange (mmq_tune
    knob 6) mmq_gibbs refuses to accumulate."""
    _need_two_gpus()
    s = synth.Synth(20260101 + 4, 300, 20000, weights=weighted)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w if weighted else None,
                             layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    ident, ni, gene, ng = _groups(h.n, 13)
    cut = [0, (h.m // 2) & ~1, h.m]
    mu0 = np.random.default_rng(0).gamma(0.5, 50.0, h.n)
    hs = []
    for r in range(2):
        a, b = cut[r], cut[r + 1]
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        hs.append(capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], None, h.len, weight=None if h.w is None else h.w[lo:hi],
                              class_id_base=a, device=r))
    capi.p2p_attach_local(hs)

    def run(r):
        H = hs[r]
        H.set_mu(mu0)
        H.count_moments_begin(ident, ni, gene, ng)
        H.gibbs(SEED, 0, 40, stride=4, trace_len=10)
        H.sweep_debug(SEED, 40, capi.MMQ_GIBBS_DEFAULT, want_x=False)
        return [_moments(H, w) for w in range(3)]
    out = _on_threads(run, 2)
    for H in hs:
        H.tune(6, 1)
    errs = _on_threads(lambda r: _refused(hs[r]), 2)
    for H in hs:
        H.close()
    assert all("knob 6" in e for e in errs), errs
    with capi.Handle(h.row_ptr, h.col, None, h.len, weight=h.w) as H:
        H.set_mu(mu0)
        H.count_moments_begin(ident, ni, gene, ng)
        H.gibbs(SEED, 0, 40, stride=4, trace_len=10)
        H.sweep_debug(SEED, 40, capi.MMQ_GIBBS_DEFAULT, want_x=False)
        one = [_moments(H, w) for w in range(3)]
    for mom in out:
        for w in range(3):
            assert mom[w][0] == one[w][0] == 41 and np.array_equal(mom[w][1], one[w][1]) and np.array_equal(mom[w][2], one[w][2]), w


def _refused(H):
    with pytest.raises(capi.MmqError) as e:
        H.gibbs(SEED, 41, 20, stride=4, trace_len=10)
    return str(e.value)
