"""The sampler kernels at shapes where every worker of their capped grid takes two or more work items.

Each kernel's grid is capped at a fixed number of CTAs per SM, and a warp, CTA or CTA pair loops over chunks, tiles or
rows, carrying state from one item to the next (mbarrier phases, bulk copies issued one chunk ahead, per-warp queues).
The parity tests elsewhere run at shapes where each worker does one item; here the same oracles (the CPU replay, bit for
bit; the EM oracle, 1e-6) check the loops.  Each test computes the caps from the device's SM count and the launch code it
cites, and asserts its shape exceeds them by the intended factor."""
import functools

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

SEED = 1234
MMQ_SEG_MAX = 96       # mmq_seg.cu: more runs of equal class size than this and the handle uses the ragged kernel
MMQ_CLS_WARPS = 4      # mmq_cls_plan.h: warps per CTA of k_alloc_cls / k_alloc_cls1
MMQ_CHAIN_CLASSES = 128  # mmq_cls.cu: classes per block pass of k_alloc_chain
MMQ_ALLOC_WARPS = 8    # mmq_internal.h: warps per CTA of the general kernel k_alloc, one tile per warp pass
MMQ_ALLOC_CAP = 320    # mmq_internal.h: CSR entries of a tile at most
MMQ_GAMMA_THREADS = 256


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _member_rows(rng, d, pool):
    """One row per entry of d: d[i] distinct, ascending members of the sorted id array `pool` (a random start, then
    gaps of 1..16)."""
    gaps = rng.integers(1, 17, int(d.sum()))
    first = np.concatenate([[0], np.cumsum(d)[:-1]])
    gaps[first] = 0
    cs = np.cumsum(gaps)
    within = cs - np.repeat(cs[first], d)
    base = rng.integers(0, len(pool) - 16 * int(d.max()), len(d))
    return pool[np.repeat(base, d) + within]


def _take_rows(d, vals, sel):
    """The rows `sel` (with repeats) of the ragged array (row lengths d, flat vals)."""
    off = np.concatenate([[0], np.cumsum(d)])
    ds = d[sel]
    start = np.concatenate([[0], np.cumsum(ds)[:-1]])
    return ds, vals[np.repeat(off[sel] - start, ds) + np.arange(int(ds.sum()))]


# ------------------------------------------------------------------ per-fragment shard, by-length layout

@functools.lru_cache(maxsize=None)
def _pf_shard(weighted):
    """~1.5 M non-singleton fragments over 200k transcripts, plus singletons.  Class sizes 2..6 (register path of
    k_alloc_seg4), 7..12 (staged pairs) and 13..40 (unstaged, read from global memory).  Fragments draw their hits from
    a pool of member sets, several fragments in a row from the same set, so that rows with identical members are
    neighbours in the layout, inside and across chunk boundaries."""
    rng = np.random.default_rng(20260404)
    T = 200_000
    d_pool = np.concatenate([rng.integers(2, 7, 200_000), rng.integers(7, 13, 120_000), rng.integers(13, 41, 80_000)])
    pool = _member_rows(rng, d_pool, np.arange(T, dtype=np.int32))
    runs = rng.integers(0, len(d_pool), 600_000)
    sel = np.repeat(runs, rng.geometric(0.4, len(runs)))
    d_frag, tid = _take_rows(d_pool, pool, sel)
    n_single = 100_000
    d_frag = np.concatenate([d_frag, np.ones(n_single, np.int64)])
    tid = np.concatenate([tid, rng.integers(0, T, n_single).astype(np.int32)])
    frag_ptr = np.concatenate([[0], np.cumsum(d_frag)]).astype(np.int64)
    w = None
    if weighted:
        w = np.exp(0.5 * rng.standard_normal(len(tid))).astype(np.float32)
        w[rng.random(len(w)) < 0.1] = 0.0                       # a hit that cannot have produced the fragment
    efflen = rng.uniform(300.0, 5000.0, T)
    return hostlib.from_records(T, efflen, frag_ptr, tid, frag_w=w, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("cid_base", [0, 3])
def test_per_fragment_kernels_many_chunks_per_warp(weighted, cid_base):
    """k_alloc_seg4 (default), k_alloc_cat (RAGGED_KERNEL), the general kernel and the transposed kernel against the CPU
    replay, bit for bit, when every warp sweeps three or more chunks; a 32-sweep graph run against gibbs_replay."""
    h = _pf_shard(weighted)
    assert (h.w is not None) == weighted
    sms = _sms()
    d = np.diff(h.row_ptr)
    per_size = np.bincount(d)
    assert (np.diff(d) >= 0).all() and per_size[1] > 0 and d.max() == 40
    assert np.count_nonzero(per_size) <= MMQ_SEG_MAX                     # else the handle silently takes the ragged kernel
    rows = int(per_size[2:].sum())
    # k_alloc_seg4, mmq_seg.cu:526,532-533: min(chunks / 4, sms * MINB) CTAs of 4 warps, MINB = 4 with weights, 6
    # without; chunks of 128 rows of one run (counted without the <= 3 alignment rows a run may add in front)
    seg_chunks = int(sum(-(-int(c) // 128) for c in per_size[2:]))
    seg_warps = sms * (4 if weighted else 6) * 4
    assert seg_chunks >= 3 * seg_warps, (seg_chunks, seg_warps)
    assert rows >= 3 * seg_warps * 128
    # k_alloc_cat, mmq_core.cu:1536,1541: min(want, 3 sms) CTAs of 8 warps, 64 classes per warp chunk
    assert h.m / 64 >= 3 * (sms * 3 * 8)
    # general and transposed k_alloc, mmq_core.cu:1512: min(tiles / 8, 3 sms) CTAs of 8 warps, tiles of <= 320 entries
    assert h.nnz / MMQ_ALLOC_CAP >= 3 * (sms * 3 * MMQ_ALLOC_WARPS)
    P = orc.Problem(h.row_ptr, h.col, None, h.len, weight=h.w)
    mu = np.random.default_rng(1).gamma(0.5, 10.0, h.n)
    mu0 = mu
    with capi.Handle(h.row_ptr, h.col, None, h.len, weight=h.w, class_id_base=cid_base) as H:
        for sweep in range(3):
            x_o, c_o, mu_o = P.sweep_replay(mu, SEED, sweep, class_id_base=cid_base)
            assert c_o.sum() == h.m
            for flags in (capi.MMQ_GIBBS_DEFAULT, capi.MMQ_GIBBS_RAGGED_KERNEL, capi.MMQ_GIBBS_GENERIC_KERNEL):
                H.set_mu(mu)
                _, c, mu_g = H.sweep_debug(SEED, sweep, flags, want_x=False)
                assert np.array_equal(c, c_o), (sweep, flags, int(np.count_nonzero(c != c_o)))
                assert np.array_equal(mu_g, mu_o), (sweep, flags)
            H.set_mu(mu)
            x, c, mu_g = H.sweep_debug(SEED, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o), (sweep, int(np.count_nonzero(x != x_o)))
            assert np.array_equal(c, c_o) and np.array_equal(mu_g, mu_o), sweep
            mu = mu_o
        if weighted and cid_base == 0:      # the replayed chain has no class-id base
            H.set_mu(mu0)
            H.gibbs(SEED, 0, 32, stride=4, trace_len=8)                  # two replays of the 16-sweep graph
            mu_end, tr_o = P.gibbs_replay(mu0, SEED, 0, 32, 4, 8)
            assert np.array_equal(H.get_trace(), tr_o) and np.array_equal(H.get_mu(), mu_end)


# ------------------------------------------------------------------ collapsed shard, class plan

def _cat_limit(d):
    """mmq_cat_limit (include/mmq_sampler.h)."""
    return np.clip(32 * (d - 1), 32, 512)


def _plan_pieces(d, k):
    """Chunks of 32 slots of the class-plan pieces, restated from mmq_cls_build_host (mmq_cls_plan.h): returns
    (lo, hi, one, chain chunks, chain packed slots, rest classes)."""
    small = (d >= 2) & (d <= 64) & (k >= 1) & (k <= _cat_limit(d))
    one = small & (k == 1)
    multi = small & (k >= 2)
    grp = np.where(d <= 8, 64, 16)
    slots = np.where(multi, -(-k // grp), 0)
    per_d = np.bincount(d[multi], weights=slots[multi], minlength=65).astype(np.int64)
    ch = -(-per_d // 32)
    one_ch = -(-np.bincount(d[one], minlength=65) // 32)
    chain = (d >= 2) & (k > _cat_limit(d)) & (d <= 16)
    chain_d = np.bincount(d[chain], minlength=17)
    chain_ch = -(-chain_d // 32)
    rest = (d >= 2) & (k >= 1) & ~small & ~chain
    return (int(ch[:9].sum()), int(ch[9:].sum()), int(one_ch.sum()), int(chain_ch.sum()),
            int((chain_ch * 32 * np.arange(17)).sum()), int(rest.sum()))


@functools.lru_cache(maxsize=None)
def _collapsed_shard():
    """About 1 M hand-made classes over 500k transcripts (every 41st never hit): every piece of the class plan several
    times the size its capped grid covers in one pass."""
    rng = np.random.default_rng(20260405)
    n = 500_000
    hit = np.setdiff1d(np.arange(n), np.arange(0, n, 41)).astype(np.int32)
    both = lambda lo_n, hi_n, lo, mid, hi: np.concatenate([rng.integers(lo, mid, lo_n), rng.integers(mid, hi, hi_n)])
    parts = []
    d1 = both(330_000, 110_000, 2, 9, 65)                               # k_alloc_cls1: k == 1, d 2..64
    parts.append((d1, np.ones_like(d1)))
    d_lo = rng.integers(2, 9, 280_000)                                  # k_alloc_cls<LO>: d 2..8, 2 <= k <= limit
    parts.append((d_lo, rng.integers(2, _cat_limit(d_lo) + 1)))
    d_hi = both(135_000, 55_000, 9, 17, 65)                             # k_alloc_cls<HI>: d 9..64, small k
    parts.append((d_hi, rng.integers(2, 25, len(d_hi))))
    d_ch = rng.integers(2, 17, 172_000)                                 # k_alloc_chain: k > limit, BINV and BTRS
    lim = _cat_limit(d_ch)
    parts.append((d_ch, np.maximum(np.exp(rng.uniform(np.log(lim + 1), np.log(20_000), len(d_ch))).astype(np.int64), lim + 1)))
    d_rest = rng.integers(65, 200, 9_200)                               # general kernel: d > 64
    parts.append((d_rest, rng.integers(1, 400, len(d_rest))))
    d_s = np.ones(3000, np.int64)                                       # singletons and empty classes
    parts.append((d_s, rng.integers(0, 50, len(d_s))))
    d = np.concatenate([p[0] for p in parts]).astype(np.int64)
    k = np.concatenate([p[1] for p in parts]).astype(np.int64)
    order = rng.permutation(len(d))
    d, k = d[order], k[order]
    k[rng.random(len(k)) < 0.002] = 0
    col = _member_rows(rng, d, hit)
    row_ptr = np.concatenate([[0], np.cumsum(d)]).astype(np.int64)
    length = rng.uniform(1e-6, 1e-2, n)
    mu = rng.gamma(0.3, 100.0, n)
    mu[hit[:200]] = 0.0                                                 # zero and denormal-range mu inside rows
    mu[hit[-200:]] = 1e-300
    return row_ptr, col, k.astype(np.int32), length, mu, _plan_pieces(d, k)


@functools.lru_cache(maxsize=None)
def _collapsed_replay(cid_base):
    row_ptr, col, k, length, mu, _ = _collapsed_shard()
    P = orc.Problem(row_ptr, col, k, length)
    out = []
    for sweep in range(3):
        out.append(P.sweep_replay(mu, 4321, sweep, class_id_base=cid_base))
        mu = out[-1][2]
    return out


@functools.lru_cache(maxsize=None)
def _collapsed_chain_and_em():
    row_ptr, col, k, length, mu, _ = _collapsed_shard()
    P = orc.Problem(row_ptr, col, k, length)
    chain = P.gibbs_replay(mu, 4321, 0, 32, 4, 8)
    mu_i, uh_i, _ = P.init_mu()
    em = P.em(mu_i, 20, 0.1)
    return chain, (mu_i, uh_i), em


@pytest.mark.parametrize("plan", ["device", "host"])
@pytest.mark.parametrize("cid_base", [0, (1 << 32) * 5 + 3])
def test_class_plan_kernels_many_chunks_per_warp(monkeypatch, plan, cid_base):
    """Every piece of the class plan (k_alloc_cls1, k_alloc_cls<LO>, k_alloc_cls<HI>, k_alloc_chain, the general kernel
    on the rest) and k_gamma with two or more passes per worker: counts, mu and X bit for bit against the CPU replay; a
    graph run with a trace against gibbs_replay; init_mu and a bounded EM against the oracle."""
    if plan == "device":
        monkeypatch.delenv("MMQ_CLS_HOST_PLAN", raising=False)
    else:
        monkeypatch.setenv("MMQ_CLS_HOST_PLAN", "1")
    row_ptr, col, k, length, mu, (lo, hi, one, chain_ch, chain_packed, rest) = _collapsed_shard()
    n = len(length)
    sms = _sms()
    # mmq_cls.cu:915-957: min(chunks / 4, sms * CTAS) CTAs of 4 warps for the three small-set kernels (9, 8 and 5 CTAs
    # per SM for cls1, LO and HI); k_alloc_chain min(chunks / 4, 3 sms) CTAs taking 4 chunks of 32 classes per pass;
    # the rest, min(tiles / 8, 3 sms) CTAs of 8 warps, one class per tile
    assert one >= 2.5 * sms * 9 * MMQ_CLS_WARPS, one
    assert lo >= 2.5 * sms * 8 * MMQ_CLS_WARPS, lo
    assert hi >= 2.5 * sms * 5 * MMQ_CLS_WARPS, hi
    assert chain_ch >= 3 * sms * 3 * (MMQ_CHAIN_CLASSES // 32), chain_ch
    assert rest >= 2.5 * sms * 3 * MMQ_ALLOC_WARPS, rest
    # k_gamma (launch_gamma in mmq_core.cu): min(n / 256, 5 sms) CTAs of 256 threads, one transcript per thread and pass
    assert n >= 2.5 * sms * 5 * MMQ_GAMMA_THREADS
    # init and EM accumulation (k_init_acc, k_em_acc): 8 sms CTAs of 8 warps, one warp per transcript
    assert n >= 3 * sms * 8 * 8
    replay = _collapsed_replay(cid_base)
    with capi.Handle(row_ptr, col, k, length, class_id_base=cid_base) as H:
        st = H.cls_stats()
        assert st["in_use"] == 1
        assert st["class_slots"] == 32 * (lo + hi + one) and st["chain_slots"] == chain_packed and st["rest_classes"] == rest
        cur = mu
        for sweep in range(3):
            x_o, c_o, mu_o = replay[sweep]
            H.set_mu(cur)
            _, c, mu_g = H.sweep_debug(4321, sweep, capi.MMQ_GIBBS_DEFAULT)
            assert np.array_equal(c, c_o), (sweep, int(np.count_nonzero(c != c_o)))
            assert np.array_equal(mu_g, mu_o), sweep
            H.set_mu(cur)
            x, c, _ = H.sweep_debug(4321, sweep, capi.MMQ_GIBBS_TRANSPOSED)
            assert np.array_equal(x, x_o), (sweep, int(np.count_nonzero(x != x_o)))
            assert np.array_equal(c, c_o), sweep
            cur = mu_o
        if cid_base != 0:                   # the replayed chain, init_mu and EM have no class-id base
            return
        (mu_end, tr_o), (mu_i, uh_i), (mu_em, it_o, ll_o, _) = _collapsed_chain_and_em()
        H.set_mu(mu)
        H.gibbs(4321, 0, 32, stride=4, trace_len=8)                      # k_gamma writes the trace column of every t
        assert np.array_equal(H.get_trace(), tr_o) and np.array_equal(H.get_mu(), mu_end)
        uh = H.init_mu()
        assert np.array_equal(uh, uh_i)
        assert np.allclose(H.get_mu(), mu_i, rtol=1e-12, atol=0.0)
        it, ll, _ = H.em(20, 0.1)
        mu_g = H.get_mu()
    assert it == it_o
    obs = mu_em > 0
    assert np.array_equal(mu_g[~obs], mu_em[~obs])                       # never-hit transcripts
    assert np.max(np.abs(mu_g[obs] / mu_em[obs] - 1)) <= 1e-6
    assert np.isclose(ll, ll_o, rtol=1e-10)
