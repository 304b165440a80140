"""The chain set of collapsed shards (classes with more than mmq_cat_limit(d) fragments, mmq_cls.cu: k_alloc_chain) on
its three depth instances (class sizes 5..16, 3..4 and 2) against the CPU replay, bit for bit over several sweeps:
k just above the limit and up to 10^5 (inversions and BTRS), nodes with p above 1/2 (the flip), members with mu = 0 and
all-zero rows, chunk ranges that cross the instances' boundaries or leave an instance empty, grids capped so that
every block takes several passes, and class ids above 2^32; the plan built on the device and on the host."""
import numpy as np
import pytest

from mmseq_b200 import capi
from oracle import oracle as orc
from tests import exact_reference as E

pytestmark = pytest.mark.gpu


def _chain_shard(counts_by_d, seed, n=30000):
    """Rows of the given sizes (every one in the chain set), sorted distinct columns; mu spread over decades with zeros."""
    rng = np.random.default_rng(seed)
    rows, ks = [], []
    for d, count in counts_by_d.items():
        start = rng.integers(0, n - 60 * d, count)
        cols = start[:, None] + np.cumsum(rng.integers(1, 60, (count, d)), axis=1)
        lim = E.cat_limit(d)
        k = np.where(rng.random(count) < 0.5, lim + 1 + rng.integers(0, 4, count),
                     np.exp(rng.uniform(np.log(lim + 1), np.log(1e5), count)).astype(np.int64))
        rows.append(cols)
        ks.append(k)
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for c in rows for r in c])]).astype(np.int64)
    col = np.concatenate([c.ravel() for c in rows]).astype(np.int32)
    k = np.concatenate(ks).astype(np.int32)
    mu = rng.gamma(0.3, 100.0, n)
    mu[rng.random(n) < 0.05] = 0.0
    # a few all-zero rows of every size
    zero_cols = np.arange(n - 16, n)
    mu[zero_cols] = 0.0
    m = len(k)
    for q in rng.choice(m, 40, replace=False):
        d = int(row_ptr[q + 1] - row_ptr[q])
        col[row_ptr[q]:row_ptr[q + 1]] = zero_cols[:d]
    return row_ptr, col, k, rng.uniform(1e-6, 1e-2, n), mu


def _check(row_ptr, col, k, l, mu, cid_base, sweeps=(0, 1, 5)):
    P = orc.Problem(row_ptr, col, k, l)
    with capi.Handle(row_ptr, col, k, l, class_id_base=cid_base) as H:
        st = H.cls_stats()
        assert st["in_use"] == 1 and st["chain_classes"] == len(k) and st["small_classes"] == 0
        for sweep in sweeps:
            H.set_mu(mu)
            _, c_o, mu_o = P.sweep_replay(mu, 9137, sweep, class_id_base=cid_base)
            _, c_f, mu_f = H.sweep_debug(9137, sweep, capi.MMQ_GIBBS_DEFAULT)
            assert np.array_equal(c_f, c_o) and np.array_equal(mu_f, mu_o), sweep
            assert c_f.sum() == k.sum()


@pytest.fixture(params=["device", "host"])
def plan(request, monkeypatch):
    if request.param == "device":
        monkeypatch.delenv("MMQ_CLS_HOST_PLAN", raising=False)
    else:
        monkeypatch.setenv("MMQ_CLS_HOST_PLAN", "1")
    return request.param


@pytest.mark.parametrize("cid_base", [0, (1 << 32) * 3 + 11])
def test_every_class_size_several_passes(plan, cid_base):
    """d = 2..16; more classes per instance than its capped grid takes in one pass (3 blocks per SM; 128 classes per
    block of the shallow instances, 64 of the deep one)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    per_deep = -(-3 * sms * 64 * 2 // 12)       # two passes of the deep instance, spread over d = 5..16
    counts = {2: 3 * sms * 128 * 2, 3: 3 * sms * 128, 4: 3 * sms * 128}
    counts.update({d: per_deep for d in range(5, 17)})
    _check(*_chain_shard(counts, seed=1), cid_base=cid_base)


@pytest.mark.parametrize("sizes", [(2,), (3, 4), (16, 9, 5), (2, 7), (3, 11), (2, 3)])
def test_instances_left_empty(plan, sizes):
    """Chain sets that leave one or two of the three instances without classes, and chunk ranges that end inside a
    chunk of 32."""
    _check(*_chain_shard({d: 1000 + 7 * d for d in sizes}, seed=sum(sizes)), cid_base=5)
