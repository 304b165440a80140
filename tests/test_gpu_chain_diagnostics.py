"""mmq_chain_diagnostics_dev and mmq_chain_diagnostics against the numpy reference (tests/chain_reference.py): every
(chains, trace length) shape the C ABI accepts at the edges and in the middle, with enough rows that every CTA of the
grid-capped loop takes several; mixed rows (iid, AR(1), shifted and scaled chains, log-normal, ties, zeros, constant,
NaN, +inf); bit-identical results under repetition, row permutation, the handle form and a second GPU."""
import ctypes
import math
import multiprocessing
import os
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from mmseq_b200 import capi, hostlib, synth
from tests import chain_reference as ref

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = [(C, L) for C in (2, 3, 4, 8) for L in (8, 64, 1024, 2048) if C * L <= 8192]
KINDS = ("iid", "ar0.5", "ar0.9", "ar0.99", "shifted", "scaled", "lognormal", "ties", "zeros", "constant", "nan", "inf")
REL = 1e-10


_POOL = []


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    for ex in _POOL:
        ex.shutdown()
    print(f"\ntest_gpu_chain_diagnostics: {time.time() - t0:.1f} s wall")


def grid_rows():
    """rows = 3 x grid + 5: every CTA of the grid (2 x SMs) takes three or four rows"""
    return 3 * 2 * torch.cuda.get_device_properties(0).multi_processor_count + 5


def ar1(rng, n, L, phi):
    x = np.empty((n, L))
    x[:, 0] = rng.standard_normal(n)
    e = rng.standard_normal((n, L)) * math.sqrt(1 - phi * phi)
    for s in range(1, L):
        x[:, s] = phi * x[:, s - 1] + e[:, s]
    return x


def mixed(rng, C, L, rows):
    """(C, rows, L) draws, row r of kind KINDS[r % len(KINDS)]"""
    x = np.empty((C, rows, L))
    for r in range(rows):
        k = KINDS[r % len(KINDS)]
        if k.startswith("ar"):
            v = ar1(rng, C, L, float(k[2:])) + 3.0
        elif k == "lognormal":
            v = np.exp(rng.normal(-2.0, 1.5, (C, L)))
        elif k == "ties":
            v = rng.choice([0.25, 1.0, 4.0], size=(C, L), p=[0.2, 0.5, 0.3])
        elif k == "zeros":
            v = rng.gamma(0.3, size=(C, L))
            v[rng.random((C, L)) < 0.1] = 0.0
        elif k == "constant":
            v = np.full((C, L), 0.7)
        else:
            v = rng.gamma(4.0, size=(C, L))
            if k == "shifted":
                v[C - 1] += 2.0
            elif k == "scaled":
                v[0] = 4.0 + 3.0 * (v[0] - 4.0)
            elif k == "nan":
                v[C // 2, L // 3] = math.nan
            elif k == "inf":
                v[0, L - 1] = math.inf
        x[:, r, :] = v
    return x


def run_dev(x):
    C, rows, L = x.shape
    chains = [torch.from_numpy(np.ascontiguousarray(x[c])).cuda() for c in range(C)]
    out = torch.empty(5 * rows, dtype=torch.float64, device="cuda")
    capi.chain_diagnostics_dev([t.data_ptr() for t in chains], rows, L, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(5, rows)


def reference(x):
    """the reference over the rows of x, split over host processes (spawned once per module: this process runs CUDA
    threads, so it does not fork)"""
    workers = max(1, min(16, os.cpu_count() or 1))
    if not _POOL:
        _POOL.append(ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")))
    parts = np.array_split(np.arange(x.shape[1]), workers * 4)
    res = list(_POOL[0].map(ref.diagnose_rows, [x[:, p, :] for p in parts if len(p)]))
    return np.stack([np.concatenate([d[k] for d, _ in res]) for k in ref.OUTPUTS]), np.concatenate([m for _, m in res])


def compare(got, want, margin):
    """all five outputs within REL (NaN where the reference has NaN); rows whose ESS decision margin is below 1e-9
    are exempt from the ESS columns, and at most 0.1 % of the rows may be."""
    exempt = margin < 1e-9
    assert exempt.sum() <= max(1, int(0.001 * len(margin))), exempt.sum()
    for q, name in enumerate(ref.OUTPUTS):
        g, w = got[q], want[q]
        skip = exempt if name.startswith("ess") else np.zeros_like(exempt)
        assert np.array_equal(np.isnan(g) | skip, np.isnan(w) | skip), name
        with np.errstate(invalid="ignore"):                              # inf - inf where both are -inf
            ok = np.isnan(w) | (g == w) | (np.abs(g - w) <= REL * np.abs(w) + 1e-13) | skip
        bad = np.flatnonzero(~ok)
        assert not len(bad), (name, bad[:5], g[bad[:5]], w[bad[:5]])


@pytest.mark.parametrize("C,L", CASES)
def test_against_reference(C, L):
    rng = np.random.default_rng(1000 * C + L)
    rows = grid_rows()
    x = mixed(rng, C, L, rows)
    got = run_dev(x)
    want, margin = reference(x)
    compare(got, want, margin)
    kinds = np.arange(rows) % len(KINDS)
    for k in ("nan", "inf"):
        assert np.isnan(got[:, kinds == KINDS.index(k)]).all()
    const = got[:, kinds == KINDS.index("constant")]
    assert np.isnan(const[:3]).all() and (const[4] < 1e-12).all()
    if L >= 1024 and C <= 4:                                             # one chain of C off: R-hat grows as C falls
        iid = kinds == KINDS.index("iid")
        assert np.abs(got[0, iid] - 1).max() < 0.05
        assert (got[0, kinds == KINDS.index("shifted")] > 1.05).all()
        assert (got[0, kinds == KINDS.index("scaled")] > 1.05).all()


def test_bits_repeat_and_row_order():
    rng = np.random.default_rng(7)
    C, L = 4, 1024
    rows = grid_rows()
    x = mixed(rng, C, L, rows)
    a, b = run_dev(x), run_dev(x)
    assert a.tobytes() == b.tobytes()
    perm = rng.permutation(rows)
    c = run_dev(x[:, perm, :])
    assert a[:, perm].tobytes() == c.tobytes()
    d = run_dev(x[:, :17, :])                                            # another grid: 17 CTAs
    assert a[:, :17].tobytes() == d.tobytes()


def test_arguments_outside_the_limits():
    lib = capi.lib()
    buf = torch.zeros(8 * 8192, dtype=torch.float64, device="cuda")
    out = torch.zeros(5 * 8, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(C, L, rows=8, null_at=-1, out_ptr=out.data_ptr()):
        ptrs = [buf.data_ptr()] * max(C, 1)
        if null_at >= 0:
            ptrs[null_at] = None
        arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        return lib.mmq_chain_diagnostics_dev(arr, C, rows, L, out_ptr, stream)
    assert call(2, 8) == 0
    for C, L in [(1, 1024), (9, 512), (0, 64), (2, 4), (2, 12), (2, 4096), (8, 2048), (5, 2048), (3, 100)]:
        assert call(C, L) == 1, (C, L)
    assert call(2, 64, rows=-1) == 1
    assert call(2, 64, null_at=1) == 1
    assert call(2, 64, out_ptr=None) == 1
    assert call(2, 64, rows=0, out_ptr=None) == 0
    torch.cuda.synchronize()


def _problem():
    s = synth.Synth(4242, 120, 6000)
    return hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)


def _chains(h, devices, L=64, seed=99):
    """one handle per device, EM start, chain c with mmq_chain_seed(seed, c), groups: identical pairs, genes of three
    with extras"""
    hs = []
    with capi.Handle(h.row_ptr, h.col, h.k, h.len, device=devices[0]) as H:
        H.init_mu()
        H.em(1000, 0.1)
        mu = H.get_mu()
    n = h.n
    iptr = np.arange(0, n - n % 2 + 1, 2, dtype=np.int64)
    imem = np.arange(n - n % 2, dtype=np.int32)
    gptr = np.append(np.arange(0, n, 3, dtype=np.int64), n)
    gmem = np.arange(n, dtype=np.int32)
    extra = np.random.default_rng(3).gamma(0.1, 1.0, (len(gptr) - 1, L))
    for c, dev in enumerate(devices):
        H = capi.Handle(h.row_ptr, h.col, h.k, h.len, device=dev)
        H.set_mu(mu)
        H.gibbs(capi.chain_seed(seed, c), 0, 16 * L, stride=16, trace_len=L)
        H.set_groups(capi.MMQ_GROUP_IDENTICAL, iptr, imem)
        H.set_groups(capi.MMQ_GROUP_GENE, gptr, gmem, extra)
        hs.append(H)
    return hs


def test_handle_form_equals_dev_form():
    hs = _chains(_problem(), [0, 0, 0, 0])
    try:
        for which in (0, 1, 2):
            got = capi.chain_diagnostics(hs, which)
            tr = np.stack([H.get_trace() if which == 0 else H.get_group_trace(which) for H in hs])
            want = run_dev(tr)
            for q, k in enumerate(capi.CHAIN_OUTPUTS):
                assert got[k].tobytes() == want[q].tobytes(), (which, k)
            assert np.isfinite(got["rhat"]).mean() > 0.5
        with pytest.raises(capi.MmqError):
            capi.chain_diagnostics(hs[:1], 0)
    finally:
        for H in hs:
            H.close()


def test_chains_on_two_devices_equal_one_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    h = _problem()
    res = []
    for devices in ([0, 0], [0, 1]):
        hs = _chains(h, devices)
        try:
            res.append([capi.chain_diagnostics(hs, w) for w in (0, 1, 2)])
        finally:
            for H in hs:
                H.close()
    for a, b in zip(*res):
        for k in capi.CHAIN_OUTPUTS:
            assert a[k].tobytes() == b[k].tobytes(), k
