"""Multi-GPU path on real devices: two ranks (torch.multiprocessing, NCCL through the library's
own communicator), each with half of the hit classes; counts all-reduced per sweep must give the
single-GPU chain bit for bit; EM within 1e-6."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, use_p2p, out_q):
    import torch
    import torch.distributed as dist
    from mmseq_b200 import capi, hostlib, synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)   # plumbing only: ships the NCCL id
    s = synth.Synth(20260101 + 1, 300, 20000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    cut = [0, h.m // 3, h.m][rank:rank + 2]
    a, b = cut
    lo, hi = h.row_ptr[a], h.row_ptr[b]
    uid = [capi.comm_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    H = capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], h.k[a:b], h.len, class_id_base=a, device=rank)
    H.comm_init(uid[0], rank, world)
    if use_p2p:   # count exchange fused into the Gamma kernel over peer memory (cudaIpc between processes)
        hs = [None] * world
        dist.all_gather_object(hs, H.p2p_export())
        H.p2p_attach(hs, rank, world)
    uh = H.init_mu()
    mu0 = H.get_mu()
    it, ll, llr = H.em(1000, 0.1)
    mu_em = H.get_mu()
    H.gibbs(1234, 0, 32, stride=4, trace_len=8)
    tr = H.get_trace()
    _, c, mu_dbg = H.sweep_debug(1234, 32, capi.MMQ_GIBBS_DEFAULT, want_x=False)
    H.close()
    out_q.put((rank, uh, mu0, it, ll, mu_em, tr, c, mu_dbg))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("use_p2p", [False, True])
def test_two_ranks_reproduce_single_gpu_chain(use_p2p):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from mmseq_b200 import capi, hostlib, synth
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, 29533 + int(use_p2p), use_p2p, out_q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([out_q.get(timeout=300) for _ in range(2)], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
    s = synth.Synth(20260101 + 1, 300, 20000)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        uh = H.init_mu(); mu0 = H.get_mu()
        it, ll, llr = H.em(1000, 0.1); mu_em = H.get_mu()
        for r in res:   # every rank holds the all-reduced quantities
            assert np.array_equal(r[1], uh) and np.allclose(r[2], mu0, rtol=1e-12)
            assert r[3] == it and np.isclose(r[4], ll, rtol=1e-10) and np.max(np.abs(r[5] / mu_em - 1)) <= 1e-6
        # the Gibbs chain: start both from rank 0's EM estimate so the comparison is exact
        H.set_mu(res[0][5])
        H.gibbs(1234, 0, 32, stride=4, trace_len=8)
        tr = H.get_trace()
        _, c, mu_dbg = H.sweep_debug(1234, 32, capi.MMQ_GIBBS_DEFAULT, want_x=False)
    assert np.array_equal(res[0][5], res[1][5])          # identical EM result on both ranks (same all-reduced sums)
    for r in res:
        assert np.array_equal(r[6], tr) and np.array_equal(r[7], c) and np.array_equal(r[8], mu_dbg)


# padded: the length array has 3 x 189,440 + 77 transcripts, most of them without hits, so that the fused Gamma kernels
# loop: k_gamma<ACC, true> runs min(n / 256, 5 sms) CTAs and k_gamma_rs min(max(n / ranks, n / 8) / 256, 4 sms) CTAs of 256
# threads (launch_gamma in mmq_core.cu).  rs: mmq_tune knob 6, the reduce-scatter exchange (k_gamma_rs + k_trace_capture).
@pytest.mark.parametrize("weighted,padded,rs", [(False, False, False), (True, False, False), (False, True, False), (True, True, True)],
                         ids=["False", "True", "padded", "padded-rs"])
def test_single_process_peer_attach_matches_single_gpu(weighted, padded, rs):
    """mmq_p2p_attach_local (what the host program uses for -gpus N): two handles in one process,
    sweeps issued from two threads; the fused peer-memory Gamma kernel gives the single-GPU chain.
    weighted = BASELINE config 4 at parity-test size: per-fragment shards with fp32 per-hit weights
    (sequence-specific / insert-size likelihoods) over several GPUs."""
    import threading
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from mmseq_b200 import capi, hostlib, synth
    s = synth.Synth(20260101 + 4, 300, 20000, weights=weighted)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w if weighted else None,
                             layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    assert (h.w is not None) == weighted
    length = h.len
    if padded:
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        length = np.concatenate([h.len, np.random.default_rng(1).uniform(1e-6, 1e-2, 3 * 189_440 + 77 - h.n)])
        assert len(length) > 2.5 * sms * 5 * 256
    cut = [0, (h.m // 2) & ~1, h.m]
    mu0 = np.random.default_rng(0).gamma(0.5, 50.0, len(length))
    hs = []
    for r in range(2):
        a, b = cut[r], cut[r + 1]
        lo, hi = h.row_ptr[a], h.row_ptr[b]
        hs.append(capi.Handle(h.row_ptr[a:b + 1] - lo, h.col[lo:hi], None, length, weight=None if h.w is None else h.w[lo:hi], class_id_base=a, device=r))
    capi.p2p_attach_local(hs)
    if rs:
        for H in hs:
            H.tune(6, 1)
    out = [None, None]

    def run(r):
        hs[r].set_mu(mu0)
        hs[r].gibbs(1234, 0, 40, stride=4, trace_len=10)
        out[r] = (hs[r].get_trace(), hs[r].get_mu())

    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for H in hs:
        H.close()
    with capi.Handle(h.row_ptr, h.col, None, length, weight=h.w) as H:
        H.set_mu(mu0)
        H.gibbs(1234, 0, 40, stride=4, trace_len=10)
        tr, mu = H.get_trace(), H.get_mu()
    for r in range(2):
        assert np.array_equal(out[r][0], tr) and np.array_equal(out[r][1], mu)
