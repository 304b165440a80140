"""bench.py --dump-outputs on the GPU: timed_run hands back mu after the last timed step and the trace slot
that step recorded, read before the kernel-timing repetition that follows."""
import numpy as np
import pytest

import bench
from mmseq_b200 import capi

pytestmark = pytest.mark.gpu


def test_timed_run_outputs_are_those_of_the_last_timed_step(small_problem):
    import torch
    h = small_problem
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    K, W, S = 3, 2, bench.SWEEPS_PER_STEP
    out = {}
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.set_stream(stream.cuda_stream)
        H.init_mu()
        mu0 = H.get_mu()
        bench.timed_run(None, H, None, stream, dev, torch.cuda.synchronize, K, W, None, capi.MMQ_GIBBS_DEFAULT, out)
        mu_end = H.get_mu()
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as R:   # the W warm-up and K timed steps, replayed
        R.set_mu(mu0)
        for j in range(W + K):
            R.gibbs(bench.SEED, j * S, S, stride=S, trace_len=2 * K + W + 1)
        mu, tr = R.get_mu(), R.get_trace()
    assert np.array_equal(out["mu"], mu)
    assert np.array_equal(out["trace_last_step"], tr[:, W + K - 1])
    assert not np.array_equal(mu_end, mu)                 # the repetition moved the chain on after the dump
