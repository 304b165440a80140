"""Cost of accumulating posterior fragment counts (mmq_count_moments_begin): device-timed Gibbs sweeps per second with
and without accumulation on the C2 sample (180k transcripts, 30 M fragments), collapsed and weighted per fragment,
over the generator's genes (no identical sets).  Two handles on the same shard, one accumulating from the start;
windows alternate between them, each 64 sweeps through the CUDA graph after a 256 MB write that evicts L2.
   python tools/gpu_counts_overhead.py [--windows 12] [--out FILE]      (on the GPU box)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from mmseq_b200 import capi, hostlib, synth  # noqa: E402

SWEEPS = 64


def measure(label, hs, gene_of, n_gene, windows, stream, flush):
    """hs: two handles on the same shard; hs[1] accumulates from the start.  Windows alternate between them."""
    mu0 = None
    for H in hs:
        H.set_stream(stream.cuda_stream)
        H.init_mu()
        mu0 = H.get_mu()
    hs[1].count_moments_begin(None, 0, gene_of, n_gene)
    times = {False: [], True: []}
    sweep = 0
    for w in range(2 * windows + 2):
        on = bool(w & 1)
        H = hs[on]
        H.set_mu(mu0)
        with torch.cuda.stream(stream):
            flush.zero_()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record(stream)
        H.gibbs(1234, sweep, SWEEPS, stride=16, trace_len=64)
        b.record(stream)
        H.synchronize()
        sweep += SWEEPS
        if w >= 2:                                   # the first window of each handle captures its graph
            times[on].append(a.elapsed_time(b) / SWEEPS)
    assert hs[1].count_moments(0)[0] == SWEEPS * (windows + 1)
    res = {}
    for on in (False, True):
        t = np.array(times[on])
        res["with" if on else "without"] = dict(us_per_sweep_median=1000 * float(np.median(t)), us_per_sweep_min=1000 * float(t.min()),
                                                us_per_sweep_max=1000 * float(t.max()), sweeps_per_s=1000.0 / float(np.median(t)))
    res["overhead_pct"] = 100.0 * (res["with"]["us_per_sweep_median"] / res["without"]["us_per_sweep_median"] - 1.0)
    res["case"] = label
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=12)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().split("\n")[0]
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = dict(gpu=gpu, sweeps_per_window=SWEEPS, windows_per_mode=args.windows, results=[])
    for weighted in (False, True):
        s = synth.Synth(20260101 + 2, 180000, 30000000, weights=weighted)
        layout = (hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH if weighted else hostlib.LAYOUT_COLLAPSED) | hostlib.LAYOUT_HEADER_ORDER_COLUMNS
        h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w if weighted else None, layout=layout)
        length = s.efflen[h.col2hdr] * s.N / 1e9
        gene_of = s.gene_of[h.col2hdr].astype(np.int32)
        hs = [capi.Handle(h.row_ptr, h.col, None if weighted else h.k, length, weight=h.w, device=0) for _ in range(2)]
        label = f"C2 {'weighted per-fragment' if weighted else 'collapsed'} (n={h.n}, rows={h.m}, genes={s.G})"
        r = measure(label, hs, gene_of, s.G, args.windows, stream, flush)
        for H in hs:
            H.close()
        print(json.dumps(r), flush=True)
        out["results"].append(r)
        del s, h
    print(json.dumps(dict(gpu=gpu)))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
