"""Time the pieces of the class-plan sweep alone (collapsed C2 sample): one workload, one handle, mmq_tune knob 0.
   python tools/gpu_tune_cls.py            (on the GPU box)"""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mmseq_b200 import capi, hostlib, synth

s = synth.Synth(20260101 + 2, 180000, 30000000)
h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
length = s.efflen[h.col2hdr] * 30000000 / 1e9
H = capi.Handle(h.row_ptr, h.col, h.k, length, device=0)
stream = torch.cuda.Stream()
H.set_stream(stream.cuda_stream)
H.init_mu()
mu0 = H.get_mu()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

def run(label, skip, steps=8):
    H.tune(0, skip)
    H.set_mu(mu0)
    sweep = 0
    for _ in range(2):
        H.gibbs(1234, sweep, 16, stride=16, trace_len=64); sweep += 16
    H.synchronize()
    tot = 0.0
    for _ in range(steps):
        with torch.cuda.stream(stream):
            flush.zero_()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(stream)
        H.gibbs(1234, sweep, 16, stride=16, trace_len=64); sweep += 16
        b.record(stream)
        H.synchronize()
        tot += a.elapsed_time(b)
    print(f"{label:44s} {1000 * tot / (steps * 16):8.2f} us per sweep", flush=True)

run("default", 0)
for name, m in (("no chain", 8), ("no large (HI)", 4), ("no small k>=2 (LO)", 1), ("no single-fragment (cls1)", 16), ("only cls1", 1 | 2 | 4 | 8),
                ("only LO", 2 | 4 | 8 | 16), ("only HI", 1 | 2 | 8 | 16), ("only chain", 1 | 2 | 4 | 16), ("none (gamma only)", 31)):
    run("skip: " + name, m)
