"""What pooling the chains costs on one B200 (mmseq -chains 4 -pool), written to profiles/pool.json with the card's name
and power limit:
  - device time (CUDA events) of mmq_pooled_summaries_dev at C2 size: n + G = 233,764 rows of the C2 sample, C = 4 chains
    of L = 1024 draws, the five default percentiles; mode 0 (draws of mu) and mode 1 (proportions), next to the
    diagnostics kernel mmq_chain_diagnostics_dev on the same draws;
  - the wall time of the handle forms on the C2 transcripts' own traces: mmq_summarize on one chain (the single-chain
    Sokal + percentile path of the tables) against mmq_pooled_summaries on four;
  - the C2 `mmseq -notraces -chains 4` wall time with and without -pool, alternated.
   python tools/gpu_pool.py [--out profiles/pool.json] [--skip-cli]      (on the GPU box)"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mmseq_b200 import capi, hostlib, synth  # noqa: E402
from tests import pool_reference as pref  # noqa: E402
from tools.gpu_chains import C2, card, draws  # noqa: E402

PCTS = (5, 25, 50, 75, 95)


def event_ms(fn, reps=5):
    st = torch.cuda.current_stream()
    fn(st)                                                               # warm-up
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn(st)
        b.record(st)
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return dict(ms_median=float(np.median(times)), ms_min=float(min(times)), ms_max=float(max(times)))


def kernel_times(rows, C=4, L=1024):
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = draws(C, rows, L, gen)
    ptrs = [x[c].data_ptr() for c in range(C)]
    idx = torch.from_numpy(pref.pct_index(PCTS, C * L)).cuda()
    out = torch.empty(5 * rows, dtype=torch.float64, device="cuda")
    pct = torch.empty(rows * len(PCTS), dtype=torch.float64, device="cuda")
    res = dict(rows=rows, chains=C, L=L)
    for mode, name in ((0, "pooled_mode0_log"), (1, "pooled_mode1_proportions")):
        res[name] = event_ms(lambda st: capi.pooled_summaries_dev(ptrs, rows, L, mode, len(PCTS), idx.data_ptr(), out.data_ptr(),
                                                                  pct.data_ptr(), st.cuda_stream))
        res[name]["us_per_row"] = 1000.0 * res[name]["ms_median"] / rows
        print(json.dumps({name: res[name]}), flush=True)
    res["chain_diagnostics"] = event_ms(lambda st: capi.chain_diagnostics_dev(ptrs, rows, L, out.data_ptr(), st.cuda_stream))
    print(json.dumps({"chain_diagnostics": res["chain_diagnostics"]}), flush=True)
    del x
    return res


def handle_times(h, length, C=4, L=1024):
    hs = [capi.Handle(h.row_ptr, h.col, h.k, length, device=0) for _ in range(C)]
    for c, H in enumerate(hs):
        H.init_mu()
        H.gibbs(capi.chain_seed(1234, c), 0, L, stride=1, trace_len=L)
    for H in hs:
        H.synchronize()
    res = {}
    for label, fn in (("summarize_one_chain", lambda: hs[0].summarize(0, pref.pct_index(PCTS, L))),
                      ("pooled_summaries_four_chains", lambda: capi.pooled_summaries(hs, 0, pref.pct_index(PCTS, C * L)))):
        fn()
        t = []
        for _ in range(3):
            t0 = time.perf_counter()
            fn()
            t.append(time.perf_counter() - t0)
        res[label] = dict(rows=h.n, wall_s_median=float(np.median(t)), note="host wall of the call: allocation, kernels and copies back")
        print(json.dumps({label: res[label]}), flush=True)
    for H in hs:
        H.close()
    return res


def cli_times(s, tmp):
    path = os.path.join(tmp, "c2.hits")
    synth.write_hits_binary(s, path)
    binary = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
    res = {}
    for label, extra in (("chains 4", []), ("chains 4 -pool", ["-pool"]), ("chains 4 (again)", []), ("chains 4 -pool (again)", ["-pool"])):
        t = time.perf_counter()
        r = subprocess.run([binary, "-notraces", "-chains", "4"] + extra + [path, os.path.join(tmp, "out")], capture_output=True, text=True)
        res[label] = dict(wall_s=time.perf_counter() - t, returncode=r.returncode,
                          stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith(("Gibbs", "EM", "Error"))])
        print(json.dumps({label: res[label]}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pool.json"))
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    out = dict(gpu=card())
    s = synth.Synth(C2["seed"], C2["transcripts"], C2["fragments"])
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    length = s.efflen[h.col2hdr] * s.N / 1e9
    out["kernels"] = kernel_times(h.n + s.G)
    out["handle_forms"] = handle_times(h, length)
    if not args.skip_cli:
        with tempfile.TemporaryDirectory() as tmp:
            out["mmseq_notraces_wall"] = cli_times(s, tmp)
    out["gpu_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"])))


if __name__ == "__main__":
    main()
