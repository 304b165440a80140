"""What several chains cost on one B200 (mmseq -chains), written to profiles/chains.json with the card's name and power
limit:
  - the diagnostics kernel (mmq_chain_diagnostics_dev) at C2 size: n + G rows of the C2 sample (180k transcripts,
    54k genes; the generator makes no identical sets), C = 4 chains of L = 1024 draws, device time by CUDA events;
  - the numpy reference (tests/chain_reference.py) on the same kind of rows: seconds per row in one host process, and
    over all host CPUs in parallel;
  - Gibbs sweeps/s per chain and in all for C = 1, 2, 4, 8 chains on one GPU (C2 collapsed shard, one handle and
    stream per chain, 64-sweep windows through the CUDA graph, enqueued round-robin);
  - the C2 `mmseq -notraces` wall time without and with -chains 4.
   python tools/gpu_chains.py [--out profiles/chains.json] [--skip-cli]      (on the GPU box)"""
import argparse
import json
import multiprocessing
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mmseq_b200 import capi, hostlib, synth  # noqa: E402
from tests import chain_reference as ref  # noqa: E402

C2 = dict(seed=20260101 + 2, transcripts=180000, fragments=30000000)
SWEEPS = 64


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().split("\n")[0]


def draws(C, rows, L, gen):
    """log-normal draws, AR(1) with phi 0.9 in the log (a slowly mixing posterior), on the device"""
    z = torch.randn((C, rows, L), dtype=torch.float64, device="cuda", generator=gen)
    for s in range(1, L):
        z[:, :, s] = 0.9 * z[:, :, s - 1] + 0.4358898943540674 * z[:, :, s]
    return torch.exp(z - 3.0)


def kernel_time(rows, C=4, L=1024, reps=5):
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = draws(C, rows, L, gen)
    out = torch.empty(5 * rows, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream()
    ptrs = [x[c].data_ptr() for c in range(C)]
    capi.chain_diagnostics_dev(ptrs, rows, L, out.data_ptr(), st.cuda_stream)       # warm-up
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        capi.chain_diagnostics_dev(ptrs, rows, L, out.data_ptr(), st.cuda_stream)
        b.record(st)
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    sample = x[:, :400].cpu().numpy()
    del x
    return dict(rows=rows, chains=C, L=L, ms_median=float(np.median(times)), ms_min=float(min(times)), ms_max=float(max(times)),
                us_per_row=1000.0 * float(np.median(times)) / rows), sample


def reference_time(sample):
    t = time.perf_counter()
    ref.diagnose_rows(sample[:, :100])
    one = (time.perf_counter() - t) / 100
    cpus = os.cpu_count() or 1
    parts = np.array_split(np.arange(sample.shape[1]), 4 * cpus)
    with ProcessPoolExecutor(cpus, mp_context=multiprocessing.get_context("spawn")) as ex:   # this process runs CUDA threads
        list(ex.map(ref.diagnose_rows, [sample[:, :2]] * cpus))                              # start the workers
        t = time.perf_counter()
        done = sum(d["rhat"].size for d, _ in ex.map(ref.diagnose_rows, [sample[:, p] for p in parts if len(p)]))
        pooled = (time.perf_counter() - t) / done
    return dict(s_per_row_one_process=one, host_cpus=cpus, s_per_row_all_cpus=pooled)


def sweep_rates(h, length):
    res = []
    for C in (1, 2, 4, 8):
        hs = [capi.Handle(h.row_ptr, h.col, h.k, length, device=0) for _ in range(C)]
        for H in hs:
            H.init_mu()
        for c, H in enumerate(hs):                                       # capture every handle's graph
            H.gibbs(capi.chain_seed(1234, c), 0, SWEEPS, stride=16, trace_len=64)
        for H in hs:
            H.synchronize()
        windows = 16
        t = time.perf_counter()
        for w in range(1, windows + 1):
            for c, H in enumerate(hs):
                H.gibbs(capi.chain_seed(1234, c), w * SWEEPS, SWEEPS, stride=16, trace_len=64)
        for H in hs:
            H.synchronize()
        sec = time.perf_counter() - t
        per = windows * SWEEPS / sec
        res.append(dict(chains=C, sweeps_per_s_per_chain=per, sweeps_per_s_total=per * C, seconds=sec, sweeps_per_chain=windows * SWEEPS))
        print(json.dumps(res[-1]), flush=True)
        for H in hs:
            H.close()
    return res


def cli_times(s, tmp):
    path = os.path.join(tmp, "c2.hits")
    synth.write_hits_binary(s, path)
    binary = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
    res = {}
    for label, extra in (("without", []), ("chains 4", ["-chains", "4"]), ("without (again)", []), ("chains 4 (again)", ["-chains", "4"])):
        t = time.perf_counter()
        r = subprocess.run([binary, "-notraces"] + extra + [path, os.path.join(tmp, "out")], capture_output=True, text=True)
        res[label] = dict(wall_s=time.perf_counter() - t, returncode=r.returncode,
                          stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith(("Gibbs", "EM", "Convergence"))])
        print(json.dumps({label: res[label]}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "chains.json"))
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    out = dict(gpu=card())
    s = synth.Synth(C2["seed"], C2["transcripts"], C2["fragments"])
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    length = s.efflen[h.col2hdr] * s.N / 1e9
    rows = h.n + s.G
    out["diagnostics_kernel"], sample = kernel_time(rows)
    print(json.dumps(out["diagnostics_kernel"]), flush=True)
    out["numpy_reference"] = reference_time(sample)
    out["numpy_reference"]["s_for_all_rows_all_cpus"] = out["numpy_reference"]["s_per_row_all_cpus"] * rows
    print(json.dumps(out["numpy_reference"]), flush=True)
    out["gibbs_one_gpu"] = dict(case=f"C2 collapsed (n={h.n}, rows={h.m})", sweeps_per_window=SWEEPS, results=sweep_rates(h, length))
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
