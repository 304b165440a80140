"""What transcripts per million cost on one B200 (mmseq -tpm), written to profiles/tpm.json with the card's name and power
limit:
  - device time (CUDA events, after a warm-up) of mmq_draw_totals_dev at C2 size: the n = 179,634 observed transcripts
    of the C2 sample, L = 1024 draws, 8 n L = 1.47 GB read once per call (11.7 times the 126 MB L2, so every call reads
    it from HBM), with its bytes over time and that rate's share of the measured HBM peak (DESIGN.md section 5);
  - device time of mmq_tpm_summaries_dev for the C2 transcripts and for its genes (the sample's gene CSR over the
    observed transcripts), at C = 1 and C = 4 chains of L = 1024, the five default percentiles;
  - the C2 `mmseq -notraces` wall time without and with -tpm, alternated, two runs each.
   python tools/gpu_tpm.py [--out profiles/tpm.json] [--skip-cli]      (on the GPU box)"""
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
from tests import tpm_reference as tref  # noqa: E402
from tools.gpu_chains import C2, card, draws  # noqa: E402
from tools.gpu_pool import event_ms  # noqa: E402

PCTS = (5, 25, 50, 75, 95)
HBM_PEAK_GBS = 6553.6  # MEASURED_PEAKS.json hbm_gbs, the peak of DESIGN.md section 5


def totals_time(n, L=1024):
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = draws(1, n, L, gen)[0]
    ws = torch.empty(max(1, capi.draw_totals_workspace_bytes(n, L) // 8), dtype=torch.float64, device="cuda")
    tot = torch.empty(L, dtype=torch.float64, device="cuda")
    res = event_ms(lambda st: capi.draw_totals_dev(x.data_ptr(), n, L, tot.data_ptr(), ws.data_ptr(), st.cuda_stream), reps=20)
    nbytes = 8 * n * L + 2 * capi.draw_totals_workspace_bytes(n, L) + 8 * L
    gbs = nbytes / (res["ms_median"] * 1e-3) / 1e9
    res.update(rows=n, L=L, bytes=nbytes, gb_per_s=gbs, share_of_hbm_peak=gbs / HBM_PEAK_GBS, hbm_peak_gbs=HBM_PEAK_GBS,
               bytes_note="the trace read once, the tile sums written and read back once, the totals written")
    exact = tref.totals_fsum(x[:2000].cpu().numpy())                    # a sanity check on a slice, not a timing
    part = torch.empty(L, dtype=torch.float64, device="cuda")
    ws2 = torch.empty(max(1, capi.draw_totals_workspace_bytes(2000, L) // 8), dtype=torch.float64, device="cuda")
    capi.draw_totals_dev(x.data_ptr(), 2000, L, part.data_ptr(), ws2.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    res["slice_max_rel_err_vs_fsum"] = float(np.max(np.abs(part.cpu().numpy() - exact) / exact))
    del x
    return res


def summaries_times(n, gptr, gmem, L=1024):
    gen = torch.Generator(device="cuda").manual_seed(4)
    res = {}
    d_ptr = torch.from_numpy(gptr).cuda()
    d_mem = torch.from_numpy(gmem).cuda()
    for C in (1, 4):
        x = draws(C, n, L, gen)
        ptrs = [x[c].data_ptr() for c in range(C)]
        tot = torch.empty(C * L, dtype=torch.float64, device="cuda")
        ws = torch.empty(max(1, capi.draw_totals_workspace_bytes(n, L) // 8), dtype=torch.float64, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        for c in range(C):
            capi.draw_totals_dev(ptrs[c], n, L, tot.data_ptr() + 8 * c * L, ws.data_ptr(), st)
        idx = torch.from_numpy(tref.pct_index(PCTS, C * L)).cuda()
        for label, rows, gp, gm in (("transcripts", n, None, None), ("genes", len(gptr) - 1, d_ptr.data_ptr(), d_mem.data_ptr())):
            out = torch.empty(2 * rows, dtype=torch.float64, device="cuda")
            pct = torch.empty(rows * len(PCTS), dtype=torch.float64, device="cuda")
            r = event_ms(lambda s: capi.tpm_summaries_dev(ptrs, tot.data_ptr(), rows, L, gp, gm, len(PCTS), idx.data_ptr(), out.data_ptr(),
                                                          pct.data_ptr(), s.cuda_stream))
            r.update(rows=rows, chains=C, L=L, us_per_row=1000.0 * r["ms_median"] / rows)
            if label == "transcripts":
                r["sum_of_means"] = float(out[:rows].sum())
            res[f"{label}_C{C}"] = r
            print(json.dumps({f"{label}_C{C}": r}), flush=True)
        del x
    return res


def cli_times(s, tmp):
    path = os.path.join(tmp, "c2.hits")
    synth.write_hits_binary(s, path)
    binary = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
    res = {}
    for label, extra in (("plain", []), ("-tpm", ["-tpm"]), ("plain (again)", []), ("-tpm (again)", ["-tpm"])):
        t = time.perf_counter()
        r = subprocess.run([binary, "-notraces"] + extra + [path, os.path.join(tmp, "out")], capture_output=True, text=True)
        res[label] = dict(wall_s=time.perf_counter() - t, returncode=r.returncode,
                          stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith(("Gibbs", "EM", "Error"))])
        print(json.dumps({label: res[label]}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tpm.json"))
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    out = dict(gpu=card())
    s = synth.Synth(C2["seed"], C2["transcripts"], C2["fragments"])
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    gptr, gmem = [0], []
    for g in range(s.G):
        gmem += [int(h.hdr2col[t]) for t in range(int(s.gene_ptr[g]), int(s.gene_ptr[g + 1])) if h.hdr2col[t] >= 0]
        gptr.append(len(gmem))
    out["draw_totals"] = totals_time(h.n)
    print(json.dumps({"draw_totals": out["draw_totals"]}), flush=True)
    out["tpm_summaries"] = summaries_times(h.n, np.array(gptr, np.int64), np.array(gmem, np.int32))
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
