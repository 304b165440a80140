"""What the isoform-pair summaries cost on one B200 (mmseq -isocorr), written to profiles/isocorr.json with the card's
name and power limit read in the same call:
  - the C2 shape: Synth(SYNTH_SEED, 180000, 30M) in the collapsed layout, its gene CSR over the observed isoforms (header
    order), its pairs, the longest hit class and the largest gene;
  - device time (CUDA events, after a warm-up) of mmq_isocorr_summaries_dev at C = 1 and C = 4 chains of L = 1024
    log-normal draws (AR(1) in the log), with the bytes the kernels must move (each member's trace row once for the
    statistics, once per work item it belongs to for the tiles, and the three outputs) over that time and its share of
    the measured HBM peak;
  - the mmq_pair_shared_counts pass (host clock around the whole call, which ends in a stream synchronise; it includes
    the copy of the three per-transcript maps to the device) on the C2 hit classes;
  - the C2 `mmseq -notraces` wall time without and with -isocorr, alternated, two runs each, and the .isocorr file size.
   python tools/gpu_isocorr.py [--out profiles/isocorr.json] [--skip-cli]      (on the GPU box)"""
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
from tests import isocorr_reference as iref  # noqa: E402
from tools.gpu_chains import C2, card, draws  # noqa: E402
from tools.gpu_pool import event_ms  # noqa: E402
from tools.gpu_tpm import HBM_PEAK_GBS  # noqa: E402

TILE = 32  # MMQ_ISO_TILE


def member_loads(gptr):
    """trace rows the tile kernel stages: per gene of k >= 2, T = ceil(k / 32) tiles; tile t is loaded once on the
    diagonal and once with each of the other T - 1 tiles"""
    k = np.diff(gptr)
    k = k[k >= 2]
    return int(k.sum() + sum(int(kk) * (int(np.ceil(kk / TILE)) - 1) for kk in k)), int(sum(int(np.ceil(kk / TILE)) * (int(np.ceil(kk / TILE)) + 1) // 2 for kk in k))


def summaries_times(n, gptr, gmem, L=1024):
    gen = torch.Generator(device="cuda").manual_seed(4)
    kk = np.diff(gptr)
    base = np.concatenate([[0], np.cumsum(kk * (kk - 1) // 2)])[:-1].astype(np.int64)
    npairs = int((kk * (kk - 1) // 2).sum())
    ngenes, nmem = len(gptr) - 1, int(gptr[-1])
    loads, items = member_loads(gptr)
    d = [torch.from_numpy(v).cuda() for v in (gptr, gmem, base)]
    ws = torch.empty(capi.isocorr_workspace_bytes(ngenes, nmem), dtype=torch.uint8, device="cuda")
    out = torch.empty(3 * npairs, dtype=torch.float64, device="cuda")
    res = {}
    for C in (1, 4):
        x = draws(C, n, L, gen)
        ptrs = [x[c].data_ptr() for c in range(C)]
        r = event_ms(lambda st: capi.isocorr_summaries_dev(ptrs, ngenes, nmem, L, *[t.data_ptr() for t in d], npairs, out.data_ptr(),
                                                           ws.data_ptr(), st.cuda_stream))
        nbytes = 8 * C * L * (nmem + loads) + 24 * npairs
        gbs = nbytes / (r["ms_median"] * 1e-3) / 1e9
        r.update(chains=C, L=L, pairs=npairs, items=items, member_rows_staged=loads, bytes=nbytes, gb_per_s=gbs,
                 share_of_hbm_peak=gbs / HBM_PEAK_GBS, hbm_peak_gbs=HBM_PEAK_GBS, nan_pairs=int(torch.isnan(out[:npairs]).sum()))
        res[f"C{C}"] = r
        print(json.dumps({f"C{C}": r}), flush=True)
        del x
    return res


def shared_times(h, gptr, gmem, reps=5):
    gene_of, local_of = iref.gene_local(gptr, gmem, h.n)
    kk = np.diff(gptr)
    base = np.concatenate([[0], np.cumsum(kk * (kk - 1) // 2)])[:-1].astype(np.int64)
    npairs = int((kk * (kk - 1) // 2).sum())
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        H.pair_shared_counts(gene_of, local_of, base, npairs)               # warm-up
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            sh = H.pair_shared_counts(gene_of, local_of, base, npairs)
            t.append(1000.0 * (time.perf_counter() - t0))
    return dict(ms_median=float(np.median(t)), ms_min=float(min(t)), ms_max=float(max(t)), pairs=npairs,
                pairs_with_shared=int((sh > 0).sum()), shared_total=int(sh.sum()))


def cli_times(s, tmp):
    path = os.path.join(tmp, "c2.hits")
    s.write_hits_fast(path, binary=True)
    binary = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
    res = {}
    for label, extra in (("plain", []), ("-isocorr", ["-isocorr"]), ("plain (again)", []), ("-isocorr (again)", ["-isocorr"])):
        base = os.path.join(tmp, "out")
        t = time.perf_counter()
        r = subprocess.run([binary, "-notraces"] + extra + [path, base], capture_output=True, text=True)
        res[label] = dict(wall_s=time.perf_counter() - t, returncode=r.returncode,
                          stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith(("Gibbs", "EM", "Error", "Note"))])
        if extra:
            res[label]["isocorr_bytes"] = os.path.getsize(base + ".isocorr")
            os.remove(base + ".isocorr")
        print(json.dumps({label: res[label]}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "isocorr.json"))
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    out = dict(gpu=card())
    s = synth.Synth(C2["seed"], C2["transcripts"], C2["fragments"])
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    gptr, gmem = [0], []
    for g in range(s.G):
        gmem += [int(h.hdr2col[t]) for t in range(int(s.gene_ptr[g]), int(s.gene_ptr[g + 1])) if h.hdr2col[t] >= 0]
        gptr.append(len(gmem))
    gptr, gmem = np.array(gptr, np.int64), np.array(gmem, np.int32)
    kk = np.diff(gptr)
    out["shape"] = dict(transcripts=s.T, observed=h.n, hit_classes=h.m, fragments=s.N, genes=s.G,
                        genes_with_pairs=int((kk >= 2).sum()), largest_gene=int(kk.max()), pairs=int((kk * (kk - 1) // 2).sum()),
                        longest_hit_class=int(np.max(np.diff(h.row_ptr))), mean_hit_class=float(h.nnz / h.m))
    print(json.dumps({"shape": out["shape"]}), flush=True)
    out["isocorr_summaries"] = summaries_times(h.n, gptr, gmem)
    out["pair_shared_counts"] = shared_times(h, gptr, gmem)
    print(json.dumps({"pair_shared_counts": out["pair_shared_counts"]}), flush=True)
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
