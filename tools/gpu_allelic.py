"""What the allelic fraction costs on one B200 (mmseq -allelic), written to profiles/allelic.json with the card's name and
power limit read in the same call:
  - the C3 shape: Synth(SYNTH_SEED + 1, 360000, 30M, haplo=True), the sample of bench.py --haplo, in the collapsed layout;
    its longest hit class (the row that k_allele_only scans), its pairs and genes;
  - device time (CUDA events, after a warm-up) of mmq_allelic_summaries_dev for the pairs and for the genes, at C = 1 and
    C = 4 chains of L = 1024 log-normal draws, with the hit-less copies as prior rows, the five default percentiles;
  - the mmq_allele_only_counts pass for the pairs and for the genes (host clock around the whole call, which ends in a
    stream synchronise; it includes the copy of the unit map to the device);
  - the `mmseq -notraces` wall time at that shape without and with -allelic, alternated, two runs each.
   python tools/gpu_allelic.py [--out profiles/allelic.json] [--skip-cli]      (on the GPU box)"""
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
from tests import allelic_reference as aref  # noqa: E402
from tools.gpu_chains import card, draws  # noqa: E402
from tools.gpu_pool import event_ms  # noqa: E402

PCTS = (5, 25, 50, 75, 95)
C3 = dict(seed=20260101 + 2 + 1, transcripts=360000, fragments=30000000)   # bench.py --haplo: SYNTH_SEED + 1


def units(s, h):
    """the pairs (header copies 2p, 2p + 1 of one gene) and the genes, in column space: hit-less copies are prior rows"""
    col = np.asarray(h.hdr2col)
    hitless = np.flatnonzero(col < 0)
    ids = col.astype(np.int64).copy()
    ids[hitless] = h.n + np.arange(len(hitless))
    P = s.T // 2
    a_ids, b_ids = ids[0::2], ids[1::2]
    pair_gene = s.gene_of[0::2]
    genes = [[] for _ in range(s.G)]
    for p in range(P):
        genes[pair_gene[p]].append(p)
    levels = {"pairs": aref.csr([[p] for p in range(P)], a_ids, b_ids), "genes": aref.csr(genes, a_ids, b_ids)}
    maps = {}
    for name, nunits, unit in (("pairs", P, np.arange(s.T) // 2), ("genes", s.G, s.gene_of)):
        unit_of = np.full(h.n, -1, np.int32)
        side = np.zeros(h.n, np.uint8)
        obs = col >= 0
        unit_of[col[obs]] = unit[obs]
        side[col[obs]] = (np.arange(s.T) % 2)[obs]
        maps[name] = (unit_of, side, nunits)
    return levels, maps, len(hitless)


def summaries_times(n, nprior, levels, L=1024):
    gen = torch.Generator(device="cuda").manual_seed(4)
    res = {}
    for C in (1, 4):
        x = draws(C, n, L, gen)
        pri = draws(C, max(nprior, 1), L, gen)
        ptrs = [x[c].data_ptr() for c in range(C)]
        pptrs = [pri[c].data_ptr() for c in range(C)]
        idx = torch.from_numpy(aref.pct_index(PCTS, C * L)).cuda()
        for label, (a_ptr, a_mem, b_ptr, b_mem) in levels.items():
            rows = len(a_ptr) - 1
            d = [torch.from_numpy(v).cuda() for v in (a_ptr, a_mem, b_ptr, b_mem)]
            out = torch.empty(3 * rows, dtype=torch.float64, device="cuda")
            pct = torch.empty(rows * len(PCTS), dtype=torch.float64, device="cuda")
            r = event_ms(lambda st: capi.allelic_summaries_dev(ptrs, pptrs, n, nprior, rows, L, *[t.data_ptr() for t in d], len(PCTS),
                                                               idx.data_ptr(), out.data_ptr(), pct.data_ptr(), st.cuda_stream))
            r.update(rows=rows, chains=C, L=L, us_per_row=1000.0 * r["ms_median"] / rows, members_per_side=len(a_mem) / rows,
                     nan_rows=int(torch.isnan(out[:rows]).sum()))
            res[f"{label}_C{C}"] = r
            print(json.dumps({f"{label}_C{C}": r}), flush=True)
        del x, pri
    return res


def allele_only_times(h, maps, reps=5):
    res = {}
    with capi.Handle(h.row_ptr, h.col, h.k, h.len) as H:
        for label, (unit_of, side, nunits) in maps.items():
            H.allele_only_counts(unit_of, side, nunits)                     # warm-up
            t = []
            for _ in range(reps):
                t0 = time.perf_counter()
                a, b = H.allele_only_counts(unit_of, side, nunits)
                t.append(1000.0 * (time.perf_counter() - t0))
            res[label] = dict(ms_median=float(np.median(t)), ms_min=float(min(t)), ms_max=float(max(t)), units=nunits,
                              a_only_total=int(a.sum()), b_only_total=int(b.sum()))
            print(json.dumps({label: res[label]}), flush=True)
    return res


def cli_times(s, tmp):
    path = os.path.join(tmp, "c3.hits")
    s.write_hits_fast(path, binary=True)
    binary = os.path.join(ROOT, "mmseq_b200", "bin", "mmseq")
    res = {}
    for label, extra in (("plain", []), ("-allelic", ["-allelic"]), ("plain (again)", []), ("-allelic (again)", ["-allelic"])):
        t = time.perf_counter()
        r = subprocess.run([binary, "-notraces"] + extra + [path, os.path.join(tmp, "out")], capture_output=True, text=True)
        res[label] = dict(wall_s=time.perf_counter() - t, returncode=r.returncode,
                          stderr_tail=[ln for ln in r.stderr.splitlines() if ln.startswith(("Gibbs", "EM", "Error", "Note"))])
        print(json.dumps({label: res[label]}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "allelic.json"))
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    out = dict(gpu=card())
    s = synth.Synth(C3["seed"], C3["transcripts"], C3["fragments"], haplo=True)
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    levels, maps, nprior = units(s, h)
    out["shape"] = dict(transcripts=s.T, observed=h.n, hit_classes=h.m, fragments=s.N, pairs=s.T // 2, genes=s.G, prior_rows=nprior,
                        longest_hit_class=int(np.max(np.diff(h.row_ptr))), mean_hit_class=float(h.nnz / h.m))
    print(json.dumps({"shape": out["shape"]}), flush=True)
    out["allelic_summaries"] = summaries_times(h.n, nprior, levels)
    out["allele_only_counts"] = allele_only_times(h, maps)
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
