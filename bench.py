#!/usr/bin/env python
"""bench.py — Gibbs sweep throughput of the mmseq hot path on B200, with its correctness gates.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload "C2-collapsed"): BASELINE.json configs[1] — a synthetic Ensembl-sized
sample, 180k transcripts / 30M paired fragments per GPU, in the REFERENCE'S OWN REPRESENTATION:
distinct hit classes with fragment counts k (src/mmseq.cpp:395-441), what the `mmseq` host
program feeds the GPU.  Both arms (ours and `--impl reference`) run the same sample in the same
representation, so value = distinct hit classes x sweeps/s is an equal-work number.

A "step" is SWEEPS_PER_STEP (= 16, the reference's trace stride, src/mmseq.cpp:192) full Gibbs
sweeps — allocation of every hit class, [count exchange when N > 1], Gamma update of every
transcript — with one trace capture per step, issued through mmq_gibbs exactly as the host program
does (CUDA graph of 16 sweeps).  Weak scaling: every rank holds its own 30M-fragment shard of the
same transcriptome.  `--scaling strong --fragments-total F` splits ONE sample of F fragments over
the ranks (config 4: `--weights --layout perfragment --fragments-total 200000000`).

After the timed region every rank runs the correctness gates of SURVEY.md section 8(d) at the
benchmark shape and rank 0 prints them in the JSON line ("gates"); a failed gate exits non-zero:
  (a) >= 3 sweeps of mmq_sweep_debug on the full shard: counts and mu bit for bit against the CPU
      replay on the shared Philox stream (every rank replays its shard, the integer counts are
      summed over ranks), and the X matrix of one sweep entry by entry;
  (b) EM: |mu_gpu / mu_oracle - 1| <= 1e-6 and equal iteration count;
  (c) N = 1: posterior mean of log mu against the reference-like GSL chain (MT19937, GSL samplers)
      within 4 Monte-Carlo standard errors (batch means) for >= 99.9 % of the transcripts, or for no
      fewer than the GPU chain against itself; posterior sd ratio within 5 %.

`--impl reference` times the reference's own algorithm and data flow on ALL host cores (oracle/:
MT19937 per OpenMP thread, GSL-style samplers, dense per-thread partials; the reference itself
needs Boost + GSL and cannot be built here), on the same N shards' worth of work.
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SWEEPS_PER_STEP = 16
SEED = 1234
SYNTH_SEED = 20260101 + 2
T_C2 = 180_000
N_C2 = 30_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--transcripts", type=int, default=T_C2)
    ap.add_argument("--fragments", type=int, default=N_C2, help="fragments per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--fragments-total", type=int, default=0, help="strong scaling: fragments of the one sample that is split over the ranks")
    ap.add_argument("--layout", default="collapsed", choices=["collapsed", "perfragment"],
                    help="collapsed = distinct classes + counts (reference semantics, default); perfragment = one row per fragment "
                         "(the only layout that can carry per-hit weights)")
    ap.add_argument("--weights", action="store_true", help="fp32 per-hit weights (config 4's extension); implies --layout perfragment")
    ap.add_argument("--haplo", action="store_true", help="config 3: haplotype-specific transcriptome (360k haplo-transcripts, deep multi-mapping)")
    ap.add_argument("--transposed", action="store_true", help="materialise X + atomic-free transposed reduction")
    ap.add_argument("--cpu-sweeps", type=int, default=768, help="most sweeps of the CPU baseline / posterior-gate chain (rank 0, N = 1)")
    ap.add_argument("--cpu-seconds", type=float, default=30.0, help="... and its time budget (at least 16 trace samples are taken)")
    ap.add_argument("--nccl-only", action="store_true", help="N > 1: exchange counts with ncclAllReduce instead of the fused peer-memory kernel")
    ap.add_argument("--p2p-rs", action="store_true", help="N > 1: reduce-scatter / all-gather variant of the fused exchange (mmq_tune knob 6)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gates", action="store_true")
    ap.add_argument("--cov-features", type=int, default=16384, help="features (columns) of the trace-covariance extra (mmcollapse candidates of one sample)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra lines (weighted per-fragment stream of the same sample)")
    ap.add_argument("--gate-sweeps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="config 5: this many independent C2-sized samples (own synthetic fragments, own chain) dealt to "
                                                         "the GPUs, each through load -> EM -> --batch-sweeps Gibbs sweeps -> Sokal summaries; reports samples/s")
    ap.add_argument("--batch-per-gpu", type=int, default=4, help="samples in flight per GPU")
    ap.add_argument("--batch-sweeps", type=int, default=16384, help="Gibbs sweeps per sample (the reference's default -gibbs_iter)")
    ap.add_argument("--batch-out", default="/tmp/mmq_batch", help="directory of the per-sample summary tables")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float64; rank 0): mu.npy, and trace_last_step.npy, the trace slot it recorded")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.batch > 0):
        ap.error("--dump-outputs writes the outputs of the timed Gibbs steps on the GPU: not with --impl reference or --batch")
    if args.weights:
        args.layout = "perfragment"
    return args


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def host_threads():
    """Host cores this process may use — NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def fragments_of(args, rank, world):
    """(fragments of this rank's shard, fragments of the whole job)."""
    if args.scaling == "strong":
        tot = args.fragments_total or args.fragments
        lo, hi = tot * rank // world, tot * (rank + 1) // world
        return hi - lo, tot
    return args.fragments, args.fragments * world


class Workload:
    pass


def make_workload(args, rank, world, weights=None, layout=None):
    """This rank's shard: its own fragments of the shared transcriptome; columns = header indices when world > 1
    (one column space across shards), header order otherwise."""
    from mmseq_b200 import hostlib, synth
    weights = args.weights if weights is None else weights
    layout = layout or args.layout
    nfrag, ntot = fragments_of(args, rank, world)
    t0 = time.time()
    s = synth.Synth(SYNTH_SEED + (1 if args.haplo else 0), args.transcripts * (2 if args.haplo else 1), nfrag, haplo=args.haplo,
                    weights=weights, frag_seed=rank, threads=max(1, host_threads() // max(1, world)))   # not OMP_NUM_THREADS (1 under torchrun)
    t1 = time.time()
    lay = hostlib.LAYOUT_COLLAPSED if layout == "collapsed" else hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH
    lay |= hostlib.LAYOUT_IDENTITY_COLUMNS if world > 1 else hostlib.LAYOUT_HEADER_ORDER_COLUMNS
    h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w if weights else None, layout=lay)
    t2 = time.time()
    w = Workload()
    w.s, w.h, w.layout, w.weights = s, h, layout, weights
    w.length = s.efflen[h.col2hdr] * ntot / 1e9   # l[t] = efflen * N_total / 1e9 over the whole job's sample, src/mmseq.cpp:603
    w.cid_base = rank * (1 << 28)                  # Philox counters of the shards do not overlap
    w.nfrag, w.ntot = nfrag, ntot
    w.prep = dict(gen_s=round(t1 - t0, 2), load_s=round(t2 - t1, 2))
    return w


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of one GPU, sampled while the timed region runs.  NVML is brought up in the constructor
    (before the region: its initialisation takes longer than the 36 ms a default run is timed for) and a last sample is
    taken when the region ends, so that there is always at least one."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm = []
        self.reasons = set()
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.dev = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.dev, nv.NVML_CLOCK_SM)
            self.names = {
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            self.get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def sample(self):
        self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM))
        r = self.get(self.dev)
        for bit, nm in self.names.items():
            if r & bit:
                self.reasons.add(nm)

    def run(self):
        if not self.ok:
            return
        try:
            while not self.stop_flag:
                self.sample()
                time.sleep(0.004)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def result(self):
        if self.ok:
            try:
                self.sample()   # the region has just ended: the clocks are still those it ran at
            except Exception:  # pragma: no cover
                pass
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


def algorithmic_bytes(h, n, weights, transposed, stride, layout, cls=None, rows=None):
    """Compulsory HBM bytes of the implemented data flow (DESIGN.md, 'Roofline'); every array once, L2-resident mu
    gathers and count reductions not counted.  Returns (allocation launch, whole sweep)."""
    m, nnz = h.m, h.nnz
    d = np.diff(h.row_ptr)
    per_entry = 4 + (4 if weights else 0)
    if rows and rows.get("in_use") and not transposed:
        # row plan (mmq_rows.cu): columns once per distinct class, weights once per fragment, 16 B of run marks per 128 rows
        alloc = rows["bytes_per_sweep"]
    elif cls and cls["in_use"] and not transposed:
        # class plan (mmq_cls.cu): packed columns (4 B) + draws (2 B) + class id (4 B) per slot of the small set; the same
        # with a 4-byte count for the chain set, 8 B per chunk descriptor; row pointer, k, class id (8 + 4 + 8 B) per class
        # and 4 B per entry of the sub-CSR left to k_alloc
        alloc = (4 * cls["packed_slots"] + 6 * cls["class_slots"] + cls["class_slots"] // 4 + 4 * cls["chain_slots"]
                 + 8 * ((cls["chain_classes"] + 31) // 32 * 32) + 20 * cls["rest_classes"] + 4 * cls["rest_nnz"])
    elif layout == "perfragment" and h.k is None and not transposed:
        alloc = per_entry * int(d[d >= 2].sum())
    else:
        alloc = 8 * (m + 1) + per_entry * nnz + (4 * m if h.k is not None else 0)
    if transposed:
        alloc += 4 * nnz
    reduce_ = (8 * nnz + 8 * (n + 1) + 4 * n) if transposed else 0
    gamma = n * (4 + 4 + 8 + 8) + (8 * n) // stride
    return int(alloc), int(alloc + reduce_ + gamma)


def workload_name(args, layout=None, weights=None):
    layout = layout or args.layout
    weights = args.weights if weights is None else weights
    base = "C3-haplotype-" if args.haplo else ("C4-" if (args.scaling == "strong" and weights) else "C2-")
    return base + layout + ("-weighted" if weights else "")


def workload_config(args, world, totals):
    """Identical in both arms (ours / reference) for the same command line."""
    nfrag, ntot = fragments_of(args, 0, world)
    return {
        "workload": workload_name(args), "transcripts": args.transcripts * (2 if args.haplo else 1),
        "fragments_per_gpu": int(nfrag), "fragments_total": int(ntot),
        "representation": "distinct hit classes with fragment counts k (src/mmseq.cpp:395-441)" if args.layout == "collapsed"
                          else "one row per fragment (k == 1)" + (", fp32 per-hit weights" if args.weights else ""),
        "n_columns": int(totals["n"]), "hit_classes_total": int(totals["m"]), "nnz_total": int(totals["nnz"]),
        "trace_stride": SWEEPS_PER_STEP, "seed": SEED, "scaling": args.scaling,
        "l2": "inputs_exceed_l2" if totals["nnz"] / world * 4 > 200e6 else "inputs_near_l2_size_flush_between_steps",
    }


def value_classes(args, w):
    """Hit classes of a shard as the metric counts them: DISTINCT transcript sets (the reference's definition of a hit
    class, src/mmseq.cpp:395-441) whatever the layout — a per-fragment shard has the same classes as its collapsed form."""
    return int(w.h.n_classes)


# ----------------------------------------------------------------------------- reference arm

def union_problem(args, world):
    """The N shards of the weak-scaling job (or the one sample of a strong-scaling job) as one problem: what a
    single CPU box has to sweep to do the same work."""
    from oracle import oracle as orc
    if args.scaling == "strong":
        sav = (args.fragments, args.scaling)
        args.fragments, args.scaling = (args.fragments_total or args.fragments), "weak"
        w = make_workload(args, 0, 1)
        args.fragments, args.scaling = sav
        return [w], orc.Problem(w.h.row_ptr, w.h.col, w.h.k, w.length, weight=w.h.w), w.h.n
    ws = [make_workload(args, r, world) for r in range(world)]
    if world == 1:
        w = ws[0]
        return ws, orc.Problem(w.h.row_ptr, w.h.col, w.h.k, w.length, weight=w.h.w), w.h.n
    n = ws[0].h.n
    rp = [np.zeros(1, np.int64)]
    off = 0
    for w in ws:
        assert w.h.n == n
        rp.append(w.h.row_ptr[1:] + off)
        off += w.h.nnz
    k = None if ws[0].h.k is None else np.concatenate([w.h.k for w in ws])
    P = orc.Problem(np.concatenate(rp), np.concatenate([w.h.col for w in ws]), k, ws[0].length)
    return ws, P, n


def run_reference(args, rank, world):
    """The reference's algorithm on the host cores (oracle/ port): the same job — all N shards — in the same
    (collapsed) representation, on every host core of the box."""
    if rank != 0:
        return
    if args.weights:
        print(json.dumps({"impl": "reference", "unavailable": "the reference has no per-hit weights (M is boolean, src/mmseq.cpp:72); "
                          "config 4's weighted stream has no CPU reference arm"}), flush=True)
        return
    ws, P, n = union_problem(args, world)
    totals = {"n": n, "m": sum(value_classes(args, w) for w in ws), "nnz": P.nnz}
    mu, _, _ = P.init_mu()
    threads = host_threads()
    mu, _, _ = P.gibbs_gsl(mu, SEED, max(1, args.warmup), threads=threads)  # warm-up sweeps
    secs = []
    for _ in range(args.steps):
        mu, _, sec = P.gibbs_gsl(mu, SEED, 1, threads=threads)  # one step of the reference arm = ONE sweep (bounded sample)
        secs.append(sec)
    tot = float(np.sum(secs))
    sweeps_per_s = args.steps / tot
    value = sweeps_per_s * totals["m"]
    line = {
        "impl": "reference", "metric": "gibbs_hit_class_allocations_per_s", "value": value, "unit": "allocations/s",
        "sweeps_per_s": sweeps_per_s, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * tot / args.steps, "sweeps_per_step": 1, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, world, totals),
        "cpu_baseline": {"value": value, "unit": "allocations/s", "sweeps_per_s": sweeps_per_s, "cores": threads, "kind": "port",
                         "layout": args.layout,
                         "sample": f"{args.steps} full sweeps (1 per step) over all {totals['m']} hit classes of the {world} shard(s)"},
        "e2e": {"value": value, "unit": "allocations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "oracle port of src/mmseq.cpp:851-918 (MT19937 per OpenMP thread, GSL-style samplers, dense per-thread partials) on "
                f"{threads} host threads; the denominator depends on the box's core count. The reference's own main() builds here only "
                "against the stand-in Boost/GSL of oracle/shim and needs minutes per sweep at this size (DESIGN.md section 9)",
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- gates

def run_gates(args, H, w, mu0_gpu, mu_em_gpu, em_iters_gpu, rank, world, dev, allreduce):
    """Correctness gates at the benchmark shape (SURVEY.md 8d).  `allreduce(np array) -> np array` sums over ranks.
    Returns the dict printed as "gates" (rank 0) — every rank computes the same verdict."""
    from mmseq_b200 import capi
    from oracle import oracle as orc
    h = w.h
    P = orc.Problem(h.row_ptr, h.col, h.k, w.length, weight=h.w)
    threads = max(1, host_threads() // max(1, world if world <= 8 else 8))
    g = {"shape": f"{h.m} rows / {h.nnz} entries per rank, {world} rank(s)"}
    t0 = time.time()
    # initial mu (src/mmseq.cpp:617-638): every shard's sum of k/|i|, summed over the ranks, over l
    mu0, _, _ = P.init_mu()
    if world > 1:
        mu0 = allreduce(mu0 * w.length) / w.length
    pos0 = mu0 > 0   # with several shards the columns are all header transcripts: those without hits start (and stay) at 0
    rel0 = float(np.max(np.abs(mu0_gpu[pos0] / mu0[pos0] - 1.0))) if np.array_equal(mu0_gpu[~pos0], mu0[~pos0]) else float("inf")
    g["init_mu"] = {"max_rel_err": rel0, "tol": 1e-9, "ok": bool(rel0 <= 1e-9)}   # fp64 sums of up to 1e8 terms in different orders
    # (b) EM from the same start: oracle iteration split over the shards (orc_em_partial = one shard's part of src/mmseq.cpp:781-802).
    # Shards above 60M entries (config 4): the first 8 iterations only (an oracle iteration is a pass over the shard on the host)
    bounded = h.nnz > 60_000_000
    if bounded:
        H.set_mu(mu0_gpu)
        em_iters_gpu, _, _ = H.em(8, -1e300)
        mu_em_gpu = H.get_mu()
    mu = mu0_gpu.copy()
    acc, ll = P.em_partial(mu, threads)
    loglik = float(allreduce(np.array([ll]))[0]) - float((mu * w.length).sum())
    llr, it = 1.1, 0
    while it < (8 if bounded else 1000) and (bounded or llr > 0.1):
        acc = allreduce(P.em_partial(mu, threads)[0])
        mu2 = mu * acc / w.length
        ll2 = float(allreduce(np.array([P.em_partial(mu2, threads)[1]]))[0]) - float((mu2 * w.length).sum())
        llr, loglik, mu = ll2 - loglik, ll2, mu2
        it += 1
    pos = mu > 0   # transcripts whose classes all lost their mass stay at exactly 0 on both sides
    rel = float(np.max(np.abs(mu_em_gpu[pos] / mu[pos] - 1.0))) if pos.any() else 0.0
    if not np.array_equal(mu_em_gpu[~pos], mu[~pos]):
        rel = float("inf")
    g["em"] = {"iters_gpu": int(em_iters_gpu), "iters_oracle": int(it), "max_rel_err": rel, "tol": 1e-6,
               "mode": "first 8 iterations (shard above 60M entries)" if bounded else "to convergence (epsilon 0.1)",
               "ok": bool(it == em_iters_gpu and rel <= 1e-6)}
    g["em_s"] = round(time.time() - t0, 2)
    # (a) bit-exact sweeps from the EM estimate
    t0 = time.time()
    H.set_mu(mu)
    cur = mu.copy()
    ok_counts = ok_mu = True
    base_sweep = 900000
    for s in range(args.gate_sweeps):
        _, c_gpu, mu_gpu = H.sweep_debug(SEED, base_sweep + s, capi.MMQ_GIBBS_DEFAULT, want_x=False)
        c_cpu = allreduce(P.sweep_counts(cur, SEED, base_sweep + s, class_id_base=w.cid_base, threads=threads).astype(np.int64)).astype(np.int32)
        mu_cpu = P.gamma_replay(c_cpu, SEED, base_sweep + s)
        ok_counts &= bool(np.array_equal(c_gpu, c_cpu))
        ok_mu &= bool(np.array_equal(mu_gpu, mu_cpu))
        cur = mu_cpu
        H.set_mu(cur)
    sha = hashlib.sha256(H.get_mu().tobytes()).hexdigest()[:16]
    g["sweeps"] = {"n": args.gate_sweeps, "counts_bit_exact": ok_counts, "mu_bit_exact": ok_mu, "mu_sha256_16": sha,
                   "fragments_conserved": bool(int(c_gpu.astype(np.int64).sum()) == int(allreduce(np.array([float(w.nfrag)]))[0]))}
    # X of one sweep, entry by entry (the X-materialising kernel + transposed reduction): own shard vs own replay
    ok_x = True
    if h.nnz <= 150_000_000:
        x_cpu, _, _ = P.sweep_replay(cur, SEED, base_sweep + 100, class_id_base=w.cid_base, do_gamma=False)
        x_gpu, c2, _ = H.sweep_debug(SEED, base_sweep + 100, capi.MMQ_GIBBS_TRANSPOSED)
        ok_x = bool(np.array_equal(x_gpu, x_cpu))
    ok_all = allreduce(np.array([float(ok_x), float(ok_counts), float(ok_mu)]))
    g["sweeps"]["x_bit_exact"] = bool(ok_all[0] == world) if h.nnz <= 150_000_000 else "skipped (shard above 150M entries)"
    g["sweeps"]["ok"] = bool(ok_all.min() == world and g["sweeps"]["fragments_conserved"])
    g["sweeps_s"] = round(time.time() - t0, 2)
    g["ok"] = bool(g["init_mu"]["ok"] and g["em"]["ok"] and g["sweeps"]["ok"])
    g["mu_em"] = mu
    return g


def posterior_gate(args, H, w, mu_em, cpu_sweeps, threads):
    """(c) posterior mean and sd of log mu: GPU chain vs the reference-like GSL chain on the host cores; also the CPU
    baseline (the same run is timed).  N = 1 only.

    Both chains start at the EM estimate, burn 16 sweeps, and then record EVERY sweep of a window of W sweeps; the statistic
    compared per transcript is the mean of log mu over that window.  Its Monte-Carlo standard error is estimated by batch
    means: the GPU chain runs on for NW more windows of the same length and the variance of their means is the sampling
    variance of exactly that statistic (no autocorrelation-time estimate, no normality of single draws needed).
    z = (mean_cpu - mean_gpu_window0) / sqrt(2 var_w).  The same estimator between two of the GPU chain's own windows gives
    the null distribution of z: with posteriors this skewed / slowly mixing (30 % of the transcripts have no fragments of
    their own) even the chain against itself leaves ~0.2 % of the transcripts beyond 4 standard errors, so the gate is
    "99.9 % within 4 se, or no worse than the chain against itself" together with the clipped rms of z."""
    from oracle import oracle as orc
    h = w.h
    P = orc.Problem(h.row_ptr, h.col, h.k, w.length)
    S = SWEEPS_PER_STEP
    burn = S
    W = 64
    while W * 2 <= min(max(cpu_sweeps, 64), 2048):
        W *= 2                                                  # a power of two: the device summaries (Sokal) need it
    NW = 32
    mu_c, _, _ = P.gibbs_gsl(mu_em, SEED, burn, threads=threads)
    mu_c, tr_c, t_cpu = P.gibbs_gsl(mu_c, SEED + 1, W, stride=1, trace_len=W, threads=threads)
    cpu_sps = W / t_cpu
    with np.errstate(divide="ignore"):
        lc = np.log(tr_c)
    del tr_c
    mean_c = lc.mean(axis=1)
    sd_c = lc.std(axis=1, ddof=1)
    del lc
    H.set_mu(mu_em)
    H.gibbs(SEED + 7, 0, burn, stride=S, trace_len=0)           # burn-in (its own stream of sweeps)
    means, variances = [], []
    for j in range(NW + 3):                                     # window 0 pairs with the CPU window, 1 and 2 make the null pair
        H.gibbs(SEED + 100 + j, 0, W, stride=1, trace_len=W)
        Sg = H.summarize(0)
        means.append(Sg["log_mean"].copy())
        variances.append(Sg["var"].copy())
    G = np.stack(means[3:])
    var_w = G.var(axis=0, ddof=1)
    se = np.sqrt(2.0 * var_w)
    with np.errstate(all="ignore"):
        z = np.abs(mean_c - means[0]) / se
        z0 = np.abs(means[1] - means[2]) / se
    finite = np.isfinite(z) & np.isfinite(z0) & (se > 0)
    z, z0 = z[finite], z0[finite]
    frac, frac0 = float((z <= 4.0).mean()), float((z0 <= 4.0).mean())
    rms, rms0 = float(np.sqrt(np.mean(np.minimum(z, 6.0) ** 2))), float(np.sqrt(np.mean(np.minimum(z0, 6.0) ** 2)))
    sd_g = np.sqrt(np.mean(np.stack(variances[1:]), axis=0))
    with np.errstate(all="ignore"):
        sd_ratio = float(np.median((sd_c / sd_g)[finite]))
    ok = bool((frac >= 0.999 or frac >= frac0 - 5e-4) and rms <= 1.05 * rms0 and abs(sd_ratio - 1.0) < 0.05)
    gate = {"chains": f"GPU and CPU (GSL-like, {threads} threads) chains from the EM estimate, {burn} burn-in sweeps, mean of log mu over the same "
                      f"window of {W} consecutive sweeps; standard error by batch means over {NW} further GPU windows",
            "frac_within_4se": frac, "need": 0.999, "self_frac_within_4se": frac0,
            "rms_z_clipped": rms, "self_rms_z_clipped": rms0, "median_sd_ratio_cpu_over_gpu": sd_ratio, "features": int(finite.sum()),
            "rule": "frac >= 0.999 or frac >= self_frac - 5e-4 (the GPU chain against itself, same estimator); rms_z <= 1.05 self_rms_z; |sd ratio - 1| < 0.05",
            "ok": ok, "hard_fail_below": 0.99}
    base = {"value": cpu_sps * value_classes(args, w), "unit": "allocations/s", "sweeps_per_s": cpu_sps, "cores": threads, "kind": "port",
            "layout": w.layout, "sample": f"{W} full sweeps of the same shard (collapsed representation) after {burn} warm-up sweeps"}
    return gate, base


# ----------------------------------------------------------------------------- ours

def timed_run(args, H, w, stream, dev, barrier, K, W, flush_buf, flags, outputs=None):
    """W warm-up steps, K timed steps through mmq_gibbs (the production launch path), then the same K steps once more
    with per-launch events for the kernel shares.  Returns (ms, alloc_ms, alloc_n, gamma_ms, gamma_n, launches, clocks).
    `outputs` (a dict): receives what a caller of the timed steps reads back after the last one, before the repetition."""
    import torch
    from mmseq_b200 import capi
    S = SWEEPS_PER_STEP
    L = 2 * K + W + 1
    sweep = 0

    def step(fl):
        nonlocal sweep
        if flush_buf is not None:
            with torch.cuda.stream(stream):
                flush_buf.zero_()
        H.gibbs(SEED, sweep, S, stride=S, trace_len=L, flags=fl)
        sweep += S

    for _ in range(W):
        step(flags)
    H.synchronize()
    launches0 = capi.launch_count()
    sampler = ClockSampler(physical_gpu_index(dev.index))
    barrier()
    sampler.start()
    # one event pair per step: the L2 flush between steps (collapsed shards are about the size of the L2) is outside
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in evs:
        if flush_buf is not None:
            with torch.cuda.stream(stream):
                flush_buf.zero_()
        a.record(stream)
        H.gibbs(SEED, sweep, S, stride=S, trace_len=L, flags=flags)
        b.record(stream)
        sweep += S
    H.synchronize()
    barrier()
    sampler.stop_flag = True
    sampler.join()
    launches = capi.launch_count() - launches0
    ms = float(sum(a.elapsed_time(b) for a, b in evs))
    if outputs is not None:
        outputs["mu"] = H.get_mu()
        outputs["trace_last_step"] = H.get_trace()[:, W + K - 1]   # step j stores its first sweep's mu into slot j
    H.kernel_times()   # drop anything pending
    for _ in range(K):
        step(flags | capi.MMQ_GIBBS_TIME_KERNELS)
    alloc_ms, alloc_n, gamma_ms, gamma_n = H.kernel_times()
    return ms, alloc_ms, alloc_n, gamma_ms, gamma_n, launches, sampler.result()


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Each array (one row per transcript) as path/<name>.npy in float64.  Above DUMP_BYTES in all, every array keeps the
    same fixed, seeded sample of rows: two builds run with the same arguments still compare output for output."""
    os.makedirs(path, exist_ok=True)
    arrays = {name: np.asarray(a, np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    rows = None
    if total > DUMP_BYTES:
        n = len(next(iter(arrays.values())))
        rows = np.sort(np.random.default_rng(SEED).choice(n, n * DUMP_BYTES // total, replace=False))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a if rows is None else a[rows])


def extra_weighted_line(args, dev, stream, peak):
    """The same sample one row per fragment with fp32 per-hit weights (config 4's stream: the only compulsory
    per-fragment traffic), device-timed, with its own roofline."""
    import torch
    from mmseq_b200 import capi
    w = make_workload(args, 0, 1, weights=True, layout="perfragment")
    h = w.h
    H = capi.Handle(h.row_ptr, h.col, None, w.length, weight=h.w, device=dev.index)
    H.set_stream(stream.cuda_stream)
    H.init_mu()
    rows = None   # the row plan (MMQ_GIBBS_ROWS_KERNEL) is not the default: measured no faster than the segment kernel
    barrier = lambda: torch.cuda.synchronize()
    ms, alloc_ms, alloc_n, gamma_ms, gamma_n, launches, clocks = timed_run(args, H, w, stream, dev, barrier, 5, 3, None, capi.MMQ_GIBBS_DEFAULT)
    H.close()
    b_alloc, _ = algorithmic_bytes(h, h.n, True, False, SWEEPS_PER_STEP, "perfragment", rows=rows)
    a = alloc_ms / max(alloc_n, 1)
    return {"workload": workload_name(args, "perfragment", True), "rows": int(h.m), "nnz": int(h.nnz),
            "kernel": "k_alloc_rows" if rows and rows.get("in_use") else "k_alloc_seg4",
            "sweeps_per_s": 5 * SWEEPS_PER_STEP / (ms / 1e3), "alloc_avg_launch_ms": a, "gamma_avg_launch_ms": gamma_ms / max(gamma_n, 1),
            "algorithmic_bytes_per_launch": b_alloc,
            "roofline": {"bound": "hbm", "achieved": b_alloc / (a * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": b_alloc / (a * 1e-3) / 1e9 / peak}, "plan": rows}


def extra_trace_cov(args, dev, stream):
    """SURVEY.md section 8 row f3 (src/mmcollapse.cpp:553-558): cov() of one sample's 1024 x C trace matrix on the tensor
    cores (mmq_trace_cov_dev), device-timed on device-resident traces, with its own roofline (bound: tensor), a gate against
    the oracle on a sub-block, the end-to-end time through the host-pointer entry point and the oracle timed beside it."""
    import torch
    from mmseq_b200 import capi
    from oracle import oracle as orc
    L, C, nsplit = 1024, args.cov_features, 2
    g = torch.Generator(device=dev); g.manual_seed(20260107)
    # posterior-trace-like columns: log-normal levels over orders of magnitude, neighbouring features anti-correlated
    base = torch.randn((C // 2, L), dtype=torch.float64, device=dev, generator=g)
    noise = torch.randn((C, L), dtype=torch.float64, device=dev, generator=g)
    level = torch.exp(3.0 * torch.randn((C, 1), dtype=torch.float64, device=dev, generator=g))
    sign = torch.tensor([1.0, -1.0], dtype=torch.float64, device=dev).repeat(C // 2).view(C, 1)
    Md = level * torch.exp(0.3 * (sign * base.repeat_interleave(2, dim=0) + 0.5 * noise))     # [C][L]: column c of the L x C matrix
    del base, noise
    Rd = torch.empty((C, C), dtype=torch.float64, device=dev)
    ws = torch.empty(capi.trace_cov_workspace_bytes(L, C, nsplit), dtype=torch.uint8, device=dev)
    K, W = 10, 3
    with torch.cuda.stream(stream):
        for _ in range(W):
            capi.trace_cov_dev(Md.data_ptr(), L, C, nsplit, Rd.data_ptr(), ws.data_ptr(), stream.cuda_stream)
        stream.synchronize()
        l0 = capi.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):   # 2.1 GB of output per launch: far larger than the L2
            capi.trace_cov_dev(Md.data_ptr(), L, C, nsplit, Rd.data_ptr(), ws.data_ptr(), stream.cuda_stream)
        e1.record(stream)
        stream.synchronize()
    ms = e0.elapsed_time(e1) / K
    launches = capi.launch_count() - l0
    nterms = nsplit * (nsplit + 1) // 2
    flops = float(C) * (C + 1) * L * nterms         # the upper triangle, one multiply-add per split product
    out_bytes = float(C) * C * 8
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tpeak = float(peaks.get("bf16_tflops", 1590.0))
    # gate: a 1024 x 1024 corner against the oracle, in correlation units
    nsub = min(C, 1024)
    sub = Rd[:nsub, :nsub].cpu().numpy()
    ref = orc.trace_cov(Md[:nsub].cpu().numpy().T)
    d = np.sqrt(np.diag(ref))
    err = float(np.max(np.abs(sub - ref) / (d[:, None] * d[None, :])))
    sym = bool(torch.equal(Rd[:2048, :2048], Rd[:2048, :2048].T))
    # CPU beside it: the oracle on a bounded sample of the same matrix
    ccpu = min(C, 3072)
    Mh = Md[:ccpu].cpu().numpy().T.copy()
    t0 = time.perf_counter()
    orc.trace_cov(Mh)
    cpu_s = time.perf_counter() - t0
    cpu_full_s = cpu_s * (float(C) * (C + 1)) / (float(ccpu) * (ccpu + 1))
    # end to end: host matrix in, host matrix out (pageable R: 2.1 GB over PCIe dominates)
    Mhost = np.asfortranarray(Md.cpu().numpy().T)
    del Md, Rd, ws
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    Rh = capi.trace_cov(Mhost, nsplit=nsplit, device=dev.index)
    e2e_s = time.perf_counter() - t0
    return {"workload": f"cov() of a {L} x {C} trace matrix (src/mmcollapse.cpp:553-558), split-bf16 x {nsplit} products, fp32 accumulation, fp64 output",
            "kernel": "k_cov_gemm2 (tcgen05.mma.cta_group::2 on CTA pairs + 2-CTA TMA + TMEM, persistent, 256 x 256 tiles of the upper triangle per pair) + k_cov_prep",
            "ms": ms, "matrices_per_s": 1e3 / ms, "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                         "frac": flops / (ms * 1e-3) / 1e12 / tpeak, "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, burst)" if peaks else "fallback",
                         "algorithmic_flops_per_launch": flops, "output_gbs": out_bytes / (ms * 1e-3) / 1e9,
                         "note": "bound by the SM's shared-memory bandwidth as a single-CTA kernel (operand reads of the 128 x 256 x 16 MMA + TMA writes + the epilogue's transposition, DESIGN.md section 4); 2.1 GB of fp64 output per launch"},
            "gate": {"max_corr_err_vs_oracle": err, "tol": 3e-5, "exactly_symmetric": sym, "ok": bool(err < 3e-5 and sym)},
            "e2e": {"seconds": e2e_s, "matrices_per_s": 1.0 / e2e_s, "h2d_bytes": int(Mhost.nbytes), "d2h_bytes": int(Rh.nbytes)},
            "cpu_baseline": {"seconds_full_matrix": cpu_full_s, "matrices_per_s": 1.0 / cpu_full_s, "cores": host_threads(), "kind": "port",
                             "sample": f"orc_cov (fp64, OpenMP) on the first {ccpu} features, scaled by the pair count"}}


def run_batch(args, rank, world, local):
    """BASELINE config 5: a batch of independent samples, no collective.  Every rank takes the samples rank, rank + N, ...;
    a producer thread makes the next samples' hit classes (synthetic fragments + the loader's class construction) while
    --batch-per-gpu worker threads, each with its own handle and stream, run EM, the Gibbs chain (trace of 1024) and the
    device summaries (log-mean, Sokal variance / IACT / MCSE inputs, percentiles) and write the sample's table."""
    import queue
    import torch
    import torch.distributed as dist
    from mmseq_b200 import capi, hostlib, synth
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    os.makedirs(args.batch_out, exist_ok=True)
    mine = [i for i in range(args.batch) if i % world == rank]
    L = 1024
    stride = max(1, args.batch_sweeps // L)
    q = queue.Queue(maxsize=args.batch_per_gpu)
    done = []
    lock = threading.Lock()

    nprod = max(1, min(args.batch_per_gpu, 3))   # class construction of the next samples on several host threads
    # the loader builds classes on all host threads it is given: share the cores between the ranks and their producers
    share = max(2, host_threads() // (max(1, world) * nprod))
    os.environ.setdefault("MMQ_LOADER_BUILDERS", str(max(1, share // 2)))
    os.environ.setdefault("MMQ_LOADER_THREADS", str(max(1, share // 2)))
    it_lock = threading.Lock()
    it_state = {"next": 0, "left": nprod}

    def producer():
        while True:
            with it_lock:
                if it_state["next"] >= len(mine):
                    it_state["left"] -= 1
                    last = it_state["left"] == 0
                    break
                i = mine[it_state["next"]]
                it_state["next"] += 1
            t0 = time.perf_counter()
            s = synth.Synth(SYNTH_SEED, args.transcripts, args.fragments, frag_seed=1000 + i, threads=share)   # not OMP_NUM_THREADS (1 under torchrun)
            h = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_COLLAPSED | hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
            length = s.efflen[h.col2hdr] * args.fragments / 1e9
            q.put((i, h, length, time.perf_counter() - t0))
        if last:
            for _ in range(args.batch_per_gpu):
                q.put(None)

    def worker():
        stream = torch.cuda.Stream(device=dev)
        while True:
            item = q.get()
            if item is None:
                return
            i, h, length, prep_s = item
            t0 = time.perf_counter()
            H = capi.Handle(h.row_ptr, h.col, h.k, length, device=local)
            H.set_stream(stream.cuda_stream)
            uh = H.init_mu()
            it, ll, _ = H.em(1000, 0.1)
            mu_em = H.get_mu()
            H.gibbs(SEED + i, 0, args.batch_sweeps, stride=stride, trace_len=L)
            S = H.summarize(0, [int(np.floor(p / 100.0 * (L - 1) + 0.5)) for p in (5, 25, 50, 75, 95)])
            H.close()
            with np.errstate(invalid="ignore"):
                sd = np.sqrt(S["var"]); mcse = np.sqrt(S["tau"] * S["var"] / L)
            tab = np.column_stack([S["log_mean"], sd, mcse, S["tau"], uh, np.log(np.maximum(mu_em, 1e-300))])
            np.savetxt(os.path.join(args.batch_out, f"sample_{i:03d}.tsv"), tab, delimiter="\t", fmt="%.6g",
                       header="log_mu\tsd\tmcse\tiact\tunique_hits\tlog_mu_em", comments="")
            with lock:
                done.append({"sample": i, "em_iters": int(it), "prep_s": round(prep_s, 2), "gpu_pipeline_s": round(time.perf_counter() - t0, 3),
                             "finite_log_mu": int(np.isfinite(S["log_mean"]).sum()), "median_iact": float(np.nanmedian(S["tau"]))})

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = capi.launch_count()
    t0 = time.perf_counter()
    th = [threading.Thread(target=producer) for _ in range(nprod)] + [threading.Thread(target=worker) for _ in range(args.batch_per_gpu)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tw = torch.tensor([wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        allres = [None] * world
        dist.all_gather_object(allres, done)
        done = [d for r in allres for d in r]
    wall = float(tw.item())
    if rank == 0:
        line = {"metric": "batch_samples_per_s", "value": args.batch / wall, "unit": "samples/s", "n_gpus": world, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "wall_s": wall,
                "sweeps_per_s_all_samples": args.batch * args.batch_sweeps / wall,
                "sweeps_per_s_per_gpu": args.batch * args.batch_sweeps / wall / world,
                "gpu_pipeline_s_median": float(np.median([d["gpu_pipeline_s"] for d in done])),
                "prep_s_median": float(np.median([d["prep_s"] for d in done])),
                "gpu_launches": int(capi.launch_count() - launches0),
                "config": {"workload": "C5-batch", "samples": args.batch, "transcripts": args.transcripts, "fragments_per_sample": args.fragments,
                           "sweeps_per_sample": args.batch_sweeps, "trace_length": L, "in_flight_per_gpu": args.batch_per_gpu,
                           "per_sample": "class construction (host) -> mmq_create -> init, EM -> Gibbs chain -> device summaries (Sokal) -> table"},
                "tables": os.path.join(args.batch_out, "sample_*.tsv"), "samples": sorted(done, key=lambda d: d["sample"])[:8]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank, world, local = dist_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.batch > 0:
        run_batch(args, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    from mmseq_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the mmseq hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(a):
        """Sum of a host array over the ranks (through the GPUs: the process group is NCCL)."""
        if world == 1:
            return a
        t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        dist.all_reduce(t)
        return t.cpu().numpy()

    w = make_workload(args, rank, world)
    h, n = w.h, w.h.n
    flags = capi.MMQ_GIBBS_TRANSPOSED if args.transposed else capi.MMQ_GIBBS_DEFAULT
    near_l2 = (4 * h.nnz) <= 200e6
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if near_l2 else None
    stream = torch.cuda.Stream(device=dev)

    def attach(Hx, reuse_from=None):
        if world == 1:
            return
        if reuse_from is not None:
            reuse_from.comm_move_to(Hx)   # the process keeps its NCCL communicator across samples
        else:
            uid = [capi.comm_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            Hx.comm_init(uid[0], rank, world)
        if not args.nccl_only and not Hx.p2p_attached():   # count exchange fused into the Gamma kernel over NVLink peer memory
            hs = [None] * world
            dist.all_gather_object(hs, Hx.p2p_export())
            Hx.p2p_attach(hs, rank, world)
        if args.p2p_rs:
            Hx.tune(6, 1)

    H = capi.Handle(h.row_ptr, h.col, h.k, w.length, weight=h.w, class_id_base=w.cid_base, device=local)
    H.set_stream(stream.cuda_stream)
    attach(H)
    H.init_mu()
    mu0 = H.get_mu()
    t0 = time.perf_counter()
    em_iters, em_ll, _ = H.em(1000, 0.1)
    em_s = time.perf_counter() - t0
    mu_em = H.get_mu()
    cls = H.cls_stats() if h.k is not None else None
    rows = None

    K, W, S = args.steps, args.warmup, SWEEPS_PER_STEP
    outputs = {} if args.dump_outputs and rank == 0 else None
    ms, alloc_ms, alloc_n, gamma_ms, gamma_n, launches, clocks = timed_run(args, H, w, stream, dev, barrier, K, W, flush_buf, flags, outputs)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    per_rank = None
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pr = [None] * world   # average kernel times of every rank: shows which rank the others wait for
        dist.all_gather_object(pr, [round(alloc_ms / max(alloc_n, 1), 5), round(gamma_ms / max(gamma_n, 1), 5), round(ms / K, 4)])
        per_rank = {"alloc_ms": [p[0] for p in pr], "gamma_ms": [p[1] for p in pr], "step_ms": [p[2] for p in pr]}
    ms_max = float(t.item())
    sweeps_per_s = K * S / (ms_max / 1000.0)
    totals = {"n": n, "m": int(allreduce(np.array([float(value_classes(args, w))]))[0]), "nnz": int(allreduce(np.array([float(h.nnz)]))[0])}
    value = sweeps_per_s * totals["m"]

    # ---- end to end through the C ABI with host buffers (pinned), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        pin = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
        rp, col, kk, ww, ll, mu_h = pin(h.row_ptr), pin(h.col), pin(h.k), pin(h.w), pin(w.length), pin(mu_em)
        mu_buf, tr_buf = pin(np.zeros(n)), pin(np.zeros((n, K)))   # pinned result buffers too
        # one repetition = a fresh handle (H2D of the shard, device plan, graph capture) + K*S sweeps + the read-back; the
        # region is ~50-100 ms of wall clock, so a single shot is at the mercy of one slow cudaMalloc: N = 1 takes the
        # median of three repetitions (all of them listed), N > 1 one (the communicator moves with the handle)
        walls, parts = [], []
        for rep in range(3 if world == 1 else 1):
            barrier()
            t0 = time.perf_counter()
            H2 = capi.Handle(rp, col, kk, ll, weight=ww, class_id_base=w.cid_base, device=local)   # H2D of the CSR shard
            attach(H2, reuse_from=H)
            H2.set_mu(mu_h)                                                                        # H2D
            t1 = time.perf_counter()
            H2.gibbs(SEED, 0, K * S, stride=S, trace_len=K, flags=flags)
            H2.synchronize()
            t2 = time.perf_counter()
            mu_out = H2.get_mu(out=mu_buf)                                                         # D2H
            tr = H2.get_trace(out=tr_buf)                                                          # D2H, n x K doubles
            barrier()
            t3 = time.perf_counter()
            walls.append(t3 - t0)
            parts.append([round(t1 - t0, 5), round(t2 - t1, 5), round(t3 - t2, 5)])
            if world == 1 and rep < 2:
                H2.close()
        wall = float(np.median(walls))
        tw = torch.tensor([wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.item())
        h2d = rp.nbytes + col.nbytes + (kk.nbytes if kk is not None else 0) + (ww.nbytes if ww is not None else 0) + ll.nbytes + mu_h.nbytes
        d2h = mu_out.nbytes + tr.nbytes
        e2e = {"value": K * S / wall * totals["m"], "unit": "allocations/s", "sweeps_per_s": K * S / wall,
               "h2d_bytes_per_step": int(h2d / K), "d2h_bytes_per_step": int(d2h / K), "wall_s": wall,
               "repetitions_wall_s": [round(x, 5) for x in walls], "create_sweeps_readback_s": parts,
               "what": "mmq_create(H2D shard, plan) + mmq_set_mu + steps*16 sweeps + mmq_get_mu + mmq_get_trace, pinned host buffers; wall clock, N = 1: median of three repetitions"}
        assert np.isfinite(tr).all() and (tr > 0).any()
        H, H2 = H2, H   # keep the handle that owns the communicator
        H2.close()

    # ---- roofline of the dominant kernel (the allocation), device time from CUDA events on its stream
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback (B200_PROFILING.md 6.65 TB/s)"
    b_alloc, b_sweep = algorithmic_bytes(h, n, args.weights, args.transposed, S, args.layout, cls, rows)
    alloc_ms_avg = alloc_ms / max(alloc_n, 1)
    gamma_ms_avg = gamma_ms / max(gamma_n, 1)
    achieved = b_alloc / (alloc_ms_avg * 1e-3) / 1e9 if alloc_n else None
    if args.transposed:
        kernel_name = "k_alloc"
    elif cls and cls["in_use"]:
        kernel_name = "k_alloc_cls"
    elif rows and rows.get("in_use"):
        kernel_name = "k_alloc_rows"
    else:
        kernel_name = "k_alloc_seg4" if h.k is None else "k_alloc"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and args.fragments == N_C2 and args.transcripts == T_C2:
        tj = json.load(open(tpath)).get(kernel_name)
        if tj and tj.get("workload") == workload_name(args):
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]   # per launch, from one ncu --set full capture
    per_sweep_ms = ms_max / (K * S)
    roofline = {"kernel": kernel_name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(b_alloc), "avg_launch_ms": alloc_ms_avg, "launches_timed": int(alloc_n),
                "share_of_sweep": alloc_ms_avg / (alloc_ms_avg + gamma_ms_avg) if alloc_n else None,
                "alloc_ms_in_graph": per_sweep_ms - gamma_ms_avg,
                "gamma_avg_launch_ms": gamma_ms_avg, "sweep_ms": per_sweep_ms,
                "graph_vs_plain_us_per_sweep": 1e3 * (per_sweep_ms - alloc_ms_avg - gamma_ms_avg),
                "sweep_bytes": int(b_sweep), "sweep_gbs": b_sweep / (per_sweep_ms * 1e-3) / 1e9,
                "how": "value: K steps through mmq_gibbs (CUDA graph of 16 sweeps), CUDA events on the handle's stream; kernel "
                       "durations: the same K steps repeated with MMQ_GIBBS_TIME_KERNELS (events around every allocation / Gamma "
                       "launch; a collapsed shard's allocation is up to four concurrent kernels timed as one)"}
    if per_rank:
        roofline["per_rank"] = per_rank
    if cls:
        roofline["class_plan"] = cls
    if rows:
        roofline["row_plan"] = rows

    line = {
        "metric": "gibbs_hit_class_allocations_per_s", "value": value, "unit": "allocations/s",
        "sweeps_per_s": sweeps_per_s, "fragments_per_s": sweeps_per_s * w.ntot,
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K, "sweeps_per_step": S, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, totals), "clocks": clocks,
        "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "prep": w.prep,
        "em": {"iters": int(em_iters), "loglik": em_ll, "wall_s": round(em_s, 4)},
        "count_path": "transposed" if args.transposed else "fused_reduction",
        "count_exchange": ("none" if world == 1 else ("nccl_allreduce" if args.nccl_only else "fused_p2p_gamma")),
    }

    # ---- correctness gates at the benchmark shape, every rank
    gates_ok = True
    if not args.no_gates:
        g = run_gates(args, H, w, mu0, mu_em, em_iters, rank, world, dev, allreduce)
        mu_oracle_em = g.pop("mu_em")
        if world == 1 and not args.no_cpu_baseline and not args.weights:
            # (c) + CPU baseline: the reference-like chain on the collapsed representation of the same sample
            wc = w if w.layout == "collapsed" else make_workload(args, 0, 1, weights=False, layout="collapsed")
            if wc is w:
                pg, base = posterior_gate(args, H, wc, mu_oracle_em, args.cpu_sweeps, host_threads())
                g["posterior"] = pg   # statistical: pg["rule"]; the run FAILS when the rule fails by a margin or on a gross miss
                g["ok"] = bool(g["ok"] and pg["frac_within_4se"] >= pg["hard_fail_below"] and
                               (pg["ok"] or pg["frac_within_4se"] >= pg["self_frac_within_4se"] - 2e-3))
            else:
                from oracle import oracle as orc
                Pc = orc.Problem(wc.h.row_ptr, wc.h.col, wc.h.k, wc.length)
                mu_c, _, _ = Pc.init_mu()
                mu_c, _, _ = Pc.gibbs_gsl(mu_c, SEED, 1, threads=host_threads())
                _, _, sec = Pc.gibbs_gsl(mu_c, SEED, 8, threads=host_threads())
                base = {"value": 8 / sec * value_classes(args, wc), "unit": "allocations/s", "sweeps_per_s": 8 / sec, "cores": host_threads(),
                        "kind": "port", "layout": "collapsed", "sample": "8 full sweeps of the collapsed form of the same sample after 1 warm-up sweep"}
            line["cpu_baseline"] = base
        line["gates"] = g
        gates_ok = g["ok"]
    elif rank == 0 and world == 1 and not args.no_cpu_baseline and not args.weights:
        from oracle import oracle as orc
        P = orc.Problem(h.row_ptr, h.col, h.k, w.length)
        mu_c, _, _ = P.gibbs_gsl(mu0, SEED, 1, threads=host_threads())
        _, _, sec = P.gibbs_gsl(mu_c, SEED, 8, threads=host_threads())
        line["cpu_baseline"] = {"value": 8 / sec * value_classes(args, w), "unit": "allocations/s", "sweeps_per_s": 8 / sec,
                                "cores": host_threads(), "kind": "port", "layout": w.layout,
                                "sample": "8 full sweeps of the same shard after 1 warm-up sweep"}
    H.close()

    # ---- the compulsory per-fragment stream of the same sample (fp32 per-hit weights), N = 1 default run only
    if rank == 0 and world == 1 and args.layout == "collapsed" and not args.no_extras and not args.haplo and args.scaling == "weak":
        try:
            line["perfragment_weighted"] = extra_weighted_line(args, dev, stream, peak)
        except Exception as e:   # an extra: never at the expense of the headline line
            line["perfragment_weighted"] = {"error": repr(e)}

    # ---- the consumer of the traces: mmcollapse's covariance step on the tensor cores (row f3), N = 1 default run only
    if rank == 0 and world == 1 and args.layout == "collapsed" and not args.no_extras and not args.haplo and args.scaling == "weak":
        try:
            line["trace_cov"] = extra_trace_cov(args, dev, stream)
            if not line["trace_cov"]["gate"]["ok"]:
                gates_ok = False
        except Exception as e:
            line["trace_cov"] = {"error": repr(e)}

    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if not gates_ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
