"""ctypes binding of include/mmq.h (libmmseq_b200.so).  One method per C entry
point, same names and argument meaning; numpy arrays in, numpy arrays out.
No fallback: a missing library or a failing call raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmseq_b200.so")

MMQ_GIBBS_DEFAULT = 0
MMQ_GIBBS_TRANSPOSED = 1
MMQ_GIBBS_NO_GRAPH = 2
MMQ_GIBBS_TIME_KERNELS = 4
MMQ_GIBBS_GENERIC_KERNEL = 8
MMQ_GIBBS_RAGGED_KERNEL = 16
MMQ_GROUP_IDENTICAL = 0
MMQ_GROUP_GENE = 1


class MmqError(RuntimeError):
    pass


class _Problem(C.Structure):
    _fields_ = [
        ("n", C.c_int64), ("m", C.c_int64), ("nnz", C.c_int64),
        ("row_ptr", C.c_void_p), ("col", C.c_void_p), ("k", C.c_void_p),
        ("weight", C.c_void_p), ("len", C.c_void_p),
        ("alpha", C.c_double), ("beta", C.c_double), ("class_id_base", C.c_int64),
        ("class_id", C.c_void_p),
    ]


def _load():
    if not os.path.exists(LIB_PATH):
        raise MmqError(
            f"{LIB_PATH} not built: run `make lib` (or __graft_entry__.build()). "
            "There is no CPU fallback for the mmseq hot path.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64, u32, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_double
    sig = {
        "mmq_create": (i32, [C.POINTER(_Problem), i32, C.POINTER(vp)]),
        "mmq_destroy": (None, [vp]),
        "mmq_last_error": (C.c_char_p, [vp]),
        "mmq_set_stream": (i32, [vp, vp]),
        "mmq_get_stream": (vp, [vp]),
        "mmq_synchronize": (i32, [vp]),
        "mmq_device_bytes": (i64, [vp]),
        "mmq_comm_id": (i32, [C.c_char_p]),
        "mmq_comm_init": (i32, [vp, C.c_char_p, i32, i32]),
        "mmq_comm_move": (i32, [vp, vp]),
        "mmq_p2p_export": (i32, [vp, C.c_char_p]),
        "mmq_p2p_attach": (i32, [vp, C.c_char_p, i32, i32]),
        "mmq_p2p_attach_local": (i32, [C.POINTER(vp), i32]),
        "mmq_p2p_attached": (i32, [vp]),
        "mmq_init_mu": (i32, [vp, vp]),
        "mmq_set_mu": (i32, [vp, vp]),
        "mmq_get_mu": (i32, [vp, vp]),
        "mmq_loglik": (i32, [vp, C.POINTER(dbl)]),
        "mmq_em": (i32, [vp, i32, dbl, C.POINTER(i32), C.POINTER(dbl), C.POINTER(dbl)]),
        "mmq_gibbs": (i32, [vp, u32, i64, i64, i32, i32, i32]),
        "mmq_sweep_debug": (i32, [vp, u32, i64, i32, vp, vp, vp]),
        "mmq_kernel_times": (i32, [vp, C.POINTER(dbl), C.POINTER(i64), C.POINTER(dbl), C.POINTER(i64)]),
        "mmq_cls_stats": (i32, [vp, C.POINTER(i64)]),
        "mmq_tune": (i32, [vp, i32, i32]),
        "mmq_count_moments_begin": (i32, [vp, vp, i64, vp, i64]),
        "mmq_count_moments_end": (i32, [vp]),
        "mmq_get_count_moments": (i32, [vp, i32, C.POINTER(i64), vp, vp, vp]),
        "mmq_expected_counts": (i32, [vp, vp]),
        "mmq_get_trace": (i32, [vp, vp]),
        "mmq_trace_len": (i32, [vp]),
        "mmq_set_groups": (i32, [vp, i32, i64, vp, vp, vp]),
        "mmq_summarize": (i32, [vp, i32, vp, vp, vp, vp, vp, i32, vp, vp]),
        "mmq_get_group_trace": (i32, [vp, i32, vp]),
        "mmq_prop_summaries": (i32, [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
        "mmq_unique_hits_sets": (i32, [vp, vp, i64, vp]),
        "mmq_sokal_batch": (i32, [i32, i64, i32, vp, vp, vp, vp, vp]),
        "mmq_chain_seed": (u32, [u32, i32]),
        "mmq_chain_diagnostics_dev": (i32, [C.POINTER(vp), i32, i64, i32, vp, vp]),
        "mmq_chain_diagnostics": (i32, [C.POINTER(vp), i32, i32, vp, vp, vp, vp, vp]),
        "mmq_pooled_summaries_dev": (i32, [C.POINTER(vp), i32, i64, i32, i32, i32, vp, vp, vp, vp]),
        "mmq_pooled_summaries": (i32, [C.POINTER(vp), i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]),
        "mmq_draw_totals_workspace_bytes": (i64, [i64, i32]),
        "mmq_draw_totals_dev": (i32, [vp, i64, i32, vp, vp, vp]),
        "mmq_tpm_summaries_dev": (i32, [C.POINTER(vp), vp, i32, i64, i32, vp, vp, i32, vp, vp, vp, vp]),
        "mmq_tpm_summaries": (i32, [C.POINTER(vp), i32, i32, i32, vp, vp, vp, vp, vp]),
        "mmq_allele_only_counts": (i32, [vp, vp, vp, i64, vp, vp]),
        "mmq_allelic_summaries_dev": (i32, [C.POINTER(vp), C.POINTER(vp), i32, i64, i64, i64, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp]),
        "mmq_allelic_summaries": (i32, [C.POINTER(vp), i32, C.POINTER(vp), i64, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]),
        "mmq_pair_shared_counts": (i32, [vp, vp, vp, vp, i64, i64, vp]),
        "mmq_isocorr_workspace_bytes": (i64, [i64, i64]),
        "mmq_isocorr_summaries_dev": (i32, [C.POINTER(vp), i32, i64, i64, i32, vp, vp, vp, i64, vp, vp, vp]),
        "mmq_isocorr_summaries": (i32, [C.POINTER(vp), i32, i64, vp, vp, vp]),
        "mmq_prior_draws": (i32, [i32, i64, vp, vp, dbl, u32, i32, vp]),
        "mmq_trace_cov": (i32, [i32, vp, i32, i64, i32, vp]),
        "mmq_trace_cov_workspace_bytes": (i64, [i32, i64, i32]),
        "mmq_trace_cov_dev": (i32, [vp, i32, i64, i32, vp, vp, vp]),
        "mmq_handle_trace_cov": (i32, [vp, vp, i64, i32, vp, vp]),
        "mmq_mean_corrs": (i32, [i32, vp, vp, i64, i32, vp, i64, dbl, vp, vp]),
        "mmq_mean_corrs_dev": (i32, [vp, vp, i64, i32, vp, i64, dbl, vp, vp, vp]),
        "mmq_release_cache": (i32, [i32]),
        "mmq_launch_count": (i64, []),
        "mmq_warmup": (i32, [i32]),
        "mmq_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


EXPORTS = [
    "mmq_create", "mmq_destroy", "mmq_last_error", "mmq_set_stream", "mmq_get_stream", "mmq_synchronize",
    "mmq_device_bytes", "mmq_comm_id", "mmq_comm_init", "mmq_comm_move", "mmq_p2p_export", "mmq_p2p_attach", "mmq_p2p_attach_local", "mmq_p2p_attached", "mmq_init_mu", "mmq_set_mu", "mmq_get_mu",
    "mmq_loglik", "mmq_em", "mmq_gibbs", "mmq_sweep_debug", "mmq_kernel_times", "mmq_cls_stats", "mmq_tune", "mmq_get_trace", "mmq_trace_len",
    "mmq_count_moments_begin", "mmq_count_moments_end", "mmq_get_count_moments", "mmq_expected_counts",
    "mmq_set_groups", "mmq_summarize", "mmq_get_group_trace", "mmq_prop_summaries",
    "mmq_unique_hits_sets", "mmq_sokal_batch", "mmq_chain_seed", "mmq_chain_diagnostics_dev", "mmq_chain_diagnostics",
    "mmq_pooled_summaries_dev", "mmq_pooled_summaries", "mmq_draw_totals_workspace_bytes", "mmq_draw_totals_dev",
    "mmq_tpm_summaries_dev", "mmq_tpm_summaries", "mmq_allele_only_counts", "mmq_allelic_summaries_dev", "mmq_allelic_summaries",
    "mmq_pair_shared_counts", "mmq_isocorr_workspace_bytes", "mmq_isocorr_summaries_dev", "mmq_isocorr_summaries",
    "mmq_prior_draws", "mmq_trace_cov", "mmq_trace_cov_workspace_bytes", "mmq_trace_cov_dev",
    "mmq_handle_trace_cov", "mmq_mean_corrs", "mmq_mean_corrs_dev", "mmq_release_cache", "mmq_launch_count", "mmq_warmup", "mmq_version",
]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype):
    if a is None:
        return None
    return np.ascontiguousarray(a, dtype=dtype)


def release_cache(device=-1):
    return int(lib().mmq_release_cache(device))


def launch_count():
    return int(lib().mmq_launch_count())


def version():
    return lib().mmq_version().decode()


def comm_id():
    buf = C.create_string_buffer(128)
    rc = lib().mmq_comm_id(buf)
    if rc:
        raise MmqError("mmq_comm_id: " + lib().mmq_last_error(None).decode())
    return buf.raw


def sokal_batch(x, device=0):
    """src/sokal.cc:33-87 on every row of x (rows, len)."""
    x = _c(x, np.float64)
    rows, ln = x.shape
    var = np.zeros(rows); tau = np.zeros(rows)
    win = np.zeros(rows, np.int32); status = np.zeros(rows, np.int32)
    rc = lib().mmq_sokal_batch(device, rows, ln, _ptr(x), _ptr(var), _ptr(tau), _ptr(win), _ptr(status))
    if rc:
        raise MmqError("mmq_sokal_batch: " + lib().mmq_last_error(None).decode())
    return var, tau, win, status


CHAIN_OUTPUTS = ("rhat", "ess_bulk", "ess_tail", "log_mean", "log_sd")


def chain_seed(seed, chain):
    """Seed of chain `chain` (0 <= chain < 8) of a run with seed `seed`; chain 0 is `seed`."""
    return int(lib().mmq_chain_seed(seed, chain))


def chain_diagnostics_dev(chain_ptrs, rows, L, out_ptr, stream_ptr):
    """mmq_chain_diagnostics_dev: chain_ptrs, device pointers (ints) of each chain's [rows, L] fp64 draws; out_ptr:
    fp64[5 * rows] on the same device.  Asynchronous on the stream."""
    arr = (C.c_void_p * len(chain_ptrs))(*chain_ptrs)
    _global_check(lib().mmq_chain_diagnostics_dev(arr, len(chain_ptrs), rows, L, out_ptr, stream_ptr), "mmq_chain_diagnostics_dev")


def chain_diagnostics(handles, which=0):
    """mmq_chain_diagnostics over the traces the handles recorded: dict of CHAIN_OUTPUTS, fp64[rows] each."""
    h0 = handles[0]
    rows = h0.n if which == 0 else h0._ng[which - 1]
    out = {k: np.zeros(rows) for k in CHAIN_OUTPUTS}
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_chain_diagnostics(arr, len(handles), which, *[_ptr(out[k]) for k in CHAIN_OUTPUTS])
    if rc:
        raise MmqError(f"mmq_chain_diagnostics failed ({rc}): " + lib().mmq_last_error(h0._h).decode())
    return out


POOL_OUTPUTS = ("mean", "sd", "ess_mean")


def pooled_summaries_dev(chain_ptrs, rows, L, mode, npct, pct_idx_ptr, out_ptr, pct_ptr, stream_ptr):
    """mmq_pooled_summaries_dev: chain_ptrs, device pointers (ints) of each chain's [rows, L] fp64 draws; pct_idx_ptr:
    int32[npct], out_ptr: fp64[3 * rows], pct_ptr: fp64[rows * npct], all on the same device.  Asynchronous on the
    stream."""
    arr = (C.c_void_p * len(chain_ptrs))(*chain_ptrs)
    _global_check(lib().mmq_pooled_summaries_dev(arr, len(chain_ptrs), rows, L, mode, npct, pct_idx_ptr, out_ptr, pct_ptr, stream_ptr),
                  "mmq_pooled_summaries_dev")


def pooled_summaries(handles, which=0, pct_idx=None, gene_of=None, multi_iso=None):
    """mmq_pooled_summaries over the traces the handles recorded: dict of POOL_OUTPUTS (fp64[rows]; sd and ess_mean stay
    NaN for which 3), pct (rows, npct) and, for which 3, sum_probit and sumsq_probit added over the chains."""
    h0 = handles[0]
    rows = h0.n if which in (0, 3) else h0._ng[which - 1]
    out = {k: np.full(rows, np.nan) for k in POOL_OUTPUTS + ("sum_probit", "sumsq_probit")}
    pct_idx = _c(pct_idx if pct_idx is not None else [], np.int32)
    out["pct"] = np.zeros((rows, len(pct_idx)))
    gene_of = _c(gene_of, np.int32); multi_iso = _c(multi_iso, np.uint8)
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_pooled_summaries(arr, len(handles), which, _ptr(gene_of), _ptr(multi_iso), len(pct_idx), _ptr(pct_idx),
                                    *[_ptr(out[k]) for k in POOL_OUTPUTS + ("sum_probit", "sumsq_probit", "pct")])
    if rc:
        raise MmqError(f"mmq_pooled_summaries failed ({rc}): " + lib().mmq_last_error(h0._h).decode())
    return out


def draw_totals_workspace_bytes(rows, L):
    return int(lib().mmq_draw_totals_workspace_bytes(rows, L))


def draw_totals_dev(trace_ptr, rows, L, totals_ptr, ws_ptr, stream_ptr):
    """mmq_draw_totals_dev: totals_ptr fp64[L] = the column sums of the [rows, L] fp64 trace at trace_ptr in the fixed
    tile order; ws_ptr: draw_totals_workspace_bytes(rows, L) bytes.  Device pointers (ints); asynchronous on the stream."""
    _global_check(lib().mmq_draw_totals_dev(trace_ptr, rows, L, totals_ptr, ws_ptr, stream_ptr), "mmq_draw_totals_dev")


def tpm_summaries_dev(chain_ptrs, totals_ptr, rows, L, group_ptr_ptr, members_ptr, npct, pct_idx_ptr, out_ptr, pct_ptr, stream_ptr):
    """mmq_tpm_summaries_dev: chain_ptrs, device pointers (ints) of each chain's transcript trace; totals_ptr
    fp64[C * L] chain-major; group_ptr_ptr / members_ptr: a CSR of features over the transcripts, or both None for one
    feature per transcript; out_ptr fp64[2 * rows] (mean, sd); pct_ptr fp64[rows * npct].  Asynchronous on the stream."""
    arr = (C.c_void_p * len(chain_ptrs))(*chain_ptrs)
    _global_check(lib().mmq_tpm_summaries_dev(arr, totals_ptr, len(chain_ptrs), rows, L, group_ptr_ptr, members_ptr, npct, pct_idx_ptr,
                                              out_ptr, pct_ptr, stream_ptr), "mmq_tpm_summaries_dev")


def tpm_summaries(handles, which=0, pct_idx=None):
    """mmq_tpm_summaries over the traces the handles recorded: dict(mean, sd: fp64[rows]; pct: (rows, npct);
    totals: (C, L), each chain's per-draw total of the observed transcripts)."""
    h0 = handles[0]
    rows = h0.n if which == 0 else getattr(h0, "_ng", {}).get(which - 1, 0)          # other values: the library refuses them
    pct_idx = _c(pct_idx if pct_idx is not None else [], np.int32)
    out = dict(mean=np.zeros(rows), sd=np.zeros(rows), pct=np.zeros((rows, len(pct_idx))),
               totals=np.zeros((len(handles), h0.trace_len())))
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_tpm_summaries(arr, len(handles), which, len(pct_idx), _ptr(pct_idx), _ptr(out["mean"]), _ptr(out["sd"]), _ptr(out["pct"]),
                                 _ptr(out["totals"]))
    if rc:
        raise MmqError(f"mmq_tpm_summaries failed ({rc}): " + lib().mmq_last_error(h0._h).decode())
    return out


def allelic_summaries_dev(chain_ptrs, prior_ptrs, n, nprior, rows, L, a_ptr_ptr, a_mem_ptr, b_ptr_ptr, b_mem_ptr, npct, pct_idx_ptr,
                         out_ptr, pct_ptr, stream_ptr):
    """mmq_allelic_summaries_dev: chain_ptrs, device pointers (ints) of each chain's transcript trace (n rows); prior_ptrs,
    of each chain's nprior prior rows (or None); the A and B member CSRs (ids < n: trace rows, n + j: prior row j);
    out_ptr fp64[3 * rows] (mean, sd, prob_a); pct_ptr fp64[rows * npct].  Asynchronous on the stream."""
    arr = (C.c_void_p * len(chain_ptrs))(*chain_ptrs)
    pri = None if prior_ptrs is None else (C.c_void_p * len(prior_ptrs))(*prior_ptrs)
    _global_check(lib().mmq_allelic_summaries_dev(arr, pri, len(chain_ptrs), n, nprior, rows, L, a_ptr_ptr, a_mem_ptr, b_ptr_ptr, b_mem_ptr,
                                                  npct, pct_idx_ptr, out_ptr, pct_ptr, stream_ptr), "mmq_allelic_summaries_dev")


def allelic_summaries(handles, a_ptr, a_mem, b_ptr, b_mem, priors=None, pct_idx=None):
    """mmq_allelic_summaries over the transcript traces the handles recorded; priors: one (nprior, L) array per chain or
    None.  Returns dict(mean, sd, prob_a: fp64[rows]; pct: (rows, npct))."""
    h0 = handles[0]
    a_ptr = _c(a_ptr, np.int64); b_ptr = _c(b_ptr, np.int64)
    a_mem = _c(a_mem, np.int32); b_mem = _c(b_mem, np.int32)
    rows = len(a_ptr) - 1
    pct_idx = _c(pct_idx if pct_idx is not None else [], np.int32)
    priors = None if priors is None else [_c(p, np.float64) for p in priors]
    nprior = 0 if priors is None else priors[0].shape[0]
    pri = None if priors is None else (C.c_void_p * len(priors))(*[p.ctypes.data for p in priors])
    out = dict(mean=np.zeros(rows), sd=np.zeros(rows), prob_a=np.zeros(rows), pct=np.zeros((rows, len(pct_idx))))
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_allelic_summaries(arr, len(handles), pri, nprior, rows, _ptr(a_ptr), _ptr(a_mem), _ptr(b_ptr), _ptr(b_mem),
                                     len(pct_idx), _ptr(pct_idx), _ptr(out["mean"]), _ptr(out["sd"]), _ptr(out["prob_a"]), _ptr(out["pct"]))
    if rc:
        raise MmqError(f"mmq_allelic_summaries failed ({rc}): " + lib().mmq_last_error(h0._h).decode())
    return out


def isocorr_workspace_bytes(ngenes, nmembers):
    return int(lib().mmq_isocorr_workspace_bytes(ngenes, nmembers))


def isocorr_summaries_dev(chain_ptrs, ngenes, nmembers, L, gene_ptr_ptr, members_ptr, pair_base_ptr, npairs, out_ptr, ws_ptr, stream_ptr):
    """mmq_isocorr_summaries_dev: chain_ptrs, device pointers (ints) of each chain's transcript trace; the gene CSR
    (int64[ngenes + 1], int32[nmembers]) and pair_base (int64[ngenes]) on the device; out_ptr fp64[3 * npairs] (corr_mu,
    corr_log_mu, prob_1_gt_2); ws_ptr isocorr_workspace_bytes(ngenes, nmembers) bytes.  Asynchronous on the stream."""
    arr = (C.c_void_p * len(chain_ptrs))(*chain_ptrs)
    _global_check(lib().mmq_isocorr_summaries_dev(arr, len(chain_ptrs), ngenes, nmembers, L, gene_ptr_ptr, members_ptr, pair_base_ptr,
                                                  npairs, out_ptr, ws_ptr, stream_ptr), "mmq_isocorr_summaries_dev")


def isocorr_summaries(handles, npairs):
    """mmq_isocorr_summaries over the transcript traces the handles recorded and handles[0]'s gene groups.  Returns
    dict(corr_mu, corr_log_mu, prob_1_gt_2: fp64[npairs])."""
    h0 = handles[0]
    out = dict(corr_mu=np.zeros(npairs), corr_log_mu=np.zeros(npairs), prob_1_gt_2=np.zeros(npairs))
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_isocorr_summaries(arr, len(handles), npairs, _ptr(out["corr_mu"]), _ptr(out["corr_log_mu"]), _ptr(out["prob_1_gt_2"]))
    if rc:
        raise MmqError(f"mmq_isocorr_summaries failed ({rc}): " + lib().mmq_last_error(h0._h).decode())
    return out


def _global_check(rc, what):
    if rc:
        raise MmqError(f"{what}: " + (lib().mmq_last_error(None) or b"").decode())


def trace_cov(M, nsplit=2, device=0):
    """mmq_trace_cov: cov() of the L x C trace matrix M[s, c] (src/mmcollapse.cpp:553-558).  Returns C x C."""
    M = np.asarray(M, np.float64)
    L, Cn = M.shape
    Mf = np.asfortranarray(M)                      # column c contiguous (Armadillo's layout)
    R = np.zeros((Cn, Cn), np.float64, order="F")
    _global_check(lib().mmq_trace_cov(device, Mf.ctypes.data_as(C.c_void_p), L, Cn, nsplit, R.ctypes.data_as(C.c_void_p)), "mmq_trace_cov")
    return R


def trace_cov_workspace_bytes(L, Cn, nsplit=2):
    return int(lib().mmq_trace_cov_workspace_bytes(L, Cn, nsplit))


def trace_cov_dev(M_ptr, L, Cn, nsplit, R_ptr, ws_ptr, stream_ptr):
    """Device pointers (ints); asynchronous on the stream."""
    _global_check(lib().mmq_trace_cov_dev(M_ptr, L, Cn, nsplit, R_ptr, ws_ptr, stream_ptr), "mmq_trace_cov_dev")


def mean_corrs(R, S, ts, sdpenalty=0.0, V=None, W=None, device=0):
    """mmq_mean_corrs (src/mmcollapse.cpp:483-511).  R: (ns, C, C) symmetric slices, S: (C, ns) 0/1."""
    R = np.ascontiguousarray(R, np.float64)
    ns, Cn, _ = R.shape
    Sf = np.asfortranarray(np.asarray(S, np.uint8))
    ts = _c(ts, np.int32)
    V = np.zeros((Cn, Cn), np.float64, order="F") if V is None else np.asfortranarray(V, np.float64)
    W = np.zeros((Cn, Cn), np.float64, order="F") if W is None else np.asfortranarray(W, np.float64)
    _global_check(lib().mmq_mean_corrs(device, _ptr(R), Sf.ctypes.data_as(C.c_void_p), Cn, ns, _ptr(ts), len(ts), float(sdpenalty),
                                       V.ctypes.data_as(C.c_void_p), W.ctypes.data_as(C.c_void_p)), "mmq_mean_corrs")
    return V, W


def mean_corrs_dev(R_ptr, S_ptr, Cn, ns, ts_ptr, nts, sdpenalty, V_ptr, W_ptr, stream_ptr):
    _global_check(lib().mmq_mean_corrs_dev(R_ptr, S_ptr, Cn, ns, ts_ptr, nts, float(sdpenalty), V_ptr, W_ptr, stream_ptr), "mmq_mean_corrs_dev")


def prior_draws(ids, rate, alpha, seed, trace_len, device=0):
    """src/mmseq.cpp:971-978 on the device: (len(ids), trace_len) Gamma(alpha, rate) draws."""
    ids = _c(ids, np.int64); rate = _c(rate, np.float64)
    out = np.zeros((len(ids), trace_len))
    rc = lib().mmq_prior_draws(device, len(ids), _ptr(ids), _ptr(rate), alpha, seed, trace_len, _ptr(out))
    if rc:
        raise MmqError("mmq_prior_draws: " + lib().mmq_last_error(None).decode())
    return out


def p2p_attach_local(handles):
    """Single process, one Handle per GPU (rank order)."""
    arr = (C.c_void_p * len(handles))(*[h._h for h in handles])
    rc = lib().mmq_p2p_attach_local(arr, len(handles))
    if rc:
        raise MmqError("mmq_p2p_attach_local: " + lib().mmq_last_error(handles[0]._h).decode())


class Handle:
    """One shard of hit classes resident on one GPU (mmq_handle)."""

    def __init__(self, row_ptr, col, k, length, alpha=0.1, beta=0.1, weight=None, n=None,
                 class_id_base=0, device=0, class_id=None):
        self._h = C.c_void_p()
        self.row_ptr = _c(row_ptr, np.int64)
        self.col = _c(col, np.int32)
        self.k = _c(k, np.int32)
        self.weight = _c(weight, np.float32)
        self.len = _c(length, np.float64)
        self.class_id = _c(class_id, np.int64)
        self.n = int(len(self.len) if n is None else n)
        self.m = int(len(self.row_ptr) - 1)
        self.nnz = int(self.row_ptr[-1]) if self.m >= 0 and len(self.row_ptr) else 0
        p = _Problem(self.n, self.m, self.nnz, _ptr(self.row_ptr), _ptr(self.col), _ptr(self.k),
                     _ptr(self.weight), _ptr(self.len), alpha, beta, class_id_base, _ptr(self.class_id))
        rc = lib().mmq_create(C.byref(p), device, C.byref(self._h))
        if rc:
            self._h = C.c_void_p()
            raise MmqError(f"mmq_create failed ({rc}): " + lib().mmq_last_error(None).decode())

    def _check(self, rc, what):
        if rc:
            raise MmqError(f"{what} failed ({rc}): " + lib().mmq_last_error(self._h).decode())

    def close(self):
        if self._h:
            lib().mmq_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream_ptr):
        self._check(lib().mmq_set_stream(self._h, C.c_void_p(cuda_stream_ptr)), "mmq_set_stream")

    def get_stream(self):
        return lib().mmq_get_stream(self._h)

    def synchronize(self):
        self._check(lib().mmq_synchronize(self._h), "mmq_synchronize")

    def device_bytes(self):
        return int(lib().mmq_device_bytes(self._h))

    def comm_init(self, uid, rank, nranks):
        self._check(lib().mmq_comm_init(self._h, uid, rank, nranks), "mmq_comm_init")

    def comm_move_to(self, other):
        self._check(lib().mmq_comm_move(self._h, other._h), "mmq_comm_move")

    def p2p_export(self):
        buf = C.create_string_buffer(64)
        self._check(lib().mmq_p2p_export(self._h, buf), "mmq_p2p_export")
        return buf.raw

    def p2p_attach(self, handles, rank, nranks):
        """handles: the 64-byte exports of all ranks, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == 64 * nranks
        self._check(lib().mmq_p2p_attach(self._h, blob, rank, nranks), "mmq_p2p_attach")

    def p2p_attached(self):
        return int(lib().mmq_p2p_attached(self._h))

    def init_mu(self):
        uh = np.zeros(self.n, np.int32)
        self._check(lib().mmq_init_mu(self._h, _ptr(uh)), "mmq_init_mu")
        return uh

    def set_mu(self, mu):
        mu = _c(mu, np.float64)
        assert mu.shape == (self.n,)
        self._check(lib().mmq_set_mu(self._h, _ptr(mu)), "mmq_set_mu")

    def get_mu(self, out=None):
        mu = np.zeros(self.n) if out is None else out
        self._check(lib().mmq_get_mu(self._h, _ptr(mu)), "mmq_get_mu")
        return mu

    def loglik(self):
        v = C.c_double()
        self._check(lib().mmq_loglik(self._h, C.byref(v)), "mmq_loglik")
        return v.value

    def em(self, max_iter=1000, eps=0.1):
        it = C.c_int(); ll = C.c_double(); llr = C.c_double()
        self._check(lib().mmq_em(self._h, max_iter, eps, C.byref(it), C.byref(ll), C.byref(llr)), "mmq_em")
        return it.value, ll.value, llr.value

    def gibbs(self, seed, first_sweep, n_sweeps, stride=16, trace_len=0, flags=0):
        self._check(lib().mmq_gibbs(self._h, seed, first_sweep, n_sweeps, stride, trace_len, flags), "mmq_gibbs")

    def kernel_times(self):
        """(alloc_ms_total, alloc_launches, gamma_ms_total, gamma_launches) since the last call."""
        a = C.c_double(); an = C.c_int64(); g = C.c_double(); gn = C.c_int64()
        self._check(lib().mmq_kernel_times(self._h, C.byref(a), C.byref(an), C.byref(g), C.byref(gn)), "mmq_kernel_times")
        return a.value, an.value, g.value, gn.value

    def cls_stats(self):
        """Class plan of a collapsed shard: dict(in_use, small_classes, packed_slots, class_slots, rest_classes, rest_nnz,
        chain_classes, chain_slots)."""
        out = (C.c_int64 * 8)()
        self._check(lib().mmq_cls_stats(self._h, out), "mmq_cls_stats")
        return dict(zip(["in_use", "small_classes", "packed_slots", "class_slots", "rest_classes", "rest_nnz", "chain_classes", "chain_slots"], [int(v) for v in out]))

    def tune(self, knob, value):
        self._check(lib().mmq_tune(self._h, knob, value), "mmq_tune")

    def sweep_debug(self, seed, sweep, flags=MMQ_GIBBS_TRANSPOSED, want_x=True):
        x = np.zeros(self.nnz, np.int32) if (want_x and (flags & MMQ_GIBBS_TRANSPOSED)) else None
        counts = np.zeros(self.n, np.int32)
        mu = np.zeros(self.n)
        self._check(lib().mmq_sweep_debug(self._h, seed, sweep, flags, _ptr(x), _ptr(counts), _ptr(mu)), "mmq_sweep_debug")
        return x, counts, mu

    def trace_len(self):
        return int(lib().mmq_trace_len(self._h))

    def count_moments_begin(self, ident_of=None, n_ident=0, gene_of=None, n_gene=0):
        """Start accumulating posterior fragment counts; ident_of / gene_of: int32[n] group of each transcript or -1."""
        ident_of = _c(ident_of, np.int32); gene_of = _c(gene_of, np.int32)
        self._cnt_rows = [self.n, int(n_ident), int(n_gene)]
        self._check(lib().mmq_count_moments_begin(self._h, _ptr(ident_of), int(n_ident), _ptr(gene_of), int(n_gene)),
                    "mmq_count_moments_begin")

    def count_moments_end(self):
        self._check(lib().mmq_count_moments_end(self._h), "mmq_count_moments_end")

    def count_moments(self, which=0):
        """(sweeps, sum, sumsq_lo, sumsq_hi) of transcripts (0), identical sets (1) or genes (2); uint64 arrays,
        sum of squares = sumsq_hi * 2**64 + sumsq_lo."""
        rows = self._cnt_rows[which] if 0 <= which <= 2 else 0
        sweeps = C.c_int64()
        s = np.zeros(rows, np.uint64); lo = np.zeros(rows, np.uint64); hi = np.zeros(rows, np.uint64)
        self._check(lib().mmq_get_count_moments(self._h, which, C.byref(sweeps), _ptr(s), _ptr(lo), _ptr(hi)), "mmq_get_count_moments")
        return sweeps.value, s, lo, hi

    def expected_counts(self):
        """One E-step at the current mu: mu[t] * sum_{i containing t} k[i] w[i,t] / D_i over all shards."""
        out = np.zeros(self.n)
        self._check(lib().mmq_expected_counts(self._h, _ptr(out)), "mmq_expected_counts")
        return out

    def get_trace(self, out=None):
        """trace[t, slot]; `out`: a caller-provided (n, trace_len) float64 buffer (e.g. pinned memory)."""
        if out is None:
            out = np.zeros((self.n, self.trace_len()))
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.size == self.n * self.trace_len()
        self._check(lib().mmq_get_trace(self._h, _ptr(out)), "mmq_get_trace")
        return out

    def trace_cov(self, features, nsplit=2):
        """mmq_handle_trace_cov: covariance of the recorded traces of the given observed transcripts (C x C)."""
        features = _c(features, np.int32)
        Cn = len(features)
        R = np.zeros((Cn, Cn), np.float64, order="F")
        self._check(lib().mmq_handle_trace_cov(self._h, _ptr(features), Cn, nsplit, R.ctypes.data_as(C.c_void_p), None), "mmq_handle_trace_cov")
        return R

    def set_groups(self, kind, group_ptr, members, extra=None):
        group_ptr = _c(group_ptr, np.int64); members = _c(members, np.int32); extra = _c(extra, np.float64)
        self._ng = getattr(self, "_ng", {})
        self._ng[kind] = len(group_ptr) - 1
        self._check(lib().mmq_set_groups(self._h, kind, len(group_ptr) - 1, _ptr(group_ptr), _ptr(members), _ptr(extra)), "mmq_set_groups")

    def summarize(self, which, pct_idx=None):
        rows = self.n if which == 0 else self._ng[which - 1]
        lm = np.zeros(rows); var = np.zeros(rows); tau = np.zeros(rows)
        win = np.zeros(rows, np.int32); st = np.zeros(rows, np.int32)
        pct_idx = _c(pct_idx if pct_idx is not None else [], np.int32)
        pct = np.zeros((rows, len(pct_idx)))
        self._check(lib().mmq_summarize(self._h, which, _ptr(lm), _ptr(var), _ptr(tau), _ptr(win), _ptr(st),
                                        len(pct_idx), _ptr(pct_idx), _ptr(pct)), "mmq_summarize")
        return dict(log_mean=lm, var=var, tau=tau, win=win, status=st, pct=pct)

    def get_group_trace(self, which):
        out = np.zeros((self._ng[which - 1], self.trace_len()))
        self._check(lib().mmq_get_group_trace(self._h, which, _ptr(out)), "mmq_get_group_trace")
        return out

    def prop_summaries(self, gene_of, multi_iso, pct_idx=None, want_trace=False):
        gene_of = _c(gene_of, np.int32); multi_iso = _c(multi_iso, np.uint8)
        mp = np.zeros(self.n); sp = np.zeros(self.n); ssp = np.zeros(self.n)
        pct_idx = _c(pct_idx if pct_idx is not None else [], np.int32)
        pct = np.zeros((self.n, len(pct_idx)))
        tr = np.zeros((self.n, self.trace_len())) if want_trace else None
        self._check(lib().mmq_prop_summaries(self._h, _ptr(gene_of), _ptr(multi_iso), _ptr(mp), _ptr(sp), _ptr(ssp),
                                             len(pct_idx), _ptr(pct_idx), _ptr(pct), _ptr(tr)), "mmq_prop_summaries")
        return dict(mean_prop=mp, sum_probit=sp, sumsq_probit=ssp, pct=pct, prop_trace=tr)

    def allele_only_counts(self, unit_of, side, nunits):
        """mmq_allele_only_counts: (a_only, b_only) int32[nunits]; unit_of int32[n] (-1: none), side uint8[n] (0 A, 1 B)."""
        unit_of = _c(unit_of, np.int32); side = _c(side, np.uint8)
        a = np.zeros(nunits, np.int32); b = np.zeros(nunits, np.int32)
        self._check(lib().mmq_allele_only_counts(self._h, _ptr(unit_of), _ptr(side), nunits, _ptr(a), _ptr(b)), "mmq_allele_only_counts")
        return a, b

    def pair_shared_counts(self, gene_of, local_of, pair_base, npairs):
        """mmq_pair_shared_counts: int64[npairs]; gene_of / local_of int32[n] (-1: no pair), pair_base int64[ngenes]."""
        gene_of = _c(gene_of, np.int32); local_of = _c(local_of, np.int32); pair_base = _c(pair_base, np.int64)
        out = np.zeros(npairs, np.int64)
        self._check(lib().mmq_pair_shared_counts(self._h, _ptr(gene_of), _ptr(local_of), _ptr(pair_base), len(pair_base), npairs, _ptr(out)),
                    "mmq_pair_shared_counts")
        return out

    def unique_hits_sets(self, set_of, nsets):
        set_of = _c(set_of, np.int32)
        out = np.zeros(nsets, np.int32)
        self._check(lib().mmq_unique_hits_sets(self._h, _ptr(set_of), nsets, _ptr(out)), "mmq_unique_hits_sets")
        return out
