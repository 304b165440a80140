"""numpy restatement of the summaries over the pooled draws of several chains (mmq_pooled_summaries_dev, include/mmq.h;
`mmseq -chains C -pool`), built on tests/chain_reference.py: the tables' log_mu, sd, mcse, iact and percentiles over
all S = C L draws, the proportion columns, and the exact sum of the chains' count moments."""
import math

import numpy as np
from scipy.special import ndtri

from tests import chain_reference as cref


def pct_index(percentiles, S):
    """round(p / 100 (S - 1)), half away from zero as C's round(): the rule of src/mmseq.cpp:1113 with S draws"""
    out = []
    for p in percentiles:
        v = p / 100.0 * (S - 1)
        f = math.floor(v)
        out.append(int(f + 1) if v - f >= 0.5 else int(f))
    return np.array(out, np.int32)


def percentiles(x, idx):
    """the pooled draws sorted ascending (NaN last) at the indices idx"""
    return np.sort(np.asarray(x, np.float64).ravel())[np.asarray(idx)]


def pooled_log(x):
    """x: (C, L) draws of one feature -> (log_mean, sd, ess_mean, smallest ESS branch margin).  log_mean and sd over all
    S draws (NaN when any x is not finite, plain IEEE otherwise); ess_mean: chain_reference.ess on the split chains of
    log x, NaN when any log x is not finite or all are equal."""
    x = np.asarray(x, np.float64)
    C, L = x.shape
    S = C * L
    if not np.isfinite(x).all():
        return math.nan, math.nan, math.nan, math.inf
    with np.errstate(divide="ignore", invalid="ignore"):
        lx = np.log(x)
        log_mean = float(np.sum(lx) / S)
        sd = math.sqrt(float(np.sum((lx - log_mean) ** 2)) / (S - 1))
    if not np.isfinite(lx).all():
        return log_mean, sd, math.nan, math.inf
    ess, margin = cref.ess(cref.split(lx))
    return log_mean, sd, ess, margin


def mcse_iact(sd, ess, S):
    """the tables' mcse = sd / sqrt(ess_mean) and iact = S / ess_mean; NaN with ess_mean"""
    if math.isnan(ess):
        return math.nan, math.nan
    return sd / math.sqrt(ess), S / ess


def pooled_rows(chains, idx):
    """chains: (C, rows, L) -> dict(log_mean, sd, ess_mean, margin: fp64[rows]; pct: (rows, len(idx)))"""
    chains = np.asarray(chains, np.float64)
    C, rows, L = chains.shape
    out = {k: np.zeros(rows) for k in ("log_mean", "sd", "ess_mean", "margin")}
    out["pct"] = np.zeros((rows, len(idx)))
    for r in range(rows):
        x = chains[:, r, :]
        out["log_mean"][r], out["sd"][r], out["ess_mean"][r], out["margin"][r] = pooled_log(x)
        out["pct"][r] = percentiles(x, idx)
    return out


def probit_sums(p, multi):
    """one chain's sum and sum of squares of Phi^-1(clamp(p, 1e-9, 1 - 1e-9)) (+inf for a single-isoform gene), as
    k_prop adds them (src/mmseq.cpp:1249-1255)"""
    if not multi:
        return math.inf, math.inf
    with np.errstate(invalid="ignore"):
        z = ndtri(np.clip(p, 1e-9, 1 - 1e-9))
    return float(np.sum(z)), float(np.sum(z * z))


def pooled_props(mu, gene, multi, idx):
    """mu, gene: (C, L) draws of a transcript and of its gene, chain by chain -> dict(mean, mean_probit, sd_probit, pct).
    Each chain's proportions are mu / its own gene trace; the chains' probit sums are added in chain order and finished
    as src/mmseq.cpp:1260-1265 with S draws: a single-isoform gene gives mean_probit inf and sd_probit NaN."""
    mu = np.asarray(mu, np.float64)
    C, L = mu.shape
    S = C * L
    with np.errstate(divide="ignore", invalid="ignore"):
        p = mu / np.asarray(gene, np.float64)
    s1 = s2 = 0.0
    for c in range(C):
        a, b = probit_sums(p[c], multi)
        s1, s2 = (a, b) if c == 0 else (s1 + a, s2 + b)
    with np.errstate(invalid="ignore"):
        sd = float(np.sqrt(np.float64((s2 - s1 * s1 / S) / (S - 1.0))))
    return dict(mean=float(np.sum(p) / S), mean_probit=s1 / S, sd_probit=sd, pct=percentiles(p, idx))


def add_count_moments(moments):
    """[(sweeps, sum, sumsq_lo, sumsq_hi) per chain] -> (S, sum, sumsq) as exact Python integers per row"""
    S = sum(int(m[0]) for m in moments)
    rows = len(moments[0][1])
    tot = [sum(int(m[1][r]) for m in moments) for r in range(rows)]
    sq = [sum((int(m[3][r]) << 64) + int(m[2][r]) for m in moments) for r in range(rows)]
    return S, tot, sq


def count_columns(S, tot, sq):
    """posterior_mean_count and posterior_sd_count from the pooled moments (count_sd of the host program)"""
    mean = [t / S for t in tot]
    sd = [math.sqrt(float(S * q - t * t) / (float(S) * float(S - 1))) if S > 1 else 0.0 for t, q in zip(tot, sq)]
    return mean, sd
