"""numpy restatement of transcripts per million over the recorded draws (mmq_draw_totals_dev, mmq_tpm_summaries_dev,
include/mmq.h; `mmseq -tpm`):
  1. the per-draw totals of the observed transcripts, exactly (math.fsum) and in the kernel's tile order;
  2. a feature's TPM draws, (w / D) * 1e6 with w its members' draws summed in CSR order;
  3. mean, two-pass sd and the NaN-last percentiles over the S = C L draws;
  4. the EM TPM from the EM estimate."""
import math

import numpy as np

from tests.pool_reference import pct_index  # noqa: F401  (the percentile rule: round(p / 100 (S - 1)))

TILE = 512  # rows per tile of k_draw_totals


def totals_fsum(trace):
    """trace (n, L) -> fp64[L], the correctly rounded sum of each column"""
    trace = np.asarray(trace, np.float64)
    return np.array([math.fsum(trace[:, s]) for s in range(trace.shape[1])])


def totals_tiled(trace):
    """trace (n, L) -> fp64[L] in the kernel's order: tiles of TILE rows, each summed in row order from 0.0, then the tile
    sums in tile order from 0.0"""
    trace = np.asarray(trace, np.float64)
    n, L = trace.shape
    tot = np.zeros(L)
    for t0 in range(0, n, TILE):
        acc = np.zeros(L)
        for t in range(t0, min(n, t0 + TILE)):
            acc = acc + trace[t]
        tot = tot + acc
    return tot


def tpm_draws(chains, totals, members):
    """chains (C, n, L) transcript traces, totals (C, L), members: the feature's transcript indices in CSR order ->
    (C, L) TPM draws, (w / D) * 1e6 in that expression order"""
    chains = np.asarray(chains, np.float64)
    w = np.zeros((chains.shape[0], chains.shape[2]))
    for m in members:
        w = w + chains[:, m, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        return (w / np.asarray(totals, np.float64)) * 1e6


def summaries(draws, idx):
    """draws (C, L) of one feature -> (mean, sd, pct[len(idx)]); mean and sd NaN when any draw is not finite; the sorted
    draws (NaN last) at idx, NaN for an index outside [0, S)"""
    x = np.asarray(draws, np.float64).ravel()
    S = x.size
    srt = np.sort(x)                                                     # numpy sorts NaN last
    pct = np.array([srt[q] if 0 <= q < S else math.nan for q in idx])
    if not np.isfinite(x).all():
        return math.nan, math.nan, pct
    mean = float(np.sum(x) / S)
    sd = math.sqrt(float(np.sum((x - mean) ** 2)) / (S - 1))
    return mean, sd, pct


def features(chains, totals, group_ptr, members, idx):
    """every feature of a CSR (group_ptr None: one feature per transcript) -> dict(mean, sd: fp64[rows]; pct (rows, npct))"""
    n = np.asarray(chains).shape[1]
    rows = n if group_ptr is None else len(group_ptr) - 1
    out = dict(mean=np.zeros(rows), sd=np.zeros(rows), pct=np.zeros((rows, len(idx))))
    for r in range(rows):
        mem = [r] if group_ptr is None else members[group_ptr[r]:group_ptr[r + 1]]
        out["mean"][r], out["sd"][r], out["pct"][r] = summaries(tpm_draws(chains, totals, mem), idx)
    return out


def em_tpm(mu_em, members):
    """(sum of the members' mu_em / sum of all mu_em) * 1e6, both sums in index order; 0 without members"""
    tot = 0.0
    for v in mu_em:
        tot += float(v)
    w = 0.0
    for m in members:
        w += float(mu_em[m])
    return (w / tot) * 1e6
