"""numpy restatement of the allelic fraction of haplotype pairs (mmq_allele_only_counts, mmq_allelic_summaries_dev,
include/mmq.h; `mmseq -allelic`):
  1. pairs: header transcripts STEM_A and STEM_B of one gene, in the header order of the _A copy; genes: the pairs
     inside each gene, in pair order;
  2. members in column space: an id m < n is row m of a chain's trace, n + j row j of its prior draws;
  3. per draw a, b = the A and B members' draws summed in CSR order from 0.0, phi = a / (a + b);
  4. over the S = C L draws: mean, two-pass sd, P(a > b) with ties counting one half, the NaN-last percentiles; every
     one NaN when any phi is not finite;
  5. the EM fraction from the EM estimate over the observed members;
  6. the allele-only fragments: sum of k over the rows holding an A member of the unit and no B member (and swapped)."""
import math

import numpy as np

from tests.pool_reference import pct_index  # noqa: F401  (the percentile rule: round(p / 100 (S - 1)))


def find_pairs(names, gene_of):
    """-> (a, b, stems, lonely): header indices of each pair's _A and _B copy, the pair ids, and the number of transcripts
    named *_A / *_B without a partner in their gene"""
    index = {}
    for t, nm in enumerate(names):
        index.setdefault(nm, t)
    a, b, stems = [], [], []
    paired = set()
    for t, nm in enumerate(names):
        if len(nm) < 2 or not nm.endswith("_A"):
            continue
        u = index.get(nm[:-2] + "_B")
        if u is None or gene_of[u] != gene_of[t]:
            continue
        a.append(t)
        b.append(u)
        stems.append(nm[:-2])
        paired.update((t, u))
    lonely = sum(1 for t, nm in enumerate(names) if len(nm) >= 2 and nm[-2:] in ("_A", "_B") and t not in paired)
    return a, b, stems, lonely


def gene_units(a, gene_of, G):
    """the pair indices inside every gene, in pair order"""
    units = [[] for _ in range(G)]
    for p, t in enumerate(a):
        units[gene_of[t]].append(p)
    return units


def csr(units, a_ids, b_ids):
    """units: a list of pair-index lists; a_ids / b_ids: each pair's member id -> (a_ptr, a_mem, b_ptr, b_mem)"""
    a_ptr, b_ptr, a_mem, b_mem = [0], [0], [], []
    for ps in units:
        a_mem += [a_ids[p] for p in ps]
        b_mem += [b_ids[p] for p in ps]
        a_ptr.append(len(a_mem))
        b_ptr.append(len(b_mem))
    return (np.array(a_ptr, np.int64), np.array(a_mem, np.int32), np.array(b_ptr, np.int64), np.array(b_mem, np.int32))


def side_sum(chains, priors, members):
    """chains (C, n, L), priors (C, nprior, L) or None -> (C, L): the members' draws summed in CSR order from 0.0"""
    chains = np.asarray(chains, np.float64)
    n = chains.shape[1]
    w = np.zeros((chains.shape[0], chains.shape[2]))
    for m in members:
        w = w + (chains[:, m, :] if m < n else np.asarray(priors, np.float64)[:, m - n, :])
    return w


def fraction(chains, priors, a_mem, b_mem):
    """-> (a, b, phi), each (C, L)"""
    a, b = side_sum(chains, priors, a_mem), side_sum(chains, priors, b_mem)
    with np.errstate(divide="ignore", invalid="ignore"):
        return a, b, a / (a + b)


def summaries(a, b, phi, idx):
    """-> (mean, sd, prob_a, pct[len(idx)]) over the S draws; all NaN when any phi is not finite"""
    x = np.asarray(phi, np.float64).ravel()
    S = x.size
    if not np.isfinite(x).all():
        return math.nan, math.nan, math.nan, np.full(len(idx), math.nan)
    srt = np.sort(x)
    pct = np.array([srt[q] if 0 <= q < S else math.nan for q in idx])
    mean = float(np.sum(x) / S)
    sd = math.sqrt(float(np.sum((x - mean) ** 2)) / (S - 1))
    a, b = np.asarray(a).ravel(), np.asarray(b).ravel()
    prob = (int(np.sum(a > b)) + 0.5 * int(np.sum(a == b))) / S
    return mean, sd, prob, pct


def units(chains, priors, a_ptr, a_mem, b_ptr, b_mem, idx):
    """every unit of the CSRs -> dict(mean, sd, prob_a: fp64[rows]; pct (rows, npct))"""
    rows = len(a_ptr) - 1
    out = dict(mean=np.zeros(rows), sd=np.zeros(rows), prob_a=np.zeros(rows), pct=np.zeros((rows, len(idx))))
    for r in range(rows):
        a, b, phi = fraction(chains, priors, a_mem[a_ptr[r]:a_ptr[r + 1]], b_mem[b_ptr[r]:b_ptr[r + 1]])
        out["mean"][r], out["sd"][r], out["prob_a"][r], out["pct"][r] = summaries(a, b, phi, idx)
    return out


def em_fraction(mu_em, a_mem, b_mem):
    """sum_A mu_em / (sum_A + sum_B) over the observed members (id < len(mu_em)) in index order; NaN when both are 0"""
    n = len(mu_em)
    sa = sb = 0.0
    for m in a_mem:
        if m < n:
            sa += float(mu_em[m])
    for m in b_mem:
        if m < n:
            sb += float(mu_em[m])
    return math.nan if sa == 0.0 and sb == 0.0 else sa / (sa + sb)


def allele_only(row_ptr, col, k, unit_of, side, nunits):
    """-> (a_only, b_only) int64[nunits]: per row (weight k[i], or 1 when k is None) the units with members of one side
    only"""
    a_only = np.zeros(nunits, np.int64)
    b_only = np.zeros(nunits, np.int64)
    for i in range(len(row_ptr) - 1):
        seen = {}
        for c in col[row_ptr[i]:row_ptr[i + 1]]:
            u = int(unit_of[c])
            if u >= 0:
                seen.setdefault(u, set()).add(int(side[c]))
        w = 1 if k is None else int(k[i])
        for u, sides in seen.items():
            if sides == {0}:
                a_only[u] += w
            elif sides == {1}:
                b_only[u] += w
    return a_only, b_only
