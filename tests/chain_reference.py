"""numpy / scipy restatement of the convergence diagnostics of several chains (mmq_chain_diagnostics_dev, include/mmq.h):
rank-normalised split-R-hat and bulk / tail ESS (Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021), and the pooled
log-scale mean and sd.  It follows the definitions line by line, with a direct-sum autocovariance (no FFT), and reports
for every row the smallest margin of the ESS's branch decisions that can change its result by more than their margin, so
that a test can exempt rows whose result depends on the last bits."""
import math

import numpy as np
from scipy.special import ndtri
from scipy.stats import rankdata

OUTPUTS = ("rhat", "ess_bulk", "ess_tail", "log_mean", "log_sd")
STREAM_CHAIN = 0x4348414E  # "CHAN"
CHAINS_MAX = 8


def philox4x32_10(ctr, k0, k1):
    """Philox4x32-10 (include/mmq_sampler.h): the four output words."""
    M0, M1, W0, W1, m32 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF
    c0, c1, c2, c3 = ctr
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> 32) ^ c3 ^ k1) & m32, p0 & m32
        k0, k1 = (k0 + W0) & m32, (k1 + W1) & m32
    return c0, c1, c2, c3


def chain_seeds(seed, nchains):
    """mmq_chain_seed(seed, c) for c < nchains: chain 0 is the seed; chain c takes word 0 of Philox at counter
    (c, j, 0, 0), key (seed, CHAN), for the first j whose value differs from the seeds of chains 0 .. c-1."""
    seeds = [seed]
    for c in range(1, nchains):
        j = 0
        while True:
            v = philox4x32_10((c, j, 0, 0), seed, STREAM_CHAIN)[0]
            if v not in seeds:
                seeds.append(v)
                break
            j += 1
    return seeds


def rank_normalise(v):
    """z = Phi^-1((r - 3/8) / (S + 1/4)), r the average ranks over all S values."""
    return ndtri((rankdata(v, method="average") - 0.375) / (v.size + 0.25))


def split(x):
    """(C, L) draws -> (2C, L/2) split chains, y[2c+h][i] = x[c][h N + i]."""
    C, L = x.shape
    return x.reshape(2 * C, L // 2)


def split_moments(y):
    """Means and variances (ddof 1) of the split chains; a split chain whose values are all equal has exactly that
    value as its mean and variance 0."""
    same = (y == y[:, :1]).all(axis=1)
    m = np.where(same, y[:, 0], y.mean(axis=1))
    w = np.where(same, 0.0, y.var(axis=1, ddof=1))
    return m, w


def rhat(y):
    N = y.shape[1]
    m, w = split_moments(y)
    W = w.mean()
    B = N * m.var(ddof=1)
    if W == 0:
        return math.nan
    return math.sqrt(((N - 1) / N * W + B / N) / W)


def ess(y):
    """Geyer's initial monotone sequence as ArviZ's _ess; (ess, smallest margin of a branch decision).  The margins are
    those of the tests on even + odd, which decide how many lags enter the sum.  The other decisions (even > 0, the
    monotone step, the floor of tau) change the result by no more than their margin, so rounding cannot move it."""
    M, N = y.shape
    if (y == y.flat[0]).all():
        return math.nan, math.inf
    m, _ = split_moments(y)
    yc = y - m[:, None]
    cache = {}

    def mean_acov(t):
        if t not in cache:
            cache[t] = float(np.mean(np.einsum("ji,ji->j", yc[:, :N - t], yc[:, t:]) / N))
        return cache[t]

    mean_var = mean_acov(0) * N / (N - 1)
    var_plus = mean_var * (N - 1) / N + m.var(ddof=1)
    if not var_plus > 0:
        return math.nan, math.inf

    def rho(t):
        return 1.0 - (mean_var - mean_acov(t)) / var_plus

    margin = math.inf
    r = np.zeros(N)
    r[0] = 1.0
    r[1] = rho(1)
    even, odd = 1.0, r[1]
    t = 1
    while True:
        if not t < N - 3:
            break
        margin = min(margin, abs(even + odd))
        if not even + odd > 0:
            break
        even, odd = rho(t + 1), rho(t + 2)
        margin = min(margin, abs(even + odd))
        if even + odd >= 0:
            r[t + 1], r[t + 2] = even, odd
        t += 2
    max_t = t - 2
    if even > 0:
        r[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        if r[t + 1] + r[t + 2] > r[t - 1] + r[t]:
            r[t + 1] = (r[t - 1] + r[t]) / 2.0
            r[t + 2] = r[t + 1]
        t += 2
    SN = M * N
    tau = -1.0 + 2.0 * float(np.sum(r[:max_t + 1])) + r[max_t + 1]
    return SN / max(tau, 1.0 / math.log10(SN)), margin


def quantile7(v_sorted, p):
    S = v_sorted.size
    h = (S - 1) * p
    f = math.floor(h)
    return v_sorted[f] + (h - f) * (v_sorted[f + 1] - v_sorted[f])


def diagnose(x):
    """x: (C, L) draws of one feature -> (dict of OUTPUTS, smallest ESS branch margin)."""
    x = np.asarray(x, np.float64)
    C, L = x.shape
    S = C * L
    nan = dict.fromkeys(OUTPUTS, math.nan)
    if not np.isfinite(x).all():
        return nan, math.inf
    v = x.ravel()
    with np.errstate(divide="ignore", invalid="ignore"):
        lx = np.log(v)
        log_mean = float(np.sum(lx) / S)
        log_sd = math.sqrt(float(np.sum((lx - log_mean) ** 2)) / (S - 1))
    vs = np.sort(v)
    med = 0.5 * (vs[S // 2 - 1] + vs[S // 2])
    zb = split(rank_normalise(v).reshape(C, L))
    zf = split(rank_normalise(np.abs(v - med)).reshape(C, L))
    rb, rf = rhat(zb), rhat(zf)
    eb, mb = ess(zb)
    tails = [ess(split((x <= quantile7(vs, p)).astype(np.float64))) for p in (0.05, 0.95)]
    et = math.nan if any(math.isnan(e) for e, _ in tails) else min(e for e, _ in tails)
    out = dict(rhat=math.nan if math.isnan(rb) or math.isnan(rf) else max(rb, rf), ess_bulk=eb, ess_tail=et,
               log_mean=log_mean, log_sd=log_sd)
    return out, min([mb] + [m for _, m in tails])


def diagnose_rows(chains):
    """chains: (C, rows, L) -> (dict of OUTPUTS, each fp64[rows]; margins fp64[rows])."""
    chains = np.asarray(chains, np.float64)
    C, rows, L = chains.shape
    out = {k: np.zeros(rows) for k in OUTPUTS}
    margin = np.zeros(rows)
    for r in range(rows):
        d, margin[r] = diagnose(chains[:, r, :])
        for k in OUTPUTS:
            out[k][r] = d[k]
    return out, margin
