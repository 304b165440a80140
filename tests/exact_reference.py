"""Exact distributions of the Gibbs sampler's steps, in plain fp64 numpy / scipy (no oracle library), and the
statistics that compare sampled values with them.

One allocation step at fixed mu
  A hit class of k fragments over d members gives x ~ Multinomial(k; p), p_j = mu_j w_j / sum.  Per-fragment rows
  (k = 1 each, own weights) that share members give a sum of independent categoricals.

One Gamma step
  mu'_t ~ Gamma(alpha + c_t, rate beta + l_t), so u = P(alpha + c_t, (beta + l_t) mu'_t) (regularised lower incomplete
  gamma function) is uniform on (0, 1) given the counts.

The stationary posterior of one component
  d members, one class of k fragments shared by all of them, and u_j fragments that only member j explains (singleton
  classes).  The sampler alternates x | mu ~ Multinomial(k; mu w / sum) and mu_j | x ~ Gamma(alpha + u_j + x_j,
  beta + l_j); its stationary law has p(x) proportional to prod_j exp(f_j(x_j)) on sum_j x_j = k, with
      f_j(x) = x log w_j - log x! + log Gamma(alpha + u_j + x) - (alpha + u_j + x) log(beta + l_j),
  and mu_j | x_j ~ Gamma(alpha + u_j + x_j, beta + l_j).  For d = 2 members and G one-fragment rows with their own
  weights, sum over the rows' choices with a DP instead: the weight of n_1 = x is the sum over x-subsets of rows of
  prod w_r1 (chosen) prod w_r2 (not chosen), and the x! terms drop out.
"""
import itertools

import numpy as np
from scipy import optimize, special, stats

Z_MAX = 5.0        # a test fails on any |z| above this
P_MIN = 1e-6       # ... or on any chi-square / KS p-value below this
# A variance or covariance statistic is only formed when its target, summed over the draws, is at least this: below it
# the statistic rests on a handful of rare events, its sample standard error is no guide, and the normal approximation
# fails (a pair that should co-occur 1.5 times in 12000 draws and never does gives z = -5).  The means of such members
# are still tested, and their binomial marginals by chi-square.
MIN_SIGNAL = 200.0


# ------------------------------------------------------------------ one allocation step

def member_probs(mu, w=None):
    """p_j = mu_j w_j / sum, in fp64."""
    p = np.asarray(mu, np.float64) * (1.0 if w is None else np.asarray(w, np.float64))
    return p / p.sum()


def multinomial_moments(k, p):
    """Mean k p_j and covariance matrix (k p_j (1 - p_j) on the diagonal, -k p_i p_j off it) of Multinomial(k; p)."""
    p = np.asarray(p, np.float64)
    cov = -float(k) * np.outer(p, p)
    cov[np.diag_indices_from(cov)] = k * p * (1.0 - p)
    return k * p, cov


def categorical_sum_moments(P):
    """Counts summed over independent categorical draws, row r picking member j with probability P[r, j]: mean
    sum_r p_rj, variance sum_r p_rj (1 - p_rj), covariance -sum_r p_ri p_rj."""
    P = np.asarray(P, np.float64)
    cov = -(P.T @ P)
    cov[np.diag_indices_from(cov)] = (P * (1.0 - P)).sum(axis=0)
    return P.sum(axis=0), cov


def binomial_marginal_pmf(k, pj):
    """pmf of x_j ~ Binomial(k, p_j) on 0..k."""
    return stats.binom.pmf(np.arange(k + 1), k, pj)


def multinomial_pmf(k, p):
    """Every composition of k into len(p) parts (rows of X) and its Multinomial(k; p) probability."""
    d = len(p)
    X = np.array([c for c in itertools.product(range(k + 1), repeat=d - 1) if sum(c) <= k], np.int64).reshape(-1, d - 1)
    X = np.hstack([X, k - X.sum(axis=1, keepdims=True)])
    return X, stats.multinomial.pmf(X, k, p)


# ------------------------------------------------------------------ one Gamma step

def gamma_pit(mu_new, counts, length, alpha, beta):
    """P(alpha + c, (beta + l) mu'): uniform on (0, 1) when mu' ~ Gamma(alpha + c, rate beta + l)."""
    return special.gammainc(alpha + np.asarray(counts, np.float64), (beta + np.asarray(length, np.float64)) * mu_new)


# ------------------------------------------------------------------ exact stationary posterior

def _logconv(a, b):
    """log of the convolution of exp(a) and exp(b) on 0..len(a)-1, by logsumexp over each antidiagonal (exact in the
    tails, where scaling and exponentiating would underflow)."""
    n = len(a)
    s = np.arange(n)
    idx = s[:, None] - s[None, :]
    M = a[None, :] + np.where(idx >= 0, b[np.clip(idx, 0, None)], -np.inf)
    return special.logsumexp(M, axis=1)


def _sample_log_pmf(rng, logp):
    """One index per row of logp (rows: unnormalised log probabilities, -inf allowed), by inversion."""
    p = np.exp(logp - logp.max(axis=1, keepdims=True))
    c = np.cumsum(p, axis=1)
    u = rng.random(len(p)) * c[:, -1]
    return np.minimum((c < u[:, None]).sum(axis=1), logp.shape[1] - 1)


class _Posterior:
    """Marginals of mu_j given the exact pmf of the member's count (self.pmf(j) on 0..K)."""

    def __init__(self, u, length, alpha, beta):
        self.u = np.asarray(u, np.float64)
        self.rate = beta + np.asarray(length, np.float64)
        self.alpha, self.beta = alpha, beta
        self.d = len(self.u)

    def shapes(self, j):
        return self.alpha + self.u[j] + np.arange(len(self.pmf(j)))

    def e_log_mu(self, j):
        """E[log mu_j] = sum_x P(x) (psi(alpha + u_j + x) - log(beta + l_j))."""
        return float(self.pmf(j) @ (special.digamma(self.shapes(j)) - np.log(self.rate[j])))

    def cdf_mu(self, j, q):
        """P(mu_j <= q): the Gamma mixture."""
        return float(self.pmf(j) @ special.gammainc(self.shapes(j), self.rate[j] * q))

    def quantile_mu(self, j, prob):
        lo, hi = 1e-300, 1.0
        while self.cdf_mu(j, hi) < prob:
            hi *= 4.0
        return optimize.brentq(lambda q: self.cdf_mu(j, q) - prob, lo, hi, xtol=1e-300, rtol=1e-14)

    def sample_mu(self, rng, R):
        """R exact stationary draws of mu (R, d): counts from sample_counts, then the Gamma step."""
        x = self.sample_counts(rng, R)
        return rng.gamma(self.alpha + self.u[None, :] + x, 1.0 / self.rate[None, :])


class SharedClass(_Posterior):
    """d members, one class of k fragments shared by all, singleton counts u_j, lengths l_j, class weights w_j."""

    def __init__(self, k, u, length, alpha, beta, w=None):
        super().__init__(u, length, alpha, beta)
        self.k = int(k)
        w = np.ones(self.d) if w is None else np.asarray(w, np.float64)
        x = np.arange(self.k + 1, dtype=np.float64)
        a = self.alpha + self.u[:, None] + x[None, :]
        self.f = x[None, :] * np.log(w)[:, None] - special.gammaln(x + 1.0)[None, :] + special.gammaln(a) - a * np.log(self.rate)[:, None]
        # pre[m]: members 0..m-1 convolved; suf[m]: members m..d-1
        zero = np.full(self.k + 1, -np.inf)
        zero[0] = 0.0
        self.pre = [zero]
        for j in range(self.d):
            self.pre.append(_logconv(self.pre[-1], self.f[j]))
        self.suf = [zero]
        for j in range(self.d - 1, -1, -1):
            self.suf.insert(0, _logconv(self.suf[0], self.f[j]))
        self._pmf = {}

    def pmf(self, j):
        if j not in self._pmf:
            others = _logconv(self.pre[j], self.suf[j + 1])
            lp = self.f[j] + others[::-1]                  # x_j = x, the others share k - x
            p = np.exp(lp - lp.max())
            self._pmf[j] = p / p.sum()
        return self._pmf[j]

    def sample_counts(self, rng, R):
        """Exact draws of x (R, d): backward through the prefix tables, member d-1 first."""
        x = np.zeros((R, self.d), np.int64)
        s = np.full(R, self.k)
        xs = np.arange(self.k + 1)
        for j in range(self.d - 1, 0, -1):
            rest = s[:, None] - xs[None, :]
            lp = self.f[j][None, :] + np.where(rest >= 0, self.pre[j][np.clip(rest, 0, None)], -np.inf)
            x[:, j] = _sample_log_pmf(rng, lp)
            s = s - x[:, j]
        x[:, 0] = s
        return x


class WeightedRowsPair(_Posterior):
    """d = 2 members, G one-fragment rows over both (row r: weights W[r, 0], W[r, 1]), singleton counts u_j."""

    def __init__(self, W, u, length, alpha, beta):
        super().__init__(u, length, alpha, beta)
        W = np.asarray(W, np.float64)
        self.G = len(W)
        # e[x] = log of the sum over x-subsets S of rows of prod_{S} W[r, 0] prod_{not S} W[r, 1]
        e = np.full(self.G + 1, -np.inf)
        e[0] = 0.0
        with np.errstate(divide="ignore"):
            lw = np.log(W)
        for r in range(self.G):
            take = np.concatenate([[-np.inf], e[:-1] + lw[r, 0]])
            e = np.logaddexp(take, e + lw[r, 1])
        x = np.arange(self.G + 1, dtype=np.float64)
        a0, a1 = self.alpha + self.u[0] + x, self.alpha + self.u[1] + self.G - x
        lp = e + special.gammaln(a0) - a0 * np.log(self.rate[0]) + special.gammaln(a1) - a1 * np.log(self.rate[1])
        p = np.exp(lp - lp.max())
        self.p0 = p / p.sum()

    def pmf(self, j):
        return self.p0 if j == 0 else self.p0[::-1]

    def sample_counts(self, rng, R):
        x0 = _sample_log_pmf(rng, np.log(np.broadcast_to(self.p0, (R, self.G + 1))))
        return np.stack([x0, self.G - x0], axis=1)


# ------------------------------------------------------------------ statistics

def moment_z(X, mean, var, cov_of):
    """z-scores of the sample means, variances and covariances of X (N draws, d members) against the exact ones.
    mean and var broadcast against X (one target for all draws, or one per draw); cov_of(i, j) gives the covariance
    (a scalar or one per draw).  The variance and covariance statistics are means of (products of) deviations from the
    EXACT mean minus their exact expectation, so each has expectation 0; their standard errors come from the sample.
    Members with zero exact variance in every draw are skipped: callers assert those exactly.  All pairs for d <= 16,
    neighbours and pairs with member 0 above.  Returns (worst z, description)."""
    X = np.asarray(X, np.float64)
    N, d = X.shape
    D = X - mean
    V = np.broadcast_to(var, X.shape)
    worst = (0.0, "none")

    def take(y, what):
        nonlocal worst
        se = y.std() / np.sqrt(N)
        z = y.mean() / se if se > 0 else (0.0 if y.mean() == 0 else np.inf)
        if abs(z) > abs(worst[0]):
            worst = (float(z), what)

    for j in range(d):
        if V[:, j].sum() > 0.0:
            z = D[:, j].sum() / np.sqrt(V[:, j].sum())
            if abs(z) > abs(worst[0]):
                worst = (float(z), f"mean of member {j}")
        if V[:, j].sum() >= MIN_SIGNAL:
            take(D[:, j] ** 2 - V[:, j], f"variance of member {j}")
    pairs = [(i, j) for i in range(d) for j in range(i + 1, d)] if d <= 16 else \
        sorted({(j, j + 1) for j in range(d - 1)} | {(0, j) for j in range(2, d)})
    for i, j in pairs:
        c = np.broadcast_to(cov_of(i, j), (N,))
        if np.abs(c).sum() >= MIN_SIGNAL:
            take(D[:, i] * D[:, j] - c, f"covariance of members {i}, {j}")
    return worst


def chi2_pvalue(values, pmf):
    """Chi-square goodness of fit of integer samples (support 0..len(pmf)-1) against pmf.  Cells whose expected count
    is below 5 are pooled into one cell."""
    values = np.asarray(values, np.int64)
    N = len(values)
    obs = np.bincount(values, minlength=len(pmf)).astype(np.float64)
    if len(obs) > len(pmf):                                # a value outside the support: certain failure
        return 0.0
    exp = N * np.asarray(pmf, np.float64)
    big = exp >= 5.0
    o = np.concatenate([obs[big], [obs[~big].sum()]])
    e = np.concatenate([exp[big], [exp[~big].sum()]])
    if e[-1] < 1e-12:
        if o[-1] > 0:
            return 0.0
        o, e = o[:-1], e[:-1]
    if len(e) < 2:
        return 1.0
    return float(stats.chi2.sf(((o - e) ** 2 / e).sum(), len(e) - 1))


def joint_chi2_pvalue(X, k, p):
    """Chi-square of whole allocation vectors (small d and k) against the multinomial pmf."""
    C, pm = multinomial_pmf(k, p)
    base = (k + 1) ** np.arange(len(p))
    where = {int(v): i for i, v in enumerate(C @ base)}
    codes = np.asarray(X, np.int64) @ base
    idx = np.array([where.get(int(c), -1) for c in codes])
    if (idx < 0).any():
        return 0.0
    return chi2_pvalue(idx, pm)


def assert_multinomial(X, k, p, what):
    """X (N, d): draws that should be Multinomial(k; p).  Exact checks: every row sums to k, members with p = 0 get
    nothing.  Statistical checks: moments; the binomial marginal of every member for k <= 1000; whole vectors for
    d <= 3, k <= 40."""
    X = np.asarray(X, np.int64)
    p = np.asarray(p, np.float64)
    assert (X.sum(axis=1) == k).all(), f"{what}: a row does not sum to k = {k}"
    assert (X[:, p == 0.0] == 0).all(), f"{what}: a member with p = 0 received a fragment"
    mean, cov = multinomial_moments(k, p)
    z, where = moment_z(X, mean, np.diag(cov), lambda i, j: cov[i, j])
    assert abs(z) <= Z_MAX, f"{what}: worst z = {z:.2f} ({where}), N = {len(X)}"
    if 1 <= k <= 1000:
        pv = [(chi2_pvalue(X[:, j], binomial_marginal_pmf(k, p[j])), j) for j in range(len(p)) if 0.0 < p[j] < 1.0]
        worst = min(pv) if pv else (1.0, -1)
        assert worst[0] >= P_MIN, f"{what}: binomial marginal of member {worst[1]}: chi-square p = {worst[0]:.3g}"
    if 2 <= len(p) <= 3 and 1 <= k <= 40:
        pj = joint_chi2_pvalue(X, k, p)
        assert pj >= P_MIN, f"{what}: joint chi-square p = {pj:.3g}"
    return z


def assert_categorical_sum(X, P, what):
    """X (N, d): counts of groups of G one-fragment rows, row r picking member j with probability P[r, j].  P is (G, d)
    for all groups, or (R, G, d) with R dividing N: group i has the rows P[i % R] (R replicas swept N / R times)."""
    X = np.asarray(X, np.int64)
    P = np.asarray(P, np.float64)
    if P.ndim == 2:
        P = P[None]
    G = P.shape[1]
    reps = len(X) // len(P)
    assert reps * len(P) == len(X)

    def per_draw(a):
        return np.tile(a, (reps,) + (1,) * (a.ndim - 1))

    assert (X.sum(axis=1) == G).all(), f"{what}: a group's counts do not sum to its {G} rows"
    never = np.broadcast_to(per_draw(P.max(axis=1) == 0.0), X.shape)
    assert (X[never] == 0).all(), f"{what}: a member with p = 0 in every row of its group received a fragment"
    mean, var = per_draw(P.sum(axis=1)), per_draw((P * (1.0 - P)).sum(axis=1))
    z, where = moment_z(X, mean, var, lambda i, j: per_draw(-(P[:, :, i] * P[:, :, j]).sum(axis=1)))
    assert abs(z) <= Z_MAX, f"{what}: worst z = {z:.2f} ({where}), N = {len(X)}"
    return z


def assert_gamma_step(mu_new, counts, length, alpha, beta, what):
    """mu_new ~ Gamma(alpha + counts, rate beta + length), elementwise: KS of the PIT values and the mean of
    mu' (beta + l) / (alpha + c), which is 1 with variance 1 / (alpha + c)."""
    a = alpha + np.asarray(counts, np.float64)
    r = beta + np.asarray(length, np.float64)
    u = gamma_pit(mu_new, counts, length, alpha, beta)
    pv = stats.kstest(u, "uniform").pvalue
    assert pv >= P_MIN, f"{what}: KS of the PIT values p = {pv:.3g}, N = {len(u)}"
    y = mu_new * r / a - 1.0
    z = y.mean() / np.sqrt(np.mean(1.0 / a) / len(y))
    assert abs(z) <= Z_MAX, f"{what}: mean of mu' (beta + l) / (alpha + c) - 1: z = {z:.2f}"
    return pv, z


def replica_mean_z(per_replica, target):
    """z of the mean over independent replicas of a per-replica statistic (rows: replicas) against target, per column;
    the standard error is the spread between replicas."""
    per_replica = np.asarray(per_replica, np.float64)
    R = per_replica.shape[0]
    se = per_replica.std(axis=0, ddof=1) / np.sqrt(R)
    return (per_replica.mean(axis=0) - target) / se


# ------------------------------------------------------------------ cases shared by the CPU and GPU tests

def cat_limit(d):
    """mmq_cat_limit (include/mmq_sampler.h): the largest k drawn as k categoricals."""
    return int(min(max(32 * (d - 1), 32), 512))


def mu_pattern(d, kind):
    """Class probabilities of d members: 'equal'; 'spread' (geometric over 10^3, 10^2 above 32 members, shuffled by a
    fixed permutation); 'zero' (equal, member d // 2 exactly 0).  Every nonzero p_j is at least 1e-4: draws use 32-bit
    uniforms, and smaller probabilities are by design not resolved to the last bit."""
    if kind == "equal":
        mu = np.ones(d)
    elif kind == "spread":
        mu = np.random.default_rng(d).permutation(np.geomspace(1.0, 1e3 if d <= 32 else 1e2, d))
    else:
        mu = np.ones(d)
        mu[d // 2] = 0.0
    p = mu / mu.sum()
    assert p[p > 0].min() >= 1e-4
    return mu


def replicated_class(R, d, k, mu):
    """R replicas of one class of k fragments over d members of its own: (row_ptr, col, k, mu over R d transcripts)."""
    row_ptr = np.arange(R + 1, dtype=np.int64) * d
    return row_ptr, np.arange(R * d, dtype=np.int32), np.full(R, k, np.int32), np.tile(np.asarray(mu, np.float64), R)


def grouped_rows(R, G, d, mu, W=None):
    """R replicas of G identical neighbouring one-fragment rows over d members of their own; W (R, G, d) per-row
    weights or None.  Returns (row_ptr, col, weight or None, mu over R d transcripts, P (R, G, d) row probabilities)."""
    mu = np.asarray(mu, np.float64)
    row_ptr = np.arange(R * G + 1, dtype=np.int64) * d
    col = np.repeat(np.arange(R, dtype=np.int32) * d, G * d) + np.tile(np.arange(d, dtype=np.int32), R * G)
    w = None if W is None else np.ascontiguousarray(W, np.float32).reshape(-1)
    q = mu[None, None, :] * (1.0 if W is None else np.asarray(W, np.float32).astype(np.float64))
    P = np.broadcast_to(q, (R, G, d)) / q.sum(axis=2, keepdims=True)
    return row_ptr, col, w, np.tile(mu, R), P


def row_weights(rng, R, G, d, zeros=True):
    """Per-row weights exp(N(0, 1/2)) in fp32, about 1 in 8 exactly 0 (never all of a row)."""
    W = np.exp(0.5 * rng.standard_normal((R, G, d))).astype(np.float32)
    if zeros:
        W[rng.random((R, G, d)) < 0.125] = 0.0
        W[..., 0] = np.where(W.max(axis=2) == 0.0, 1.0, W[..., 0])
    return W


POSTERIOR_ALPHA = POSTERIOR_BETA = 0.1


def posterior_components():
    """One component per allocation regime (kind, spec): 'rows' components are d = 2 with G one-fragment rows (weights
    W, or unweighted when W is None), 'class' components one class of k fragments over d members.  Singleton counts u
    and lengths l vary between members so that no two members share a marginal."""
    rng = np.random.default_rng(20261020)

    def ul(d):
        return rng.integers(0, 6, d).astype(np.float64), rng.uniform(0.5, 2.0, d)

    out = {}
    u, l = ul(2)
    out["cls1"] = ("rows", dict(W=None, G=6, u=u, l=l))                    # k = 1 classes: k_alloc_cls1
    u, l = ul(3)
    out["lo"] = ("class", dict(d=3, k=20, u=u, l=l))                        # k_alloc_cls<LO>
    u, l = ul(12)
    out["hi"] = ("class", dict(d=12, k=40, u=u, l=l))                       # k_alloc_cls<HI>
    u, l = ul(7)
    out["chain"] = ("class", dict(d=7, k=cat_limit(7) + 1, u=u, l=l))      # k_alloc_chain
    u, l = ul(65)
    out["general"] = ("class", dict(d=65, k=100, u=u, l=l))                 # the general kernel
    u, l = ul(2)
    W = np.exp(0.7 * rng.standard_normal((8, 2))).astype(np.float32)
    out["weighted"] = ("rows", dict(W=W, G=8, u=u, l=l))                    # per-fragment, weighted
    return out


def posterior_of(kind, spec):
    if kind == "rows":
        W = np.ones((spec["G"], 2)) if spec["W"] is None else spec["W"].astype(np.float64)
        return WeightedRowsPair(W, spec["u"], spec["l"], POSTERIOR_ALPHA, POSTERIOR_BETA)
    return SharedClass(spec["k"], spec["u"], spec["l"], POSTERIOR_ALPHA, POSTERIOR_BETA)


def posterior_problem(kind, spec, R):
    """R replicas of a component in one shard: (row_ptr, col, k or None, weight or None, length).  Member j of replica
    r is transcript r d + j.  Singleton classes carry u_j (k = u_j collapsed, u_j one-member rows per fragment);
    'class' components are collapsed, 'rows' components collapsed when unweighted (one k = 1 class per row) and per
    fragment when weighted."""
    d = 2 if kind == "rows" else spec["d"]
    u = spec["u"].astype(np.int64)
    per_fragment = kind == "rows" and spec["W"] is not None
    rows, ks, ws = [], [], []
    for r in range(R):
        base = r * d
        if kind == "rows":
            for g in range(spec["G"]):
                rows.append([base, base + 1]); ks.append(1)
                if per_fragment:
                    ws.append(spec["W"][g])
        else:
            rows.append(list(range(base, base + d))); ks.append(spec["k"])
        for j in range(d):
            if per_fragment:
                for _ in range(u[j]):
                    rows.append([base + j]); ks.append(1); ws.append(np.ones(1, np.float32))
            elif u[j] > 0:
                rows.append([base + j]); ks.append(int(u[j]))
    if per_fragment:                     # the by-length layout: rows grouped by class size, singletons first
        order = sorted(range(len(rows)), key=lambda i: len(rows[i]))
        rows = [rows[i] for i in order]; ws = [ws[i] for i in order]
    row_ptr = np.concatenate([[0], np.cumsum([len(x) for x in rows])]).astype(np.int64)
    col = np.concatenate(rows).astype(np.int32)
    k = None if per_fragment else np.array(ks, np.int32)
    w = np.concatenate(ws).astype(np.float32) if per_fragment else None
    return row_ptr, col, k, w, np.tile(spec["l"], R)


def posterior_z(post, trace, R, quartiles=(0.25, 0.5, 0.75)):
    """trace (R d, S): mu of every member of every replica after each sweep, from an exact stationary start.  Per member
    the replica's time-averages of log mu_j and of 1{mu_j <= q} at the exact quartiles q, against the exact values;
    the standard error comes from the spread between replicas.  Returns (worst |z|, description)."""
    d = post.d
    T = np.asarray(trace, np.float64).reshape(R, d, -1)
    worst = (0.0, "none")
    for j in range(d):
        z = replica_mean_z(np.log(T[:, j, :]).mean(axis=1), post.e_log_mu(j))
        if abs(z) > abs(worst[0]):
            worst = (float(z), f"E log mu of member {j}")
        for q in quartiles:
            qv = post.quantile_mu(j, q)
            z = replica_mean_z((T[:, j, :] <= qv).mean(axis=1), q)
            if abs(z) > abs(worst[0]):
                worst = (float(z), f"P(mu <= q{q:g}) of member {j}")
    return worst
