/* mmq_post.cu — posterior summaries on the device (sm_100a): group (gene /
 * identical-set) traces, log-scale means, batched Sokal IACT, percentiles,
 * isoform-proportion and probit moments, unique hits of transcript sets.
 *
 * Reference code replaced (eturro/mmseq 1.0.11, /root/reference):
 *   k_group_trace      src/mmseq.cpp:938-982   identical-set and gene trace sums
 *   k_row_sokal        src/mmseq.cpp:1203-1227 (log + mean), :1308-1363 and
 *                      src/sokal.cc:33-87      (var, tau, window)
 *   k_row_percentiles  src/mmseq.cpp:1111-1172 (sort each trace, pick indices)
 *   k_prop             src/mmseq.cpp:985-1008, :1236-1257
 *   k_uh_sets          src/uh.cpp:3-26 restated O(nnz)
 * and, with no reference counterpart, the diagnostics of several chains (k_chain_diag), the summaries of their
 * pooled draws (k_pool_summ), transcripts per million (k_draw_totals, k_totals_fold, k_tpm_summ), the allelic fraction
 * of haplotype pairs (k_allele_only, k_allelic_summ) and the isoform pairs within a gene (k_pair_shared, k_isocorr_prep,
 * k_isocorr_items, k_isocorr).
 * All traces are [row * trace_len + slot] (the reference's mu_trace layout).
 */
#include <algorithm>
#include <cstdio>
#include <vector>

#include "../../include/mmq_sampler.h"
#include "mmq_internal.h"

#define MMQ_POST_THREADS 256
#define MMQ_MAX_ROW_LEN 2048

__device__ __forceinline__ double post_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

/* deterministic block sum, result broadcast to every thread */
__device__ __forceinline__ double post_block_sum(double v) {
  __shared__ double s_part[33];
  v = post_warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_part[wid] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double r = 0.0;
    const int nw = (blockDim.x + 31) >> 5;
    for (int i = 0; i < nw; ++i) r += s_part[i];
    s_part[32] = r;
  }
  __syncthreads();
  return s_part[32];
}

/* group_trace[g*L+s] = sum_{t in group g} trace[t*L+s] (+ extra[g*L+s]) */
__global__ void k_group_trace(const double* __restrict__ trace, const int64_t* __restrict__ gptr,
                              const int32_t* __restrict__ members, const double* __restrict__ extra,
                              double* __restrict__ out, int64_t ngroups, int L) {
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t b = gptr[g], e = gptr[g + 1];
    for (int s = threadIdx.x; s < L; s += blockDim.x) {
      double v = 0.0;
      for (int64_t q = b; q < e; ++q) v += trace[(int64_t)members[q] * L + s];
      if (extra) v += extra[g * L + s];
      out[g * L + s] = v;
    }
  }
}

/* In-place forward FFT of (re, im) in shared memory, length len = 2^lg.
 * dif = true : natural order in, bit-reversed order out (Gentleman-Sande)
 * dif = false: bit-reversed order in, natural order out (Cooley-Tukey) */
__device__ void smem_fft(double* re, double* im, int len, bool dif) {
  const int nb = len >> 1;
  if (dif) {
    for (int half = nb; half >= 1; half >>= 1) {
      for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        const int j = b & (half - 1);
        const int a = ((b - j) << 1) + j;
        const int c = a + half;
        double sn, cs;
        sincospi(-(double)j / (double)half, &sn, &cs);
        const double xr = re[a] - re[c], xi = im[a] - im[c];
        re[a] += re[c]; im[a] += im[c];
        re[c] = xr * cs - xi * sn;
        im[c] = xr * sn + xi * cs;
      }
      __syncthreads();
    }
  } else {
    for (int half = 1; half <= nb; half <<= 1) {
      for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        const int j = b & (half - 1);
        const int a = ((b - j) << 1) + j;
        const int c = a + half;
        double sn, cs;
        sincospi(-(double)j / (double)half, &sn, &cs);
        const double xr = re[c] * cs - im[c] * sn, xi = re[c] * sn + im[c] * cs;
        re[c] = re[a] - xr; im[c] = im[a] - xi;
        re[a] += xr; im[a] += xi;
      }
      __syncthreads();
    }
  }
}

/* One CTA per row: optional log, mean, then Sokal's estimator (src/sokal.cc:33-87):
 * FFT -> |.|^2 -> zero DC -> FFT -> var = acov0/(n(n-1)) -> rho -> adaptive window. */
__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_row_sokal(const double* __restrict__ src, int64_t rows, int len, int do_log, double* __restrict__ mean_out,
            double* __restrict__ var_out, double* __restrict__ tau_out, int32_t* __restrict__ win_out,
            int32_t* __restrict__ status_out) {
  extern __shared__ double sh[];
  double* re = sh;
  double* im = sh + len;
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    double part = 0.0;
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
      double v = src[row * len + i];
      if (do_log) v = log(v);
      re[i] = v;
      im[i] = 0.0;
      part += v;
    }
    const double total = post_block_sum(part); /* also orders the smem writes */
    if (threadIdx.x == 0 && mean_out) mean_out[row] = total / (double)len;
    smem_fft(re, im, len, true);
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
      const double p = re[i] * re[i] + im[i] * im[i];
      re[i] = (i == 0) ? 0.0 : p; /* bit-reversal maps bin 0 to slot 0 */
      im[i] = 0.0;
    }
    __syncthreads();
    smem_fft(re, im, len, false);
    if (threadIdx.x == 0) {
      const double x0 = re[0];
      const double var = x0 / ((double)len * (double)(len - 1));
      const double c = 1.0 / x0;
      double sum = -0.333333333333333333333;
      int m = len + 1;
      for (int i = 0; i < len; ++i) {
        sum += re[i] * c - 0.166666666666666666666;
        if (sum < 0) { m = i + 1; break; }
      }
      if (var_out) var_out[row] = var;
      if (tau_out) tau_out[row] = 2 * (sum + (m - 1.0) / 6.0);
      if (win_out) win_out[row] = m;
      if (status_out) status_out[row] = 0;
    }
    __syncthreads();
  }
}

/* One CTA per row: bitonic sort of the row in shared memory (len a power of two),
 * then pct[row*npct + j] = sorted[idx[j]].  src/mmseq.cpp:1139-1146. */
__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_row_percentiles(const double* __restrict__ src, int64_t rows, int len, int npct,
                  const int32_t* __restrict__ idx, double* __restrict__ pct) {
  extern __shared__ double sh[];
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    for (int i = threadIdx.x; i < len; i += blockDim.x) sh[i] = src[row * len + i];
    __syncthreads();
    for (int k = 2; k <= len; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < len; i += blockDim.x) {
          const int p = i ^ j;
          if (p > i) {
            const double a = sh[i], b = sh[p];
            const bool up = (i & k) == 0;
            if ((a > b) == up) { sh[i] = b; sh[p] = a; }
          }
        }
        __syncthreads();
      }
    for (int j = threadIdx.x; j < npct; j += blockDim.x) pct[row * npct + j] = sh[idx[j]];
    __syncthreads();
  }
}

/* prop[s] = trace[t][s] / gene_trace[gene_of[t]][s]  (src/mmseq.cpp:995-996);
 * mean (:1244, :1258), probit sum / sum of squares (:1249-1255). */
__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_prop(const double* __restrict__ trace, const double* __restrict__ gene_trace, const int32_t* __restrict__ gene_of,
       const uint8_t* __restrict__ multi_iso, int64_t n, int L, double* __restrict__ prop_trace,
       double* __restrict__ mean_prop, double* __restrict__ sum_probit, double* __restrict__ sumsq_probit) {
  for (int64_t t = blockIdx.x; t < n; t += gridDim.x) {
    const int64_t g = gene_of[t];
    const bool multi = multi_iso[t] != 0;
    double sp = 0.0, sz = 0.0, szz = 0.0;
    for (int s = threadIdx.x; s < L; s += blockDim.x) {
      const double p = trace[t * L + s] / gene_trace[g * L + s];
      prop_trace[t * L + s] = p;
      sp += p;
      double z;
      if (multi) {
        double pc = p; /* min(max(p,1e-9),1-1e-9); a NaN passes through both, as with std::max/min */
        if (pc < 0.000000001) pc = 0.000000001;
        if (pc > 0.999999999) pc = 0.999999999;
        z = mmq_ndtri(pc);
      } else {
        z = mmq_u2d(0x7ff0000000000000ull);
      }
      sz += z;
      szz += z * z;
    }
    sp = post_block_sum(sp);
    sz = post_block_sum(sz);
    szz = post_block_sum(szz);
    if (threadIdx.x == 0) {
      mean_prop[t] = sp / (double)L;
      sum_probit[t] = sz;
      sumsq_probit[t] = szz;
    }
  }
}

/* uh(): a class counts for set s when all its members lie in s. src/uh.cpp:12-23. */
template <bool HAS_K>
__global__ void k_uh_sets(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                          const int32_t* __restrict__ kk, const int32_t* __restrict__ set_of, int64_t m,
                          int32_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = row_ptr[i], e = row_ptr[i + 1];
    const int32_t s0 = set_of[col[b]];
    bool uniq = s0 >= 0;
    for (int64_t q = b + 1; q < e && uniq; ++q) uniq = set_of[col[q]] == s0;
    if (uniq) atomicAdd(out + s0, HAS_K ? kk[i] : 1);
  }
}

/* Gamma(alpha, rate_u) prior draws, one thread per (transcript, slot). src/mmseq.cpp:971-978. */
__global__ void k_prior(const int64_t* __restrict__ ids, const double* __restrict__ rate, int64_t count, int L,
                        double alpha, uint32_t seed, double* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count * L; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t u = i / L;
    const int s = (int)(i - u * L);
    mmq_rng g;
    mmq_rng_init(&g, seed, MMQ_STREAM_PRIOR, (uint64_t)ids[u], (uint32_t)s);
    out[i] = mmq_gamma(&g, alpha, rate[u]);
  }
}

/* ------------------------------------------------ convergence of several chains
 * Rank-normalised split-R-hat and bulk / tail ESS (Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021), one CTA per
 * feature.  Definitions: include/mmq.h (mmq_chain_diagnostics_dev); tests/chain_reference.py restates them in numpy.
 * Shared memory, P = the power of two >= S = C L draws:  key fp64[P] | z fp64[S] | idx int32[P] | run int32[S].
 * key/idx: the (value, draw) pairs being sorted; z: the series under study, in draw order; run: the first sorted
 * position of each value's run of ties.  The ESS step reuses key as the FFT's (re, im), idx as the summed
 * autocovariance and run as the autocorrelation sequence: 12 (P + S) bytes in all, 192 KB at S = 8192. */
#define MMQ_CHAIN_SMAX 8192

struct mmq_chain_ptrs { const double* p[MMQ_CHAINS_MAX]; };

static int chain_pow2_at_least(int s) { int p = 1; while (p < s) p <<= 1; return p; }
static size_t chain_smem_bytes(int S) { return (size_t)12 * (size_t)(chain_pow2_at_least(S) + S); }
/* The caps on dynamic shared memory that k_chain_diag and k_pool_summ are given: the largest request of any accepted
 * shape (S = 8192; for k_pool_summ with L = 2048).  The cap is a per-device property of the function that any host thread
 * can change between another thread's set and its launch, so it never depends on the call: a cap sized to one call's
 * request could be lowered under a concurrent larger one, whose launch would then fail. */
#define MMQ_CHAIN_DIAG_SMEM_CAP (12 * (8192 + 8192))
#define MMQ_POOL_SMEM_CAP (8 * (8192 + 8192 + 2048))

/* draw k (< S) of the row: chain k >> lgL, sweep slot k & (L - 1) */
__device__ __forceinline__ double chain_x(const mmq_chain_ptrs& cp, int64_t row, int lgL, int k) {
  return cp.p[k >> lgL][(row << lgL) + (k & ((1 << lgL) - 1))];
}

/* bitonic sort of (key, idx) pairs, ascending by key then idx; P a power of two */
__device__ __forceinline__ void chain_sort(double* key, int32_t* idx, int P) {
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const double a = key[i], b = key[p];
          const int32_t ia = idx[i], ib = idx[p];
          const bool gt = a > b || (a == b && ia > ib);
          if (gt == ((i & k) == 0)) { key[i] = b; key[p] = a; idx[i] = ib; idx[p] = ia; }
        }
      }
      __syncthreads();
    }
}

/* z[draw] = Phi^-1((r - 3/8) / (S + 1/4)), r the average 1-based rank of the draw's value among the S sorted keys.
 * Each thread owns a contiguous range of sorted positions; the run of ties that crosses into it from the left (right)
 * starts (ends) at the last head (first tail) of the threads before (after) it. */
__device__ __forceinline__ void chain_rank_normalise(const double* key, const int32_t* idx, int32_t* run, double* z, int S) {
  __shared__ int32_t s_head[MMQ_POST_THREADS], s_tail[MMQ_POST_THREADS];
  const int T = blockDim.x, t = threadIdx.x;
  const int chunk = (S + T - 1) / T;
  const int a = min(S, t * chunk), b = min(S, a + chunk);
  auto head = [&](int i) { return i == 0 || key[i] != key[i - 1]; };
  auto tail = [&](int i) { return i == S - 1 || key[i] != key[i + 1]; };
  int last_head = -1, first_tail = 0x7fffffff;
  for (int i = a; i < b; ++i) if (head(i)) last_head = i;
  for (int i = b - 1; i >= a; --i) if (tail(i)) first_tail = i;
  s_head[t] = last_head;
  s_tail[t] = first_tail;
  __syncthreads();
  if (t == 0) { /* exclusive prefix max of the heads, exclusive suffix min of the tails */
    int c = -1;
    for (int u = 0; u < T; ++u) { const int v = s_head[u]; s_head[u] = c; c = max(c, v); }
    c = 0x7fffffff;
    for (int u = T - 1; u >= 0; --u) { const int v = s_tail[u]; s_tail[u] = c; c = min(c, v); }
  }
  __syncthreads();
  int start = s_head[t];
  for (int i = a; i < b; ++i) { if (head(i)) start = i; run[i] = start; }
  int end = s_tail[t];
  const double denom = (double)S + 0.25;
  for (int i = b - 1; i >= a; --i) {
    if (tail(i)) end = i;
    const double r = 0.5 * (double)(run[i] + end + 2);
    z[idx[i]] = mmq_ndtri((r - 0.375) / denom);
  }
  __syncthreads();
}

/* mean and variance (ddof 1) of each of the M split chains y[j N .. j N + N), one warp per chain.  A split chain whose
 * values are all equal has exactly that mean and variance 0. */
__device__ __forceinline__ void chain_split_moments(const double* y, int M, int N, double* s_m, double* s_w) {
  const int lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int j = threadIdx.x >> 5; j < M; j += nw) {
    const double* q = y + (size_t)j * N;
    const double y0 = q[0];
    double s = 0.0;
    bool same = true;
    for (int i = lane; i < N; i += 32) { s += q[i]; same &= q[i] == y0; }
    s = post_warp_sum(s);
    same = __all_sync(0xffffffffu, same);
    const double m = same ? y0 : __shfl_sync(0xffffffffu, s, 0) / (double)N;
    double v = 0.0;
    if (!same) {
      for (int i = lane; i < N; i += 32) { const double d = q[i] - m; v += d * d; }
      v = post_warp_sum(v);
    }
    if (lane == 0) { s_m[j] = m; s_w[j] = same ? 0.0 : v / (double)(N - 1); }
  }
  __syncthreads();
}

/* split R-hat from the split chains' moments; NaN when the within-chain variance W is 0 */
__device__ __forceinline__ double chain_rhat(const double* s_m, const double* s_w, int M, int N) {
  double W = 0.0, mm = 0.0, B = 0.0;
  for (int j = 0; j < M; ++j) { W += s_w[j]; mm += s_m[j]; }
  W /= (double)M;
  mm /= (double)M;
  for (int j = 0; j < M; ++j) { const double d = s_m[j] - mm; B += d * d; }
  B = (double)N * (B / (double)(M - 1));
  if (W == 0.0) return mmq_u2d(0x7ff8000000000000ull);
  return sqrt((((double)(N - 1) / (double)N) * W + B / (double)N) / W);
}

/* ESS of the split chains y (moments s_m from chain_split_moments): autocovariances by FFT (zero-padded to 2N = L,
 * as k_row_sokal), then Geyer's initial monotone sequence.  The result is valid in thread 0; NaN when `constant`.
 * Shared scratch: key fp64[2 L], the FFT's (re, im); acc fp64[N], the sum over split chains of L * sum_i yc[i] yc[i + t];
 * r fp64[N], the autocorrelation sequence. */
__device__ __forceinline__ double chain_ess(const double* y, int M, int N, const double* s_m, bool constant, double* key, double* acc,
                            double* r) {
  const int L = 2 * N;
  double* re = key;
  double* im = key + L;
  double out = mmq_u2d(0x7ff8000000000000ull);
  if (constant) return out;
  for (int t = threadIdx.x; t < N; t += blockDim.x) acc[t] = 0.0;
  for (int j = 0; j < M; ++j) {
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
      re[i] = i < N ? y[(size_t)j * N + i] - s_m[j] : 0.0;
      im[i] = 0.0;
    }
    __syncthreads();
    smem_fft(re, im, L, true);
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
      re[i] = re[i] * re[i] + im[i] * im[i];
      im[i] = 0.0;
    }
    __syncthreads();
    smem_fft(re, im, L, false);
    for (int t = threadIdx.x; t < N; t += blockDim.x) acc[t] += re[t];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double scale = 1.0 / ((double)M * (double)L * (double)N); /* acc -> mean over chains of acov_j */
    double mm = 0.0, vm = 0.0;
    for (int j = 0; j < M; ++j) mm += s_m[j];
    mm /= (double)M;
    for (int j = 0; j < M; ++j) { const double d = s_m[j] - mm; vm += d * d; }
    vm /= (double)(M - 1);
    const double mean_var = acc[0] * scale * ((double)N / (double)(N - 1));
    const double var_plus = mean_var * ((double)(N - 1) / (double)N) + vm;
    if (var_plus > 0.0) {
      auto rho = [&](int t) { return 1.0 - (mean_var - acc[t] * scale) / var_plus; };
      for (int t = 0; t < N; ++t) r[t] = 0.0;
      r[0] = 1.0;
      r[1] = rho(1);
      double even = 1.0, odd = r[1];
      int t = 1;
      while (t < N - 3 && even + odd > 0.0) {
        even = rho(t + 1);
        odd = rho(t + 2);
        if (even + odd >= 0.0) { r[t + 1] = even; r[t + 2] = odd; }
        t += 2;
      }
      const int max_t = t - 2;
      if (even > 0.0) r[max_t + 1] = even;
      for (t = 1; t <= max_t - 2; t += 2)
        if (r[t + 1] + r[t + 2] > r[t - 1] + r[t]) { r[t + 1] = (r[t - 1] + r[t]) / 2.0; r[t + 2] = r[t + 1]; }
      double sum = 0.0;
      for (t = 0; t <= max_t; ++t) sum += r[t];
      const double SN = (double)M * (double)N;
      double tau = -1.0 + 2.0 * sum + r[max_t + 1];
      const double floor_tau = 1.0 / log10(SN);
      if (tau < floor_tau) tau = floor_tau;
      out = SN / tau;
    }
  }
  __syncthreads(); /* the scratch areas are free again */
  return out;
}

__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_chain_diag(const __grid_constant__ mmq_chain_ptrs cp, int C, int64_t rows, int lgL, double* __restrict__ out) {
  extern __shared__ double sh[];
  __shared__ double s_m[2 * MMQ_CHAINS_MAX], s_w[2 * MMQ_CHAINS_MAX];
  const int L = 1 << lgL, N = L >> 1, M = 2 * C, S = C * L;
  int P = 1;
  while (P < S) P <<= 1;
  double* key = sh;
  double* z = sh + P;
  int32_t* idx = reinterpret_cast<int32_t*>(sh + P + S);
  int32_t* run = idx + P;
  const double nan = mmq_u2d(0x7ff8000000000000ull), inf = mmq_u2d(0x7ff0000000000000ull);
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    /* finiteness and the log-scale mean */
    double bad = 0.0, ls = 0.0;
    for (int k = threadIdx.x; k < S; k += blockDim.x) {
      const double x = chain_x(cp, row, lgL, k);
      bad += isfinite(x) ? 0.0 : 1.0;
      ls += log(x);
    }
    bad = post_block_sum(bad);
    if (bad > 0.0) {
      if (threadIdx.x == 0) for (int q = 0; q < 5; ++q) out[q * rows + row] = nan;
      continue;
    }
    ls = post_block_sum(ls);
    const double log_mean = ls / (double)S;
    double lv = 0.0;
    for (int k = threadIdx.x; k < S; k += blockDim.x) { const double d = log(chain_x(cp, row, lgL, k)) - log_mean; lv += d * d; }
    lv = post_block_sum(lv);
    const double log_sd = sqrt(lv / (double)(S - 1));

    /* bulk: rank-normalised draws */
    for (int i = threadIdx.x; i < P; i += blockDim.x) { key[i] = i < S ? chain_x(cp, row, lgL, i) : inf; idx[i] = i; }
    chain_sort(key, idx, P);
    const double med = 0.5 * (key[S / 2 - 1] + key[S / 2]);
    auto quantile = [&](double p) { /* type 7 */
      const double h = (double)(S - 1) * p, f = floor(h);
      const int lo = (int)f;
      return key[lo] + (h - f) * (key[lo + 1] - key[lo]);
    };
    const double q05 = quantile(0.05), q95 = quantile(0.95);
    bool constant = key[0] == key[S - 1];
    chain_rank_normalise(key, idx, run, z, S);
    chain_split_moments(z, M, N, s_m, s_w);
    const double rhat_bulk = chain_rhat(s_m, s_w, M, N);
    /* the idx and run areas (4 P and 4 S bytes) hold the N fp64 of acc and of r */
    const double ess_bulk = chain_ess(z, M, N, s_m, constant, key, reinterpret_cast<double*>(idx), reinterpret_cast<double*>(run));

    /* folded: rank-normalised |x - median| */
    for (int i = threadIdx.x; i < P; i += blockDim.x) { key[i] = i < S ? fabs(chain_x(cp, row, lgL, i) - med) : inf; idx[i] = i; }
    chain_sort(key, idx, P);
    chain_rank_normalise(key, idx, run, z, S);
    chain_split_moments(z, M, N, s_m, s_w);
    const double rhat_fold = chain_rhat(s_m, s_w, M, N);

    /* tails: indicators of x <= q05 and x <= q95 */
    double ess_tail = inf;
    for (int side = 0; side < 2; ++side) {
      const double q = side ? q95 : q05;
      double cnt = 0.0;
      for (int k = threadIdx.x; k < S; k += blockDim.x) { z[k] = chain_x(cp, row, lgL, k) <= q ? 1.0 : 0.0; cnt += z[k]; }
      cnt = post_block_sum(cnt); /* also orders the writes of z */
      constant = cnt == 0.0 || cnt == (double)S;
      chain_split_moments(z, M, N, s_m, s_w);
      const double e = chain_ess(z, M, N, s_m, constant, key, reinterpret_cast<double*>(idx), reinterpret_cast<double*>(run));
      ess_tail = (isnan(e) || isnan(ess_tail)) ? nan : fmin(ess_tail, e);
    }
    if (threadIdx.x == 0) {
      out[row] = (isnan(rhat_bulk) || isnan(rhat_fold)) ? nan : fmax(rhat_bulk, rhat_fold);
      out[rows + row] = ess_bulk;
      out[2 * rows + row] = ess_tail;
      out[3 * rows + row] = log_mean;
      out[4 * rows + row] = log_sd;
    }
    __syncthreads();
  }
}

/* bitonic sort of key[0 .. P) ascending with NaN last, P a power of two; opens with a barrier that orders the caller's
 * writes of key and ends with one after the last exchange */
__device__ __forceinline__ void sort_nan_last(double* key, int P) {
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const double a = key[i], b = key[p];
          const bool gt = a > b || (isnan(a) && !isnan(b));
          if (gt == ((i & k) == 0)) { key[i] = b; key[p] = a; }
        }
      }
      __syncthreads();
    }
}

/* ------------------------------------------------ summaries of the pooled draws of several chains
 * The posterior columns of the tables over all S = C L draws of a feature (mmseq -pool), one CTA per feature.
 * Definitions: include/mmq.h (mmq_pooled_summaries_dev); tests/pool_reference.py restates them in numpy.
 * mode 0: log mean and sd (the sums of k_chain_diag, in its order, so the bits equal its log_mean / log_sd), the sorted
 * draws at the percentile indices, and the ESS of the split chains of log x.  mode 1 (proportion draws): plain mean and
 * percentiles.  Shared memory: key fp64[P] | y fp64[S] | acc fp64[L/2] | r fp64[L/2], 8 (P + S + L) bytes, 144 KB at
 * S = 8192 (mode 1: key only).  key holds the values being sorted (padded with NaN, which sorts last), then the
 * FFT's (re, im); y is log x in draw order. */
__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_pool_summ(const __grid_constant__ mmq_chain_ptrs cp, int C, int64_t rows, int lgL, int mode, int npct,
            const int32_t* __restrict__ pct_idx, double* __restrict__ out, double* __restrict__ pct) {
  extern __shared__ double sh[];
  __shared__ double s_m[2 * MMQ_CHAINS_MAX], s_w[2 * MMQ_CHAINS_MAX];
  const int L = 1 << lgL, N = L >> 1, M = 2 * C, S = C * L;
  int P = 1;
  while (P < S) P <<= 1;
  double* key = sh;
  double* y = sh + P;
  double* acc = y + S;
  double* r = acc + N;
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    double mean = nan, sd = nan, ess = nan;
    bool logs_finite = false;
    if (mode == 0) {
      double bad = 0.0, badlog = 0.0, ls = 0.0;
      for (int k = threadIdx.x; k < S; k += blockDim.x) {
        const double x = chain_x(cp, row, lgL, k), lx = log(x);
        bad += isfinite(x) ? 0.0 : 1.0;
        badlog += isfinite(lx) ? 0.0 : 1.0;
        ls += lx;
        y[k] = lx;
      }
      bad = post_block_sum(bad);
      badlog = post_block_sum(badlog);
      ls = post_block_sum(ls);
      if (bad == 0.0) {
        mean = ls / (double)S;
        double lv = 0.0;
        for (int k = threadIdx.x; k < S; k += blockDim.x) { const double d = y[k] - mean; lv += d * d; }
        lv = post_block_sum(lv);
        sd = sqrt(lv / (double)(S - 1));
      }
      logs_finite = badlog == 0.0;
    } else {
      double s = 0.0;
      for (int k = threadIdx.x; k < S; k += blockDim.x) s += chain_x(cp, row, lgL, k);
      mean = post_block_sum(s) / (double)S;
    }

    /* percentiles: bitonic sort of the values, NaN last */
    for (int i = threadIdx.x; i < P; i += blockDim.x) key[i] = i < S ? chain_x(cp, row, lgL, i) : nan;
    sort_nan_last(key, P);
    for (int j = threadIdx.x; j < npct; j += blockDim.x) {
      const int q = pct_idx[j];
      pct[row * npct + j] = q >= 0 && q < S ? key[q] : nan;
    }

    /* ESS of log x over the 2C split chains */
    if (logs_finite) {
      const bool constant = key[0] == key[S - 1];
      chain_split_moments(y, M, N, s_m, s_w); /* its barrier also ends the reads of key above */
      ess = chain_ess(y, M, N, s_m, constant, key, acc, r);
    }
    if (threadIdx.x == 0) {
      out[row] = mean;
      if (mode == 0) { out[rows + row] = sd; out[2 * rows + row] = ess; }
    }
    __syncthreads();
  }
}

/* ------------------------------------------------ transcripts per million (mmseq -tpm)
 * Definitions: include/mmq.h (mmq_draw_totals_dev, mmq_tpm_summaries_dev); tests/tpm_reference.py restates them in numpy.
 * k_draw_totals + k_totals_fold: D[s] = sum over the rows of a trace [row * L + s], in a fixed order that depends on
 * (rows, L) only: tiles of MMQ_TOTALS_TILE rows, each summed in row order per slot from 0.0, then the tile sums in tile
 * order from 0.0.  A warp reads 32 consecutive slots of one row (the trace is row-major), so every load is coalesced;
 * each thread keeps eight loads in flight ahead of its in-order adds. */
#define MMQ_TOTALS_TILE 512
#define MMQ_TOTALS_THREADS 256

__global__ void __launch_bounds__(MMQ_TOTALS_THREADS)
k_draw_totals(const double* __restrict__ trace, int64_t rows, int L, double* __restrict__ partial) {
  const int s = blockIdx.y * blockDim.x + threadIdx.x;
  if (s >= L) return;
  const int64_t t0 = (int64_t)blockIdx.x * MMQ_TOTALS_TILE;
  const int nt = rows - t0 < MMQ_TOTALS_TILE ? (int)(rows - t0) : MMQ_TOTALS_TILE;
  const double* p = trace + t0 * L + s;
  double acc = 0.0;
  int t = 0;
  for (; t + 8 <= nt; t += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = p[(int64_t)(t + u) * L];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc += v[u];
  }
  for (; t < nt; ++t) acc += p[(int64_t)t * L];
  partial[(int64_t)blockIdx.x * L + s] = acc;
}

__global__ void __launch_bounds__(MMQ_TOTALS_THREADS)
k_totals_fold(const double* __restrict__ partial, int64_t ntiles, int L, double* __restrict__ totals) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= L) return;
  double acc = 0.0;
  int64_t k = 0;
  for (; k + 8 <= ntiles; k += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = partial[(k + u) * L + s];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc += v[u];
  }
  for (; k < ntiles; ++k) acc += partial[k * L + s];
  totals[s] = acc;
}

/* One CTA per feature, grid-capped as k_pool_summ: draw k (< S = C L) of the feature is (w / D[k]) 1e6, w the sum of its
 * members' draws at chain k >> lgL, slot k & (L - 1) in CSR order from 0.0 (gptr NULL: the feature is row `row` alone);
 * D chain-major, so D[k] is that chain's total at that slot.  The member sum and the normalisation happen in the load,
 * so no TPM trace is stored anywhere.  Then the mean, the two-pass sd and the percentiles of the NaN-last sort.  Shared
 * memory: key fp64[P], the draws in draw order padded with NaN, sorted in place; 8 P bytes, 64 KB at S = 8192. */
#define MMQ_TPM_SMEM_CAP (8 * 8192)

/* The tail that k_tpm_summ and k_allelic_summ share.  key[0 .. P) holds the row's S draws in draw order, padded with NaN;
 * `finite`: no draw is NaN or infinite; `sum`: the draws' block sum.  mean = sum / S and the two-pass sd (S - 1), both
 * NaN unless `finite`; then the NaN-last sort and pct[row npct + j] = sorted[pct_idx[j]], NaN for an index outside [0, S).
 * Every thread gets mean and sd. */
__device__ __forceinline__ void draws_mean_sd_pct(double* key, int P, int S, bool finite, double sum, int64_t row, int npct,
                                                  const int32_t* __restrict__ pct_idx, double* __restrict__ pct, double& mean,
                                                  double& sd) {
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  mean = nan;
  sd = nan;
  if (finite) {
    mean = sum / (double)S;
    double ss = 0.0;
    for (int k = threadIdx.x; k < S; k += blockDim.x) { const double d = key[k] - mean; ss += d * d; }
    sd = sqrt(post_block_sum(ss) / (double)(S - 1));
  }
  sort_nan_last(key, P);
  for (int j = threadIdx.x; j < npct; j += blockDim.x) {
    const int q = pct_idx[j];
    pct[row * npct + j] = q >= 0 && q < S ? key[q] : nan;
  }
}

__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_tpm_summ(const __grid_constant__ mmq_chain_ptrs cp, const double* __restrict__ totals, int C, int64_t rows, int lgL,
           const int64_t* __restrict__ gptr, const int32_t* __restrict__ members, int npct, const int32_t* __restrict__ pct_idx,
           double* __restrict__ out, double* __restrict__ pct) {
  extern __shared__ double sh[];
  const int L = 1 << lgL, S = C * L;
  int P = 1;
  while (P < S) P <<= 1;
  double* key = sh;
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    const int64_t b = gptr ? gptr[row] : row, e = gptr ? gptr[row + 1] : row + 1;
    double bad = 0.0, sum = 0.0;
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
      double v = nan;
      if (k < S) {
        const double* x = cp.p[k >> lgL] + (k & (L - 1));
        double w = 0.0;
        for (int64_t q = b; q < e; ++q) w += x[(int64_t)(gptr ? members[q] : q) << lgL];
        v = (w / totals[k]) * 1e6;
        bad += isfinite(v) ? 0.0 : 1.0;
        sum += v;
      }
      key[k] = v;
    }
    bad = post_block_sum(bad); /* also orders the writes of key */
    sum = post_block_sum(sum);
    double mean, sd;
    draws_mean_sd_pct(key, P, S, bad == 0.0, sum, row, npct, pct_idx, pct, mean, sd);
    if (threadIdx.x == 0) { out[row] = mean; out[rows + row] = sd; }
    __syncthreads();
  }
}

/* ------------------------------------------------ allelic fraction of haplotype pairs (mmseq -allelic)
 * Definitions: include/mmq.h (mmq_allele_only_counts, mmq_allelic_summaries_dev); tests/allelic_reference.py restates
 * them in numpy.
 * k_allele_only, the shape of k_uh_sets (one thread per hit class or fragment row, grid-capped): a row counts for side A
 * (B) of unit u when it holds an A (B) member of u and no B (A) member of u; each (unit, side) of the row is counted once,
 * by its first position.  The check scans the row for every member, O(len^2) on rows that are a few entries long. */
template <bool HAS_K>
__global__ void k_allele_only(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const int32_t* __restrict__ kk,
                              const int32_t* __restrict__ unit_of, const uint8_t* __restrict__ side, int64_t m,
                              int32_t* __restrict__ a_only, int32_t* __restrict__ b_only) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = row_ptr[i], e = row_ptr[i + 1];
    for (int64_t q = b; q < e; ++q) {
      const int32_t u = unit_of[col[q]];
      if (u < 0) continue;
      const uint8_t s = side[col[q]];
      bool first = true, opposite = false;
      for (int64_t r = b; r < e && !opposite; ++r) {
        if (r == q || unit_of[col[r]] != u) continue;
        if (side[col[r]] != s) opposite = true;
        else if (r < q) first = false;
      }
      if (first && !opposite) atomicAdd((s ? b_only : a_only) + u, HAS_K ? kk[i] : 1);
    }
  }
}

/* One CTA per unit, grid-capped, the layout of k_tpm_summ.  Draw k (< S = C L) is chain c = k >> lgL, slot k & (L - 1); a
 * member id m < n is row m of chain c's trace, m >= n row m - n of chain c's prior draws.  a (b) = the sum of the A (B)
 * members' draws in CSR order from 0.0 and phi = a / (a + b), fused into the load that fills key, so no fraction trace is
 * stored.  Block sums: the non-finite phi, the sum of phi and 2 #{a > b} + #{a = b}.  A unit with a non-finite phi gets
 * NaN in every output; otherwise draws_mean_sd_pct.  Shared memory: key fp64[P]; 8 P bytes, 64 KB at S = 8192. */
#define MMQ_ALLELIC_SMEM_CAP (8 * 8192)

__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_allelic_summ(const __grid_constant__ mmq_chain_ptrs cp, const __grid_constant__ mmq_chain_ptrs pp, int C, int64_t n, int64_t rows, int lgL,
               const int64_t* __restrict__ a_ptr, const int32_t* __restrict__ a_mem, const int64_t* __restrict__ b_ptr,
               const int32_t* __restrict__ b_mem, int npct, const int32_t* __restrict__ pct_idx, double* __restrict__ out,
               double* __restrict__ pct) {
  extern __shared__ double sh[];
  const int L = 1 << lgL, S = C * L;
  int P = 1;
  while (P < S) P <<= 1;
  double* key = sh;
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    const int64_t ab = a_ptr[row], ae = a_ptr[row + 1], bb = b_ptr[row], be = b_ptr[row + 1];
    double bad = 0.0, sum = 0.0, gt = 0.0;
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
      double v = nan;
      if (k < S) {
        const int c = k >> lgL, s = k & (L - 1);
        auto draw = [&](int32_t m) { return m < n ? cp.p[c][((int64_t)m << lgL) + s] : pp.p[c][(((int64_t)m - n) << lgL) + s]; };
        double a = 0.0, b = 0.0;
        for (int64_t q = ab; q < ae; ++q) a += draw(a_mem[q]);
        for (int64_t q = bb; q < be; ++q) b += draw(b_mem[q]);
        v = a / (a + b);
        bad += isfinite(v) ? 0.0 : 1.0;
        sum += v;
        gt += a > b ? 2.0 : a == b ? 1.0 : 0.0;
      }
      key[k] = v;
    }
    bad = post_block_sum(bad); /* also orders the writes of key */
    if (bad > 0.0) {
      if (threadIdx.x == 0) { out[row] = nan; out[rows + row] = nan; out[2 * rows + row] = nan; }
      for (int j = threadIdx.x; j < npct; j += blockDim.x) pct[row * npct + j] = nan;
      continue;
    }
    sum = post_block_sum(sum);
    gt = post_block_sum(gt);
    double mean, sd;
    draws_mean_sd_pct(key, P, S, true, sum, row, npct, pct_idx, pct, mean, sd);
    if (threadIdx.x == 0) { out[row] = mean; out[rows + row] = sd; out[2 * rows + row] = gt / (2.0 * (double)S); }
    __syncthreads();
  }
}

/* ------------------------------------------------ isoform pairs within a gene (mmseq -isocorr)
 * Definitions: include/mmq.h (mmq_pair_shared_counts, mmq_isocorr_summaries_dev); tests/isocorr_reference.py restates
 * them in numpy.
 * k_pair_shared, the shape of k_allele_only: one thread per hit class or fragment row, grid-capped.  Every two positions
 * q < r of the row whose transcripts are observed isoforms of one gene add k (or 1) at the pair's index, rowbase[t_a] +
 * local_of[t_b] with a < b the two local indices; O(len^2) on the row. */
template <bool HAS_K>
__global__ void k_pair_shared(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const int32_t* __restrict__ kk,
                              const int32_t* __restrict__ gene_of, const int32_t* __restrict__ local_of,
                              const int64_t* __restrict__ rowbase, int64_t m, unsigned long long* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = row_ptr[i], e = row_ptr[i + 1];
    const unsigned long long w = HAS_K ? (unsigned long long)kk[i] : 1ull;
    for (int64_t q = b; q < e; ++q) {
      const int32_t t = col[q], g = gene_of[t];
      if (g < 0) continue;
      for (int64_t r = q + 1; r < e; ++r) {
        const int32_t u = col[r];
        if (gene_of[u] != g) continue;
        const int32_t la = local_of[t], lb = local_of[u];
        if (la == lb) continue;
        atomicAdd(out + (la < lb ? rowbase[t] + lb : rowbase[u] + la), w);
      }
    }
  }
}

/* The pair summaries.  S = C L draws; draw k is chain k >> lgL, slot k & (L - 1).  Work in three kernels:
 *   k_isocorr_prep   one warp per CSR position q (every gene's observed members): mean and two-pass centred sum of
 *                    squares of x and of log x over the S draws, lanes strided by 32 in draw order, then a fixed shuffle
 *                    tree.  st[5 q ..]: mean x (NaN if a draw is not finite), ss x, mean log x (NaN if a draw is not
 *                    finite or <= 0), ss log x, 1.0 if a draw is NaN.
 *   k_isocorr_items  one CTA: items[g] = the exclusive prefix of T(T + 1) / 2 over the genes, T = ceil(k / 32) tiles of a
 *                    gene of k >= 2 members; items[ngenes] = the total.
 *   k_isocorr        a work item is (gene, tile row ta <= tile column tb), 32 x 32 members, in a grid-capped loop.  The
 *                    two tiles' draws, centred draws and centred logs are staged in shared memory MMQ_ISO_CHUNK draws at
 *                    a time ([draw][member], padded to 33); each thread owns four pairs (rows i0, i0 + 8, .., column j =
 *                    its lane) and adds their three sums in draw order.  Every member's trace row is read once per item.
 * Nothing depends on gridDim or on the gene order, so the bits are the same on any grid, device or repeat. */
#define MMQ_ISO_TILE 32
#define MMQ_ISO_CHUNK 32
#define MMQ_ISO_PAD (MMQ_ISO_TILE + 1)
#define MMQ_ISO_SMEM (3 * 2 * MMQ_ISO_CHUNK * MMQ_ISO_PAD * 8)

__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_isocorr_prep(const __grid_constant__ mmq_chain_ptrs cp, int C, int lgL, const int32_t* __restrict__ members, int64_t nmem,
               double* __restrict__ st) {
  const int S = C << lgL, lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  auto warp_total = [&](double v) { return __shfl_sync(0xffffffffu, post_warp_sum(v), 0); };
  for (int64_t q = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); q < nmem; q += warps) {
    const int64_t row = members[q];
    double sx = 0.0, sl = 0.0, nonfin = 0.0, badlog = 0.0, isnanv = 0.0;
    for (int k = lane; k < S; k += 32) {
      const double x = chain_x(cp, row, lgL, k);
      sx += x;
      sl += log(x);
      nonfin += isfinite(x) ? 0.0 : 1.0;
      badlog += isfinite(x) && x > 0.0 ? 0.0 : 1.0;
      isnanv += isnan(x) ? 1.0 : 0.0;
    }
    nonfin = warp_total(nonfin);
    badlog = warp_total(badlog);
    isnanv = warp_total(isnanv);
    const double mx = nonfin == 0.0 ? warp_total(sx) / (double)S : nan;
    const double ml = badlog == 0.0 ? warp_total(sl) / (double)S : nan;
    double ssx = 0.0, ssl = 0.0;
    for (int k = lane; k < S; k += 32) {
      const double x = chain_x(cp, row, lgL, k), dx = x - mx, dl = log(x) - ml;
      ssx += dx * dx;
      ssl += dl * dl;
    }
    ssx = warp_total(ssx);
    ssl = warp_total(ssl);
    if (lane == 0) {
      double* o = st + 5 * q;
      o[0] = mx; o[1] = ssx; o[2] = ml; o[3] = ssl; o[4] = isnanv > 0.0 ? 1.0 : 0.0;
    }
  }
}

__device__ __forceinline__ int64_t iso_items_of(int64_t k) {
  const int64_t T = (k + MMQ_ISO_TILE - 1) / MMQ_ISO_TILE;
  return k >= 2 ? T * (T + 1) / 2 : 0;
}

#define MMQ_ISO_SCAN 1024
__global__ void __launch_bounds__(MMQ_ISO_SCAN)
k_isocorr_items(const int64_t* __restrict__ gene_ptr, int64_t ngenes, int64_t* __restrict__ items) {
  __shared__ int64_t part[MMQ_ISO_SCAN];
  const int64_t g0 = ngenes * threadIdx.x / MMQ_ISO_SCAN, g1 = ngenes * (threadIdx.x + 1) / MMQ_ISO_SCAN;
  int64_t s = 0;
  for (int64_t g = g0; g < g1; ++g) s += iso_items_of(gene_ptr[g + 1] - gene_ptr[g]);
  part[threadIdx.x] = s;
  __syncthreads();
  for (int d = 1; d < MMQ_ISO_SCAN; d <<= 1) { /* inclusive Hillis-Steele scan */
    const int64_t v = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  s = part[threadIdx.x] - s;
  for (int64_t g = g0; g < g1; ++g) { items[g] = s; s += iso_items_of(gene_ptr[g + 1] - gene_ptr[g]); }
  if (threadIdx.x == MMQ_ISO_SCAN - 1) items[ngenes] = s;
}

__global__ void __launch_bounds__(MMQ_POST_THREADS)
k_isocorr(const __grid_constant__ mmq_chain_ptrs cp, int C, int lgL, int64_t ngenes, const int64_t* __restrict__ gene_ptr,
          const int32_t* __restrict__ members, const int64_t* __restrict__ pair_base, int64_t npairs,
          const double* __restrict__ st, const int64_t* __restrict__ items, double* __restrict__ out) {
  extern __shared__ double sh[];
  typedef double tile_t[MMQ_ISO_CHUNK][MMQ_ISO_PAD];
  tile_t* X = reinterpret_cast<tile_t*>(sh);  /* [2]: the draws of tile row / tile column */
  tile_t* D = X + 2;                          /* [2]: x - mean x */
  tile_t* E = X + 4;                          /* [2]: log x - mean log x */
  __shared__ int64_t s_row[2][MMQ_ISO_TILE];
  __shared__ double s_mx[2][MMQ_ISO_TILE], s_ml[2][MMQ_ISO_TILE];
  const int S = C << lgL, j = threadIdx.x & 31, i0 = threadIdx.x >> 5;
  const double nan = mmq_u2d(0x7ff8000000000000ull);
  const int64_t nitems = items[ngenes];
  for (int64_t it = blockIdx.x; it < nitems; it += gridDim.x) {
    int64_t lo = 0, hi = ngenes; /* items[lo] <= it < items[hi] */
    while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (items[mid] <= it) lo = mid; else hi = mid; }
    const int64_t g = lo, q0 = gene_ptr[g], k = gene_ptr[g + 1] - q0;
    const int T = (int)((k + MMQ_ISO_TILE - 1) / MMQ_ISO_TILE);
    int r = (int)(it - items[g]), ta = 0;
    while (r >= T - ta) { r -= T - ta; ++ta; }
    const int tb = ta + r;
    const bool diag = ta == tb;
    const int ka = (int)min((int64_t)MMQ_ISO_TILE, k - (int64_t)ta * MMQ_ISO_TILE);
    const int kb = (int)min((int64_t)MMQ_ISO_TILE, k - (int64_t)tb * MMQ_ISO_TILE);
    const int64_t qa = q0 + (int64_t)ta * MMQ_ISO_TILE, qb = q0 + (int64_t)tb * MMQ_ISO_TILE;
    const int nside = diag ? 1 : 2, B = diag ? 0 : 1;
    __syncthreads(); /* the previous item is done with the staging arrays */
    if (threadIdx.x < 2 * MMQ_ISO_TILE) {
      const int sd = threadIdx.x / MMQ_ISO_TILE, i = threadIdx.x % MMQ_ISO_TILE;
      if (sd < nside && i < (sd ? kb : ka)) {
        const int64_t q = (sd ? qb : qa) + i;
        s_row[sd][i] = members[q];
        s_mx[sd][i] = st[5 * q];
        s_ml[sd][i] = st[5 * q + 2];
      }
    }
    double sxy[4] = {0.0, 0.0, 0.0, 0.0}, sll[4] = {0.0, 0.0, 0.0, 0.0}, gt[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = 0; k0 < S; k0 += MMQ_ISO_CHUNK) {
      const int cn = min(MMQ_ISO_CHUNK, S - k0);
      __syncthreads();
      for (int v = threadIdx.x; v < nside * MMQ_ISO_TILE * MMQ_ISO_CHUNK; v += blockDim.x) {
        const int sd = v / (MMQ_ISO_TILE * MMQ_ISO_CHUNK), i = (v / MMQ_ISO_CHUNK) % MMQ_ISO_TILE, s = v % MMQ_ISO_CHUNK;
        if (i < (sd ? kb : ka) && s < cn) {
          const double x = chain_x(cp, s_row[sd][i], lgL, k0 + s);
          X[sd][s][i] = x;
          D[sd][s][i] = x - s_mx[sd][i];
          E[sd][s][i] = log(x) - s_ml[sd][i];
        }
      }
      __syncthreads();
      for (int s = 0; s < cn && i0 < ka; ++s) { /* warps without a row of the tile skip the chunk */
        const double xb = X[B][s][j], db = D[B][s][j], eb = E[B][s][j];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + 8 * u;
          if (i >= ka) break;
          const double xa = X[0][s][i];
          sxy[u] = fma(D[0][s][i], db, sxy[u]);
          sll[u] = fma(E[0][s][i], eb, sll[u]);
          gt[u] += xa > xb ? 2.0 : xa == xb ? 1.0 : 0.0;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + 8 * u;
      if (i >= ka || j >= kb || (diag && i >= j)) continue;
      const int64_t a = (int64_t)ta * MMQ_ISO_TILE + i, b = (int64_t)tb * MMQ_ISO_TILE + j;
      const int64_t p = pair_base[g] + a * (2 * k - a - 1) / 2 + (b - a - 1);
      const double* sa = st + 5 * (qa + i);
      const double* sb = st + 5 * (qb + j);
      auto corr = [&](double sum, double m1, double ss1, double m2, double ss2) {
        if (isnan(m1) || isnan(m2) || ss1 == 0.0 || ss2 == 0.0) return nan;
        const double c = sum / sqrt(ss1 * ss2);
        return c > 1.0 ? 1.0 : c < -1.0 ? -1.0 : c;
      };
      const bool bad = sa[4] != 0.0 || sb[4] != 0.0;
      out[p] = bad ? nan : corr(sxy[u], sa[0], sa[1], sb[0], sb[1]);
      out[npairs + p] = bad ? nan : corr(sll[u], sa[2], sa[3], sb[2], sb[3]);
      out[2 * npairs + p] = bad ? nan : gt[u] / (2.0 * (double)S);
    }
  }
}

/* ------------------------------------------------------------------ host */

static bool pow2_ok(int len) { return len >= 4 && len <= MMQ_MAX_ROW_LEN && (len & (len - 1)) == 0; }

int mmq_ensure_trace_groups(mmq_handle* h) {
  for (int kind = 0; kind < 2; ++kind) {
    mmq_group_set& g = h->groups[kind];
    if (g.ngroups == 0 || g.trace_valid) continue;
    if (!h->trace) return mmq_fail(h, MMQ_ERR_STATE, "no trace recorded yet");
    if (!g.trace_dev) {
      int rc = mmq_dev_alloc(h, (void**)&g.trace_dev, sizeof(double) * (size_t)g.ngroups * (size_t)h->trace_len);
      if (rc) return rc;
    }
    const int grid = (int)std::min<int64_t>(g.ngroups, (int64_t)h->num_sms * 16);
    k_group_trace<<<grid, 128, 0, h->stream>>>(h->trace, g.ptr_dev, g.members_dev, g.extra_dev, g.trace_dev, g.ngroups, h->trace_len);
    MMQ_LAUNCHED(h);
    g.trace_valid = true;
  }
  return MMQ_OK;
}

static int run_row_summaries(mmq_handle* h, cudaStream_t st, const double* src_dev, int64_t rows, int len, int do_log,
                             double* log_mean, double* var, double* tau, int32_t* win, int32_t* status, int npct,
                             const int32_t* pct_idx, double* pct) {
  if (rows <= 0) return MMQ_OK;
  double *d_mean = nullptr, *d_var = nullptr, *d_tau = nullptr, *d_pct = nullptr;
  int32_t *d_win = nullptr, *d_status = nullptr, *d_idx = nullptr;
  cudaError_t e = cudaSuccess;
  auto A = [&](void** p, size_t b) { if (e == cudaSuccess) e = cudaMalloc(p, b ? b : 16); };
  const bool want_sokal = log_mean || var || tau || win || status;
  int ret = MMQ_OK;
  if (want_sokal) {
    A((void**)&d_mean, sizeof(double) * rows); A((void**)&d_var, sizeof(double) * rows); A((void**)&d_tau, sizeof(double) * rows);
    A((void**)&d_win, sizeof(int32_t) * rows); A((void**)&d_status, sizeof(int32_t) * rows);
  }
  if (npct > 0 && pct) { A((void**)&d_pct, sizeof(double) * rows * npct); A((void**)&d_idx, sizeof(int32_t) * npct); }
  if (e == cudaSuccess && want_sokal) {
    const int grid = (int)std::min<int64_t>(rows, 148 * 8);
    k_row_sokal<<<grid, MMQ_POST_THREADS, sizeof(double) * 2 * len, st>>>(src_dev, rows, len, do_log, d_mean, d_var, d_tau, d_win, d_status);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
    auto D = [&](void* dst, const void* src, size_t b) { if (e == cudaSuccess && dst) e = cudaMemcpyAsync(dst, src, b, cudaMemcpyDeviceToHost, st); };
    D(log_mean, d_mean, sizeof(double) * rows); D(var, d_var, sizeof(double) * rows); D(tau, d_tau, sizeof(double) * rows);
    D(win, d_win, sizeof(int32_t) * rows); D(status, d_status, sizeof(int32_t) * rows);
  }
  if (e == cudaSuccess && npct > 0 && pct) {
    e = cudaMemcpyAsync(d_idx, pct_idx, sizeof(int32_t) * npct, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
      const int grid = (int)std::min<int64_t>(rows, 148 * 8);
      k_row_percentiles<<<grid, MMQ_POST_THREADS, sizeof(double) * len, st>>>(src_dev, rows, len, npct, d_idx, d_pct);
      g_mmq_launches.fetch_add(1);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(pct, d_pct, sizeof(double) * rows * npct, cudaMemcpyDeviceToHost, st);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) ret = mmq_cuda_fail(h, e, "row summaries", __FILE__, __LINE__);
  cudaFree(d_mean); cudaFree(d_var); cudaFree(d_tau); cudaFree(d_win); cudaFree(d_status); cudaFree(d_pct); cudaFree(d_idx);
  return ret;
}

extern "C" {

int mmq_set_groups(mmq_handle* h, int kind, int64_t ngroups, const int64_t* group_ptr, const int32_t* members, const double* extra) {
  if (!h || kind < 0 || kind > 1 || ngroups < 0 || (ngroups > 0 && (!group_ptr || group_ptr[0] != 0)))
    return mmq_fail(h, MMQ_ERR_ARG, "mmq_set_groups: bad arguments");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  mmq_group_set& g = h->groups[kind];
  if (g.ptr_dev) { mmq_dev_free(h, g.ptr_dev); g.ptr_dev = nullptr; }
  if (g.members_dev) { mmq_dev_free(h, g.members_dev); g.members_dev = nullptr; }
  if (g.extra_dev) { mmq_dev_free(h, g.extra_dev); g.extra_dev = nullptr; }
  if (g.trace_dev) { mmq_dev_free(h, g.trace_dev); g.trace_dev = nullptr; }
  g.ngroups = ngroups;
  g.trace_valid = false;
  if (ngroups == 0) return MMQ_OK;
  const int64_t nm = group_ptr[ngroups];
  for (int64_t q = 0; q < nm; ++q)
    if (members[q] < 0 || members[q] >= h->n) return mmq_fail(h, MMQ_ERR_ARG, "mmq_set_groups: member index out of range");
  int rc;
  if ((rc = mmq_dev_alloc(h, (void**)&g.ptr_dev, sizeof(int64_t) * (size_t)(ngroups + 1)))) return rc;
  if ((rc = mmq_dev_alloc(h, (void**)&g.members_dev, sizeof(int32_t) * (size_t)std::max<int64_t>(nm, 1)))) return rc;
  MMQ_CUDA(h, cudaMemcpyAsync(g.ptr_dev, group_ptr, sizeof(int64_t) * (size_t)(ngroups + 1), cudaMemcpyHostToDevice, h->stream));
  if (nm) MMQ_CUDA(h, cudaMemcpyAsync(g.members_dev, members, sizeof(int32_t) * (size_t)nm, cudaMemcpyHostToDevice, h->stream));
  if (extra) {
    if (h->trace_len <= 0) return mmq_fail(h, MMQ_ERR_STATE, "mmq_set_groups: extra given before any trace exists");
    const size_t b = sizeof(double) * (size_t)ngroups * (size_t)h->trace_len;
    if ((rc = mmq_dev_alloc(h, (void**)&g.extra_dev, b))) return rc;
    MMQ_CUDA(h, cudaMemcpyAsync(g.extra_dev, extra, b, cudaMemcpyHostToDevice, h->stream));
  }
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_summarize(mmq_handle* h, int which, double* log_mean, double* var, double* tau, int32_t* win,
                  int32_t* sokal_status, int npct, const int32_t* pct_idx, double* pct) {
  if (!h || which < 0 || which > 2) return mmq_fail(h, MMQ_ERR_ARG, "mmq_summarize: bad arguments");
  if (!h->trace) return mmq_fail(h, MMQ_ERR_STATE, "mmq_summarize: no trace recorded");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  const int L = h->trace_len;
  for (int j = 0; j < npct; ++j)
    if (pct_idx[j] < 0 || pct_idx[j] >= L) return mmq_fail(h, MMQ_ERR_ARG, "mmq_summarize: percentile index out of range");
  int rc = mmq_ensure_trace_groups(h);
  if (rc) return rc;
  const double* src = which == 0 ? h->trace : h->groups[which - 1].trace_dev;
  const int64_t rows = which == 0 ? h->n : h->groups[which - 1].ngroups;
  if (rows == 0) return MMQ_OK;
  if (!pow2_ok(L)) {
    /* sokal() fails for such lengths (src/sokal.cc:36-40, :108-126); callers map
     * failure to mcse = trace_length, iact = NaN (src/mmseq.cpp:1316-1318).
     * Percentiles and log means are not produced either. */
    if (sokal_status) for (int64_t r = 0; r < rows; ++r) sokal_status[r] = L < 4 ? 200 : (L > MMQ_MAX_ROW_LEN ? 100 : 201);
    return mmq_fail(h, MMQ_ERR_ARG, "mmq_summarize: trace_len must be a power of two in [4, 2048]");
  }
  return run_row_summaries(h, h->stream, src, rows, L, 1, log_mean, var, tau, win, sokal_status, npct, pct_idx, pct);
}

int mmq_get_group_trace(mmq_handle* h, int which, double* out) {
  if (!h || !out || which < 1 || which > 2) return mmq_fail(h, MMQ_ERR_ARG, "mmq_get_group_trace: bad arguments");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int rc = mmq_ensure_trace_groups(h);
  if (rc) return rc;
  mmq_group_set& g = h->groups[which - 1];
  if (g.ngroups == 0) return MMQ_OK;
  MMQ_CUDA(h, cudaMemcpyAsync(out, g.trace_dev, sizeof(double) * (size_t)g.ngroups * (size_t)h->trace_len, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_prop_summaries(mmq_handle* h, const int32_t* gene_of, const uint8_t* multi_iso, double* mean_prop,
                       double* sum_probit, double* sumsq_probit, int npct, const int32_t* pct_idx, double* pct,
                       double* prop_trace_out) {
  if (!h || !gene_of || !multi_iso) return mmq_fail(h, MMQ_ERR_ARG, "mmq_prop_summaries: NULL argument");
  if (!h->trace) return mmq_fail(h, MMQ_ERR_STATE, "mmq_prop_summaries: no trace recorded");
  mmq_group_set& G = h->groups[MMQ_GROUP_GENE];
  if (G.ngroups == 0) return mmq_fail(h, MMQ_ERR_STATE, "mmq_prop_summaries: gene groups not set");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  const int L = h->trace_len;
  const int64_t n = h->n;
  for (int64_t t = 0; t < n; ++t)
    if (gene_of[t] < 0 || gene_of[t] >= G.ngroups) return mmq_fail(h, MMQ_ERR_ARG, "mmq_prop_summaries: gene index out of range");
  int rc = mmq_ensure_trace_groups(h);
  if (rc) return rc;
  int32_t* d_gene = nullptr; uint8_t* d_multi = nullptr;
  double *d_prop = nullptr, *d_mean = nullptr, *d_s = nullptr, *d_ss = nullptr;
  cudaError_t e = cudaSuccess;
  auto A = [&](void** p, size_t b) { if (e == cudaSuccess) e = cudaMalloc(p, b ? b : 16); };
  A((void**)&d_gene, sizeof(int32_t) * n); A((void**)&d_multi, n); A((void**)&d_prop, sizeof(double) * n * L);
  A((void**)&d_mean, sizeof(double) * n); A((void**)&d_s, sizeof(double) * n); A((void**)&d_ss, sizeof(double) * n);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_gene, gene_of, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_multi, multi_iso, n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) {
    const int grid = (int)std::min<int64_t>(n, (int64_t)h->num_sms * 8);
    k_prop<<<grid, MMQ_POST_THREADS, 0, h->stream>>>(h->trace, G.trace_dev, d_gene, d_multi, n, L, d_prop, d_mean, d_s, d_ss);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  auto D = [&](void* dst, const void* src, size_t b) { if (e == cudaSuccess && dst) e = cudaMemcpyAsync(dst, src, b, cudaMemcpyDeviceToHost, h->stream); };
  D(mean_prop, d_mean, sizeof(double) * n); D(sum_probit, d_s, sizeof(double) * n); D(sumsq_probit, d_ss, sizeof(double) * n);
  D(prop_trace_out, d_prop, sizeof(double) * n * L);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  int ret = MMQ_OK;
  if (e != cudaSuccess) ret = mmq_cuda_fail(h, e, "mmq_prop_summaries", __FILE__, __LINE__);
  if (ret == MMQ_OK && npct > 0 && pct) {
    if (!pow2_ok(L)) ret = mmq_fail(h, MMQ_ERR_ARG, "mmq_prop_summaries: trace_len must be a power of two in [4, 2048]");
    else ret = run_row_summaries(h, h->stream, d_prop, n, L, 0, nullptr, nullptr, nullptr, nullptr, nullptr, npct, pct_idx, pct);
  }
  cudaFree(d_gene); cudaFree(d_multi); cudaFree(d_prop); cudaFree(d_mean); cudaFree(d_s); cudaFree(d_ss);
  return ret;
}

int mmq_unique_hits_sets(mmq_handle* h, const int32_t* set_of, int64_t nsets, int32_t* out) {
  if (!h || !set_of || !out || nsets < 0) return mmq_fail(h, MMQ_ERR_ARG, "mmq_unique_hits_sets: bad arguments");
  if (nsets == 0) return MMQ_OK;
  for (int64_t t = 0; t < h->n; ++t)
    if (set_of[t] >= nsets) return mmq_fail(h, MMQ_ERR_ARG, "mmq_unique_hits_sets: set index out of range");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int32_t *d_set = nullptr, *d_out = nullptr;
  MMQ_CUDA(h, cudaMalloc(&d_set, sizeof(int32_t) * (size_t)h->n));
  cudaError_t e = cudaMalloc(&d_out, sizeof(int32_t) * (size_t)nsets);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_set, set_of, sizeof(int32_t) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_out, 0, sizeof(int32_t) * (size_t)nsets, h->stream);
  int ret = MMQ_OK;
  if (e == cudaSuccess && h->m > 0) {
    const int grid = mmq_grid_for(h->m, 256, h->num_sms * 8);
    if (h->has_k) k_uh_sets<true><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_set, h->m, d_out);
    else k_uh_sets<false><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_set, h->m, d_out);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) ret = mmq_allreduce(h, d_out, (size_t)nsets, 0);
  if (e == cudaSuccess && ret == MMQ_OK) e = cudaMemcpyAsync(out, d_out, sizeof(int32_t) * (size_t)nsets, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) ret = mmq_cuda_fail(h, e, "mmq_unique_hits_sets", __FILE__, __LINE__);
  cudaFree(d_set); cudaFree(d_out);
  return ret;
}

int mmq_prior_draws(int device, int64_t count, const int64_t* ids, const double* rate, double alpha, uint32_t seed,
                    int trace_len, double* out) {
  if (count < 0 || trace_len <= 0 || (count > 0 && (!ids || !rate || !out)) || !(alpha > 0.0))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_prior_draws: bad arguments");
  if (count == 0) return MMQ_OK;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "cudaSetDevice", __FILE__, __LINE__);
  int64_t* d_ids = nullptr; double *d_rate = nullptr, *d_out = nullptr;
  auto A = [&](void** p, size_t b) { if (e == cudaSuccess) e = cudaMalloc(p, b); };
  A((void**)&d_ids, sizeof(int64_t) * count); A((void**)&d_rate, sizeof(double) * count);
  A((void**)&d_out, sizeof(double) * count * trace_len);
  if (e == cudaSuccess) e = cudaMemcpy(d_ids, ids, sizeof(int64_t) * count, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d_rate, rate, sizeof(double) * count, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_prior<<<mmq_grid_for(count * trace_len, 128, 148 * 16), 128>>>(d_ids, d_rate, count, trace_len, alpha, seed, d_out);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, sizeof(double) * count * trace_len, cudaMemcpyDeviceToHost);
  cudaFree(d_ids); cudaFree(d_rate); cudaFree(d_out);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_prior_draws", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_sokal_batch(int device, int64_t rows, int len, const double* x, double* var, double* tau, int32_t* win, int32_t* status) {
  if (rows < 0 || !x) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_sokal_batch: bad arguments");
  if (!pow2_ok(len)) {
    /* the reference's return codes: src/sokal.cc:36-40 (100), :108-111 (200), :119-126 (201) */
    const int code = len < 4 ? 200 : (len > MMQ_MAX_ROW_LEN ? 100 : 201);
    if (status) for (int64_t r = 0; r < rows; ++r) status[r] = code;
    return MMQ_OK;
  }
  if (rows == 0) return MMQ_OK;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "cudaSetDevice", __FILE__, __LINE__);
  double* d_x = nullptr;
  e = cudaMalloc(&d_x, sizeof(double) * (size_t)rows * (size_t)len);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "cudaMalloc", __FILE__, __LINE__);
  e = cudaMemcpy(d_x, x, sizeof(double) * (size_t)rows * (size_t)len, cudaMemcpyHostToDevice);
  int ret = MMQ_OK;
  if (e != cudaSuccess) ret = mmq_cuda_fail(nullptr, e, "cudaMemcpy", __FILE__, __LINE__);
  else ret = run_row_summaries(nullptr, 0, d_x, rows, len, 0, nullptr, var, tau, win, status, 0, nullptr, nullptr);
  cudaFree(d_x);
  return ret;
}

int mmq_chain_diagnostics_dev(const double* const* chain_dev, int nchains, int64_t rows, int L, double* out_dev, void* cuda_stream) {
  if (!chain_dev || nchains < 2 || nchains > MMQ_CHAINS_MAX || rows < 0 || L < 8 || L > MMQ_MAX_ROW_LEN || (L & (L - 1)) != 0 ||
      nchains * L > MMQ_CHAIN_SMAX || (rows > 0 && !out_dev))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_chain_diagnostics_dev: bad arguments");
  mmq_chain_ptrs cp = {};
  for (int c = 0; c < nchains; ++c) {
    if (!chain_dev[c]) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_chain_diagnostics_dev: NULL chain");
    cp.p[c] = chain_dev[c];
  }
  if (rows == 0) return MMQ_OK;
  int dev = 0, sms = 0, lgL = 0;
  while ((1 << lgL) < L) ++lgL;
  const size_t smem = chain_smem_bytes(nchains * L);
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, MMQ_CHAIN_DIAG_SMEM_CAP);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_chain_diagnostics_dev", __FILE__, __LINE__);
  const int grid = (int)std::min<int64_t>(rows, 2 * (int64_t)sms);
  k_chain_diag<<<grid, MMQ_POST_THREADS, smem, (cudaStream_t)cuda_stream>>>(cp, nchains, rows, lgL, out_dev);
  g_mmq_launches.fetch_add(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_chain_diag", __FILE__, __LINE__);
  return MMQ_OK;
}

/* The checks of the handle forms (fn: the caller's name): no NULL handle, a trace on every chain, the same n, trace_len
 * and group counts, and a trace_len within the limits of the kernels (a power of two in [min_len, 2048]). */
static int chain_handles_check(mmq_handle* const* chains, int nchains, const char* fn, int min_len = 8) {
  auto fail = [&](mmq_handle* h, int code, const char* what) { return mmq_fail(h, code, std::string(fn) + ": " + what); };
  for (int c = 0; c < nchains; ++c)
    if (!chains[c]) return fail(nullptr, MMQ_ERR_ARG, "NULL handle");
  mmq_handle* h0 = chains[0];
  for (int c = 0; c < nchains; ++c) {
    mmq_handle* h = chains[c];
    if (!h->trace) return fail(h0, MMQ_ERR_STATE, "a chain has no trace recorded");
    if (h->n != h0->n || h->trace_len != h0->trace_len || h->groups[0].ngroups != h0->groups[0].ngroups ||
        h->groups[1].ngroups != h0->groups[1].ngroups)
      return fail(h0, MMQ_ERR_ARG, "the chains differ in n, trace_len or group counts");
  }
  const int L = h0->trace_len;
  if (L < min_len || L > MMQ_MAX_ROW_LEN || (L & (L - 1)) != 0 || nchains * L > MMQ_CHAIN_SMAX)
    return fail(h0, MMQ_ERR_ARG, ("trace_len must be a power of two in [" + std::to_string(min_len) +
                                  ", 2048] with nchains * trace_len <= 8192").c_str());
  return MMQ_OK;
}

/* Chain c's draws t[c] (rows x L, on chains[c]'s device) as pointers src[c] on chains[0]'s device: read in place there,
 * copied from other devices with cudaMemcpyPeerAsync on chains[0]'s stream into *ws, a block-cache workspace of rows L 8
 * bytes per such chain that the caller frees.  Runs with chains[0]'s device current. */
static cudaError_t chain_gather(mmq_handle* const* chains, int nchains, const double* const* t, int64_t rows, int L, double** ws,
                                const double** src) {
  mmq_handle* h0 = chains[0];
  const size_t tbytes = sizeof(double) * (size_t)rows * (size_t)L;
  int remote = 0;
  for (int c = 1; c < nchains; ++c) remote += chains[c]->device != h0->device;
  cudaError_t e = remote ? mmq_cache_malloc(ws, tbytes * (size_t)remote) : cudaSuccess;
  for (int c = 0, r = 0; c < nchains && e == cudaSuccess; ++c) {
    if (chains[c]->device == h0->device) { src[c] = t[c]; continue; }
    double* dst = *ws + (size_t)r++ * (size_t)rows * (size_t)L;
    e = cudaMemcpyPeerAsync(dst, h0->device, t[c], chains[c]->device, tbytes, h0->stream);
    src[c] = dst;
  }
  return e;
}

int mmq_chain_diagnostics(mmq_handle* const* chains, int nchains, int which, double* rhat, double* ess_bulk, double* ess_tail,
                          double* log_mean, double* log_sd) {
  if (!chains || nchains < 2 || nchains > MMQ_CHAINS_MAX || which < 0 || which > 2)
    return mmq_fail(chains ? chains[0] : nullptr, MMQ_ERR_ARG, "mmq_chain_diagnostics: bad arguments");
  if (const int rc = chain_handles_check(chains, nchains, "mmq_chain_diagnostics")) return rc;
  mmq_handle* h0 = chains[0];
  const int L = h0->trace_len;
  const int64_t rows = which == 0 ? h0->n : h0->groups[which - 1].ngroups;
  if (rows == 0) return MMQ_OK;
  /* every chain's trace complete on its own device */
  for (int c = 0; c < nchains; ++c) {
    mmq_handle* h = chains[c];
    MMQ_CUDA(h0, cudaSetDevice(h->device));
    if (which > 0) { const int rc = mmq_ensure_trace_groups(h); if (rc) return mmq_fail(h0, rc, mmq_last_error(h)); }
    MMQ_CUDA(h0, cudaStreamSynchronize(h->stream));
  }
  MMQ_CUDA(h0, cudaSetDevice(h0->device));
  double *ws = nullptr, *out = nullptr;
  const double *t[MMQ_CHAINS_MAX] = {}, *src[MMQ_CHAINS_MAX] = {};
  for (int c = 0; c < nchains; ++c) t[c] = which == 0 ? chains[c]->trace : chains[c]->groups[which - 1].trace_dev;
  cudaError_t e = mmq_cache_malloc(&out, sizeof(double) * 5 * (size_t)rows);
  if (e == cudaSuccess) e = chain_gather(chains, nchains, t, rows, L, &ws, src);
  int ret = MMQ_OK;
  if (e == cudaSuccess) {
    ret = mmq_chain_diagnostics_dev(src, nchains, rows, L, out, h0->stream);
    if (ret) ret = mmq_fail(h0, ret, mmq_last_error(nullptr));
  }
  double* dst[5] = {rhat, ess_bulk, ess_tail, log_mean, log_sd};
  for (int q = 0; q < 5 && e == cudaSuccess && ret == MMQ_OK; ++q)
    if (dst[q]) e = cudaMemcpyAsync(dst[q], out + (size_t)q * (size_t)rows, sizeof(double) * (size_t)rows, cudaMemcpyDeviceToHost, h0->stream);
  const cudaError_t es = cudaStreamSynchronize(h0->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h0, e, "mmq_chain_diagnostics", __FILE__, __LINE__);
  mmq_cache_free(out);
  mmq_cache_free(ws);
  return ret;
}

int mmq_pooled_summaries_dev(const double* const* chain_dev, int nchains, int64_t rows, int L, int mode, int npct,
                             const int32_t* pct_idx_dev, double* out_dev, double* pct_dev, void* cuda_stream) {
  if (!chain_dev || nchains < 2 || nchains > MMQ_CHAINS_MAX || rows < 0 || L < 8 || L > MMQ_MAX_ROW_LEN || (L & (L - 1)) != 0 ||
      nchains * L > MMQ_CHAIN_SMAX || (mode != 0 && mode != 1) || npct < 0 || (rows > 0 && !out_dev) ||
      (rows > 0 && npct > 0 && (!pct_idx_dev || !pct_dev)))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_pooled_summaries_dev: bad arguments");
  mmq_chain_ptrs cp = {};
  for (int c = 0; c < nchains; ++c) {
    if (!chain_dev[c]) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_pooled_summaries_dev: NULL chain");
    cp.p[c] = chain_dev[c];
  }
  if (rows == 0) return MMQ_OK;
  int dev = 0, sms = 0, lgL = 0;
  while ((1 << lgL) < L) ++lgL;
  const int S = nchains * L, P = chain_pow2_at_least(S);
  const size_t smem = sizeof(double) * (size_t)(mode == 0 ? P + S + L : P);
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_pool_summ, cudaFuncAttributeMaxDynamicSharedMemorySize, MMQ_POOL_SMEM_CAP);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_pooled_summaries_dev", __FILE__, __LINE__);
  const int grid = (int)std::min<int64_t>(rows, 2 * (int64_t)sms);
  k_pool_summ<<<grid, MMQ_POST_THREADS, smem, (cudaStream_t)cuda_stream>>>(cp, nchains, rows, lgL, mode, npct, pct_idx_dev, out_dev, pct_dev);
  g_mmq_launches.fetch_add(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_pool_summ", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_pooled_summaries(mmq_handle* const* chains, int nchains, int which, const int32_t* gene_of, const uint8_t* multi_iso,
                         int npct, const int32_t* pct_idx, double* mean, double* sd, double* ess_mean, double* sum_probit,
                         double* sumsq_probit, double* pct) {
  if (!chains || nchains < 2 || nchains > MMQ_CHAINS_MAX || which < 0 || which > 3 || npct < 0 || (npct > 0 && (!pct_idx || !pct)) ||
      (which == 3 && (!gene_of || !multi_iso)))
    return mmq_fail(chains ? chains[0] : nullptr, MMQ_ERR_ARG, "mmq_pooled_summaries: bad arguments");
  if (const int rc = chain_handles_check(chains, nchains, "mmq_pooled_summaries")) return rc;
  mmq_handle* h0 = chains[0];
  const int L = h0->trace_len;
  const int64_t n = h0->n;
  const int64_t rows = which == 0 || which == 3 ? n : h0->groups[which - 1].ngroups;
  for (int j = 0; j < npct; ++j)
    if (pct_idx[j] < 0 || pct_idx[j] >= nchains * L) return mmq_fail(h0, MMQ_ERR_ARG, "mmq_pooled_summaries: percentile index out of range");
  if (which == 3) {
    if (h0->groups[MMQ_GROUP_GENE].ngroups == 0) return mmq_fail(h0, MMQ_ERR_STATE, "mmq_pooled_summaries: gene groups not set");
    for (int64_t t = 0; t < n; ++t)
      if (gene_of[t] < 0 || gene_of[t] >= h0->groups[MMQ_GROUP_GENE].ngroups)
        return mmq_fail(h0, MMQ_ERR_ARG, "mmq_pooled_summaries: gene index out of range");
  }
  if (rows == 0) return MMQ_OK;
  const size_t tbytes = sizeof(double) * (size_t)rows * (size_t)L;
  /* every chain's draws complete on its own device; proportions: k_prop on each chain's device, into prop[c] */
  double* prop[MMQ_CHAINS_MAX] = {};
  double* part[MMQ_CHAINS_MAX] = {}; /* per chain: mean, sum and sum of squares of the probits, fp64[3 n] */
  int32_t* gdev[MMQ_CHAINS_MAX] = {};
  uint8_t* mdev[MMQ_CHAINS_MAX] = {};
  std::vector<double> sums(which == 3 ? (size_t)nchains * 3 * (size_t)n : 0);
  cudaError_t e = cudaSuccess;
  int ret = MMQ_OK;
  for (int c = 0; c < nchains && e == cudaSuccess && ret == MMQ_OK; ++c) {
    mmq_handle* h = chains[c];
    e = cudaSetDevice(h->device);
    if (e != cudaSuccess) break;
    if (which > 0) { const int rc = mmq_ensure_trace_groups(h); if (rc) { ret = mmq_fail(h0, rc, mmq_last_error(h)); break; } }
    if (which == 3) {
      e = mmq_cache_malloc(&prop[c], tbytes);
      if (e == cudaSuccess) e = mmq_cache_malloc(&part[c], sizeof(double) * 3 * (size_t)n);
      if (e == cudaSuccess) e = mmq_cache_malloc(&gdev[c], sizeof(int32_t) * (size_t)n);
      if (e == cudaSuccess) e = mmq_cache_malloc(&mdev[c], (size_t)n);
      if (e == cudaSuccess) e = cudaMemcpyAsync(gdev[c], gene_of, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = cudaMemcpyAsync(mdev[c], multi_iso, (size_t)n, cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) {
        const int grid = (int)std::min<int64_t>(n, (int64_t)h->num_sms * 8);
        k_prop<<<grid, MMQ_POST_THREADS, 0, h->stream>>>(h->trace, h->groups[MMQ_GROUP_GENE].trace_dev, gdev[c], mdev[c], n, L, prop[c],
                                                          part[c], part[c] + n, part[c] + 2 * n);
        g_mmq_launches.fetch_add(1);
        e = cudaGetLastError();
      }
      if (e == cudaSuccess) e = cudaMemcpyAsync(sums.data() + (size_t)c * 3 * (size_t)n, part[c], sizeof(double) * 3 * (size_t)n,
                                                cudaMemcpyDeviceToHost, h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  }
  double *ws = nullptr, *out = nullptr, *d_pct = nullptr;
  int32_t* d_idx = nullptr;
  const double *t[MMQ_CHAINS_MAX] = {}, *src[MMQ_CHAINS_MAX] = {};
  for (int c = 0; c < nchains; ++c) t[c] = which == 3 ? prop[c] : which == 0 ? chains[c]->trace : chains[c]->groups[which - 1].trace_dev;
  if (e == cudaSuccess && ret == MMQ_OK) e = cudaSetDevice(h0->device);
  if (e == cudaSuccess && ret == MMQ_OK) e = mmq_cache_malloc(&out, sizeof(double) * 3 * (size_t)rows);
  if (e == cudaSuccess && ret == MMQ_OK && npct > 0) {
    e = mmq_cache_malloc(&d_pct, sizeof(double) * (size_t)rows * (size_t)npct);
    if (e == cudaSuccess) e = mmq_cache_malloc(&d_idx, sizeof(int32_t) * (size_t)npct);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_idx, pct_idx, sizeof(int32_t) * (size_t)npct, cudaMemcpyHostToDevice, h0->stream);
  }
  if (e == cudaSuccess && ret == MMQ_OK) e = chain_gather(chains, nchains, t, rows, L, &ws, src);
  if (e == cudaSuccess && ret == MMQ_OK) {
    ret = mmq_pooled_summaries_dev(src, nchains, rows, L, which == 3 ? 1 : 0, npct, d_idx, out, d_pct, h0->stream);
    if (ret) ret = mmq_fail(h0, ret, mmq_last_error(nullptr));
  }
  double* dst[3] = {mean, which == 3 ? nullptr : sd, which == 3 ? nullptr : ess_mean};
  for (int q = 0; q < 3 && e == cudaSuccess && ret == MMQ_OK; ++q)
    if (dst[q]) e = cudaMemcpyAsync(dst[q], out + (size_t)q * (size_t)rows, sizeof(double) * (size_t)rows, cudaMemcpyDeviceToHost, h0->stream);
  if (e == cudaSuccess && ret == MMQ_OK && npct > 0)
    e = cudaMemcpyAsync(pct, d_pct, sizeof(double) * (size_t)rows * (size_t)npct, cudaMemcpyDeviceToHost, h0->stream);
  const cudaError_t es = cudaStreamSynchronize(h0->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h0, e, "mmq_pooled_summaries", __FILE__, __LINE__);
  /* the probit sums of the chains, added in chain order */
  if (ret == MMQ_OK && which == 3)
    for (int64_t t = 0; t < n; ++t) {
      double s = 0.0, ss = 0.0;
      for (int c = 0; c < nchains; ++c) {
        s += sums[((size_t)c * 3 + 1) * (size_t)n + (size_t)t];
        ss += sums[((size_t)c * 3 + 2) * (size_t)n + (size_t)t];
      }
      if (sum_probit) sum_probit[t] = s;
      if (sumsq_probit) sumsq_probit[t] = ss;
    }
  mmq_cache_free(out); mmq_cache_free(ws); mmq_cache_free(d_pct); mmq_cache_free(d_idx);
  for (int c = 0; c < nchains; ++c) { /* into the cache of the device each block came from */
    if (!prop[c] && !part[c] && !gdev[c] && !mdev[c]) continue;
    cudaSetDevice(chains[c]->device);
    mmq_cache_free(prop[c]); mmq_cache_free(part[c]); mmq_cache_free(gdev[c]); mmq_cache_free(mdev[c]);
  }
  cudaSetDevice(h0->device);
  return ret;
}

static bool tpm_len_ok(int nchains, int L) {
  return nchains >= 1 && nchains <= MMQ_CHAINS_MAX && pow2_ok(L) && nchains * L <= MMQ_CHAIN_SMAX;
}

int64_t mmq_draw_totals_workspace_bytes(int64_t rows, int L) {
  if (rows < 0 || !pow2_ok(L)) return 0;
  const int64_t ntiles = (rows + MMQ_TOTALS_TILE - 1) / MMQ_TOTALS_TILE;
  return (int64_t)sizeof(double) * ntiles * L;
}

int mmq_draw_totals_dev(const double* trace_dev, int64_t rows, int L, double* totals_dev, void* workspace_dev, void* cuda_stream) {
  if (rows < 0 || !pow2_ok(L) || !totals_dev || (rows > 0 && (!trace_dev || !workspace_dev)))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_draw_totals_dev: bad arguments");
  const cudaStream_t st = (cudaStream_t)cuda_stream;
  const int64_t ntiles = (rows + MMQ_TOTALS_TILE - 1) / MMQ_TOTALS_TILE;
  const int block = std::min(L, MMQ_TOTALS_THREADS), chunks = (L + block - 1) / block;
  double* partial = static_cast<double*>(workspace_dev);
  if (ntiles > 0) {
    k_draw_totals<<<dim3((unsigned)ntiles, (unsigned)chunks), block, 0, st>>>(trace_dev, rows, L, partial);
    g_mmq_launches.fetch_add(1);
  }
  k_totals_fold<<<chunks, block, 0, st>>>(partial, ntiles, L, totals_dev);
  g_mmq_launches.fetch_add(1);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_draw_totals", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_tpm_summaries_dev(const double* const* chain_dev, const double* totals_dev, int nchains, int64_t rows, int L,
                          const int64_t* group_ptr_dev, const int32_t* members_dev, int npct, const int32_t* pct_idx_dev,
                          double* out_dev, double* pct_dev, void* cuda_stream) {
  if (!chain_dev || !tpm_len_ok(nchains, L) || rows < 0 || npct < 0 || (!group_ptr_dev) != (!members_dev) ||
      (rows > 0 && (!out_dev || !totals_dev)) || (rows > 0 && npct > 0 && (!pct_idx_dev || !pct_dev)))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_tpm_summaries_dev: bad arguments");
  mmq_chain_ptrs cp = {};
  for (int c = 0; c < nchains; ++c) {
    if (!chain_dev[c]) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_tpm_summaries_dev: NULL chain");
    cp.p[c] = chain_dev[c];
  }
  if (rows == 0) return MMQ_OK;
  int dev = 0, sms = 0, lgL = 0;
  while ((1 << lgL) < L) ++lgL;
  const size_t smem = sizeof(double) * (size_t)chain_pow2_at_least(nchains * L);
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tpm_summ, cudaFuncAttributeMaxDynamicSharedMemorySize, MMQ_TPM_SMEM_CAP);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_tpm_summaries_dev", __FILE__, __LINE__);
  const int grid = (int)std::min<int64_t>(rows, 2 * (int64_t)sms);
  k_tpm_summ<<<grid, MMQ_POST_THREADS, smem, (cudaStream_t)cuda_stream>>>(cp, totals_dev, nchains, rows, lgL, group_ptr_dev, members_dev,
                                                                          npct, pct_idx_dev, out_dev, pct_dev);
  g_mmq_launches.fetch_add(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_tpm_summ", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_tpm_summaries(mmq_handle* const* chains, int nchains, int which, int npct, const int32_t* pct_idx, double* mean, double* sd,
                      double* pct, double* totals_out) {
  if (!chains || nchains < 1 || nchains > MMQ_CHAINS_MAX || which < 0 || which > 2 || npct < 0 || (npct > 0 && !pct_idx))
    return mmq_fail(chains ? chains[0] : nullptr, MMQ_ERR_ARG, "mmq_tpm_summaries: bad arguments");
  if (const int rc = chain_handles_check(chains, nchains, "mmq_tpm_summaries", 4)) return rc;
  mmq_handle* h0 = chains[0];
  const int L = h0->trace_len;
  const int64_t n = h0->n;
  for (int j = 0; j < npct; ++j)
    if (pct_idx[j] < 0 || pct_idx[j] >= nchains * L) return mmq_fail(h0, MMQ_ERR_ARG, "mmq_tpm_summaries: percentile index out of range");
  const mmq_group_set* g = which == 0 ? nullptr : &h0->groups[which - 1];
  const int64_t rows = which == 0 ? n : g->ngroups;
  /* every chain's draws complete on its own device */
  for (int c = 0; c < nchains; ++c) {
    MMQ_CUDA(h0, cudaSetDevice(chains[c]->device));
    MMQ_CUDA(h0, cudaStreamSynchronize(chains[c]->stream));
  }
  MMQ_CUDA(h0, cudaSetDevice(h0->device));
  double *ws = nullptr, *work = nullptr, *totals = nullptr, *out = nullptr, *d_pct = nullptr;
  int32_t* d_idx = nullptr;
  const double *t[MMQ_CHAINS_MAX] = {}, *src[MMQ_CHAINS_MAX] = {};
  for (int c = 0; c < nchains; ++c) t[c] = chains[c]->trace;
  const int64_t wbytes = mmq_draw_totals_workspace_bytes(n, L);
  cudaError_t e = mmq_cache_malloc(&work, (size_t)std::max<int64_t>(wbytes, 8));
  if (e == cudaSuccess) e = mmq_cache_malloc(&totals, sizeof(double) * (size_t)nchains * (size_t)L);
  if (e == cudaSuccess) e = mmq_cache_malloc(&out, sizeof(double) * 2 * (size_t)std::max<int64_t>(rows, 1));
  if (e == cudaSuccess && npct > 0) {
    e = mmq_cache_malloc(&d_pct, sizeof(double) * (size_t)std::max<int64_t>(rows, 1) * (size_t)npct);
    if (e == cudaSuccess) e = mmq_cache_malloc(&d_idx, sizeof(int32_t) * (size_t)npct);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_idx, pct_idx, sizeof(int32_t) * (size_t)npct, cudaMemcpyHostToDevice, h0->stream);
  }
  if (e == cudaSuccess) e = chain_gather(chains, nchains, t, n, L, &ws, src);
  int ret = MMQ_OK;
  for (int c = 0; c < nchains && e == cudaSuccess && ret == MMQ_OK; ++c) /* one workspace, reused in stream order */
    ret = mmq_draw_totals_dev(src[c], n, L, totals + (size_t)c * (size_t)L, work, h0->stream);
  if (e == cudaSuccess && ret == MMQ_OK)
    ret = mmq_tpm_summaries_dev(src, totals, nchains, rows, L, g ? g->ptr_dev : nullptr, g ? g->members_dev : nullptr, npct, d_idx, out, d_pct,
                                h0->stream);
  if (ret) ret = mmq_fail(h0, ret, mmq_last_error(nullptr));
  auto D = [&](void* dst, const void* from, size_t b) {
    if (e == cudaSuccess && ret == MMQ_OK && dst && b) e = cudaMemcpyAsync(dst, from, b, cudaMemcpyDeviceToHost, h0->stream);
  };
  D(mean, out, sizeof(double) * (size_t)rows);
  D(sd, out + rows, sizeof(double) * (size_t)rows);
  if (npct > 0) D(pct, d_pct, sizeof(double) * (size_t)rows * (size_t)npct);
  D(totals_out, totals, sizeof(double) * (size_t)nchains * (size_t)L);
  const cudaError_t es = cudaStreamSynchronize(h0->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h0, e, "mmq_tpm_summaries", __FILE__, __LINE__);
  mmq_cache_free(ws); mmq_cache_free(work); mmq_cache_free(totals); mmq_cache_free(out); mmq_cache_free(d_pct); mmq_cache_free(d_idx);
  return ret;
}

int mmq_allele_only_counts(mmq_handle* h, const int32_t* unit_of, const uint8_t* side, int64_t nunits, int32_t* a_only, int32_t* b_only) {
  if (!h || !unit_of || !side || !a_only || !b_only || nunits < 0) return mmq_fail(h, MMQ_ERR_ARG, "mmq_allele_only_counts: bad arguments");
  for (int64_t t = 0; t < h->n; ++t)
    if (unit_of[t] < -1 || unit_of[t] >= nunits || side[t] > 1)
      return mmq_fail(h, MMQ_ERR_ARG, "mmq_allele_only_counts: unit index or side out of range");
  if (nunits == 0) return MMQ_OK;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int32_t *d_unit = nullptr, *d_out = nullptr;
  uint8_t* d_side = nullptr;
  cudaError_t e = mmq_cache_malloc(&d_unit, sizeof(int32_t) * (size_t)std::max<int64_t>(h->n, 1));
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_side, (size_t)std::max<int64_t>(h->n, 1));
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_out, sizeof(int32_t) * 2 * (size_t)nunits);
  if (e == cudaSuccess && h->n > 0) e = cudaMemcpyAsync(d_unit, unit_of, sizeof(int32_t) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess && h->n > 0) e = cudaMemcpyAsync(d_side, side, (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_out, 0, sizeof(int32_t) * 2 * (size_t)nunits, h->stream);
  int ret = MMQ_OK;
  if (e == cudaSuccess && h->m > 0) {
    const int grid = mmq_grid_for(h->m, 256, h->num_sms * 8);
    if (h->has_k) k_allele_only<true><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_unit, d_side, h->m, d_out, d_out + nunits);
    else k_allele_only<false><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_unit, d_side, h->m, d_out, d_out + nunits);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) ret = mmq_allreduce(h, d_out, 2 * (size_t)nunits, 0);
  if (e == cudaSuccess && ret == MMQ_OK) e = cudaMemcpyAsync(a_only, d_out, sizeof(int32_t) * (size_t)nunits, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && ret == MMQ_OK) e = cudaMemcpyAsync(b_only, d_out + nunits, sizeof(int32_t) * (size_t)nunits, cudaMemcpyDeviceToHost, h->stream);
  const cudaError_t es = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h, e, "mmq_allele_only_counts", __FILE__, __LINE__);
  mmq_cache_free(d_unit); mmq_cache_free(d_side); mmq_cache_free(d_out);
  return ret;
}

int mmq_allelic_summaries_dev(const double* const* chain_dev, const double* const* prior_dev, int nchains, int64_t n, int64_t nprior,
                              int64_t rows, int L, const int64_t* a_ptr_dev, const int32_t* a_mem_dev, const int64_t* b_ptr_dev,
                              const int32_t* b_mem_dev, int npct, const int32_t* pct_idx_dev, double* out_dev, double* pct_dev,
                              void* cuda_stream) {
  if (!chain_dev || !tpm_len_ok(nchains, L) || n < 0 || nprior < 0 || n + nprior > INT32_MAX || rows < 0 || npct < 0 ||
      (nprior > 0 && !prior_dev) ||
      (rows > 0 && (!a_ptr_dev || !a_mem_dev || !b_ptr_dev || !b_mem_dev || !out_dev)) || (rows > 0 && npct > 0 && (!pct_idx_dev || !pct_dev)))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_allelic_summaries_dev: bad arguments");
  mmq_chain_ptrs cp = {}, pp = {};
  for (int c = 0; c < nchains; ++c) {
    if (!chain_dev[c] || (nprior > 0 && !prior_dev[c])) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_allelic_summaries_dev: NULL chain or prior");
    cp.p[c] = chain_dev[c];
    pp.p[c] = nprior > 0 ? prior_dev[c] : nullptr;
  }
  if (rows == 0) return MMQ_OK;
  int dev = 0, sms = 0, lgL = 0;
  while ((1 << lgL) < L) ++lgL;
  const size_t smem = sizeof(double) * (size_t)chain_pow2_at_least(nchains * L);
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_allelic_summ, cudaFuncAttributeMaxDynamicSharedMemorySize, MMQ_ALLELIC_SMEM_CAP);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_allelic_summaries_dev", __FILE__, __LINE__);
  const int grid = (int)std::min<int64_t>(rows, 2 * (int64_t)sms);
  k_allelic_summ<<<grid, MMQ_POST_THREADS, smem, (cudaStream_t)cuda_stream>>>(cp, pp, nchains, n, rows, lgL, a_ptr_dev, a_mem_dev, b_ptr_dev,
                                                                              b_mem_dev, npct, pct_idx_dev, out_dev, pct_dev);
  g_mmq_launches.fetch_add(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_allelic_summ", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_allelic_summaries(mmq_handle* const* chains, int nchains, const double* const* prior_host, int64_t nprior, int64_t rows,
                          const int64_t* a_ptr, const int32_t* a_mem, const int64_t* b_ptr, const int32_t* b_mem, int npct,
                          const int32_t* pct_idx, double* mean, double* sd, double* prob_a, double* pct) {
  if (!chains || nchains < 1 || nchains > MMQ_CHAINS_MAX || nprior < 0 || rows < 0 || npct < 0 || (npct > 0 && !pct_idx) ||
      (nprior > 0 && !prior_host) || (rows > 0 && (!a_ptr || !a_mem || !b_ptr || !b_mem)))
    return mmq_fail(chains ? chains[0] : nullptr, MMQ_ERR_ARG, "mmq_allelic_summaries: bad arguments");
  if (const int rc = chain_handles_check(chains, nchains, "mmq_allelic_summaries", 4)) return rc;
  mmq_handle* h0 = chains[0];
  const int L = h0->trace_len;
  const int64_t n = h0->n;
  auto fail = [&](const char* what) { return mmq_fail(h0, MMQ_ERR_ARG, std::string("mmq_allelic_summaries: ") + what); };
  for (int c = 0; c < nchains; ++c)
    if (nprior > 0 && !prior_host[c]) return fail("NULL prior draws");
  for (int j = 0; j < npct; ++j)
    if (pct_idx[j] < 0 || pct_idx[j] >= nchains * L) return fail("percentile index out of range");
  if (n + nprior > INT32_MAX) return fail("too many rows");
  if (rows == 0) return MMQ_OK;
  if (a_ptr[0] != 0 || b_ptr[0] != 0) return fail("a unit CSR must start at 0");
  for (int64_t r = 0; r < rows; ++r)
    if (a_ptr[r + 1] < a_ptr[r] || b_ptr[r + 1] < b_ptr[r]) return fail("a unit CSR must not decrease");
  const int64_t na = a_ptr[rows], nb = b_ptr[rows];
  for (int64_t q = 0; q < na; ++q)
    if (a_mem[q] < 0 || a_mem[q] >= n + nprior) return fail("member id out of range");
  for (int64_t q = 0; q < nb; ++q)
    if (b_mem[q] < 0 || b_mem[q] >= n + nprior) return fail("member id out of range");
  /* every chain's draws complete on its own device */
  for (int c = 0; c < nchains; ++c) {
    MMQ_CUDA(h0, cudaSetDevice(chains[c]->device));
    MMQ_CUDA(h0, cudaStreamSynchronize(chains[c]->stream));
  }
  MMQ_CUDA(h0, cudaSetDevice(h0->device));
  double *ws = nullptr, *prior = nullptr, *out = nullptr, *d_pct = nullptr;
  int64_t *d_aptr = nullptr, *d_bptr = nullptr;
  int32_t *d_amem = nullptr, *d_bmem = nullptr, *d_idx = nullptr;
  const double *t[MMQ_CHAINS_MAX] = {}, *src[MMQ_CHAINS_MAX] = {}, *pri[MMQ_CHAINS_MAX] = {};
  for (int c = 0; c < nchains; ++c) t[c] = chains[c]->trace;
  const size_t pbytes = sizeof(double) * (size_t)nprior * (size_t)L;
  cudaError_t e = cudaSuccess;
  auto A = [&](auto** p, size_t b) { if (e == cudaSuccess) e = mmq_cache_malloc(p, std::max<size_t>(b, 8)); };
  auto H2D = [&](void* dst, const void* from, size_t b) {
    if (e == cudaSuccess && b) e = cudaMemcpyAsync(dst, from, b, cudaMemcpyHostToDevice, h0->stream);
  };
  A(&prior, pbytes * (size_t)nchains);
  A(&out, sizeof(double) * 3 * (size_t)rows);
  A(&d_aptr, sizeof(int64_t) * (size_t)(rows + 1)); A(&d_bptr, sizeof(int64_t) * (size_t)(rows + 1));
  A(&d_amem, sizeof(int32_t) * (size_t)na); A(&d_bmem, sizeof(int32_t) * (size_t)nb);
  if (npct > 0) { A(&d_pct, sizeof(double) * (size_t)rows * (size_t)npct); A(&d_idx, sizeof(int32_t) * (size_t)npct); }
  for (int c = 0; c < nchains && nprior > 0; ++c) {
    pri[c] = prior + (size_t)c * (size_t)nprior * (size_t)L;
    H2D(prior + (size_t)c * (size_t)nprior * (size_t)L, prior_host[c], pbytes);
  }
  H2D(d_aptr, a_ptr, sizeof(int64_t) * (size_t)(rows + 1)); H2D(d_bptr, b_ptr, sizeof(int64_t) * (size_t)(rows + 1));
  H2D(d_amem, a_mem, sizeof(int32_t) * (size_t)na); H2D(d_bmem, b_mem, sizeof(int32_t) * (size_t)nb);
  if (npct > 0) H2D(d_idx, pct_idx, sizeof(int32_t) * (size_t)npct);
  if (e == cudaSuccess) e = chain_gather(chains, nchains, t, n, L, &ws, src);
  int ret = MMQ_OK;
  if (e == cudaSuccess) {
    ret = mmq_allelic_summaries_dev(src, pri, nchains, n, nprior, rows, L, d_aptr, d_amem, d_bptr, d_bmem, npct, d_idx, out, d_pct, h0->stream);
    if (ret) ret = mmq_fail(h0, ret, mmq_last_error(nullptr));
  }
  auto D = [&](void* dst, const void* from, size_t b) {
    if (e == cudaSuccess && ret == MMQ_OK && dst && b) e = cudaMemcpyAsync(dst, from, b, cudaMemcpyDeviceToHost, h0->stream);
  };
  D(mean, out, sizeof(double) * (size_t)rows);
  D(sd, out + rows, sizeof(double) * (size_t)rows);
  D(prob_a, out + 2 * rows, sizeof(double) * (size_t)rows);
  if (npct > 0) D(pct, d_pct, sizeof(double) * (size_t)rows * (size_t)npct);
  const cudaError_t es = cudaStreamSynchronize(h0->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h0, e, "mmq_allelic_summaries", __FILE__, __LINE__);
  mmq_cache_free(ws); mmq_cache_free(prior); mmq_cache_free(out); mmq_cache_free(d_pct); mmq_cache_free(d_idx);
  mmq_cache_free(d_aptr); mmq_cache_free(d_bptr); mmq_cache_free(d_amem); mmq_cache_free(d_bmem);
  return ret;
}

int mmq_pair_shared_counts(mmq_handle* h, const int32_t* gene_of, const int32_t* local_of, const int64_t* pair_base, int64_t ngenes,
                           int64_t npairs, int64_t* out) {
  if (!h || !gene_of || !local_of || (!out && npairs > 0) || ngenes < 0 || npairs < 0 || (ngenes > 0 && !pair_base) || (ngenes == 0 && npairs > 0))
    return mmq_fail(h, MMQ_ERR_ARG, "mmq_pair_shared_counts: bad arguments");
  auto fail = [&](const char* what) { return mmq_fail(h, MMQ_ERR_ARG, std::string("mmq_pair_shared_counts: ") + what); };
  if (ngenes > 0 && pair_base[0] != 0) return fail("pair_base must start at 0");
  std::vector<int64_t> kof((size_t)ngenes);
  for (int64_t g = 0; g < ngenes; ++g) {
    const int64_t end = g + 1 < ngenes ? pair_base[g + 1] : npairs, d = end - pair_base[g];
    if (d < 0) return fail("pair_base must not decrease or exceed npairs");
    int64_t k = (int64_t)((1.0 + std::sqrt(1.0 + 8.0 * (double)d)) / 2.0);
    while (k * (k - 1) / 2 > d) --k;
    while (k * (k - 1) / 2 < d) ++k;
    if (k * (k - 1) / 2 != d) return fail("a gene's pair count is not k (k - 1) / 2");
    kof[(size_t)g] = d == 0 ? 0 : k;
  }
  std::vector<int64_t> rowbase((size_t)std::max<int64_t>(h->n, 1));
  for (int64_t t = 0; t < h->n; ++t) {
    const int32_t g = gene_of[t];
    if (g < -1 || g >= ngenes) return fail("gene index out of range");
    if (g < 0) continue;
    const int64_t a = local_of[t], k = kof[(size_t)g];
    if (a < 0 || a >= k) return fail("local index out of range");
    rowbase[(size_t)t] = pair_base[g] + a * (2 * k - a - 1) / 2 - a - 1;
  }
  if (npairs == 0) return MMQ_OK;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int32_t *d_gene = nullptr, *d_local = nullptr;
  int64_t* d_base = nullptr;
  unsigned long long* d_out = nullptr;
  const size_t nb = (size_t)std::max<int64_t>(h->n, 1);
  cudaError_t e = mmq_cache_malloc(&d_gene, sizeof(int32_t) * nb);
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_local, sizeof(int32_t) * nb);
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_base, sizeof(int64_t) * nb);
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_out, sizeof(int64_t) * (size_t)npairs);
  if (e == cudaSuccess && h->n > 0) e = cudaMemcpyAsync(d_gene, gene_of, sizeof(int32_t) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess && h->n > 0) e = cudaMemcpyAsync(d_local, local_of, sizeof(int32_t) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess && h->n > 0) e = cudaMemcpyAsync(d_base, rowbase.data(), sizeof(int64_t) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)npairs, h->stream);
  int ret = MMQ_OK;
  if (e == cudaSuccess && h->m > 0) {
    const int grid = mmq_grid_for(h->m, 256, h->num_sms * 8);
    if (h->has_k) k_pair_shared<true><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_gene, d_local, d_base, h->m, d_out);
    else k_pair_shared<false><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, d_gene, d_local, d_base, h->m, d_out);
    g_mmq_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) ret = mmq_allreduce(h, d_out, (size_t)npairs, 2);
  if (e == cudaSuccess && ret == MMQ_OK) e = cudaMemcpyAsync(out, d_out, sizeof(int64_t) * (size_t)npairs, cudaMemcpyDeviceToHost, h->stream);
  const cudaError_t es = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h, e, "mmq_pair_shared_counts", __FILE__, __LINE__);
  mmq_cache_free(d_gene); mmq_cache_free(d_local); mmq_cache_free(d_base); mmq_cache_free(d_out);
  return ret;
}

int64_t mmq_isocorr_workspace_bytes(int64_t ngenes, int64_t nmembers) {
  if (ngenes < 0 || nmembers < 0) return 0;
  return (int64_t)sizeof(double) * 5 * nmembers + (int64_t)sizeof(int64_t) * (ngenes + 1);
}

int mmq_isocorr_summaries_dev(const double* const* chain_dev, int nchains, int64_t ngenes, int64_t nmembers, int L,
                              const int64_t* gene_ptr_dev, const int32_t* members_dev, const int64_t* pair_base_dev, int64_t npairs,
                              double* out_dev, void* workspace_dev, void* cuda_stream) {
  if (!chain_dev || !tpm_len_ok(nchains, L) || ngenes < 0 || nmembers < 0 || npairs < 0 ||
      (npairs > 0 && (!gene_ptr_dev || !members_dev || !pair_base_dev || !out_dev || !workspace_dev)))
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_isocorr_summaries_dev: bad arguments");
  mmq_chain_ptrs cp = {};
  for (int c = 0; c < nchains; ++c) {
    if (!chain_dev[c]) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_isocorr_summaries_dev: NULL chain");
    cp.p[c] = chain_dev[c];
  }
  if (npairs == 0) return MMQ_OK;
  int dev = 0, sms = 0, lgL = 0;
  while ((1 << lgL) < L) ++lgL;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_isocorr, cudaFuncAttributeMaxDynamicSharedMemorySize, MMQ_ISO_SMEM);
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "mmq_isocorr_summaries_dev", __FILE__, __LINE__);
  const cudaStream_t st = (cudaStream_t)cuda_stream;
  double* stats = static_cast<double*>(workspace_dev);
  int64_t* items = reinterpret_cast<int64_t*>(stats + 5 * nmembers);
  if (nmembers > 0) {
    k_isocorr_prep<<<mmq_grid_for(nmembers, MMQ_POST_THREADS / 32, 8 * sms), MMQ_POST_THREADS, 0, st>>>(cp, nchains, lgL, members_dev, nmembers, stats);
    g_mmq_launches.fetch_add(1);
  }
  k_isocorr_items<<<1, MMQ_ISO_SCAN, 0, st>>>(gene_ptr_dev, ngenes, items);
  g_mmq_launches.fetch_add(1);
  const int grid = (int)std::min<int64_t>(npairs, 2 * (int64_t)sms); /* npairs >= work items */
  k_isocorr<<<grid, MMQ_POST_THREADS, MMQ_ISO_SMEM, st>>>(cp, nchains, lgL, ngenes, gene_ptr_dev, members_dev, pair_base_dev, npairs, stats,
                                                          items, out_dev);
  g_mmq_launches.fetch_add(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return mmq_cuda_fail(nullptr, e, "k_isocorr", __FILE__, __LINE__);
  return MMQ_OK;
}

int mmq_isocorr_summaries(mmq_handle* const* chains, int nchains, int64_t npairs, double* corr_mu, double* corr_log_mu, double* prob_gt) {
  if (!chains || nchains < 1 || nchains > MMQ_CHAINS_MAX || npairs < 0)
    return mmq_fail(chains ? chains[0] : nullptr, MMQ_ERR_ARG, "mmq_isocorr_summaries: bad arguments");
  if (const int rc = chain_handles_check(chains, nchains, "mmq_isocorr_summaries", 4)) return rc;
  mmq_handle* h0 = chains[0];
  const int L = h0->trace_len;
  const mmq_group_set& G = h0->groups[MMQ_GROUP_GENE];
  const int64_t ngenes = G.ngroups;
  /* every chain's draws complete on its own device */
  for (int c = 0; c < nchains; ++c) {
    MMQ_CUDA(h0, cudaSetDevice(chains[c]->device));
    MMQ_CUDA(h0, cudaStreamSynchronize(chains[c]->stream));
  }
  MMQ_CUDA(h0, cudaSetDevice(h0->device));
  /* pair_base from the gene CSR */
  std::vector<int64_t> gptr((size_t)ngenes + 1, 0), pb((size_t)std::max<int64_t>(ngenes, 1), 0);
  if (ngenes > 0) {
    MMQ_CUDA(h0, cudaMemcpyAsync(gptr.data(), G.ptr_dev, sizeof(int64_t) * (size_t)(ngenes + 1), cudaMemcpyDeviceToHost, h0->stream));
    MMQ_CUDA(h0, cudaStreamSynchronize(h0->stream));
  }
  int64_t total = 0;
  for (int64_t g = 0; g < ngenes; ++g) {
    const int64_t k = gptr[(size_t)g + 1] - gptr[(size_t)g];
    pb[(size_t)g] = total;
    total += k * (k - 1) / 2;
  }
  if (total != npairs)
    return mmq_fail(h0, MMQ_ERR_ARG, "mmq_isocorr_summaries: npairs is " + std::to_string(npairs) + ", the gene groups have " +
                                         std::to_string(total) + " pairs");
  if (npairs == 0) return MMQ_OK;
  const int64_t n = h0->n, nmem = gptr[(size_t)ngenes];
  double *ws = nullptr, *work = nullptr, *out = nullptr;
  int64_t* d_pb = nullptr;
  const double *t[MMQ_CHAINS_MAX] = {}, *src[MMQ_CHAINS_MAX] = {};
  for (int c = 0; c < nchains; ++c) t[c] = chains[c]->trace;
  cudaError_t e = mmq_cache_malloc(&work, (size_t)mmq_isocorr_workspace_bytes(ngenes, nmem));
  if (e == cudaSuccess) e = mmq_cache_malloc(&out, sizeof(double) * 3 * (size_t)npairs);
  if (e == cudaSuccess) e = mmq_cache_malloc(&d_pb, sizeof(int64_t) * (size_t)ngenes);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_pb, pb.data(), sizeof(int64_t) * (size_t)ngenes, cudaMemcpyHostToDevice, h0->stream);
  if (e == cudaSuccess) e = chain_gather(chains, nchains, t, n, L, &ws, src);
  int ret = MMQ_OK;
  if (e == cudaSuccess) {
    ret = mmq_isocorr_summaries_dev(src, nchains, ngenes, nmem, L, G.ptr_dev, G.members_dev, d_pb, npairs, out, work, h0->stream);
    if (ret) ret = mmq_fail(h0, ret, mmq_last_error(nullptr));
  }
  double* dst[3] = {corr_mu, corr_log_mu, prob_gt};
  for (int q = 0; q < 3 && e == cudaSuccess && ret == MMQ_OK; ++q)
    if (dst[q]) e = cudaMemcpyAsync(dst[q], out + (size_t)q * (size_t)npairs, sizeof(double) * (size_t)npairs, cudaMemcpyDeviceToHost, h0->stream);
  const cudaError_t es = cudaStreamSynchronize(h0->stream);
  if (e == cudaSuccess) e = es;
  if (e != cudaSuccess && ret == MMQ_OK) ret = mmq_cuda_fail(h0, e, "mmq_isocorr_summaries", __FILE__, __LINE__);
  mmq_cache_free(ws); mmq_cache_free(work); mmq_cache_free(out); mmq_cache_free(d_pb);
  return ret;
}

/* exported under the name of include/mmq_sampler.h's inline function, which this file sees (so mmq.h does not declare it here) */
extern "C" uint32_t mmq_chain_seed_export(uint32_t seed, int chain) __asm__("mmq_chain_seed");
uint32_t mmq_chain_seed_export(uint32_t seed, int chain) { return mmq_chain_seed(seed, chain); }

} /* extern "C" */
