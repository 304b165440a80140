/* mmq_sampler.h — counter-based RNG and exact samplers shared by the sm_100a
 * kernels (mmseq_b200/csrc) and by the CPU replay in oracle/.
 *
 * Everything in this header is built only from IEEE-754 binary64 add, sub,
 * mul, div, sqrt, floor and integer/bit operations, so that the SAME source
 * compiled by nvcc (-fmad=false) and by gcc (-ffp-contract=off) produces
 * bit-identical results for the same (seed, sweep, id) Philox counter.  No
 * libm transcendental is used: mmq_log / mmq_exp are fdlibm-style polynomial
 * kernels written out here.  That is what makes north_star's correctness
 * part (a) — allocations and counts bit-exact against a CPU replay — possible.
 *
 * What is sampled, and which reference call each sampler stands in for
 * (paths relative to /root/reference):
 *   mmq_alloc_row    Multinomial(k_i; mu_j/sum mu) for one hit class
 *                    src/mmseq.cpp:871-889 (gsl_ran_multinomial at :880:
 *                    a chain of conditional binomials with running
 *                    norm - sum_p, zero-probability categories skipped)
 *   mmq_gamma        Gamma(shape, scale 1/rate), Marsaglia-Tsang
 *                    src/mmseq.cpp:907 and :974 (gsl_ran_gamma)
 *   mmq_ndtri        inverse standard normal CDF, Wichura AS241 PPND16
 *                    src/mmseq.cpp:1250, :1286 (gsl_cdf_ugaussian_Pinv)
 * The DISTRIBUTIONS are those of the reference; the bit streams are not
 * GSL's MT19937 streams (those depend on the OpenMP thread count in the
 * reference, src/mmseq.cpp:834-838, so no fixed stream exists to match).
 */
#ifndef MMQ_SAMPLER_H
#define MMQ_SAMPLER_H

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define MMQ_HD __host__ __device__ __forceinline__
#else
#define MMQ_HD static inline
#endif

/* Philox key word 1: which of the path's independent streams a counter is on. */
#define MMQ_STREAM_ALLOC 0x414c4c4fu /* per hit class, per sweep   */
#define MMQ_STREAM_GAMMA 0x47414d4du /* per transcript, per sweep  */
#define MMQ_STREAM_PRIOR 0x5052494fu /* per unobserved transcript, per trace slot */
/* A class with d members and k fragments: k categorical draws (four 32-bit uniforms per Philox block), O(k d), up to
 * mmq_cat_limit(d) fragments; above that gsl_ran_multinomial's chain of d - 1 conditional binomials, O(d).  The limit
 * grows with d because a chain is serial in the members (a binomial costs about as much as 32 categorical draws):
 * 32 (d - 1), at least 32 and at most MMQ_CAT_KMAX.  Round 1 drew up to 8192 categoricals whatever d: 54 % of a sweep's
 * draws on the config-2 sample belonged to classes above 64. */
#define MMQ_CAT_KMAX 512
#define MMQ_CAT_GROUP 64 /* categorical draws are generated in groups of at most 64 (16 blocks): one slot of the class-plan kernel */
#define MMQ_STREAM_CAT 0x43415431u   /* k == 1 classes: one block per QUAD of classes (one 32-bit word each) */

MMQ_HD int64_t mmq_cat_limit(int d) {
  const int64_t v = 32 * (int64_t)(d - 1);
  return v < 32 ? 32 : v > MMQ_CAT_KMAX ? MMQ_CAT_KMAX : v;
}

/* ------------------------------------------------------------------ bits */

/* Fused multiply-add, spelled out: the sources are compiled with contraction OFF (nvcc -fmad=false, gcc
 * -ffp-contract=off) so that a * b + c rounds twice on both sides; where one rounding is wanted (polynomial
 * evaluation: half the instructions and half the dependent latency on the GPU) it is asked for explicitly.  IEEE fma
 * is correctly rounded everywhere (DFMA on the device; the FMA unit, or glibc's exact software fma, on the host). */
MMQ_HD double mmq_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  return __builtin_fma(a, b, c);
#endif
}

MMQ_HD uint64_t mmq_d2u(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t u;
  memcpy(&u, &x, 8);
  return u;
#endif
}

MMQ_HD double mmq_u2d(uint64_t u) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)u);
#else
  double x;
  memcpy(&x, &u, 8);
  return x;
#endif
}

MMQ_HD uint32_t mmq_mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

/* ---------------------------------------------------------------- Philox */

/* Philox4x32-10 (Salmon et al., SC'11).  ctr and key are updated in place:
 * on return ctr[0..3] holds the 128 output bits. */
MMQ_HD void mmq_philox4x32_10(uint32_t ctr[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mmq_mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mmq_mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  ctr[0] = c0; ctr[1] = c1; ctr[2] = c2; ctr[3] = c3;
}

/* Seed of chain `chain` (0 <= chain < MMQ_CHAINS_MAX) of a run with several independent Gibbs chains (mmseq -chains):
 * chain 0 is `seed` itself, so a single chain is the chain of the run without chains.  Chain c >= 1 takes word 0 of
 * Philox4x32-10 at counter (c, j, 0, 0) under key (seed, MMQ_STREAM_CHAIN), for the first j = 0, 1, ... whose value
 * differs from the seeds of chains 0 .. c-1: the seeds of one run are distinct.  A chain outside the range gets `seed`. */
#define MMQ_STREAM_CHAIN 0x4348414eu /* "CHAN" */
#define MMQ_CHAINS_MAX 8
MMQ_HD uint32_t mmq_chain_seed(uint32_t seed, int chain) {
  if (chain <= 0 || chain >= MMQ_CHAINS_MAX) return seed;
  uint32_t s[MMQ_CHAINS_MAX];
  s[0] = seed;
  for (int c = 1; c <= chain; ++c)
    for (uint32_t j = 0;; ++j) {
      uint32_t w[4] = {(uint32_t)c, j, 0u, 0u};
      mmq_philox4x32_10(w, seed, MMQ_STREAM_CHAIN);
      int dup = 0;
      for (int d = 0; d < c; ++d) dup |= w[0] == s[d];
      if (!dup) { s[c] = w[0]; break; }
    }
  return s[chain];
}

/* A stream = (seed, stream tag) key and (id_lo, id_hi, sweep, block) counter.
 * Each block yields two 52-bit uniforms; `block` counts upwards from 0, so a
 * draw is a pure function of (seed, stream, id, sweep, how many uniforms the
 * same (id, sweep) consumed before it). */
typedef struct {
  uint32_t seed, stream;
  uint32_t id_lo, id_hi, sweep, block;
  uint32_t w[4];
  int left; /* uniforms left in w: 0, 1 or 2 */
} mmq_rng;

MMQ_HD void mmq_rng_init(mmq_rng* g, uint32_t seed, uint32_t stream, uint64_t id, uint32_t sweep) {
  g->seed = seed; g->stream = stream;
  g->id_lo = (uint32_t)id; g->id_hi = (uint32_t)(id >> 32);
  g->sweep = sweep; g->block = 0; g->left = 0;
  g->w[0] = g->w[1] = g->w[2] = g->w[3] = 0;
}

/* Uniform on the open interval (0,1): (j + 1/2) * 2^-52, j a 52-bit integer.
 * Never 0 and never 1, exactly representable, identical on host and device. */
MMQ_HD double mmq_uniform(mmq_rng* g) {
  if (g->left == 0) {
    g->w[0] = g->id_lo; g->w[1] = g->id_hi; g->w[2] = g->sweep; g->w[3] = g->block;
    mmq_philox4x32_10(g->w, g->seed, g->stream);
    g->block += 1;
    g->left = 2;
  }
  uint32_t hi, lo;
  if (g->left == 2) { hi = g->w[0]; lo = g->w[1]; } else { hi = g->w[2]; lo = g->w[3]; }
  g->left -= 1;
  uint64_t j = (((uint64_t)hi << 32) | (uint64_t)lo) >> 12;
  return ((double)j + 0.5) * 2.220446049250313080847263336181640625e-16; /* 2^-52 */
}

/* Uniform on (0,1) from ONE 32-bit word: (w + 1/2) * 2^-32.  Used by the k == 1 categorical
 * draw only: 2^-32 is the granularity of gsl_rng_uniform on mt19937, i.e. of every draw the
 * reference's gsl_ran_multinomial makes (src/mmseq.cpp:872), and it lets one Philox block serve
 * four classes.  All three steps are exact, so host and device agree bit for bit. */
MMQ_HD double mmq_uniform32(uint32_t w) {
#if defined(__CUDA_ARCH__)
  /* the same number without a conversion instruction and with one addition: (1 + w 2^-32) - (1 - 2^-33)
   * = (2w + 1) 2^-33 has 33 significant bits, so the subtraction is exact */
  return __hiloint2double((int)(0x3ff00000u | (w >> 12)), (int)(w << 20)) - 0.99999999988358467817306518554688;
#else
  return ((double)w + 0.5) * 2.3283064365386962890625e-10; /* 2^-32 */
#endif
}

/* ------------------------------------------------------- log / exp kernels */

/* Natural logarithm, fdlibm e_log.c scheme: x = 2^k (1+f), sqrt(1/2) < 1+f <
 * sqrt(2); s = f/(2+f); log(1+f) = f - hfsq + s (hfsq + R(s^2)).  < 1 ulp.
 * Domain here: x > 0 finite (callers never pass 0, negatives or NaN, but the
 * edge values are still mapped the IEEE way). */
MMQ_HD double mmq_log(double x) {
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01,
               Lg3 = 2.857142874366239149e-01, Lg4 = 2.222219843214978396e-01,
               Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
               Lg7 = 1.479819860511658591e-01;
  uint64_t u = mmq_d2u(x);
  int k = 0;
  if (x != x) return x;
  if ((u >> 63) != 0 && x != 0.0) return mmq_u2d(0x7ff8000000000000ull); /* log(<0) = nan */
  if (x == 0.0) return mmq_u2d(0xfff0000000000000ull);                    /* -inf */
  if ((u >> 52) == 0x7ffull) return x;                                    /* +inf */
  if ((u >> 52) == 0) { /* subnormal: scale up by 2^54 */
    x = x * 18014398509481984.0;
    u = mmq_d2u(x);
    k = -54;
  }
  uint32_t hx = (uint32_t)(u >> 32);
  /* normalise so that the mantissa lies in [sqrt(2)/2, sqrt(2)) */
  hx += 0x3ff00000u - 0x3fe6a09eu;
  k += (int)(hx >> 20) - 0x3ff;
  hx = (hx & 0x000fffffu) + 0x3fe6a09eu;
  u = ((uint64_t)hx << 32) | (u & 0xffffffffull);
  double f = mmq_u2d(u) - 1.0;
  double hfsq = 0.5 * f * f;
  double s = f / (2.0 + f);
  double z = s * s;
  double w = z * z;
  double t1 = w * mmq_fma(w, mmq_fma(w, Lg6, Lg4), Lg2);
  double t2 = z * mmq_fma(w, mmq_fma(w, mmq_fma(w, Lg7, Lg5), Lg3), Lg1);
  double R = t2 + t1;
  double dk = (double)k;
  return mmq_fma(dk, ln2_hi, mmq_fma(s, hfsq + R, dk * ln2_lo) - hfsq + f);
}

/* log(1+x) for |x| < 1 through log(): log(u) * x / (u - 1), u = 1 + x
 * (the rounding error of u cancels between log(u) and u - 1). */
MMQ_HD double mmq_log1p(double x) {
  double u = 1.0 + x;
  if (u == 1.0) return x;
  return mmq_log(u) * x / (u - 1.0);
}

/* 2^k as a double for -1022 <= k <= 1023 */
MMQ_HD double mmq_pow2i(int k) { return mmq_u2d((uint64_t)(k + 1023) << 52); }

/* exp(x), fdlibm e_exp.c scheme: x = k ln2 + r, |r| <= ln2/2;
 * exp(r) = 1 + r + r c/(2 - c), c = r - r^2 P(r^2).  < 1 ulp. */
MMQ_HD double mmq_exp(double x) {
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  const double invln2 = 1.44269504088896338700e+00;
  const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03,
               P3 = 6.61375632143793436117e-05, P4 = -1.65339022054652515390e-06,
               P5 = 4.13813679705723846039e-08;
  if (x != x) return x;
  if (x > 709.782712893383973096) return mmq_u2d(0x7ff0000000000000ull);
  if (x < -745.13321910194110842) return 0.0;
  double fk = floor(invln2 * x + 0.5);
  int k = (int)fk;
  double hi = x - fk * ln2_hi;
  double lo = fk * ln2_lo;
  double r = hi - lo;
  double t = r * r;
  double c = r - t * mmq_fma(t, mmq_fma(t, mmq_fma(t, mmq_fma(t, P5, P4), P3), P2), P1);
  double y = 1.0 - ((lo - (r * c) / (2.0 - c)) - hi);
  if (k >= -1021 && k <= 1023) return y * mmq_pow2i(k);
  if (k > 1023) return y * mmq_pow2i(1023) * mmq_pow2i(k - 1023);
  return y * mmq_pow2i(k + 1000) * mmq_pow2i(-1000); /* gradual underflow */
}

/* ------------------------------------------------------------- normal */

/* Inverse of the standard normal CDF, Wichura's AS241 PPND16 (relative
 * accuracy about 1e-16).  GSL's gsl_cdf_ugaussian_Pinv (cdf/gaussinv.c) is an
 * implementation of the same algorithm; the reference calls it at
 * src/mmseq.cpp:1250 and :1286. */
MMQ_HD double mmq_ndtri(double p) {
  double q = p - 0.5, r, val;
  if (q >= -0.425 && q <= 0.425) {
    r = 0.180625 - q * q;
    val = q * (((((((2.5090809287301226727e+3 * r + 3.3430575583588128105e+4) * r +
                    6.7265770927008700853e+4) * r + 4.5921953931549871457e+4) * r +
                  1.3731693765509461125e+4) * r + 1.9715909503065514427e+3) * r +
                1.3314166789178437745e+2) * r + 3.3871328727963666080e0) /
          (((((((5.2264952788528545610e+3 * r + 2.8729085735721942674e+4) * r +
                3.9307895800092710610e+4) * r + 2.1213794301586595867e+4) * r +
              5.3941960214247511077e+3) * r + 6.8718700749205790830e+2) * r +
            4.2313330701600911252e+1) * r + 1.0);
    return val;
  }
  r = (q < 0.0) ? p : 1.0 - p;
  if (r <= 0.0) return (q < 0.0) ? mmq_u2d(0xfff0000000000000ull) : mmq_u2d(0x7ff0000000000000ull);
  r = sqrt(-mmq_log(r));
  if (r <= 5.0) {
    r -= 1.6;
    val = (((((((7.74545014278341407640e-4 * r + 2.27238449892691845833e-2) * r +
                2.41780725177450611770e-1) * r + 1.27045825245236838258e0) * r +
              3.64784832476320460504e0) * r + 5.76949722146069140550e0) * r +
            4.63033784615654529590e0) * r + 1.42343711074968357734e0) /
          (((((((1.05075007164441684324e-9 * r + 5.47593808499534494600e-4) * r +
                1.51986665636164571966e-2) * r + 1.48103976427480074590e-1) * r +
              6.89767334985100004550e-1) * r + 1.67638483018380384940e0) * r +
            2.05319162663775882187e0) * r + 1.0);
  } else {
    r -= 5.0;
    val = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r +
                1.24266094738807843860e-3) * r + 2.65321895265761230930e-2) * r +
              2.96560571828504891230e-1) * r + 1.78482653991729133580e0) * r +
            5.46378491116411436990e0) * r + 6.65790464350110377720e0) /
          (((((((2.04426310338993978564e-15 * r + 1.42151175831644588870e-7) * r +
                1.84631831751005468180e-5) * r + 7.86869131145613259100e-4) * r +
              1.48753612908506148525e-2) * r + 1.36929880922735805310e-1) * r +
            5.99832206555887937690e-1) * r + 1.0);
  }
  return (q < 0.0) ? -val : val;
}

/* ---------------------------------------------------- attempt-indexed blocks */

/* Every rejection sampler below numbers its attempts and takes the random numbers of attempt r from ONE Philox
 * block whose index is a function of r alone (not of how many numbers earlier attempts consumed).  An attempt is
 * then a pure function of (seed, stream, id, sweep, block): a kernel may run the attempts of many draws in any
 * order, re-queue the rejected ones and process them densely (mmq_cls.cu: k_alloc_chain, mmq_core.cu: k_gamma)
 * and still produce, bit for bit, what the sequential loops of mmq_gamma / mmq_binomial produce on the CPU. */
MMQ_HD void mmq_rng_block(const mmq_rng* g, uint32_t block, uint32_t w[4]) {
  w[0] = g->id_lo; w[1] = g->id_hi; w[2] = g->sweep; w[3] = block;
  mmq_philox4x32_10(w, g->seed, g->stream);
}
/* 52-bit uniform on (0,1) from two words: (j + 1/2) 2^-52 */
MMQ_HD double mmq_uniform52(uint32_t hi, uint32_t lo) {
  const uint64_t j = (((uint64_t)hi << 32) | (uint64_t)lo) >> 12;
  return ((double)j + 0.5) * 2.220446049250313080847263336181640625e-16; /* 2^-52 */
}

/* ------------------------------------------------------------- normal */

/* cos(2 pi (w + 1/2) / 2^32) from the 32-bit word itself: the top three bits pick the octant, the other 29 the
 * position inside it, mirrored in the odd octants so that the polynomial argument is phi = (q + 1/2) 2^-30 pi/2
 * with an integer q in [0, 2^30): cos(phi) on (0, pi/2) by its Taylor polynomial in phi^2 up to phi^24
 * (truncation error 3e-22), Horner form with explicit fused multiply-adds, no branches: identical on host and device. */
MMQ_HD double mmq_cos2pi_u32(uint32_t w) {
  const uint32_t o = w >> 29, f = w & 0x1fffffffu;
  const uint32_t fm = (o & 1u) ? (0x1fffffffu - f) : f;             /* distance to the nearer octant boundary */
  const uint32_t use_sin = ((o + 1u) >> 1) & 1u, neg = ((o + 2u) >> 2) & 1u;
  const uint32_t q = use_sin ? (0x3fffffffu - fm) : fm;              /* sin(t) = cos(pi/2 - t) */
  const double phi = ((double)q + 0.5) * 1.4629180792671596e-09;     /* 2^-30 pi/2 */
  const double z = phi * phi;
  double c = 1.6117375710961184e-24;                                  /* 1/24! */
  c = mmq_fma(c, z, -8.8967913924505741e-22);                         /* -1/22! */
  c = mmq_fma(c, z, 4.1103176233121648e-19);                          /* 1/20! */
  c = mmq_fma(c, z, -1.5619206968586225e-16);                         /* -1/18! */
  c = mmq_fma(c, z, 4.7794773323873853e-14);                          /* 1/16! */
  c = mmq_fma(c, z, -1.1470745597729725e-11);                         /* -1/14! */
  c = mmq_fma(c, z, 2.08767569878681e-09);                            /* 1/12! */
  c = mmq_fma(c, z, -2.7557319223985888e-07);                         /* -1/10! */
  c = mmq_fma(c, z, 2.48015873015873e-05);                            /* 1/8! */
  c = mmq_fma(c, z, -0.001388888888888889);                           /* -1/6! */
  c = mmq_fma(c, z, 0.041666666666666664);                            /* 1/4! */
  c = mmq_fma(c, z, -0.5);
  c = mmq_fma(c, z, 1.0);
  return neg ? -c : c;
}

/* Standard normal variate, Box-Muller: sqrt(-2 log u) cos(2 pi v) with u a 52-bit uniform (words 0, 1 of a block)
 * and v a 32-bit one (word 2).  Branch-free, unlike an inverse-CDF with separate tail formulas: all lanes of a
 * warp do the same work. */
MMQ_HD double mmq_normal_bm(uint32_t w0, uint32_t w1, uint32_t w2) {
  return sqrt(-2.0 * mmq_log(mmq_uniform52(w0, w1))) * mmq_cos2pi_u32(w2);
}

/* -------------------------------------------------------------- gamma */

/* Gamma(shape a > 0, rate b > 0): Marsaglia & Tsang (2000), with the Gamma(a+1) U^(1/a) boost for a < 1 — the
 * algorithm of gsl_ran_gamma, which the reference calls as gsl_ran_gamma(rg, alpha + Xcolsum[t], 1/(beta+l[t]))
 * at src/mmseq.cpp:907.  Blocks of the draw's stream: 0 = the boost uniform (words 0, 1; only read when a < 1),
 * 1 + r = attempt r (words 0, 1, 2: the normal; word 3: the acceptance uniform, 32 bits like gsl_rng_uniform). */
typedef struct { double d, c; } mmq_gamma_par;
MMQ_HD mmq_gamma_par mmq_gamma_setup(double a_ge_1) {
  mmq_gamma_par q;
  q.d = a_ge_1 - 1.0 / 3.0;
  q.c = (1.0 / 3.0) / sqrt(q.d);
  return q;
}
/* attempt r, first part: 1 accepted (squeeze), 0 rejected (v <= 0), 2 undecided: mmq_gamma_logtest(u, x2, v, d) decides.
 * *v_out = v^3.  The two parts are separate so that a kernel can run the (rare, expensive) log tests of a block densely. */
MMQ_HD int mmq_gamma_try(const mmq_rng* g, uint32_t r, mmq_gamma_par q, double* v_out, double* x2_out, double* u_out) {
  uint32_t w[4];
  mmq_rng_block(g, 1u + r, w);
  const double x = mmq_normal_bm(w[0], w[1], w[2]);
  double v = 1.0 + q.c * x;
  if (v <= 0.0) return 0;
  v = v * v * v;
  const double u = mmq_uniform32(w[3]);
  const double x2 = x * x;
  *v_out = v; *x2_out = x2; *u_out = u;
  return (u < 1.0 - 0.0331 * x2 * x2) ? 1 : 2;
}
MMQ_HD int mmq_gamma_logtest(double u, double x2, double v, double d) {
  return mmq_log(u) < 0.5 * x2 + d * (1.0 - v + mmq_log(v));
}
MMQ_HD int mmq_gamma_attempt(const mmq_rng* g, uint32_t r, mmq_gamma_par q, double* v_out) {
  double x2 = 0.0, u = 0.0;
  const int st = mmq_gamma_try(g, r, q, v_out, &x2, &u);
  return st == 2 ? mmq_gamma_logtest(u, x2, *v_out, q.d) : st;
}
/* U^(1/a) for a < 1 */
MMQ_HD double mmq_gamma_boost(const mmq_rng* g, double a_lt_1) {
  uint32_t w[4];
  mmq_rng_block(g, 0u, w);
  return mmq_exp(mmq_log(mmq_uniform52(w[0], w[1])) / a_lt_1);
}
MMQ_HD double mmq_gamma(const mmq_rng* g, double a, double rate) {
  double boost = 1.0;
  if (a < 1.0) {
    boost = mmq_gamma_boost(g, a);
    a += 1.0;
  }
  const mmq_gamma_par q = mmq_gamma_setup(a);
  double v = 0.0;
  for (uint32_t r = 0; !mmq_gamma_attempt(g, r, q, &v); ++r) { }
  return boost * q.d * v / rate;
}

/* ------------------------------------------------------------ binomial */

/* log(k!) - [ (k+1/2) log(k+1) - (k+1) + log(2 pi)/2 ] */
MMQ_HD double mmq_stirling_tail(double k) {
  if (k <= 9.0) {
    switch ((int)k) {
      case 0: return 0.08106146679532726;
      case 1: return 0.04134069595540929;
      case 2: return 0.02767792568499834;
      case 3: return 0.02079067210376509;
      case 4: return 0.01664469118982119;
      case 5: return 0.01387612882307075;
      case 6: return 0.01189670994589177;
      case 7: return 0.01041126526197209;
      case 8: return 0.009255462182712733;
      default: return 0.008330563433362871;
    }
  }
  double kp1 = k + 1.0;
  double kp1sq = kp1 * kp1;
  return (1.0 / 12.0 - (1.0 / 360.0 - 1.0 / 1260.0 / kp1sq) / kp1sq) / kp1;
}

/* Binomial(n, p) for 0 <= p <= 1/2, n >= 2.
 *   n*p <  10 : sequential inversion (BINV, Kachitvichyanukul & Schmeiser 1988)
 *   n*p >= 10 : transformed rejection BTRS (Hoermann 1993)
 * Both are exact samplers; GSL's gsl_ran_binomial (BTPE + inversion) samples the same distribution.
 * Attempt r of a draw reads block block0 + r of the stream: words 0, 1 = the first 52-bit uniform, words 2, 3 the
 * second (BTRS only). */
#define MMQ_BINV_MEAN 10.0
/* 1/x for x = 1..63, correctly rounded (the compiler folds the divisions): the inversion loop multiplies instead of
 * dividing (a division is ~20 dependent instructions on the GPU) */
#define MMQ_INV_ROW(b) 1.0 / ((b) + 0), 1.0 / ((b) + 1), 1.0 / ((b) + 2), 1.0 / ((b) + 3), 1.0 / ((b) + 4), 1.0 / ((b) + 5), 1.0 / ((b) + 6), 1.0 / ((b) + 7)
#define MMQ_INV_INIT {0.0, 1.0 / 1, 1.0 / 2, 1.0 / 3, 1.0 / 4, 1.0 / 5, 1.0 / 6, 1.0 / 7, MMQ_INV_ROW(8), MMQ_INV_ROW(16), MMQ_INV_ROW(24), \
                      MMQ_INV_ROW(32), MMQ_INV_ROW(40), MMQ_INV_ROW(48), MMQ_INV_ROW(56)}
#if defined(__CUDACC__)
static __constant__ double mmq_inv_dev[64] = MMQ_INV_INIT;
#endif
static const double mmq_inv_host[64] = MMQ_INV_INIT;
MMQ_HD double mmq_inv_small(int64_t x) { /* 1 <= x */
#if defined(__CUDA_ARCH__)
  return x < 64 ? mmq_inv_dev[x] : 1.0 / (double)x;
#else
  return x < 64 ? mmq_inv_host[x] : 1.0 / (double)x;
#endif
}
/* BINV in two parts, like BTRS below: the per-draw constants (one log and one exp among them), then one inversion per
 * attempt.  A kernel that runs the attempts of a draw apart from its setup computes the constants once per draw. */
typedef struct { double q, s, a, r0; } mmq_binv_par;
MMQ_HD mmq_binv_par mmq_binv_setup(int64_t n, double p) {
  mmq_binv_par t;
  const double dn = (double)n;
  t.q = 1.0 - p;
  t.s = p / t.q;
  t.a = (dn + 1.0) * t.s;
  t.r0 = mmq_exp(dn * mmq_log1p(-p));
  return t;
}
/* one inversion from block `block`: returns 1 and *x_out when it ends at x <= n, 0 when it runs past n */
MMQ_HD int mmq_binv_attempt(const mmq_rng* g, uint32_t block, int64_t n, const mmq_binv_par t, int64_t* x_out) {
  uint32_t w[4];
  mmq_rng_block(g, block, w);
  double r = t.r0;
  double u = mmq_uniform52(w[0], w[1]);
  int64_t x = 0;
  while (u > r) {
    u -= r;
    x += 1;
    if (x > n) return 0;
    r *= (t.a * mmq_inv_small(x) - t.s);
  }
  *x_out = x;
  return 1;
}
typedef struct { double dn, b, a, c, vr, r, alpha, m; } mmq_btrs_par;
MMQ_HD mmq_btrs_par mmq_btrs_setup(int64_t n, double p) {
  mmq_btrs_par t;
  t.dn = (double)n;
  const double q = 1.0 - p;
  const double spq = sqrt(t.dn * p * q);
  t.b = 1.15 + 2.53 * spq;
  t.a = -0.0873 + 0.0248 * t.b + 0.01 * p;
  t.c = t.dn * p + 0.5;
  t.vr = 0.92 - 4.2 / t.b;
  t.r = p / q;
  t.alpha = (2.83 + 5.1 / t.b) * spq;
  t.m = floor((t.dn + 1.0) * p);
  return t;
}
/* one BTRS attempt from block `block`: returns 1 and *x_out when accepted */
MMQ_HD int mmq_btrs_attempt(const mmq_rng* g, uint32_t block, const mmq_btrs_par t, int64_t* x_out) {
  uint32_t w[4];
  mmq_rng_block(g, block, w);
  const double u = mmq_uniform52(w[0], w[1]) - 0.5;
  const double v = mmq_uniform52(w[2], w[3]);
  const double us = 0.5 - fabs(u);
  const double kk = floor((2.0 * t.a / us + t.b) * u + t.c);
  if (kk < 0.0 || kk > t.dn) return 0;
  *x_out = (int64_t)kk;
  if (us >= 0.07 && v <= t.vr) return 1;
  const double lv = mmq_log(v * t.alpha / (t.a / (us * us) + t.b));
  const double ub = (t.m + 0.5) * mmq_log((t.m + 1.0) / (t.r * (t.dn - t.m + 1.0))) +
                    (t.dn + 1.0) * mmq_log((t.dn - t.m + 1.0) / (t.dn - kk + 1.0)) +
                    (kk + 0.5) * mmq_log(t.r * (t.dn - kk + 1.0) / (kk + 1.0)) +
                    mmq_stirling_tail(t.m) + mmq_stirling_tail(t.dn - t.m) -
                    mmq_stirling_tail(kk) - mmq_stirling_tail(t.dn - kk);
  return lv <= ub;
}
MMQ_HD int64_t mmq_binomial_half(const mmq_rng* g, uint32_t block0, int64_t n, double p) {
  int64_t x = 0;
  if ((double)n * p < MMQ_BINV_MEAN) {
    const mmq_binv_par t = mmq_binv_setup(n, p);
    for (uint32_t r = 0; !mmq_binv_attempt(g, block0 + r, n, t, &x); ++r) { }
    return x;
  }
  const mmq_btrs_par t = mmq_btrs_setup(n, p);
  for (uint32_t r = 0; !mmq_btrs_attempt(g, block0 + r, t, &x); ++r) { }
  return x;
}

/* Binomial(n, p), any p in [0,1], from the blocks block0, block0 + 1, ... of the stream. */
MMQ_HD int64_t mmq_binomial(const mmq_rng* g, uint32_t block0, int64_t n, double p) {
  if (n <= 0 || !(p > 0.0)) return 0;
  if (p >= 1.0) return n;
  if (n == 1) {
    uint32_t w[4];
    mmq_rng_block(g, block0, w);
    return (mmq_uniform52(w[0], w[1]) < p) ? 1 : 0;
  }
  if (p > 0.5) return n - mmq_binomial_half(g, block0, n, 1.0 - p);
  return mmq_binomial_half(g, block0, n, p);
}

/* ---------------------------------------------------- one hit class */

/* blocks of node h (heap index (1 << level) + position) of a chain class: (h << 8) + attempt */
#define MMQ_CHAIN_BLOCK(j) ((uint32_t)(j) << 8)

/* Multinomial(k; p) for a class with many fragments, as gsl_ran_multinomial (src/mmseq.cpp:880) draws it: by conditional
 * binomials.  GSL walks the members left to right (x_j ~ Bin(rest, p_j / P(j..d-1))): d - 1 binomials that each wait for
 * the one before.  The same distribution is obtained from any binary splitting of the member range, and a BALANCED one
 * has depth ceil(log2 d) instead of d - 1 — what bounds the time of a sweep on the GPU, where the binomials of a level
 * are drawn side by side (mmq_cls.cu: k_alloc_chain).  Node i of level L covers the members [(i d) >> L, ((i+1) d) >> L);
 * its count n splits into Bin(n, left / (left + right)) for the left half and the rest for the right half, the two
 * range sums formed left to right.  Members with zero probability never receive fragments (an all-zero node hands
 * everything to its right half, so an all-zero row ends in its last member).  The binomial of node (L, i) reads the
 * blocks MMQ_CHAIN_BLOCK((1 << L) + i) + attempt of the class's ALLOC stream, so nodes can be drawn in any order.
 * x[j] is assigned exactly once per member. */
#define MMQ_NODE_LO(i, L, d) ((int)(((int64_t)(i) * (int64_t)(d)) >> (L)))
template <typename PIt>
MMQ_HD double mmq_node_prob(PIt p, int lo, int mid, int hi) {
  double left = 0.0, right = 0.0;
  for (int j = lo; j < mid; ++j) left += p[j];
  for (int j = mid; j < hi; ++j) right += p[j];
  const double tot = left + right;
  double pr = tot > 0.0 ? left / tot : 0.0;
  return pr > 1.0 ? 1.0 : pr;
}
template <typename PIt, typename XIt>
MMQ_HD void mmq_alloc_chain(PIt p, XIt x, int d, int64_t k, const mmq_rng* g) {
  int sl[40], si[40];
  int64_t sn[40];
  int top = 0;
  sl[0] = 0; si[0] = 0; sn[0] = k; top = 1;
  while (top > 0) {
    --top;
    const int L = sl[top], i = si[top];
    const int64_t n = sn[top];
    const int lo = MMQ_NODE_LO(i, L, d), hi = MMQ_NODE_LO(i + 1, L, d);
    if (hi <= lo) continue;
    if (hi - lo == 1) { x[lo] = (int32_t)n; continue; }
    const int mid = MMQ_NODE_LO(2 * i + 1, L + 1, d);
    int64_t nl;
    if (mid == lo) nl = 0;
    else if (mid == hi) nl = n;
    else if (n == 0) nl = 0;
    else nl = mmq_binomial(g, MMQ_CHAIN_BLOCK((1u << L) + (uint32_t)i), n, mmq_node_prob(p, lo, mid, hi));
    sl[top] = L + 1; si[top] = 2 * i + 1; sn[top] = n - nl; ++top;
    sl[top] = L + 1; si[top] = 2 * i; sn[top] = nl; ++top;
  }
}

/* How mmq_alloc_row accumulates into its output: plain arrays are zeroed and added to; an output
 * that is itself a reduction (the kernels' counts[] adaptor) overloads these two. */
template <typename XIt>
MMQ_HD void mmq_x_zero(XIt x, int d) {
  for (int j = 0; j < d; ++j) x[j] = 0;
}
template <typename XIt>
MMQ_HD void mmq_x_add(XIt x, int j, int32_t v) {
  x[j] = x[j] + v;
}


/* Allocate the k fragments of one hit class among its d member transcripts.
 *   p[j]  unnormalised probability of member j (mu[col_j], times the per-hit
 *         weight when weights are present); read twice, never written
 *   x[j]  out: number of fragments given to member j; sum_j x[j] == k
 * d == 1 consumes no random numbers (x = k).  k == 1 is one categorical draw
 * (one 32-bit uniform of the CAT stream: chosen = first j with u * sum_p < p_0 + ... + p_j); 2 <= k <= mmq_cat_limit(d) is k
 * such draws from the class's own stream (32-bit uniforms, four per block).  Larger k is gsl_ran_multinomial's chain of conditional
 * binomials x_j ~ Bin(k - sum_{<j} x, p_j / (P - sum_{<j} p)).
 * The arithmetic order (left-to-right sums) is part of the contract: the CPU
 * replay and every kernel variant walk the row in the same order. */
template <typename PIt, typename XIt>
MMQ_HD void mmq_alloc_row(PIt p, XIt x, int d, int64_t k, uint32_t seed, uint64_t class_id,
                          uint32_t sweep) {
  if (d <= 0) return;
  if (d == 1) { x[0] = (int32_t)k; return; }
  double norm = 0.0;
  int last_pos = d - 1; /* last member with p > 0 (d-1 if none) */
  {
    int lp = -1;
    for (int j = 0; j < d; ++j) {
      const double pj = p[j];
      norm += pj;
      if (pj > 0.0) lp = j;
    }
    if (lp >= 0) last_pos = lp;
  }
  mmq_rng g;
  if (k == 1) {
    /* one categorical draw needs one uniform of 32 bits; a Philox block holds four words, so
     * classes 4c .. 4c+3 share block c of the CAT stream (word class_id & 3).  A kernel thread
     * that owns four consecutive classes runs Philox once. */
    uint32_t wd[4] = {(uint32_t)(class_id >> 2), (uint32_t)(class_id >> 34), sweep, 0u};
    mmq_philox4x32_10(wd, seed, MMQ_STREAM_CAT);
    const uint32_t sel = (uint32_t)(class_id & 3);
    const double u = mmq_uniform32(sel == 0 ? wd[0] : sel == 1 ? wd[1] : sel == 2 ? wd[2] : wd[3]);
    const double target = u * norm;
    double acc = 0.0;
    int chosen = -1;
    for (int j = 0; j < d; ++j) {
      acc += p[j];
      x[j] = 0;
      if (chosen < 0 && target < acc) chosen = j;
    }
    if (chosen < 0) chosen = last_pos; /* rounding at the top end, or norm == 0 */
    x[chosen] = 1;
    return;
  }
  mmq_rng_init(&g, seed, MMQ_STREAM_ALLOC, class_id, sweep);
  if (k <= mmq_cat_limit(d)) {
    /* k independent categorical draws — the same Multinomial(k; p) as the binomial chain below,
     * without log/exp and without a serial dependence between members.  Draw t uses word t & 3 of
     * block t >> 2 of the class's own stream as one 32-bit uniform (the granularity of the k == 1
     * draw), so a kernel thread runs Philox once per four fragments and the draws of a large class
     * can be shared out between threads in groups of MMQ_CAT_GROUP (mmq_cls.cu). */
    mmq_x_zero(x, d);
    for (int t0 = 0; t0 < (int)k; t0 += MMQ_CAT_GROUP) {
      const int cnt = ((int)k - t0 < MMQ_CAT_GROUP) ? (int)k - t0 : MMQ_CAT_GROUP;
      int32_t ch[MMQ_CAT_GROUP];
      uint32_t wd[4] = {0u, 0u, 0u, 0u};
      for (int q = 0; q < cnt; ++q) {
        const int t = t0 + q;
        if ((t & 3) == 0) {
          wd[0] = g.id_lo; wd[1] = g.id_hi; wd[2] = sweep; wd[3] = (uint32_t)(t >> 2);
          mmq_philox4x32_10(wd, seed, MMQ_STREAM_ALLOC);
        }
        const int r = t & 3;
        const double target = mmq_uniform32(r == 0 ? wd[0] : r == 1 ? wd[1] : r == 2 ? wd[2] : wd[3]) * norm;
        double acc = 0.0;
        int chosen = -1;
        for (int j = 0; j < d; ++j) {
          acc += p[j];
          if (chosen < 0 && target < acc) chosen = j;
        }
        ch[q] = chosen < 0 ? last_pos : chosen;
      }
      for (int j = 0; j < d; ++j) {
        int32_t v = 0;
        for (int q = 0; q < cnt; ++q) v += (ch[q] == j) ? 1 : 0;
        mmq_x_add(x, j, v);
      }
    }
    return;
  }
  mmq_alloc_chain(p, x, d, k, &g);
}

#endif /* MMQ_SAMPLER_H */
