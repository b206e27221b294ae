// rc_math.h -- deterministic fp64 elementary functions shared by the CUDA kernels and the
// CPU oracle.
//
// Bit-exact replay between the sm_100a kernels and the CPU oracle needs every transcendental
// to be the SAME sequence of IEEE-754 binary64 operations on both sides.  libm / libdevice
// differ by an ulp here and there, so neither side calls them: everything below is built from
// + - * / sqrt and explicit fma(), all of which are correctly rounded on x86-64 and on sm_100a.
// Build rules that make this hold:
//   nvcc : -fmad=false           (no implicit contraction; explicit fma() stays an FMA)
//   g++  : -ffp-contract=off -mfma (ditto; fma() compiles to vfmadd, correctly rounded)
//
// These replace, for the sampler hot path, the third-party functions the reference calls:
//   Base.log / Base.exp / Base.log1p (Julia),  SpecialFunctions.loggamma (openlibm lgamma_r)
//   at /root/reference/src/mcmc.jl:17-20,35,51,73,75,117-121,186-191,223-241,293-297,323-329,
//   348-351,427-430,448-451 and src/utils.jl:5.  Agreement with libm is ~1 ulp
//   (tests/test_oracle_golden.py::test_math_accuracy).
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define RC_HD __host__ __device__ __forceinline__
#else
#define RC_HD static inline
#endif

#define RC_INF (__builtin_huge_val())
#define RC_NAN (__builtin_nan(""))

RC_HD double rc_from_bits(uint64_t u) {
  union { uint64_t u; double d; } c; c.u = u; return c.d;
}
RC_HD uint64_t rc_to_bits(double d) {
  union { uint64_t u; double d; } c; c.d = d; return c.u;
}
RC_HD bool rc_isnan(double x) { return x != x; }

// x * 2^k for |k| <= ~2100, by exact power-of-two multiplies (deterministic everywhere).
RC_HD double rc_scalbn(double x, int k) {
  if (k > 1023) { x *= 0x1p1023; k -= 1023; if (k > 1023) { x *= 0x1p1023; k -= 1023; if (k > 1023) k = 1023; } }
  else if (k < -1022) { x *= 0x1p-969; k += 969; if (k < -1022) { x *= 0x1p-969; k += 969; if (k < -1022) k = -1022; } }
  return x * rc_from_bits((uint64_t)(0x3ff + k) << 52);
}

// Natural logarithm.  x = 2^k m with m in [sqrt(1/2), sqrt(2)) (fdlibm's normalisation, so k = 0 around 1);
// F = round(128 m) / 128, f = m - F (exact), u = f * (1/F) from a table, log x = k ln2 + log F + log1p(u) with
// log1p(u) - u as a degree-7 polynomial (|u| < 0.0056) in Estrin form.  k ln2_hi + head(log F) is exact (both carry
// 21 trailing zero bits), so the result is within ~1 ulp.  No division and a dependent chain of ~14 operations
// (the fdlibm form it replaces had ~45 with a division): this function sits on the sampler's sequential paths.
// Straight-line: the main path is always evaluated (subnormals are pre-scaled by a select) and the special
// cases (NaN, negative, zero, +Inf) override the result at the end, so independent calls interleave.
#include "rc_logtab.h"
static const double rc_logtab_h[][3] = {RC_LOGTAB_ROWS};
#if defined(__CUDACC__)
static __device__ const double rc_logtab_d[][3] = {RC_LOGTAB_ROWS};
#endif
RC_HD double rc_log(double x) {
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  const uint64_t ix0 = rc_to_bits(x);
  const bool sub = ix0 < 0x0010000000000000ULL;          // subnormal (or +0): pre-scale
  const double xs = sub ? x * 0x1p54 : x;
  uint64_t ix = rc_to_bits(xs);
  int k = sub ? -54 : 0;
  // bring mantissa into [sqrt(1/2), sqrt(2))
  uint32_t hx = (uint32_t)(ix >> 32);
  hx += 0x3ff00000 - 0x3fe6a09e;
  k += (int)(hx >> 20) - 0x3ff;
  hx = (hx & 0x000fffff) + 0x3fe6a09e;
  ix = ((uint64_t)hx << 32) | (ix & 0xffffffffULL);
  const double m = rc_from_bits(ix);
  int j = (int)(m * 128.0 + 0.5);
  j = j < RC_LOGTAB_J0 ? RC_LOGTAB_J0 : (j > RC_LOGTAB_J0 + 92 ? RC_LOGTAB_J0 + 92 : j);   // only NaN / Inf patterns leave the range
#if defined(__CUDA_ARCH__)
  const double* T = rc_logtab_d[j - RC_LOGTAB_J0];
#else
  const double* T = rc_logtab_h[j - RC_LOGTAB_J0];
#endif
  const double f = m - (double)j * 0.0078125;            // exact
  const double u = f * T[0];
  const double u2 = u * u;
  const double u4 = u2 * u2;
  const double p01 = -0.5 + u * 3.33333333333333314830e-01;
  const double p23 = -0.25 + u * 2.00000000000000011102e-01;
  const double p45 = -1.66666666666666657415e-01 + u * 1.42857142857142849213e-01;
  const double q = u2 * ((p01 + u2 * p23) + u4 * p45);   // log1p(u) - u
  const double dk = (double)k;
  double res = (dk * ln2_hi + T[1]) + (u + ((dk * ln2_lo + T[2]) + q));
  if (ix0 >= 0x7ff0000000000000ULL) res = x;              // +Inf, and every negative / NaN pattern lands here too
  if ((int64_t)ix0 < 0) res = ((ix0 << 1) == 0) ? -RC_INF : RC_NAN;   // -0 -> -Inf, negative -> NaN
  if (ix0 == 0) res = -RC_INF;
  if (rc_isnan(x)) res = x;
  return res;
}

// log(1+x), Kahan's compensated form on top of rc_log.
RC_HD double rc_log1p(double x) {
  double u = 1.0 + x;
  double d = u - 1.0;
  if (d == 0.0) return x;
  return rc_log(u) * (x / d);
}

// e^x, fdlibm-style: x = k ln2 + r, rational approximation of exp(r).
RC_HD double rc_exp(double x) {
  const double o_threshold = 7.09782712893383973096e+02, u_threshold = -7.45133219101941108420e+02;
  const double ln2hi = 6.93147180369123816490e-01, ln2lo = 1.90821492927058770002e-10,
               invln2 = 1.44269504088896338700e+00;
  const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03,
               P3 = 6.61375632143793436117e-05, P4 = -1.65339022054652515390e-06,
               P5 = 4.13813679705723846039e-08;
  if (rc_isnan(x)) return x;
  if (x > o_threshold) return RC_INF;
  if (x < u_threshold) return 0.0;
  double ax = x < 0 ? -x : x;
  int k = 0;
  double hi = x, lo = 0.0, r = x;
  if (ax > 0.34657359027997264) {                        // |x| > 0.5 ln2
    double kf = invln2 * x + (x < 0 ? -0.5 : 0.5);
    k = (int)kf;                                        // truncation toward zero
    hi = x - (double)k * ln2hi;
    lo = (double)k * ln2lo;
    r = hi - lo;
  } else if (ax < 0x1p-28) {
    return 1.0 + x;
  }
  double xx = r * r;
  double c = r - xx * (P1 + xx * (P2 + xx * (P3 + xx * (P4 + xx * P5))));
  double y = 1.0 + (r * c / (2.0 - c) - lo + hi);
  if (k == 0) return y;
  return rc_scalbn(y, k);
}

// log Gamma(x) for x > 0: recurrence up to x >= 16, then Stirling's series.
// x <= 0 returns +Inf (the sampler only ever evaluates positive arguments; x = 0 is the pole).
RC_HD double rc_lgamma(double x) {
  if (rc_isnan(x)) return x;
  if (x <= 0.0) return RC_INF;
  if (x >= 0x1p1000) return RC_INF;
  double prod = 1.0;
  while (x < 16.0) { prod *= x; x += 1.0; }
  double w = 1.0 / x;
  double w2 = w * w;
  double ser = w * (8.3333333333333333333e-02 - w2 * (2.7777777777777777778e-03 - w2 * (7.9365079365079365079e-04 -
               w2 * (5.9523809523809523810e-04 - w2 * (8.4175084175084175084e-04 - w2 * (1.9175269175269175269e-03 -
               w2 * 6.4102564102564102564e-03))))));
  double st = (x - 0.5) * rc_log(x) - x + 9.1893853320467274178e-01 + ser;
  if (prod != 1.0) st -= rc_log(prod);
  return st;
}

// erfc(x): series for |x| < 3, continued fraction beyond.  ~1e-15 absolute.
RC_HD double rc_erfc(double x) {
  if (rc_isnan(x)) return x;
  double ax = x < 0 ? -x : x;
  double r;
  if (ax < 3.0) {
    // erf(x) = 2/sqrt(pi) e^{-x^2} sum_{n>=0} 2^n x^{2n+1} / (2n+1)!!   (all terms positive)
    double x2 = ax * ax;
    double term = ax, sum = ax;
    for (int n = 1; n < 200; ++n) {
      term = term * (2.0 * x2) / (double)(2 * n + 1);
      sum += term;
      if (term < 1e-17 * sum) break;
    }
    double erfv = 1.1283791670955125739 * rc_exp(-x2) * sum;
    r = 1.0 - erfv;
  } else if (ax > 27.0) {
    r = 0.0;
  } else {
    // erfc(x) = e^{-x^2}/sqrt(pi) * 1/(x + (1/2)/(x + 1/(x + (3/2)/(x + ...))))
    double t = ax;
    for (int k = 60; k >= 1; --k) t = ax + (0.5 * (double)k) / t;
    r = rc_exp(-ax * ax) * 5.6418958354775628695e-01 / t;
  }
  return x < 0 ? 2.0 - r : r;
}

// Standard normal cdf.
RC_HD double rc_normcdf(double z) { return 0.5 * rc_erfc(-z * 7.0710678118654752440e-01); }

// Standard normal quantile for p in (0,1): Acklam's rational approximation + one Halley step.
RC_HD double rc_norminv(double p) {
  const double a1 = -3.969683028665376e+01, a2 = 2.209460984245205e+02, a3 = -2.759285104469687e+02,
               a4 = 1.383577518672690e+02, a5 = -3.066479806614716e+01, a6 = 2.506628277459239e+00;
  const double b1 = -5.447609879822406e+01, b2 = 1.615858368580409e+02, b3 = -1.556989798598866e+02,
               b4 = 6.680131188771972e+01, b5 = -1.328068155288572e+01;
  const double c1 = -7.784894002430293e-03, c2 = -3.223964580411365e-01, c3 = -2.400758277161838e+00,
               c4 = -2.549732539343734e+00, c5 = 4.374664141464968e+00, c6 = 2.938163982698783e+00;
  const double d1 = 7.784695709041462e-03, d2 = 3.224671290700398e-01, d3 = 2.445134137142996e+00,
               d4 = 3.754408661907416e+00;
  const double plow = 0.02425, phigh = 1.0 - 0.02425;
  double x;
  if (p <= 0.0) return -RC_INF;
  if (p >= 1.0) return RC_INF;
  if (p < plow) {
    double q = sqrt(-2.0 * rc_log(p));
    x = (((((c1 * q + c2) * q + c3) * q + c4) * q + c5) * q + c6) / ((((d1 * q + d2) * q + d3) * q + d4) * q + 1.0);
  } else if (p <= phigh) {
    double q = p - 0.5, r = q * q;
    x = (((((a1 * r + a2) * r + a3) * r + a4) * r + a5) * r + a6) * q /
        (((((b1 * r + b2) * r + b3) * r + b4) * r + b5) * r + 1.0);
  } else {
    double q = sqrt(-2.0 * rc_log(1.0 - p));
    x = -(((((c1 * q + c2) * q + c3) * q + c4) * q + c5) * q + c6) / ((((d1 * q + d2) * q + d3) * q + d4) * q + 1.0);
  }
  // Halley refinement against rc_normcdf
  double e = rc_normcdf(x) - p;
  double u = e * 2.5066282746310005024 * rc_exp(0.5 * x * x);
  x = x - u / (1.0 + 0.5 * x * u);
  return x;
}

// Julia `minimum([0, x])` (NaN-propagating), /root/reference/src/mcmc.jl:131,467-468.
RC_HD double rc_min0(double x) {
  if (rc_isnan(x)) return x;
  return x < 0.0 ? x : 0.0;
}

// shape * log(rate) - lgamma(shape): the log normalising constant of the Gamma(shape, rate) priors of the within- and
// between-cluster dissimilarities, abratio = (alpha, beta) and zgratio = (zeta, gamma) at /root/reference/src/mcmc.jl:17-18,186-187,293-294.
RC_HD double rc_gamma_lognorm(double shape, double rate) { return shape * rc_log(rate) - rc_lgamma(shape); }

// ---- Euclidean distance entries -------------------------------------------------------------
// Every distance path computes v = |x_i|^2 + |x_j|^2 - 2 x_i.x_j (the Gram form of Distances.jl's pairwise).  Its
// rounding error is up to ~dim u (|x_i|^2 + |x_j|^2), which swamps v when the two points are close relative to their
// norms (offset data such as geographic coordinates, near-duplicates): the Gram form can then return 0 for two distinct
// points.  An entry with v < tau (|x_i|^2 + |x_j|^2), tau = 2^-6, is recomputed from the differences, as Distances.jl's
// Euclidean(thresh) does; a kept entry then has relative error <= (dim + 2) u / tau, a recomputed one <= (dim / 2 + 2) u.
// s = |x_i|^2 + |x_j|^2 (commutes, so the decision does not depend on the operand order).
RC_HD bool rc_dist_unresolved(double v, double s) { return v < 0x1p-6 * s; }
// sum_t (x_t - y_t)^2 in ascending coordinates; (x_t - y_t)^2 == (y_t - x_t)^2 bitwise, so it is symmetric too.
RC_HD double rc_dist_direct2(const double* x, const double* y, int64_t dim) {
  double a = 0.0;
  for (int64_t t = 0; t < dim; ++t) { const double d = x[t] - y[t]; a += d * d; }
  return a;
}

// ---- fixed-point images of D and log D ------------------------------------------------------
// Row/cluster sums of D and log D are accumulated as exact 64-bit integers of q-bit fixed-point
// images (order-independent => identical on CPU and GPU for any tiling).  Block totals for the
// log-likelihood use 128 bits.
RC_HD int64_t rc_quantize(double v, int q) {
  // round-half-even of v * 2^q; caller guarantees |v| * 2^q < 2^62
  double s = v * rc_from_bits((uint64_t)(0x3ff + q) << 52);
  return (int64_t)rint(s);
}
RC_HD double rc_dequant(int64_t s, int q) {
  return (double)s * rc_from_bits((uint64_t)(0x3ff - q) << 52);
}
// 128-bit two's complement (hi signed, lo unsigned) -> double * 2^-q, same formula on both sides.
RC_HD double rc_dequant128(int64_t hi, uint64_t lo, int q) {
  double d = (double)hi * 0x1p64 + (double)lo;
  return d * rc_from_bits((uint64_t)(0x3ff - q) << 52);
}

// Fixed-point scale: the largest q with n * maxabs * 2^q < 2^61, so that every sum of n image
// entries fits an int64 and its resolution follows the data's scale (host side, both the library
// and the oracle call this so the images are identical).  q is clamped to [-1022, 1022] so that
// 2^q and 2^-q stay normal doubles; the upper clamp binds only for n * maxabs < 2^-961.  All-zero
// data gets 50.  Returns RC_Q_NONE when n * maxabs is not finite.
#define RC_Q_NONE INT32_MIN
#if defined(__CUDACC__)
__host__
#endif
static inline int rc_choose_q(double maxabs, int64_t n) {
  double v = maxabs * (double)n;
  if (v == 0.0) return 50;
  if (!(v > 0.0 && v < RC_INF)) return RC_Q_NONE;
  int e = 0;
  (void)frexp(v, &e);            // v = m * 2^e, m in [0.5, 1)  =>  v < 2^e
  int q = 61 - e;
  return q > 1022 ? 1022 : (q < -1022 ? -1022 : q);
}
