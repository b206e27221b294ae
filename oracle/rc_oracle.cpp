// rc_oracle.cpp -- CPU ORACLE (TEST INFRASTRUCTURE ONLY -- never imported by the product path).
//
// A single-threaded restatement, function by function, of the sampler hot path of
// RedClust.jl v1.2.2 (/root/reference/src/mcmc.jl:1-479,537-555, src/utils.jl:2-6,59-74,
// src/types.jl:131-157).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// --impl reference legs may load the library built from this file.
//
// PARITY STATUS: the reference's own tests hold no golden vectors for the sampler
// (test/test_sampler.jl is no-throw only) and Julia is not installed, so for the sampler this
// oracle is "parity unpinned" against a real RedClust.jl run; it is pinned only by reading
// (every function cites the lines it follows) and by the statistical checks in tests/.
// The distance-matrix restatement IS pinned against the reference fixture
// data/example_datasets.h5 (tests/golden/, tests/test_oracle_golden.py).
//
// Two deliberate, documented departures from the reference's arithmetic (DESIGN.md section 3):
//   (1) elementary functions come from rc_math.h (deterministic, ~1 ulp from Julia's);
//   (2) sum_mode 0 accumulates cluster sums of D / log D as exact integers of fixed-point
//       images (order-independent, so the GPU can match bit-for-bit); sum_mode 1 is the plain
//       ascending-index fp64 summation closest to the reference's matsum (utils.jl:9-17).
//   Random draws come from the structured Philox stream of rc_rng.h at the draw sites the
//   reference has (SURVEY.md A.5).
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include <thread>
#include <chrono>
#include "../include/rcb200.h"
#include "../redclust.jl_b200/csrc/rc_math.h"
#include "../redclust.jl_b200/csrc/rc_rng.h"

typedef __int128 i128;

namespace {

struct Data {
  int64_t n;
  const double* D;            // n x n
  std::vector<double> logD;   // types.jl:155
  std::vector<int64_t> Dq, Lq;
  int qD, qL;
  int sum_mode;
};

struct State {                 // MCMCState, types.jl:131-137 (slots are 1..n, index 0 unused)
  std::vector<int64_t> clusts; // 0-based point index -> slot id in 1..n, or -1 when detached
  double r, p;
  std::vector<int64_t> sizes;  // sizes[slot], slot in 1..n
  int64_t K;
};

void build_data(Data& d, const double* D, int64_t n, int sum_mode) {
  d.n = n; d.D = D; d.sum_mode = sum_mode;
  d.logD.resize((size_t)n * n);
  double maxD = 0, maxL = 0;
  for (int64_t i = 0; i < n; ++i)
    for (int64_t j = 0; j < n; ++j) {
      // log.(D .- Diagonal(D) .+ I): off-diagonal log(D_ij - 0 + 0), diagonal log(D_ii - D_ii + 1)
      double v = (i == j) ? (D[i * n + i] - D[i * n + i] + 1.0) : (D[i * n + j] - 0.0 + 0.0);
      double l = rc_log(v);
      d.logD[i * n + j] = l;
      maxD = std::max(maxD, std::fabs(D[i * n + j]));
      maxL = std::max(maxL, std::fabs(l));
    }
  d.qD = rc_choose_q(maxD, n);
  d.qL = rc_choose_q(maxL, n);
  if (sum_mode == 0) {
    d.Dq.resize((size_t)n * n); d.Lq.resize((size_t)n * n);
    for (size_t t = 0; t < (size_t)n * n; ++t) {
      d.Dq[t] = rc_quantize(D[t], d.qD);
      d.Lq[t] = rc_quantize(d.logD[t], d.qL);
    }
  }
}

// matsum(x, [i], clust_k) for every slot k at once (utils.jl:9-17 with inds1 = [i]):
// sD[k], sL[k] = sum over j with clusts[j] == k of D[i,j], logD[i,j].
void rowsums(const Data& d, const State& s, int64_t i, std::vector<double>& sD, std::vector<double>& sL,
             std::vector<int64_t>& accD, std::vector<int64_t>& accL) {
  const int64_t n = d.n;
  if (d.sum_mode == 0) {
    std::fill(accD.begin(), accD.end(), 0); std::fill(accL.begin(), accL.end(), 0);
    const int64_t* rd = &d.Dq[i * n]; const int64_t* rl = &d.Lq[i * n];
    for (int64_t j = 0; j < n; ++j) { int64_t k = s.clusts[j]; if (k > 0) { accD[k] += rd[j]; accL[k] += rl[j]; } }
    for (int64_t k = 1; k <= n; ++k) { sD[k] = rc_dequant(accD[k], d.qD); sL[k] = rc_dequant(accL[k], d.qL); }
  } else {
    std::fill(sD.begin(), sD.end(), 0.0); std::fill(sL.begin(), sL.end(), 0.0);
    const double* rd = &d.D[i * n]; const double* rl = &d.logD[i * n];
    for (int64_t j = 0; j < n; ++j) { int64_t k = s.clusts[j]; if (k > 0) { sD[k] += rd[j]; sL[k] += rl[j]; } }
  }
}

// vecsum(x, inds) (utils.jl:25-31).  @turbo's reduction order is unspecified; the canonical
// order of this build is: slot s (1-based) lives in lane (s-1)%32, each lane adds its slots in
// ascending order, then an xor-butterfly (16,8,4,2,1) combines the 32 lanes.  Absent slots add 0.0.
double vecsum_canonical(const std::vector<double>& x, const std::vector<int64_t>& inds) {
  double lane[32];
  for (int l = 0; l < 32; ++l) lane[l] = 0.0;
  for (int64_t s : inds) lane[(s - 1) % 32] += x[s];   // inds ascending => per-lane ascending
  for (int off = 16; off >= 1; off >>= 1) {
    double t[32];
    for (int l = 0; l < 32; ++l) t[l] = lane[l] + lane[l ^ off];
    for (int l = 0; l < 32; ++l) lane[l] = t[l];
  }
  return lane[0];
}

// sample_logweights, utils.jl:2-6 (mutates logprobs).  Uniform j comes from address (site, mh, a, j)
// or, for the two-candidate restricted scan, both from one address.
int64_t sample_logweights(std::vector<double>& lp, const std::vector<double>& u) {
  size_t m = lp.size();
  double mn = lp[0];
  for (size_t k = 1; k < m; ++k) { if (rc_isnan(mn)) break; if (rc_isnan(lp[k]) || lp[k] < mn) mn = lp[k]; }
  for (size_t k = 0; k < m; ++k) lp[k] -= mn;
  size_t best = 0; double bv = 0; bool have = false;
  for (size_t k = 0; k < m; ++k) {
    double g = -rc_log(-rc_log(u[k])) + lp[k];
    if (!have) { best = k; bv = g; have = true; if (rc_isnan(g)) break; continue; }
    if (rc_isnan(g)) { best = k; break; }            // argmax: NaN is maximal, first one wins
    if (g > bv) { best = k; bv = g; }
  }
  return (int64_t)best;                                // 0-based
}

struct Consts {
  double abratio, zgratio, lgd1, lgd2;
};
Consts make_consts(const rc_params& P) {
  Consts c;
  c.abratio = P.alpha * rc_log(P.beta) - rc_lgamma(P.alpha);   // mcmc.jl:17,186,293
  c.zgratio = P.zeta * rc_log(P.gamma) - rc_lgamma(P.zeta);    // mcmc.jl:18,187,294
  c.lgd1 = rc_lgamma(P.delta1);
  c.lgd2 = rc_lgamma(P.delta2);
  return c;
}

// loglik, mcmc.jl:1-56
double loglik(const Data& d, const State& s, const rc_params& P) {
  const int64_t n = d.n;
  Consts c = make_consts(P);
  std::vector<int64_t> C;
  for (int64_t k = 1; k <= n; ++k) if (s.sizes[k] > 0) C.push_back(k);
  const int64_t K = s.K;
  std::vector<std::vector<int64_t>> mem(K);
  for (int64_t k = 0; k < K; ++k)
    for (int64_t j = 0; j < n; ++j) if (s.clusts[j] == C[k]) mem[k].push_back(j);
  auto matsum2 = [&](bool logm, const std::vector<int64_t>& a, const std::vector<int64_t>& b) -> double {
    if (d.sum_mode == 0) {
      const std::vector<int64_t>& M = logm ? d.Lq : d.Dq;
      i128 acc = 0;
      for (int64_t x : a) for (int64_t y : b) acc += (i128)M[x * n + y];
      return rc_dequant128((int64_t)(acc >> 64), (uint64_t)acc, logm ? d.qL : d.qD);
    } else {
      const double* M = logm ? d.logD.data() : d.D;
      double acc = 0.0;
      for (int64_t x : a) for (int64_t y : b) acc += M[x * n + y];
      return acc;
    }
  };
  double L1 = 0;
  for (int64_t k = 0; k < K; ++k) {                                   // mcmc.jl:26-36
    int64_t sz = s.sizes[C[k]];
    double pairs = (double)(sz * (sz - 1) / 2);
    double a = P.alpha + P.delta1 * pairs;
    double b = P.beta + matsum2(false, mem[k], mem[k]) / 2;
    L1 += (P.delta1 - 1) * matsum2(true, mem[k], mem[k]) / 2 - pairs * c.lgd1 + c.abratio + rc_lgamma(a) - a * rc_log(b);
  }
  double L2 = 0;
  for (int64_t k = 0; k < K; ++k) {                                   // mcmc.jl:40-53
    int64_t szk = s.sizes[C[k]];
    for (int64_t t = k + 1; t < K; ++t) {
      int64_t szt = s.sizes[C[t]];
      double pairs = (double)(szk * szt);
      double z = P.zeta + P.delta2 * pairs;
      double g = P.gamma + matsum2(false, mem[k], mem[t]);
      L2 += (P.delta2 - 1) * matsum2(true, mem[k], mem[t]) - pairs * c.lgd2 + c.zgratio + rc_lgamma(z) - z * rc_log(g);
    }
  }
  return P.repulsion ? (L1 + L2) : (L1 + copysign(0.0, L2));          // L2 * repulsion, Bool strong zero
}

double xlogy(double a, double b) { return (a == 0.0 && !rc_isnan(b)) ? 0.0 : a * rc_log(b); }
double xlog1py(double a, double b) { return (a == 0.0 && !rc_isnan(b)) ? 0.0 : a * rc_log1p(b); }

// logprior, mcmc.jl:58-78.  logpdf(Gamma), logpdf(Beta) restate StatsFuns' gammalogpdf / betalogpdf.
double logprior(const State& s, const rc_params& P) {
  const int64_t n = (int64_t)s.clusts.size();
  const double K = (double)s.K, r = s.r, p = s.p;
  double theta = 1 / P.sigma;
  double xt = (r > 0 ? r : 0.0) / theta;
  double gl = -rc_lgamma(P.eta) - rc_log(theta) - xt;
  if (std::isfinite(xt)) gl += xlogy(P.eta - 1, xt);
  if (r < 0) gl = -RC_INF;
  double y = p < 0 ? 0.0 : (p > 1 ? 1.0 : p);
  double bl = xlogy(P.u - 1, y) + xlog1py(P.v - 1, -y) - (rc_lgamma(P.u) + rc_lgamma(P.v) - rc_lgamma(P.u + P.v));
  if (p < 0 || p > 1) bl = -RC_INF;
  double L = rc_lgamma(K + 1) + ((double)n - K) * rc_log(p) + (r * K) * rc_log(1 - p) - K * rc_lgamma(r) + gl + bl;
  for (int64_t k = 1; k <= n; ++k)
    if (s.sizes[k] > 0) { double nj = (double)s.sizes[k]; L += rc_log(nj) + rc_lgamma(nj + r - 1); }
  return L;
}

// rand(truncated(Normal(r, sd), lower = 0)): rejection of r + sd*z against the lower bound (mcmc.jl:104-109)
double draw_truncnorm0(double r, double sd, uint64_t key, uint32_t it) {
  double lb = (0.0 - r) / sd;
  double z = 0;
  for (uint32_t att = 0; att < 100000u; ++att) {
    z = rc_norminv(rc_open01(rc_draw1(key, it, RC_SITE_R_NORMAL, 0, att, 0)));
    if (z >= lb) break;
  }
  return r + sd * z;
}

// sample_r! / sample_r, mcmc.jl:80-136
bool sample_r(State& s, const rc_params& P, uint64_t key, uint32_t it) {
  const int64_t n = (int64_t)s.clusts.size();
  const double r = s.r, p = s.p, sd = P.proposalsd_r;
  const double K = (double)s.K;
  double cand = draw_truncnorm0(r, sd, key, it);
  double l1mp = rc_log(1 - p);
  double lpc = (P.eta - 1) * rc_log(cand) + K * (cand * l1mp - rc_lgamma(cand)) - cand * P.sigma;   // :117
  double lpr = (P.eta - 1) * rc_log(r) + K * (r * l1mp - rc_lgamma(r)) - r * P.sigma;               // :118
  for (int64_t k = 1; k <= n; ++k)
    if (s.sizes[k] > 0) {
      double nk1 = (double)(s.sizes[k] - 1);
      lpc = lpc + rc_lgamma(nk1 + cand);
      lpr = lpr + rc_lgamma(nk1 + r);
    }
  // logpdf(truncated Normal) = normlogpdf(z) - log(sd) - log(tp), tp = 1 - cdf(lower)   (:124-125)
  const double log2pi = 1.8378770664093454836;
  auto trunc_logpdf = [&](double mu, double x) {
    double zz = (x - mu) / sd;
    double lcdf = rc_normcdf((0.0 - mu) / sd);
    double logtp = rc_log(1.0 - lcdf);
    return -(zz * zz + log2pi) / 2 - rc_log(sd) - logtp;
  };
  double lratio = trunc_logpdf(r, cand) - trunc_logpdf(cand, r);
  double lu = rc_log(rc_draw1(key, it, RC_SITE_R_ACCEPT, 0, 0, 0));
  bool accept = lu < rc_min0(lpc - lpr - lratio);                                                    // :130-131
  if (accept) s.r = cand;
  return accept;
}

// sample_p! / sample_p, mcmc.jl:138-155
void sample_p(State& s, const rc_params& P, uint64_t key, uint32_t it) {
  const int64_t n = (int64_t)s.clusts.size();
  double a = (double)(n - s.K) + P.u;
  double b = s.r * (double)s.K + P.v;
  s.p = rc_beta(a, b, key, it);
}

// sample_labels_Gibbs!, mcmc.jl:158-256
struct GibbsProbe { int64_t i; std::vector<int64_t> cand; std::vector<double> lp; };   // tests: candidates / log-probabilities of one step
void gibbs_full(const Data& d, State& s, const rc_params& P, uint64_t key, uint32_t it, GibbsProbe* probe = nullptr) {
  const int64_t n = d.n;
  const double r = s.r, p = s.p;
  Consts c = make_consts(P);
  const double logp = rc_log(p), log1mp = rc_log(1 - p);
  std::vector<double> a_i(n + 1, 0.0), b_i(n + 1, 0.0), z_i(n + 1, 0.0), g_i(n + 1, 0.0), sl_i(n + 1, 0.0), L2p(n + 1, 0.0);
  std::vector<double> sD(n + 1), sL(n + 1);
  std::vector<int64_t> accD(n + 1), accL(n + 1);
  for (int64_t i = 0; i < n; ++i) {
    s.sizes[s.clusts[i]] -= 1;                                                       // :193
    s.clusts[i] = -1;                                                                // :194
    std::vector<int64_t> Ci;
    for (int64_t k = 1; k <= n; ++k) if (s.sizes[k] > 0) Ci.push_back(k);            // :195
    const int64_t Ki = (int64_t)Ci.size();
    std::vector<int64_t> cand = Ci;
    if ((P.maxK == 0 || Ki < P.maxK) && Ki < n) {                                    // :198-202
      for (int64_t k = 1; k <= n; ++k) if (s.sizes[k] == 0) { cand.push_back(k); break; }
    }
    const int64_t m = (int64_t)cand.size();
    rowsums(d, s, i, sD, sL, accD, accL);
    for (int64_t k : Ci) {                                                           // :206-214
      double sz = (double)s.sizes[k];
      a_i[k] = P.alpha + P.delta1 * sz;
      b_i[k] = P.beta + sD[k];
      z_i[k] = P.zeta + P.delta2 * sz;
      g_i[k] = P.gamma + sD[k];
      sl_i[k] = sL[k];
    }
    std::vector<double> L1(m, 0.0), L2(m, 0.0), lpr(m, 0.0), lp(m, 0.0);
    auto existing = [&](int64_t kk) {
      int64_t ck = cand[kk];
      double sz = (double)s.sizes[ck];
      L1[kk] = rc_lgamma(a_i[ck]) + c.abratio - a_i[ck] * rc_log(b_i[ck]) + (P.delta1 - 1) * sl_i[ck] - sz * c.lgd1;   // :223-225
      lpr[kk] = rc_log((double)(s.sizes[ck] + 1)) + logp + rc_log((double)(s.sizes[ck] - 1) + r) - rc_log(sz);          // :226
    };
    for (int64_t kk = 0; kk < m - 1; ++kk) existing(kk);                             // :221-227
    if (s.sizes[cand[m - 1]] == 0) {                                                 // :228-230
      lpr[m - 1] = rc_log((double)(Ki + 1)) + r * log1mp;
      L1[m - 1] = 0;
    } else existing(m - 1);                                                          // :231-237
    for (int64_t t : Ci) {                                                           // :239-242
      L2p[t] = rc_lgamma(z_i[t]) - z_i[t] * rc_log(g_i[t]) + c.zgratio + (P.delta2 - 1) * sl_i[t] - (double)s.sizes[t] * c.lgd2;
    }
    double L2i = vecsum_canonical(L2p, Ci);                                          // :243
    for (int64_t kk = 0; kk < m; ++kk) {                                             // :244-246
      bool live = s.sizes[cand[kk]] != 0;
      L2[kk] = live ? (L2i - L2p[cand[kk]]) : (L2i - copysign(0.0, L2p[cand[kk]]));
    }
    for (int64_t kk = 0; kk < m; ++kk)                                               // :247
      lp[kk] = lpr[kk] + (L1[kk] + (P.repulsion ? L2[kk] : copysign(0.0, L2[kk])));
    if (probe && probe->i == i) { probe->cand = cand; probe->lp = lp; }
    std::vector<double> u(m);
    for (int64_t kk = 0; kk < m; ++kk) {   // candidates 2q and 2q+1 share one Philox block (u0, u1)
      rc_draw dr = rc_draw2(key, it, RC_SITE_SCAN, 0, (uint32_t)i, (uint32_t)(kk >> 1));
      u[kk] = (kk & 1) ? dr.u1 : dr.u0;
    }
    int64_t k = sample_logweights(lp, u);                                            // :249
    int64_t cnew = cand[k];
    s.clusts[i] = cnew;                                                              // :251-252
    s.sizes[cnew] += 1;
  }
  int64_t K = 0;
  for (int64_t k = 1; k <= n; ++k) K += s.sizes[k] > 0;                              // :254
  s.K = K;
}

// sample_labels_Gibbs_restricted!, mcmc.jl:259-354.  `forced` empty => free allocation.
double gibbs_restricted(const Data& d, State& s, const rc_params& P, const std::vector<int64_t>& items,
                        const int64_t cands[2], const std::vector<int64_t>* forced,
                        uint64_t key, uint32_t it, uint32_t mh, uint32_t scan) {
  const int64_t n = d.n;
  const int64_t K = s.K;
  std::vector<int64_t> C;
  for (int64_t k = 1; k <= n; ++k) if (s.sizes[k] > 0) C.push_back(k);               // :273
  int64_t cind[2];
  for (int q = 0; q < 2; ++q) { cind[q] = -1; for (int64_t t = 0; t < (int64_t)C.size(); ++t) if (C[t] == cands[q]) { cind[q] = t; break; } }  // :274
  const double r = s.r, p = s.p;
  const bool free_alloc = (forced == nullptr);
  double ltp = 0;
  Consts c = make_consts(P);
  const double logp = rc_log(p);
  double a_i[2], b_i[2], L1[2], L2[2], lpr[2];
  std::vector<double> z_i(K, 0.0), g_i(K, 0.0), sl_i(K, 0.0), L2p(K, 0.0);
  std::vector<double> sD(n + 1), sL(n + 1);
  std::vector<int64_t> accD(n + 1), accL(n + 1);
  for (size_t pos = 0; pos < items.size(); ++pos) {
    const int64_t i = items[pos];
    s.sizes[s.clusts[i]] -= 1;                                                       // :303-304
    s.clusts[i] = -1;
    rowsums(d, s, i, sD, sL, accD, accL);
    for (int q = 0; q < 2; ++q) {                                                    // :307-312
      a_i[q] = P.alpha + P.delta1 * (double)s.sizes[cands[q]];
      b_i[q] = P.beta + sD[cands[q]];
    }
    for (int64_t k = 0; k < K; ++k) {                                                // :313-319
      z_i[k] = P.zeta + P.delta2 * (double)s.sizes[C[k]];
      g_i[k] = P.gamma + sD[C[k]];
      sl_i[k] = sL[C[k]];
    }
    for (int q = 0; q < 2; ++q) {                                                    // :321-326
      double sz = (double)s.sizes[cands[q]];
      L1[q] = rc_lgamma(a_i[q]) + c.abratio - a_i[q] * rc_log(b_i[q]) + (P.delta1 - 1) * sl_i[cind[q]] - sz * c.lgd1;
      lpr[q] = rc_log((double)(s.sizes[cands[q]] + 1)) + logp + rc_log((double)(s.sizes[cands[q]] - 1) + r) - rc_log(sz);
    }
    for (int64_t t = 0; t < K; ++t)                                                  // :327-330
      L2p[t] = rc_lgamma(z_i[t]) - z_i[t] * rc_log(g_i[t]) + c.zgratio + (P.delta2 - 1) * sl_i[t] - (double)s.sizes[C[t]] * c.lgd2;
    double L2i = L2p[0] + L2p[1];                                                    // :331 (quirk Q2)
    for (int q = 0; q < 2; ++q) L2[q] = L2i - L2p[cind[q]];                          // :332-334
    std::vector<double> lp(2);
    for (int q = 0; q < 2; ++q) lp[q] = lpr[q] + (L1[q] + (P.repulsion ? L2[q] : copysign(0.0, L2[q])));  // :335
    int64_t k, cnew;
    if (free_alloc) {                                                                // :336-338
      rc_draw dr = rc_draw2(key, it, RC_SITE_SM_RGIBBS, mh, scan, (uint32_t)pos);
      std::vector<double> u = {dr.u0, dr.u1};
      k = sample_logweights(lp, u);
      cnew = cands[k];
    } else {                                                                         // :339-342
      cnew = (*forced)[i];
      k = (cands[0] == cnew) ? 0 : 1;
    }
    s.clusts[i] = cnew;                                                              // :344-345
    s.sizes[cnew] += 1;
    double mn = lp[0];                                                               // :348 (quirk Q3: ADDS the minimum)
    if (!rc_isnan(mn)) { if (rc_isnan(lp[1]) || lp[1] < mn) mn = lp[1]; }
    lp[0] += mn; lp[1] += mn;
    double p0 = rc_exp(lp[0]), p1 = rc_exp(lp[1]);                                   // :349
    double den = p0 + p1;
    p0 /= den; p1 /= den;                                                            // :350
    ltp += rc_log(k == 0 ? p0 : p1);                                                 // :351
  }
  return ltp;
}

// sample_labels!, mcmc.jl:356-479.  Returns through accept[] / split[] (numMH entries each).
void sample_labels(const Data& d, State& caller, const rc_params& P, const rc_options& O, uint64_t key, uint32_t it,
                   uint8_t* accept, uint8_t* split) {
  const int64_t n = d.n;
  const double r = caller.r, p = caller.p;                                            // :365-366
  State* state = &caller;               // Julia's local `state`; rebinding it does not touch the caller (quirk Q1)
  std::vector<State> keep;              // keeps accepted final states alive
  keep.reserve((size_t)O.numMH + 1);
  for (int64_t mh = 0; mh < O.numMH; ++mh) {
    accept[mh] = 0; split[mh] = 0;
    const std::vector<int64_t>& clusts = state->clusts;
    const std::vector<int64_t>& sizes = state->sizes;
    const int64_t K = state->K;
    // (i, j) = sample(1:n, 2, replace=false): StatsBase samplepair (:379)
    rc_draw dr = rc_draw2(key, it, RC_SITE_SM_PAIR, (uint32_t)mh, 0, 0);
    int64_t i1 = rc_randint(dr.u0, n), i2 = rc_randint(dr.u1, n - 1);
    if (i2 == i1) i2 = n;
    const int64_t i = i1 - 1, j = i2 - 1;
    const int64_t ci = clusts[i], cj = clusts[j];
    if (P.maxK > 0 && ci == cj) {                                                     // :384-386
      int64_t live = 0; for (int64_t k = 1; k <= n; ++k) live += sizes[k] > 0;
      if (live >= P.maxK) continue;
    }
    std::vector<int64_t> S;                                                           // :389-390
    for (int64_t k = 0; k < n; ++k) if ((clusts[k] == ci || clusts[k] == cj) && k != i && k != j) S.push_back(k);
    State launch;                                                                     // :393-408
    launch.clusts = clusts; launch.sizes = sizes; launch.r = r; launch.p = p; launch.K = K;
    if (ci == cj) {
      int64_t e = 0; for (int64_t k = 1; k <= n; ++k) if (sizes[k] == 0) { e = k; break; }
      launch.clusts[i] = e;
      launch.sizes[ci] -= 1;
      launch.sizes[e] += 1;
      launch.K = K + 1;
    }
    const int64_t cands[2] = {launch.clusts[i], launch.clusts[j]};
    for (size_t pos = 0; pos < S.size(); ++pos) {
      int64_t k = S[pos];
      double u = rc_draw1(key, it, RC_SITE_SM_LAUNCH, (uint32_t)mh, (uint32_t)pos, 0);
      launch.clusts[k] = cands[rc_randint(u, 2) - 1];
      launch.sizes[clusts[k]] -= 1;
      launch.sizes[launch.clusts[k]] += 1;
    }
    for (int64_t g = 0; g < O.numGibbs; ++g)                                          // :411-414
      gibbs_restricted(d, launch, P, S, cands, nullptr, key, it, (uint32_t)mh, (uint32_t)g);
    double log_prior_ratio, log_proposal_ratio;
    State fin;
    if (ci == cj) {                                                                   // split, :416-434
      split[mh] = 1;
      double ltp = gibbs_restricted(d, launch, P, S, cands, nullptr, key, it, (uint32_t)mh, (uint32_t)O.numGibbs);
      fin = launch;
      const std::vector<int64_t>& cf = fin.clusts; const std::vector<int64_t>& szf = fin.sizes;
      log_prior_ratio = rc_log((double)(K + 1)) + r * rc_log(1 - p) - rc_log(p) - rc_lgamma(r) +
                        rc_lgamma((double)(szf[cf[i]] - 1) + r) + rc_lgamma((double)(szf[cf[j]] - 1) + r) +
                        rc_log((double)szf[cf[i]]) + rc_log((double)szf[cf[j]]) +
                        -(rc_lgamma((double)(sizes[ci] - 1) + r) + rc_log((double)sizes[ci]));   // :427-430
      log_proposal_ratio = ltp;                                                       // :433
    } else {                                                                          // merge, :435-459
      fin.clusts = launch.clusts; fin.sizes = launch.sizes; fin.r = r; fin.p = p; fin.K = launch.K;
      int64_t szi = 0;
      for (int64_t k = 0; k < n; ++k) if (fin.clusts[k] == ci) { fin.clusts[k] = cj; ++szi; }
      fin.sizes[ci] = 0;
      fin.sizes[cj] += szi;
      fin.K -= 1;
      const std::vector<int64_t>& szf = fin.sizes;
      log_prior_ratio = -(rc_log((double)K) + r * rc_log(1 - p) - rc_log(p) - rc_lgamma(r)) +
                        rc_lgamma((double)(szf[cj] - 1) + r) + rc_log((double)szf[cj]) +
                        -(rc_lgamma((double)(sizes[ci] - 1) + r) + rc_lgamma((double)(sizes[cj] - 1) + r) +
                          rc_log((double)sizes[ci]) + rc_log((double)sizes[cj]));              // :448-451
      double ltp = gibbs_restricted(d, launch, P, S, cands, &clusts, key, it, (uint32_t)mh, (uint32_t)O.numGibbs);  // :454-455
      log_proposal_ratio = -ltp;                                                      // :457
    }
    double log_lik_ratio = loglik(d, fin, P) - loglik(d, *state, P);                  // :462-464
    double lar = rc_min0(log_prior_ratio + log_lik_ratio - log_proposal_ratio);       // :467-468
    double lu = rc_log(rc_draw1(key, it, RC_SITE_SM_ACCEPT, (uint32_t)mh, 0, 0));
    if (lu < lar) {                                                                   // :469-472
      keep.push_back(fin);
      state = &keep.back();
      accept[mh] = 1;
    }
  }
  gibbs_full(d, *state, P, key, it);                                                  // :477 (on the LOCAL state)
}

// sortlabels, utils.jl:69-74 (StatsBase.levelsmap = first-appearance numbering)
void sortlabels(const std::vector<int64_t>& x, int64_t* out) {
  const int64_t n = (int64_t)x.size();
  std::vector<int64_t> map(n + 2, 0);
  int64_t next = 0;
  for (int64_t i = 0; i < n; ++i) { if (map[x[i]] == 0) map[x[i]] = ++next; out[i] = map[x[i]]; }
}

State make_state(const int64_t* labels, int64_t n, double r, double p) {              // types.jl:131-137
  State s; s.clusts.assign(labels, labels + n); s.r = r; s.p = p;
  s.sizes.assign(n + 1, 0);
  for (int64_t i = 0; i < n; ++i) s.sizes[labels[i]] += 1;
  s.K = 0; for (int64_t k = 1; k <= n; ++k) s.K += s.sizes[k] > 0;
  return s;
}

}  // namespace

extern "C" {

// runsampler's iteration loop + record step, mcmc.jl:537-555, for ONE chain.
int rco_run(const double* D, int64_t n, const rc_options* O, const rc_params* P, const int64_t* init_labels,
            double init_r, double init_p, uint64_t seed, uint64_t chain, int sum_mode,
            int64_t* out_labels, int64_t* out_K, double* out_r, double* out_p, double* out_loglik, double* out_logpost,
            uint8_t* r_acc, uint8_t* sm_acc, uint8_t* sm_split, int64_t* final_labels, double* final_rp) {
  Data d; build_data(d, D, n, sum_mode);
  State s = make_state(init_labels, n, init_r, init_p);
  const uint64_t key = rc_chain_key(seed, chain);
  int64_t j = 0;
  std::vector<uint8_t> acc((size_t)std::max<int64_t>(O->numMH, 1)), spl((size_t)std::max<int64_t>(O->numMH, 1));
  for (int64_t i = 1; i <= O->numiters; ++i) {
    bool ra = sample_r(s, *P, key, (uint32_t)i);                                       // :538
    if (r_acc) r_acc[i - 1] = ra;
    sample_p(s, *P, key, (uint32_t)i);                                                 // :539
    sample_labels(d, s, *P, *O, key, (uint32_t)i, acc.data(), spl.data());             // :540
    for (int64_t m = 0; m < O->numMH; ++m) {                                           // :541-543
      if (sm_acc) sm_acc[(i - 1) * O->numMH + m] = acc[m];
      if (sm_split) sm_split[(i - 1) * O->numMH + m] = spl[m];
    }
    if (i > O->burnin && (i - O->burnin) % O->thin == 0) {                             // :546-554
      if (out_labels) sortlabels(s.clusts, out_labels + j * n);
      if (out_K) out_K[j] = s.K;
      if (out_r) out_r[j] = s.r;
      if (out_p) out_p[j] = s.p;
      double ll = loglik(d, s, *P);
      if (out_loglik) out_loglik[j] = ll;
      if (out_logpost) out_logpost[j] = ll + logprior(s, *P);
      ++j;
    }
  }
  if (final_labels) for (int64_t k = 0; k < n; ++k) final_labels[k] = s.clusts[k];
  if (final_rp) { final_rp[0] = s.r; final_rp[1] = s.p; }
  return 0;
}

double rco_loglik(const double* D, int64_t n, const rc_params* P, const int64_t* labels, int sum_mode) {
  Data d; build_data(d, D, n, sum_mode);
  State s = make_state(labels, n, 1.0, 0.5);
  return loglik(d, s, *P);
}
double rco_logprior(int64_t n, const rc_params* P, const int64_t* labels, double r, double p) {
  State s = make_state(labels, n, r, p);
  return logprior(s, *P);
}
void rco_logdist(const double* D, int64_t n, double* out) {
  Data d; build_data(d, D, n, 1);
  std::memcpy(out, d.logD.data(), sizeof(double) * (size_t)n * n);
}
void rco_init_rp(const rc_params* P, uint64_t seed, uint64_t chain, double* r, double* p) {
  // r ~ Gamma(eta, 1/sigma), p ~ Beta(u, v): mcmc.jl:524-525 (iteration 0 of the stream)
  rc_init_rp_draw(P->eta, P->sigma, P->u, P->v, seed, chain, r, p);
}

// pairwise(Euclidean(), X, dims=2), types.jl:160 / utils.jl:144-145 / prior.jl:51,180.
// Restates the Gram formulation of Distances.jl 0.10 (not vendored in /root/reference):
// D_ij = sqrt(max(|x_i|^2 + |x_j|^2 - 2 x_i.x_j, 0)), one triangle mirrored, zero diagonal; an entry the Gram form
// cannot resolve is recomputed from the differences (rc_dist_unresolved, Distances.jl's Euclidean(thresh)).
void rco_distm(const double* X, int64_t dim, int64_t n, double* D) {
  std::vector<double> sq(n);
  for (int64_t i = 0; i < n; ++i) { double a = 0; for (int64_t t = 0; t < dim; ++t) a += X[i * dim + t] * X[i * dim + t]; sq[i] = a; }
  for (int64_t i = 0; i < n; ++i) {
    D[i * n + i] = 0.0;
    for (int64_t j = i + 1; j < n; ++j) {
      double dot = 0;
      for (int64_t t = 0; t < dim; ++t) dot += X[i * dim + t] * X[j * dim + t];
      double v = sq[i] + sq[j] - 2 * dot;
      if (rc_dist_unresolved(v, sq[i] + sq[j])) v = rc_dist_direct2(X + i * dim, X + j * dim, dim);
      double r = sqrt(v > 0 ? v : 0.0);
      D[i * n + j] = r; D[j * n + i] = r;
    }
  }
}

// Timed multi-chain driver for bench.py's cpu_baseline / --impl reference legs: the data images are built
// once (untimed), then `nchains` independent chains run `sweeps` iterations of the loop at mcmc.jl:537-555
// on `nthreads` host threads (one chain per thread at a time; the reference itself is single-threaded,
// so this is the "one independent chain per core" figure of BASELINE.md section 4).  Returns the seconds
// spent in the iteration loops (wall clock over all threads) and each chain's final K.
double rco_time_chains(const double* D, int64_t n, const rc_options* O, const rc_params* P, const int64_t* init_labels,
                       const double* init_r, const double* init_p, uint64_t seed, int64_t chain0, int64_t nchains,
                       int nthreads, int sum_mode, int64_t* final_K) {
  Data d; build_data(d, D, n, sum_mode);
  std::vector<std::thread> th;
  auto t0 = std::chrono::steady_clock::now();
  for (int t = 0; t < nthreads; ++t)
    th.emplace_back([&, t]() {
      for (int64_t c = t; c < nchains; c += nthreads) {
        State s = make_state(init_labels, n, init_r[c], init_p[c]);
        const uint64_t key = rc_chain_key(seed, (uint64_t)(chain0 + c));
        std::vector<uint8_t> acc((size_t)std::max<int64_t>(O->numMH, 1)), spl((size_t)std::max<int64_t>(O->numMH, 1));
        double sink = 0;
        for (int64_t i = 1; i <= O->numiters; ++i) {
          sample_r(s, *P, key, (uint32_t)i);
          sample_p(s, *P, key, (uint32_t)i);
          sample_labels(d, s, *P, *O, key, (uint32_t)i, acc.data(), spl.data());
          if (i > O->burnin && (i - O->burnin) % O->thin == 0) sink += loglik(d, s, *P) + logprior(s, *P);
        }
        if (final_K) final_K[c] = s.K + (sink != sink ? 0 : 0);
      }
    });
  for (auto& x : th) x.join();
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// sample_rp, mcmc.jl:592-636: the (r, p)-only chain on fixed cluster sizes (fitprior, prior.jl:80).
void rco_sample_rp(const int64_t* clustsizes, int64_t nsizes, const rc_options* O, const rc_params* P, uint64_t seed,
                   double* out_r, double* out_p, uint8_t* r_acc) {
  std::vector<int64_t> labels;                                       // C = clustsizes[findall(clustsizes .> 0)]  (:613)
  int64_t k = 0;
  for (int64_t t = 0; t < nsizes; ++t)
    if (clustsizes[t] > 0) { ++k; for (int64_t q = 0; q < clustsizes[t]; ++q) labels.push_back(k); }
  const uint64_t key = rc_chain_key(seed, 0);
  const double r0 = rc_gamma_mt(P->eta, key, 0, RC_SITE_INIT, 2) * P->sigma;   // :617 rand(Gamma(eta, sigma)): scale sigma
  const double p0 = rc_beta(P->u, P->v, key, 0);                                // :618
  State s = make_state(labels.data(), (int64_t)labels.size(), r0, p0);
  int64_t j = 0;
  for (int64_t i = 1; i <= O->numiters; ++i) {
    bool ra = sample_r(s, *P, key, (uint32_t)i);                                 // :623
    sample_p(s, *P, key, (uint32_t)i);                                           // :625
    if (r_acc) r_acc[i - 1] = ra;
    if (i > O->burnin && (i - O->burnin) % O->thin == 0) { out_r[j] = s.r; out_p[j] = s.p; ++j; }
  }
}

// ---- probes for tests/test_oracle_pins.py ----------------------------------------------------------------
// `iters` full Gibbs scans (mcmc.jl:158-256) at FIXED (r, p): the Markov chain on partitions whose exact transition
// matrix the test builds from an independent numpy statement of the conditionals.  states: iters x n, sortlabels'd.
void rco_scan_only(const double* D, int64_t n, const rc_params* P, const int64_t* labels, double r, double p, uint64_t seed,
                   uint64_t chain, int64_t iters, int sum_mode, int64_t* states) {
  Data d; build_data(d, D, n, sum_mode);
  State s = make_state(labels, n, r, p);
  const uint64_t key = rc_chain_key(seed, chain);
  for (int64_t it = 1; it <= iters; ++it) {
    gibbs_full(d, s, *P, key, (uint32_t)it);
    sortlabels(s.clusts, states + (it - 1) * n);
  }
}
// Candidate slots and un-normalised log-probabilities (mcmc.jl:247) of the scan step of point i (0-based) when the
// points before it keep their labels: returns the number of candidates m; cand / lp hold m entries.
int64_t rco_gibbs_logprobs(const double* D, int64_t n, const rc_params* P, const int64_t* labels, double r, double p, int64_t i,
                           int sum_mode, int64_t* cand, double* lp) {
  // gibbs_full visits the points in index order, so point i is swapped with point 0 (rows / columns of D and the
  // labels): it is then visited first, in exactly the given state; slot ids -- hence the candidate order -- are unchanged
  std::vector<double> Dp((size_t)n * n);
  std::vector<int64_t> perm(n), lab(n);
  for (int64_t t = 0; t < n; ++t) perm[t] = t;
  std::swap(perm[0], perm[i]);
  for (int64_t a = 0; a < n; ++a)
    for (int64_t b = 0; b < n; ++b) Dp[a * n + b] = D[perm[a] * n + perm[b]];
  for (int64_t t = 0; t < n; ++t) lab[t] = labels[perm[t]];
  Data dp; build_data(dp, Dp.data(), n, sum_mode);
  State sp = make_state(lab.data(), n, r, p);
  GibbsProbe q; q.i = 0;
  gibbs_full(dp, sp, *P, 12345u, 1u, &q);
  for (size_t t = 0; t < q.cand.size(); ++t) { cand[t] = q.cand[t]; lp[t] = q.lp[t]; }
  return (int64_t)q.cand.size();
}
// Raw draws of the samplers shared by the oracle and the kernels (rc_rng.h), one per iteration index, for
// goodness-of-fit tests against scipy: kind 0 Gamma(a, 1) (Marsaglia-Tsang, mcmc.jl:154 / :524), 1 Beta(a, b)
// (mcmc.jl:154), 2 truncated(Normal(a, b), lower = 0) (mcmc.jl:104-109), 3 rand(1:a) (mcmc.jl:379, 404).
void rco_draws(int kind, double a, double b, uint64_t seed, int64_t count, double* out) {
  const uint64_t key = rc_chain_key(seed, 0);
  for (int64_t t = 0; t < count; ++t) {
    const uint32_t it = (uint32_t)(t + 1);
    if (kind == 0) out[t] = rc_gamma_mt(a, key, it, RC_SITE_P_GAMMA_A, 0);
    else if (kind == 1) out[t] = rc_beta(a, b, key, it);
    else if (kind == 2) out[t] = draw_truncnorm0(a, b, key, it);
    else out[t] = (double)rc_randint(rc_draw1(key, it, RC_SITE_SM_PAIR, 0, 0, 0), (int64_t)a);
  }
}

// probes for tests/test_math.py
double rco_log(double x) { return rc_log(x); }
double rco_exp(double x) { return rc_exp(x); }
double rco_log1p(double x) { return rc_log1p(x); }
double rco_lgamma(double x) { return rc_lgamma(x); }
double rco_erfc(double x) { return rc_erfc(x); }
double rco_normcdf(double x) { return rc_normcdf(x); }
double rco_norminv(double x) { return rc_norminv(x); }
void rco_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
  rc_u4 o = rc_philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
  out[0] = o.x; out[1] = o.y; out[2] = o.z; out[3] = o.w;
}
void rco_draw2(uint64_t seed, uint64_t chain, uint32_t it, uint32_t site, uint32_t mh, uint32_t a, uint32_t b, double* out) {
  rc_draw d = rc_draw2(rc_chain_key(seed, chain), it, site, mh, a, b);
  out[0] = d.u0; out[1] = d.u1;
}
int rco_fixedpoint_scales(const double* D, int64_t n, int* qD, int* qL) {
  Data d; build_data(d, D, n, 1);
  *qD = d.qD; *qL = d.qL; return 0;
}

}  // extern "C"
