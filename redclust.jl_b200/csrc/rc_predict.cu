// rc_predict.cu -- posterior predictive allocation of new observations.
//
// For a new point x and a recorded state s = (labels, r, p), P_s(x, k) is the scan-step conditional of src/mcmc.jl:193-247
// for x as point n + 1 of the augmented data [[D, Dnew[x]'], [Dnew[x], 0]], normalised as sample_logweights draws from it
// (src/utils.jl:2-6): softmax over the existing slots 1..K_s and, unless maxK forbids it, the new slot K_s + 1.  The
// predictive co-clustering with training point j is the mean over samples of P_s(x, c_s(j)).  The reference has no such
// call; this is the quantity its sampler would produce if x were in the data and visited at that state.
//
// The arithmetic is the oracle's scan step (oracle/rc_oracle.cpp gibbs_full, sum_mode 0) term for term:
//   - per-slot sums of Dnew[x] and log Dnew[x] are exact int64 sums of fixed-point images at the augmented data's scales
//     qD = rc_choose_q(max(max|D|, max Dnew[x]), n + 1), qL likewise over |log|;
//   - the repulsion total L2i is vecsum_canonical: slot k on lane (k - 1) % 32, lane sums ascending, xor butterfly;
//   - the normaliser of the softmax is summed the same way.
// Kernels, in launch order (DESIGN.md 3.5):
//   k_pred_scan   domain check and per-row maxima of Dnew
//   k_pred_image  {Dq, Lq} image of Dnew at each row's scales (m x n longlong2)
//   per chunk of samples:
//   k_pred_terms  cluster sizes and the per-(sample, slot) terms that do not depend on x
//   k_pred_sums   per-(x, sample, slot) sums in shared memory, then lp and P (one warp per (x, sample))
//   k_pred_cocl   ascending-sample accumulation of P_s(x, c_s(j)) into the m x n output
#include <vector>
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include "rc_common.cuh"
#include "rc_labels.h"

namespace {

#define PX 4                          // new points per CTA of k_pred_sums and k_pred_cocl
#define PT_MAX 64                     // samples per CTA of k_pred_sums (fewer when the slot count is large)
#define PSUM_THREADS 256
#define PSMEM_BUDGET (96 * 1024)      // accumulators of one k_pred_sums CTA: two CTAs per SM
#define PCHUNK_BYTES (256ull << 20)   // probabilities of one chunk of samples
#define FULL 0xffffffffu

struct PConst {                       // mcmc.jl:17-18,186-187 constants and the hyperparameters the scan step reads
  double alpha, beta, zeta, gamma, delta1, delta2;
  double abratio, zgratio, lgd1, lgd2;
  long long maxK;
  int repulsion;
};

// Domain check (the rules of rc_data.cu's k_scan for off-diagonal entries) and the row maxima of max |d|, max |log d|.
__global__ void __launch_bounds__(256) k_pred_scan(const double* __restrict__ Dn, int64_t n, int* __restrict__ bad,
                                                   double2* __restrict__ rowmax) {
  const double* row = Dn + (int64_t)blockIdx.x * n;
  double mD = 0.0, mL = 0.0;
  int b = 0;
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    const double v = row[j];
    if (!(v > 0.0) || !(v < RC_INF)) { b = 1; continue; }
    mD = fmax(mD, v);
    mL = fmax(mL, fabs(rc_log(v)));
  }
  __shared__ double sD[8], sL[8];
  for (int off = 16; off; off >>= 1) {
    mD = fmax(mD, __shfl_xor_sync(FULL, mD, off));
    mL = fmax(mL, __shfl_xor_sync(FULL, mL, off));
  }
  b = __syncthreads_or(b);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { sD[w] = mD; sL[w] = mL; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 1; q < (int)(blockDim.x >> 5); ++q) { mD = fmax(mD, sD[q]); mL = fmax(mL, sL[q]); }
    rowmax[blockIdx.x] = make_double2(mD, mL);
    if (b) atomicOr(bad, 1);
  }
}

// The fixed-point image of each new row at its own scales, as rc_data.cu's k_build_dl for an off-diagonal entry.
__global__ void k_pred_image(const double* __restrict__ Dn, int64_t m, int64_t n, const int2* __restrict__ q,
                             longlong2* __restrict__ img) {
  const int64_t total = m * n;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int2 s = q[t / n];
    const double v = Dn[t];
    longlong2 o;
    o.x = rc_quantize(v, s.x);
    o.y = rc_quantize(rc_log(v - 0.0 + 0.0), s.y);
    img[t] = o;
  }
}

// Per sample of the chunk: K, the cluster sizes, and the terms of the scan step that depend only on the size of a slot and
// (r, p): TA = lgamma(alpha + delta1 n_k) + abratio, TZ = lgamma(zeta + delta2 n_k), TL = the prior term of an existing slot
// (mcmc.jl:226), TN = that of the new slot (mcmc.jl:229), NaN when maxK leaves no new slot (mcmc.jl:198-202).
__global__ void __launch_bounds__(256) k_pred_terms(const uint8_t* __restrict__ lab, int64_t n, const double* __restrict__ r,
                                                    const double* __restrict__ p, PConst c, int* __restrict__ Kt,
                                                    int* __restrict__ szt, double* __restrict__ TA, double* __restrict__ TZ,
                                                    double* __restrict__ TL, double* __restrict__ TN) {
  __shared__ int h[256];
  __shared__ int Ks;
  const int s = blockIdx.x;
  h[threadIdx.x] = 0;
  if (threadIdx.x == 0) Ks = 0;
  __syncthreads();
  const uint8_t* l = lab + (int64_t)s * n;
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) atomicAdd(&h[l[j]], 1);
  __syncthreads();
  if (threadIdx.x > 0 && h[threadIdx.x] > 0) atomicMax(&Ks, (int)threadIdx.x);
  __syncthreads();
  const int K = Ks;
  const double rs = r[s], ps = p[s];
  const double logp = rc_log(ps), log1mp = rc_log(1 - ps);
  const int k = threadIdx.x + 1;
  const size_t o = (size_t)s * 256 + threadIdx.x;
  if (k <= K) {
    const int nk = h[k];
    const double sz = (double)nk;
    szt[o] = nk;
    TA[o] = rc_lgamma(c.alpha + c.delta1 * sz) + c.abratio;
    TZ[o] = rc_lgamma(c.zeta + c.delta2 * sz);
    TL[o] = rc_log((double)(nk + 1)) + logp + rc_log((double)(nk - 1) + rs) - rc_log(sz);
  }
  if (threadIdx.x == 0) {
    Kt[s] = K;
    TN[s] = (c.maxK == 0 || K < c.maxK) ? rc_log((double)(K + 1)) + rs * log1mp : RC_NAN;   // K < n + 1 always
  }
}

// Every label byte of the samples lies in 1..Kc (flag otherwise): the accumulators and the probability rows are indexed by it.
__global__ void k_pred_check(const uint8_t* __restrict__ lab, size_t total, int Kc, int* __restrict__ bad) {
  int b = 0;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int l = lab[t];
    b |= (l == 0) | (l > Kc);
  }
  if (__syncthreads_or(b) && threadIdx.x == 0) atomicOr(bad, 1);
}

// acc += v modulo 2^64 on a {lo, hi} pair of 32-bit shared words with two native atomics (a 64-bit shared atomicAdd is a
// compare-and-swap loop on sm_100a): the low add returns the old word, which tells whether it carried.
__device__ __forceinline__ void atomic_add64(unsigned* acc, long long v) {
  const unsigned lo = (unsigned)v, hi = (unsigned)((unsigned long long)v >> 32);
  const unsigned old = atomicAdd(acc, lo);
  atomicAdd(acc + 1, hi + (old + lo < old ? 1u : 0u));
}

// Sum of eight 64-bit words over the warp, scattered: afterwards lane 4v (v = 0..7) holds the total of word v.
__device__ __forceinline__ long long warp_sum8(const long long (&v)[8], int lane) {
  long long w4[4], w2[2], w1;
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long keep = b4 ? v[4 + i] : v[i], give = b4 ? v[i] : v[4 + i];
    w4[i] = keep + __shfl_xor_sync(FULL, give, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const long long keep = b3 ? w4[2 + i] : w4[i], give = b3 ? w4[i] : w4[2 + i];
    w2[i] = keep + __shfl_xor_sync(FULL, give, 8);
  }
  {
    const long long keep = b2 ? w2[1] : w2[0], give = b2 ? w2[0] : w2[1];
    w1 = keep + __shfl_xor_sync(FULL, give, 4);
  }
  w1 += __shfl_xor_sync(FULL, w1, 2);
  w1 += __shfl_xor_sync(FULL, w1, 1);
  return w1;
}

// One CTA per (block of PX new points, block of T samples).  Pass 1 walks every training column once: each thread owns a
// column, holds its PX image entries in registers and adds them into the (x, sample, slot) accumulators in shared memory
// -- one 64-bit atomic per lane, or, when the whole warp shares the label (training data is often stored by cluster),
// one per word after a warp sum.  Integer sums are exact, so the order is free.  Pass 2: one warp per (x, sample)
// evaluates the scan step's log-probabilities and their softmax.
__global__ void __launch_bounds__(PSUM_THREADS) k_pred_sums(const longlong2* __restrict__ img, const int2* __restrict__ q, int64_t m,
                                                            int64_t n, const uint8_t* __restrict__ lab, int nsc, int SC, int T, int Kc,
                                                            const int* __restrict__ Kt, const int* __restrict__ szt,
                                                            const double* __restrict__ TA, const double* __restrict__ TZ,
                                                            const double* __restrict__ TL, const double* __restrict__ TN, PConst c,
                                                            double* __restrict__ Pb, double* __restrict__ PN,
                                                            double* __restrict__ lp_out) {
  extern __shared__ unsigned acc[];                      // [PX][T][Kc] x {D, L} x {lo, hi}
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t x0 = (int64_t)blockIdx.x * PX;
  const int t0 = blockIdx.y * T;
  const int nx = (int)min((int64_t)PX, m - x0), nt = min(T, nsc - t0);
  const int words = PX * T * Kc * 4;
  for (int i = threadIdx.x; i < words; i += PSUM_THREADS) acc[i] = 0u;
  __syncthreads();
  for (int64_t j0 = 0; j0 < n; j0 += PSUM_THREADS) {
    const int64_t j = j0 + threadIdx.x;
    const bool ok = j < n;
    long long v[2 * PX];
#pragma unroll
    for (int xi = 0; xi < PX; ++xi) {
      const longlong2 e = (ok && xi < nx) ? img[(x0 + xi) * n + j] : make_longlong2(0, 0);
      v[2 * xi] = e.x; v[2 * xi + 1] = e.y;
    }
    for (int tb = 0; tb < nt; tb += 4) {
      int cls[4];                                        // four samples' labels in flight at once
#pragma unroll
      for (int u = 0; u < 4; ++u) cls[u] = (ok && tb + u < nt) ? lab[(int64_t)(t0 + tb + u) * n + j] : 0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = tb + u, cl = cls[u];
        const int c0 = __shfl_sync(FULL, cl, 0);
        if (__all_sync(FULL, cl == c0)) {
          if (c0 == 0) continue;
          const long long w = warp_sum8(v, lane);
          const int vi = lane >> 2, xi = vi >> 1;
          if ((lane & 3) == 0 && xi < nx) atomic_add64(&acc[((((size_t)xi * T + t) * Kc + c0 - 1) * 2 + (vi & 1)) * 2], w);
        } else if (cl) {
#pragma unroll
          for (int xi = 0; xi < PX; ++xi)
            if (xi < nx) {
              unsigned* a = &acc[(((size_t)xi * T + t) * Kc + cl - 1) * 4];
              atomic_add64(a, v[2 * xi]);
              atomic_add64(a + 2, v[2 * xi + 1]);
            }
        }
      }
    }
  }
  __syncthreads();
  const long long* sums = reinterpret_cast<const long long*>(acc);
  for (int pr = warp; pr < nx * nt; pr += PSUM_THREADS / 32) {
    const int xi = pr / nt, t = pr - xi * nt, tg = t0 + t;
    const int64_t x = x0 + xi;
    const int K = Kt[tg];
    const double tn = TN[tg];
    const bool has_new = !rc_isnan(tn);
    const int2 qx = q[x];
    double L1[8], L2p[8];
    double lane_sum = 0.0;                               // vecsum_canonical of the L2' terms (mcmc.jl:243)
#pragma unroll
    for (int qq = 0; qq < 8; ++qq) {
      const int k = lane + 1 + 32 * qq;
      L1[qq] = 0.0; L2p[qq] = 0.0;
      if (k <= K) {
        const size_t o = (size_t)tg * 256 + k - 1;
        const long long* a = sums + (((size_t)xi * T + t) * Kc + k - 1) * 2;
        const double sD = rc_dequant(a[0], qx.x), sL = rc_dequant(a[1], qx.y);
        const double sz = (double)szt[o];
        const double ai = c.alpha + c.delta1 * sz, bi = c.beta + sD;           // mcmc.jl:206-214
        const double zi = c.zeta + c.delta2 * sz, gi = c.gamma + sD;
        L1[qq] = TA[o] - ai * rc_log(bi) + (c.delta1 - 1) * sL - sz * c.lgd1;      // mcmc.jl:223-225
        L2p[qq] = TZ[o] - zi * rc_log(gi) + c.zgratio + (c.delta2 - 1) * sL - sz * c.lgd2;   // mcmc.jl:239-242
        lane_sum += L2p[qq];
      }
    }
    for (int off = 16; off; off >>= 1) lane_sum = lane_sum + __shfl_xor_sync(FULL, lane_sum, off);
    const double L2i = __shfl_sync(FULL, lane_sum, 0);
    double lp[8];
    double mx = -RC_INF;
#pragma unroll
    for (int qq = 0; qq < 8; ++qq) {
      const int k = lane + 1 + 32 * qq;
      lp[qq] = RC_NAN;
      if (k <= K) {
        const double L2 = L2i - L2p[qq];                                      // mcmc.jl:244-246
        lp[qq] = TL[(size_t)tg * 256 + k - 1] + (L1[qq] + (c.repulsion ? L2 : copysign(0.0, L2)));   // mcmc.jl:247
      } else if (k == K + 1 && has_new) {
        const double L2 = L2i - copysign(0.0, 0.0);                           // the new slot's L2' is +0
        lp[qq] = tn + (0.0 + (c.repulsion ? L2 : copysign(0.0, L2)));
      }
      if (k <= K + (has_new ? 1 : 0)) mx = lp[qq] > mx ? lp[qq] : mx;
    }
    for (int off = 16; off; off >>= 1) { const double o = __shfl_xor_sync(FULL, mx, off); mx = o > mx ? o : mx; }
    double e[8];
    double zsum = 0.0;                                   // normaliser, canonical lane order
#pragma unroll
    for (int qq = 0; qq < 8; ++qq) {
      const int k = lane + 1 + 32 * qq;
      e[qq] = 0.0;
      if (k <= K + (has_new ? 1 : 0)) { e[qq] = rc_exp(lp[qq] - mx); zsum += e[qq]; }
    }
    for (int off = 16; off; off >>= 1) zsum = zsum + __shfl_xor_sync(FULL, zsum, off);
    const double Z = __shfl_sync(FULL, zsum, 0);
    double* prow = Pb + ((size_t)x * SC + tg) * Kc;
#pragma unroll
    for (int qq = 0; qq < 8; ++qq) {
      const int k = lane + 1 + 32 * qq;
      if (k <= K) prow[k - 1] = e[qq] / Z;
      if (k == K + 1) PN[(size_t)x * SC + tg] = has_new ? e[qq] / Z : 0.0;
      if (lp_out) lp_out[((size_t)tg * m + x) * 256 + k - 1] = lp[qq];
    }
  }
}

// Thread (block of PX new points, training column j): P_s(x, c_s(j)) of the chunk's samples added in ascending order to
// the running sums in `cocl` (fp64, the output buffer); `newcl` likewise; the last chunk divides by the sample count.
__global__ void __launch_bounds__(256) k_pred_cocl(const uint8_t* __restrict__ lab, int64_t n, int64_t m, int nsc, int SC, int Kc,
                                                   const double* __restrict__ Pb, const double* __restrict__ PN,
                                                   double* __restrict__ cocl, double* __restrict__ newcl, double Stot, int last) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t x0 = (int64_t)blockIdx.y * PX;
  const int nx = (int)min((int64_t)PX, m - x0);
  if (j < n) {
    double a[PX];
#pragma unroll
    for (int xi = 0; xi < PX; ++xi) a[xi] = xi < nx ? cocl[(x0 + xi) * n + j] : 0.0;
    for (int t = 0; t < nsc; ++t) {
      const int cl = lab[(int64_t)t * n + j];
#pragma unroll
      for (int xi = 0; xi < PX; ++xi)
        if (xi < nx) a[xi] += __ldg(&Pb[((size_t)(x0 + xi) * SC + t) * Kc + cl - 1]);
    }
#pragma unroll
    for (int xi = 0; xi < PX; ++xi)
      if (xi < nx) cocl[(x0 + xi) * n + j] = last ? a[xi] / Stot : a[xi];
  }
  if (blockIdx.x == 0 && threadIdx.x < nx) {
    const int64_t x = x0 + threadIdx.x;
    double a = newcl[x];
    for (int t = 0; t < nsc; ++t) a += PN[(size_t)x * SC + t];
    newcl[x] = last ? a / Stot : a;
  }
}

PConst make_pconst(const rc_params& P) {
  PConst c;
  c.alpha = P.alpha; c.beta = P.beta; c.zeta = P.zeta; c.gamma = P.gamma; c.delta1 = P.delta1; c.delta2 = P.delta2;
  c.abratio = rc_gamma_lognorm(P.alpha, P.beta);               // mcmc.jl:17,186
  c.zgratio = rc_gamma_lognorm(P.zeta, P.gamma);                // mcmc.jl:18,187
  c.lgd1 = rc_lgamma(P.delta1);
  c.lgd2 = rc_lgamma(P.delta2);
  c.maxK = P.maxK; c.repulsion = P.repulsion ? 1 : 0;
  return c;
}

// Per-kernel device times of one call (CUDA events), printed to stderr with RCB200_VERBOSE.
struct PTimer {
  bool on = getenv("RCB200_VERBOSE") != nullptr;
  std::vector<cudaEvent_t> ev;
  void mark() { if (on) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, 0); ev.push_back(e); } }
  float span(size_t i) const { float ms = 0.f; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); return ms; }
  ~PTimer() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

// Validate Dnew (m x n host) and build its fixed-point image at each row's augmented-data scales.
int new_image(const rc_data* d, const double* Dnew, int64_t m, Bufs& B, longlong2** img, int2** qdev, PTimer& tm) {
  const int64_t n = d->n;
  double* Dn; int* bad; double2* rowmax;
  TRYP(B.get(&Dn, (size_t)m * n)); TRYP(B.get(&bad, 1)); TRYP(B.get(&rowmax, (size_t)m)); TRYP(B.get(qdev, (size_t)m));
  TRYP(B.get(img, (size_t)m * n));
  RC_CUDA(cudaMemcpy(Dn, Dnew, sizeof(double) * (size_t)m * n, cudaMemcpyHostToDevice));
  RC_CUDA(cudaMemset(bad, 0, sizeof(int)));
  tm.mark();
  k_pred_scan<<<(unsigned)m, 256>>>(Dn, n, bad, rowmax);
  tm.mark();
  RC_CUDA(cudaGetLastError());
  int hbad = 0;
  std::vector<double2> hm((size_t)m);
  RC_CUDA(cudaMemcpy(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost));
  if (hbad) { rc_set_error(RC_DOMAIN_MSG); return RC_ERR_DOMAIN; }
  RC_CUDA(cudaMemcpy(hm.data(), rowmax, sizeof(double2) * (size_t)m, cudaMemcpyDeviceToHost));
  std::vector<int2> hq((size_t)m);
  for (int64_t x = 0; x < m; ++x) {
    hq[x].x = rc_choose_q(std::max(d->mD, hm[x].x), n + 1);   // scales of the augmented data, n + 1 points
    hq[x].y = rc_choose_q(std::max(d->mL, hm[x].y), n + 1);
    if (hq[x].x == RC_Q_NONE || hq[x].y == RC_Q_NONE) { rc_set_error("dissimilarities too large for the fixed-point image."); return RC_ERR_DOMAIN; }
  }
  RC_CUDA(cudaMemcpy(*qdev, hq.data(), sizeof(int2) * (size_t)m, cudaMemcpyHostToDevice));
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, d->device);
  tm.mark();
  k_pred_image<<<nsm * 8, 256>>>(Dn, m, n, *qdev, *img);
  tm.mark();
  RC_CUDA(cudaGetLastError());
  return RC_OK;
}

// The chunked pipeline over S device-resident samples (labels S x n bytes 1..K_s, r, p), Kmax = max K_s.
int predict_core(const rc_data* d, const rc_params& P, const longlong2* img, const int2* q, int64_t m, const uint8_t* lab,
                 const double* r, const double* p, int64_t S, int Kmax, double* cocl_out, double* newcl_out, double* lp_out, Bufs& B,
                 PTimer& tm) {
  const int64_t n = d->n;
  if (S == 0) {                                          // (1/S) sum over no samples: NaN, as rc_sampler_psm
    std::fill(cocl_out, cocl_out + (size_t)m * n, RC_NAN);
    std::fill(newcl_out, newcl_out + (size_t)m, RC_NAN);
    return RC_OK;
  }
  const int Kc = std::max(Kmax, 1);
  const int T = std::max(1, std::min(PT_MAX, (int)(PSMEM_BUDGET / ((size_t)PX * Kc * 16))));
  const size_t smem = (size_t)PX * T * Kc * 16;
  const int64_t per_T = (int64_t)(PCHUNK_BYTES / ((size_t)m * T * Kc * 8));
  int64_t SC = std::min<int64_t>((S + T - 1) / T * T, (int64_t)T * std::max<int64_t>(1, std::min<int64_t>(per_T, 4096)));
  if (const char* e = getenv("RCB200_PREDICT_CHUNK")) SC = std::min<int64_t>(SC, std::max(1, atoi(e)));   // smaller chunks: same bits
  double *cocl, *newcl, *Pb, *PN, *TA, *TZ, *TL, *TN, *lpd = nullptr;
  int *Kt, *szt;
  TRYP(B.get(&cocl, (size_t)m * n)); TRYP(B.get(&newcl, (size_t)m));
  TRYP(B.get(&Pb, (size_t)m * SC * Kc)); TRYP(B.get(&PN, (size_t)m * SC));
  TRYP(B.get(&TA, (size_t)SC * 256)); TRYP(B.get(&TZ, (size_t)SC * 256)); TRYP(B.get(&TL, (size_t)SC * 256));
  TRYP(B.get(&TN, (size_t)SC)); TRYP(B.get(&Kt, (size_t)SC)); TRYP(B.get(&szt, (size_t)SC * 256));
  if (lp_out) TRYP(B.get(&lpd, (size_t)SC * m * 256));
  int* bad;
  TRYP(B.get(&bad, 1));
  RC_CUDA(cudaMemset(bad, 0, sizeof(int)));
  k_pred_check<<<148 * 4, 256>>>(lab, (size_t)S * n, Kc, bad);
  int hbad = 0;
  RC_CUDA(cudaMemcpy(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost));
  if (hbad) { rc_set_error("sample labels outside 1..%d (the largest K of the samples)", Kc); return RC_ERR_STATE; }
  RC_CUDA(cudaMemset(cocl, 0, sizeof(double) * (size_t)m * n));
  RC_CUDA(cudaMemset(newcl, 0, sizeof(double) * (size_t)m));
  RC_CUDA(cudaFuncSetAttribute(k_pred_sums, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const PConst c = make_pconst(P);
  for (int64_t s0 = 0; s0 < S; s0 += SC) {
    const int nsc = (int)std::min<int64_t>(SC, S - s0);
    const uint8_t* L = lab + (size_t)s0 * n;
    tm.mark();
    k_pred_terms<<<nsc, 256>>>(L, n, r + s0, p + s0, c, Kt, szt, TA, TZ, TL, TN);
    tm.mark();
    k_pred_sums<<<dim3((unsigned)((m + PX - 1) / PX), (unsigned)((nsc + T - 1) / T)), PSUM_THREADS, smem>>>(
        img, q, m, n, L, nsc, (int)SC, T, Kc, Kt, szt, TA, TZ, TL, TN, c, Pb, PN, lpd);
    tm.mark();
    k_pred_cocl<<<dim3((unsigned)((n + 255) / 256), (unsigned)((m + PX - 1) / PX)), 256>>>(
        L, n, m, nsc, (int)SC, Kc, Pb, PN, cocl, newcl, (double)S, s0 + nsc == S);
    tm.mark();
    RC_CUDA(cudaGetLastError());
    if (lpd) RC_CUDA(cudaMemcpy(lp_out + (size_t)s0 * m * 256, lpd, sizeof(double) * (size_t)nsc * m * 256, cudaMemcpyDeviceToHost));
  }
  RC_CUDA(cudaMemcpy(cocl_out, cocl, sizeof(double) * (size_t)m * n, cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(newcl_out, newcl, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost));
  if (tm.on) {                                           // events: scan, image, then (terms, sums, cocl) per chunk
    float t[5] = {tm.span(0), tm.span(2), 0.f, 0.f, 0.f};
    for (size_t i = 4; i + 3 < tm.ev.size(); i += 4) { t[2] += tm.span(i); t[3] += tm.span(i + 1); t[4] += tm.span(i + 2); }
    fprintf(stderr, "[rcb200] rc_predict m=%lld n=%lld S=%lld K=%d T=%d chunk=%lld (CUDA events, ms): k_pred_scan %.4f k_pred_image %.4f "
            "k_pred_terms %.4f k_pred_sums %.4f k_pred_cocl %.4f\n", (long long)m, (long long)n, (long long)S, Kc, T, (long long)SC,
            t[0], t[1], t[2], t[3], t[4]);
  }
  return RC_OK;
}

int check_rp(const double* r, const double* p, int64_t S) {
  for (int64_t s = 0; s < S; ++s) {
    if (!(r[s] > 0.0) || !(r[s] < RC_INF)) { rc_set_error("r must be positive and finite (sample %lld)", (long long)s); return RC_ERR_ARG; }
    if (!(p[s] > 0.0 && p[s] < 1.0)) { rc_set_error("p must lie in (0, 1) (sample %lld)", (long long)s); return RC_ERR_ARG; }
  }
  return RC_OK;
}

}  // namespace

extern "C" {

int32_t rc_predict(const rc_data* d, const rc_params* par, const double* Dnew, int64_t m, const int64_t* labels, const double* r,
                   const double* p, int64_t S, double* cocl_out, double* newcl_out, double* lp_out) {
  if (!d || !par || !Dnew || !cocl_out || !newcl_out || m < 1 || S < 0 || (S > 0 && (!labels || !r || !p))) {
    rc_set_error("rc_predict: null pointer or bad size"); return RC_ERR_ARG;
  }
  TRYP(check_rp(r, p, S));
  TRYP(rc_select_device(d->device));
  Bufs B;
  uint8_t* dl = nullptr; std::vector<int> K;
  if (S > 0) TRYP(upload_labels(labels, S, d->n, B, &dl, K));
  PTimer tm;
  longlong2* img; int2* q;
  TRYP(new_image(d, Dnew, m, B, &img, &q, tm));
  double *dr, *dp;
  TRYP(B.get(&dr, (size_t)S)); TRYP(B.get(&dp, (size_t)S));
  if (S > 0) {
    RC_CUDA(cudaMemcpy(dr, r, sizeof(double) * (size_t)S, cudaMemcpyHostToDevice));
    RC_CUDA(cudaMemcpy(dp, p, sizeof(double) * (size_t)S, cudaMemcpyHostToDevice));
  }
  const int Kmax = K.empty() ? 1 : *std::max_element(K.begin(), K.end());
  return predict_core(d, *par, img, q, m, dl, dr, dp, S, Kmax, cocl_out, newcl_out, lp_out, B, tm);
}

int32_t rc_sampler_predict(const rc_sampler* s, const double* Dnew, int64_t m, int64_t chain0, int64_t nch, double* cocl_out,
                           double* newcl_out) {
  if (!s || !Dnew || !cocl_out || !newcl_out || m < 1) { rc_set_error("rc_sampler_predict: null pointer or bad size"); return RC_ERR_ARG; }
  rc_sample_range v;
  TRYP(rc_sampler_range(s, chain0, nch, "rc_sampler_predict", v));
  Bufs B;
  PTimer tm;
  longlong2* img; int2* q;
  TRYP(new_image(v.d, Dnew, m, B, &img, &q, tm));
  std::vector<int> K((size_t)v.R);
  if (v.R > 0) RC_CUDA(cudaMemcpy(K.data(), v.K, sizeof(int) * (size_t)v.R, cudaMemcpyDeviceToHost));
  const int Kmax = K.empty() ? 1 : *std::max_element(K.begin(), K.end());
  if (Kmax > RC_MAXCAP_INC) { rc_set_error("rc_sampler_predict: recorded K = %d exceeds %d", Kmax, RC_MAXCAP_INC); return RC_ERR_STATE; }
  return predict_core(v.d, v.par, img, q, m, v.labels, v.r, v.p, v.R, Kmax, cocl_out, newcl_out, nullptr, B, tm);
}

int32_t rc_crossdist(const double* X, int64_t n, const double* Y, int64_t m, int64_t dim, int32_t device, double* out) {
  if (!X || !Y || !out || n < 1 || m < 1 || dim < 1) { rc_set_error("rc_crossdist: null pointer or empty input"); return RC_ERR_ARG; }
  std::vector<double> XY((size_t)(n + m) * dim);
  std::memcpy(XY.data(), X, sizeof(double) * (size_t)n * dim);
  std::memcpy(XY.data() + (size_t)n * dim, Y, sizeof(double) * (size_t)m * dim);
  TRYP(rc_select_device(device));
  Bufs B;
  double* rows;
  TRYP(B.get(&rows, (size_t)m * (n + m)));
  TRYP(rc_distm_rows_dev(XY.data(), dim, n + m, n, m, device, rows));   // rows n.. of the stacked points' matrix
  RC_CUDA(cudaMemcpy2D(out, sizeof(double) * (size_t)n, rows, sizeof(double) * (size_t)(n + m), sizeof(double) * (size_t)n, (size_t)m,
                       cudaMemcpyDeviceToHost));
  return RC_OK;
}

}  // extern "C"
