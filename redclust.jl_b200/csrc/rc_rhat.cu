// rc_rhat.cu -- convergence across chains from the co-clustering counts (no reference equivalent; the reference's
// diagnostics are per chain, src/mcmc.jl:564-573).  Cluster labels switch between chains, but the co-clustering
// indicator [c(a) = c(b)] of a point pair does not, so its split-R-hat (BDA3 section 11.4) compares chains.
//
// C chains of S samples, L = floor(S / 2): chain c gives group 2c = samples [0, L) and group 2c + 1 = samples [S - L, S)
// (the middle sample of an odd S is dropped), m = 2C groups.  For a pair a < b, N_g counts the samples of group g in
// which a and b share a label, and with N = sum_g N_g, Q = sum_g N_g^2 (exact int64):
//   Wn = L N - Q,  Bn = m Q - N^2,
//   R  = sqrt((L-1)/L + ((L-1) Bn) / ((m-1) L Wn))  for Wn > 0;  1 for Wn = Bn = 0;  +Inf for Wn = 0 < Bn,
// which is BDA3's sqrt(var+ / W) for a 0/1 variable.  Chain deviation from the pooled PSM: d_ab = |m N_c - 2 N| with
// N_c = N_2c + N_2c+1, so that p_c - pbar = +-d / (2 m L); meandev[c] = sum d / (2 m L C(n, 2)), maxdev[c] = max d / (2 m L).
//
//   pass 1  N: psm_counts_device over every sample of the range, minus the counts of the C middle samples for odd S
//   pass 2  per chain: the counts of its two halves, then k_rhat_acc over the upper triangle (Q, sum d, max d)
//   finish  k_rhat_finish: R per pair, the optional n x n matrix, per-CTA max / argmax / count above 1.01
//
// Bounds (rhat_check_args): 2 <= n <= 65 535 and m L < 2^31, so N^2, m Q and L N are below 2^62 and d < 2^32,
// sum d < 2^63.  Everything is an integer until the final divisions: results do not depend on tiling, grid or atomic order.
#include <cmath>
#include <cstdlib>
#include "rc_common.cuh"
#include "rc_labels.h"

namespace {

#define RT 256   // threads per CTA of the two triangle kernels

__global__ void k_sub_counts(int* __restrict__ N, const int* __restrict__ M, size_t total) {
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) N[t] -= M[t];
}

// CTA i walks rows i and n - 1 - i of the strict upper triangle (n - 1 pairs per CTA, (n + 1) / 2 CTAs); lane-contiguous b.
// Bytes per pair: the two halves' counts (4 + 4), the pooled N (4), Q read and written (8 + 8) = 28.
__global__ void __launch_bounds__(RT) k_rhat_acc(const int* __restrict__ Na, const int* __restrict__ Nb, const int* __restrict__ N,
                                                 long long* __restrict__ Q, int64_t n, long long m, unsigned long long* __restrict__ dsum,
                                                 unsigned long long* __restrict__ dmax) {
  unsigned long long s = 0, mx = 0;
  for (int h = 0; h < 2; ++h) {
    const int64_t a = h ? n - 1 - (int64_t)blockIdx.x : (int64_t)blockIdx.x;
    if (h && a == (int64_t)blockIdx.x) break;
    const int64_t row = a * n;
    for (int64_t b = a + 1 + threadIdx.x; b < n; b += RT) {
      const long long x = Na[row + b], y = Nb[row + b];
      Q[row + b] += x * x + y * y;
      const long long e = m * (x + y) - 2LL * (long long)N[row + b];
      const unsigned long long d = (unsigned long long)(e < 0 ? -e : e);
      s += d;
      mx = d > mx ? d : mx;
    }
  }
  __shared__ unsigned long long rs[RT / 32], rm[RT / 32];
  for (int off = 16; off; off >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, off);
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, mx, off);
    mx = o > mx ? o : mx;
  }
  if ((threadIdx.x & 31) == 0) { rs[threadIdx.x >> 5] = s; rm[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < RT / 32; ++w) { s += rs[w]; mx = rm[w] > mx ? rm[w] : mx; }
    if (s) atomicAdd(dsum, s);
    if (mx) atomicMax(dmax, mx);
  }
}

// (v, i) beats (w, j): larger value, then smaller pair index
__device__ __forceinline__ bool beats(double v, long long i, double w, long long j) { return v > w || (v == w && i < j); }

// R of every pair a < b from N and Q; R_out (may be NULL) gets the symmetric n x n matrix with a unit diagonal.  Per CTA:
// the largest R with its row-major pair index a n + b (-1 and INT64_MAX when the CTA has no pair) and the count above 1.01.
__global__ void __launch_bounds__(RT) k_rhat_finish(const int* __restrict__ N, const long long* __restrict__ Q, int64_t n, long long L,
                                                    long long m, double* __restrict__ R_out, double* __restrict__ cta_max,
                                                    long long* __restrict__ cta_idx, long long* __restrict__ cta_above) {
  double best = -1.0;
  long long bi = 0x7fffffffffffffffLL, above = 0;
  for (int h = 0; h < 2; ++h) {
    const int64_t a = h ? n - 1 - (int64_t)blockIdx.x : (int64_t)blockIdx.x;
    if (h && a == (int64_t)blockIdx.x) break;
    const int64_t row = a * n;
    if (R_out && threadIdx.x == 0) R_out[row + a] = 1.0;
    for (int64_t b = a + 1 + threadIdx.x; b < n; b += RT) {
      const long long Nv = N[row + b], Qv = Q[row + b];
      const long long Wn = L * Nv - Qv, Bn = m * Qv - Nv * Nv;
      double r;
      if (Wn > 0) r = sqrt((double)(L - 1) / (double)L + ((double)(L - 1) * (double)Bn) / ((double)(m - 1) * (double)L * (double)Wn));
      else r = Bn == 0 ? 1.0 : INFINITY;
      if (R_out) { R_out[row + b] = r; R_out[b * n + a] = r; }
      above += r > 1.01;
      if (beats(r, row + b, best, bi)) { best = r; bi = row + b; }
    }
  }
  __shared__ double sv[RT / 32];
  __shared__ long long si[RT / 32], sa[RT / 32];
  for (int off = 16; off; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, off);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, off);
    if (beats(ov, oi, best, bi)) { best = ov; bi = oi; }
    above += __shfl_xor_sync(0xffffffffu, above, off);
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; sa[threadIdx.x >> 5] = above; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < RT / 32; ++w) {
      if (beats(sv[w], si[w], best, bi)) { best = sv[w]; bi = si[w]; }
      above += sa[w];
    }
    cta_max[blockIdx.x] = best; cta_idx[blockIdx.x] = bi; cta_above[blockIdx.x] = above;
  }
}

struct Timer {            // CUDA events on the legacy stream, only with RCB200_VERBOSE
  bool on = getenv("RCB200_VERBOSE") != nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  Timer() { if (on) { cudaEventCreate(&e0); cudaEventCreate(&e1); } }
  ~Timer() { if (on) { cudaEventDestroy(e0); cudaEventDestroy(e1); } }
  void start() { if (on) cudaEventRecord(e0, 0); }
  float stop() {
    if (!on) return 0.f;
    float ms = 0; cudaEventRecord(e1, 0); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
    return ms;
  }
};

}  // namespace

int rhat_check_args(int64_t C, int64_t S, int64_t n, const char* who) {
  const int64_t L = S / 2;
  const int64_t lim = (int64_t)1 << 31;
  if (C < 1 || S < 4 || n < 2 || n > 65535 || C >= lim || S >= lim || 2 * C * L >= lim || C * S >= lim) {
    rc_set_error("%s: needs at least one chain, S >= 4 samples per chain, 2 <= n <= 65535 and fewer than 2^31 samples "
                 "(chains = %lld, S = %lld, n = %lld)", who, (long long)C, (long long)S, (long long)n);
    return RC_ERR_ARG;
  }
  return RC_OK;
}

// Device buffers of one call (Cl local chains): N, Q, the two halves' counts, the per-chain {sum d, max d}, and the matrix
// when asked for.  Refuses with the sizes when they and the largest counts call's transposed labels do not fit the free memory.
int rhat_alloc(int64_t Cl, int64_t S, int64_t n, bool matrix, Bufs& B, RhatDev& d, const char* who) {
  const double nn = (double)n * (double)n, GB = 1e9;
  const int64_t R = Cl * S, odd = S & 1;
  const double cN = 4 * nn, cH = 8 * nn, cQ = 8 * nn, cM = matrix ? 8 * nn : 0.0;
  const double lt = (double)n * (double)((R + 63) & ~63LL) + (odd ? 4 * nn + (double)n * (double)(((Cl + 63) & ~63LL) + Cl) : 0.0);
  const double need = cN + cH + cQ + cM + lt;
  size_t free_b = 0, total_b = 0;
  RC_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (need > (double)free_b) {
    rc_set_error("%s: needs %.2f GB of device memory (pooled counts %.2f GB, the two halves' counts %.2f GB, Q %.2f GB, "
                 "transposed labels%s %.2f GB, R matrix %.2f GB); %.2f GB are free", who, need / GB, cN / GB, cH / GB, cQ / GB,
                 odd ? " and middle-sample counts" : "", lt / GB, cM / GB, (double)free_b / GB);
    return RC_ERR_CUDA;
  }
  TRYP(B.get(&d.N, (size_t)(n * n))); TRYP(B.get(&d.Q, (size_t)(n * n)));
  TRYP(B.get(&d.Na, (size_t)(n * n))); TRYP(B.get(&d.Nb, (size_t)(n * n)));
  TRYP(B.get(&d.dev, 2 * (size_t)Cl));
  d.R = nullptr;
  if (matrix) TRYP(B.get(&d.R, (size_t)(n * n)));
  RC_CUDA(cudaMemset(d.Q, 0, sizeof(long long) * (size_t)(n * n)));
  RC_CUDA(cudaMemset(d.dev, 0, sizeof(unsigned long long) * 2 * (size_t)Cl));
  return RC_OK;
}

// Pass 1: the pooled counts N of the split halves of Cl chains (sample-major device labels L, chain-major).
int rhat_pass1(const uint8_t* L, int64_t Cl, int64_t S, int64_t n, RhatDev& d, RhatTimes& t) {
  Timer tm;
  tm.start();
  {
    Bufs B;
    TRYP(psm_counts_device(L, Cl * S, n, d.N, B));
  }
  if (S & 1) {                                      // subtract the C middle samples, gathered into one buffer
    Bufs B;
    uint8_t* mid; int* Nm;
    TRYP(B.get(&mid, (size_t)(Cl * n))); TRYP(B.get(&Nm, (size_t)(n * n)));
    RC_CUDA(cudaMemcpy2DAsync(mid, (size_t)n, L + (S / 2) * n, (size_t)(S * n), (size_t)n, (size_t)Cl, cudaMemcpyDeviceToDevice, 0));
    TRYP(psm_counts_device(mid, Cl, n, Nm, B));
    k_sub_counts<<<148 * 8, 256>>>(d.N, Nm, (size_t)(n * n));
    RC_CUDA(cudaGetLastError());
    RC_CUDA(cudaDeviceSynchronize());
  }
  t.pass1_ms = tm.stop();
  return RC_OK;
}

// Pass 2: for each of the Cl chains, the counts of its two halves and one k_rhat_acc over the upper triangle against the
// pooled N of m groups in all: Q += N_2c^2 + N_2c+1^2, and chain c's {sum d, max d} in d.dev[2c], d.dev[2c + 1].
int rhat_pass2(const uint8_t* L, int64_t Cl, int64_t S, int64_t n, int64_t m, RhatDev& d, RhatTimes& t) {
  const int64_t Lh = S / 2;
  Timer tc, ta;
  for (int64_t c = 0; c < Cl; ++c) {
    tc.start();
    {
      Bufs B;
      TRYP(psm_counts_device(L + c * S * n, Lh, n, d.Na, B));
      TRYP(psm_counts_device(L + (c * S + S - Lh) * n, Lh, n, d.Nb, B));
    }
    t.pass2_counts_ms += tc.stop();
    ta.start();
    k_rhat_acc<<<(unsigned)((n + 1) / 2), RT>>>(d.Na, d.Nb, d.N, d.Q, n, (long long)m, d.dev + 2 * c, d.dev + 2 * c + 1);
    RC_CUDA(cudaGetLastError());
    t.acc_ms += ta.stop();
  }
  RC_CUDA(cudaDeviceSynchronize());
  return RC_OK;
}

// R from N and Q of m groups of L = S / 2 samples: the summary (and the matrix into rhat_out when both are non-NULL).
int rhat_finish(const RhatDev& d, int64_t S, int64_t n, int64_t m, rc_rhat_summary* sum, double* rhat_out, RhatTimes& t) {
  const unsigned ncta = (unsigned)((n + 1) / 2);
  Bufs B;
  double* cmax; long long *cidx, *cab;
  TRYP(B.get(&cmax, ncta)); TRYP(B.get(&cidx, ncta)); TRYP(B.get(&cab, ncta));
  Timer tm;
  tm.start();
  k_rhat_finish<<<ncta, RT>>>(d.N, d.Q, n, (long long)(S / 2), (long long)m, rhat_out ? d.R : nullptr, cmax, cidx, cab);
  RC_CUDA(cudaGetLastError());
  t.finish_ms = tm.stop();
  std::vector<double> hmax(ncta);
  std::vector<long long> hidx(ncta), hab(ncta);
  RC_CUDA(cudaMemcpy(hmax.data(), cmax, sizeof(double) * ncta, cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(hidx.data(), cidx, sizeof(long long) * ncta, cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(hab.data(), cab, sizeof(long long) * ncta, cudaMemcpyDeviceToHost));
  double best = -1.0;
  long long bi = 0x7fffffffffffffffLL, above = 0;
  for (unsigned q = 0; q < ncta; ++q) {
    if (hmax[q] > best || (hmax[q] == best && hidx[q] < bi)) { best = hmax[q]; bi = hidx[q]; }
    above += hab[q];
  }
  if (sum) { sum->max = best; sum->a = bi / n; sum->b = bi % n; sum->above = above; }
  if (rhat_out) RC_CUDA(cudaMemcpy(rhat_out, d.R, sizeof(double) * (size_t)(n * n), cudaMemcpyDeviceToHost));
  return RC_OK;
}

// meandev / maxdev (each may be NULL) of C chains from their {sum d, max d} (host, 2 per chain).
void rhat_deviations(const unsigned long long* dev, int64_t C, int64_t S, int64_t n, int64_t m, double* meandev, double* maxdev) {
  const int64_t twomL = 2 * m * (S / 2), pairs = n * (n - 1) / 2;
  for (int64_t c = 0; c < C; ++c) {
    if (meandev) meandev[c] = (double)dev[2 * c] / ((double)twomL * (double)pairs);
    if (maxdev) maxdev[c] = (double)dev[2 * c + 1] / (double)twomL;
  }
}

void rhat_report(const RhatTimes& t, int64_t C, int64_t S, int64_t n) {
  if (!getenv("RCB200_VERBOSE")) return;
  const double pairs = 0.5 * (double)n * (double)(n - 1), bytes = 28.0 * pairs * (double)C;
  fprintf(stderr, "[rcb200] cocl rhat: n=%lld chains=%lld S=%lld pass1 %.3f ms, pass2 counts %.3f ms, k_rhat_acc %.3f ms "
                  "(%.3e B, %.1f %% of 7.7 TB/s), k_rhat_finish %.3f ms\n", (long long)n, (long long)C, (long long)S, t.pass1_ms,
          t.pass2_counts_ms, t.acc_ms, bytes, t.acc_ms > 0 ? 100.0 * bytes / (t.acc_ms * 1e-3) / 7.7e12 : 0.0, t.finish_ms);
}

// Passes 1 and 2, the finish and the deviations of the Cl chains of device labels L (every chain of the call).
static int rhat_device(const uint8_t* L, int64_t C, int64_t S, int64_t n, rc_rhat_summary* sum, double* rhat_out, double* meandev,
                       double* maxdev, const char* who) {
  Bufs B;
  RhatDev d;
  RhatTimes t;
  TRYP(rhat_alloc(C, S, n, rhat_out != nullptr, B, d, who));
  TRYP(rhat_pass1(L, C, S, n, d, t));
  TRYP(rhat_pass2(L, C, S, n, 2 * C, d, t));
  TRYP(rhat_finish(d, S, n, 2 * C, sum, rhat_out, t));
  std::vector<unsigned long long> dev(2 * (size_t)C);
  RC_CUDA(cudaMemcpy(dev.data(), d.dev, sizeof(unsigned long long) * dev.size(), cudaMemcpyDeviceToHost));
  rhat_deviations(dev.data(), C, S, n, 2 * C, meandev, maxdev);
  rhat_report(t, C, S, n);
  return RC_OK;
}

extern "C" {

int32_t rc_cocl_rhat(const int64_t* labels, int64_t nchains, int64_t S, int64_t n, int32_t device, rc_rhat_summary* sum,
                     double* rhat_out, double* meandev, double* maxdev) {
  if (!labels) { rc_set_error("rc_cocl_rhat: null pointer"); return RC_ERR_ARG; }
  TRYP(rhat_check_args(nchains, S, n, "rc_cocl_rhat"));
  TRYP(rc_select_device(device));
  Bufs B;
  uint8_t* dL; std::vector<int> K;
  TRYP(upload_labels(labels, nchains * S, n, B, &dL, K));
  return rhat_device(dL, nchains, S, n, sum, rhat_out, meandev, maxdev, "rc_cocl_rhat");
}

int32_t rc_sampler_cocl_rhat(const rc_sampler* s, int64_t chain0, int64_t nch, rc_rhat_summary* sum, double* rhat_out,
                             double* meandev, double* maxdev) {
  if (!s) { rc_set_error("rc_sampler_cocl_rhat: null handle"); return RC_ERR_ARG; }
  rc_sample_range v;
  TRYP(rc_sampler_range(s, chain0, nch, "rc_sampler_cocl_rhat", v));
  const int64_t S = rc_sampler_numsamples(s);
  TRYP(rhat_check_args(nch, S, v.n, "rc_sampler_cocl_rhat"));
  return rhat_device(v.labels, nch, S, v.n, sum, rhat_out, meandev, maxdev, "rc_sampler_cocl_rhat");
}

}  // extern "C"
