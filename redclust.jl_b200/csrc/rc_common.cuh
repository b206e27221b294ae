// rc_common.cuh -- shared declarations of the sm_100a implementation (internal, not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <algorithm>
#include "../../include/rcb200.h"
#include "rc_math.h"
#include "rc_rng.h"

// ---- error plumbing ----------------------------------------------------------------------------
void rc_set_error(const char* fmt, ...);
int rc_select_device(int32_t device);   // rc_data.cu
// Device memory of the long-lived handles comes from the device's stream-ordered pool with a bounded release
// threshold (32 GB, RCB200_POOL_KEEP_GB): a destroyed handle's gigabytes are reused by the next one instead of going back
// to the driver (RCB200_NO_POOL=1: plain cudaMalloc / cudaFree).
cudaError_t rc_dev_malloc(void** p, size_t bytes);
void rc_dev_free(void* p);
#define RC_CUDA(call)                                                                          \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      rc_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__,     \
                   cudaGetErrorString(e_));                                                    \
      return RC_ERR_CUDA;                                                                      \
    }                                                                                          \
  } while (0)

#define TRYP(x) do { int st_ = (x); if (st_) return st_; } while (0)

// Device buffers of one call, released on every return path.
struct Bufs {
  std::vector<void*> p;
  template <class T> int get(T** out, size_t count) {
    *out = nullptr;
    cudaError_t e = cudaMalloc((void**)out, sizeof(T) * std::max<size_t>(count, 1));
    if (e != cudaSuccess) { (void)cudaGetLastError(); rc_set_error("out of device memory (%zu bytes)", sizeof(T) * count); return RC_ERR_CUDA; }
    p.push_back(*out);
    return RC_OK;
  }
  ~Bufs() { for (void* q : p) cudaFree(q); }
};

// The recorded samples of chains [chain0, chain0 + nch) of a sampler, on its device (rc_api.cu): R = nch * numsamples
// label vectors of n bytes (1..K, chain-major, sample-minor) and their K, r, p, with the sampler's data and hyperparameters.
struct rc_sample_range {
  const rc_data* d;
  rc_params par;
  const uint8_t* labels;
  const int* K;
  const double *r, *p;
  int64_t R, n;
};
// Selects the sampler's device and fills v.  A range outside the chains: RC_ERR_ARG; a run that has not reached numiters
// (the samples are not all recorded): RC_ERR_STATE; a chain of the range that stopped at the slot capacity: RC_ERR_SLOTS.
int rc_sampler_range(const rc_sampler* s, int64_t chain0, int64_t nch, const char* who, rc_sample_range& v);

// pairwise Euclidean distances on the FP64 tensor cores (rc_gram.cu): X_dev n x dim row-major -> rows [row0, row0 + nrows) in D_dev (nrows x n)
int rc_distm_dmma(const double* X_dev, int64_t dim, int64_t n, int64_t row0, int64_t nrows, double* D_dev);
// int32 co-clustering counts on the device -> host fp64 counts / denom (rc_post.cu)
int rc_counts_to_host_psm(const int* counts, size_t total, double denom, double* out);
// co-clustering counts of R device label vectors (sample-major) into counts (n x n int32), rc_post.cu.  The transposed
// labels live in B; Lt (may be NULL) receives them for binder_wp.
int psm_counts_device(const uint8_t* L, int64_t R, int64_t n, int* counts, Bufs& B, const uint8_t** Lt = nullptr);
// posterior expected Binder loss from the counts (rc_post.cu): the sample and size limits, W and P of R label vectors (L and
// its transpose Lt from psm_counts_device) against counts of at most nmax samples, and the exact totals
// T_s = S P_s + sum_t P_t - 2 W_s with their first argmin
int rc_binder_check_args(int64_t S, int64_t n, const char* who);
int binder_wp(const uint8_t* L, const uint8_t* Lt, int64_t R, int64_t n, const int* counts, int64_t nmax, unsigned long long* W_out,
              unsigned long long* P_out, float* w_ms);
int rc_binder_finish(const unsigned long long* W, const unsigned long long* P, int64_t S, int64_t n, double* loss_sums,
                     int64_t* best, int64_t* totals);

// distances from reference partitions to samples (rc_post.cu).  PartitionRefs: the references relabelled and uploaded
// (bytes nref x n, their K, the largest K) with the loss code, after the argument checks of the entry points.  PairLaunch:
// the launch geometry of k_pair_loss; pair_geometry checks that a krow x kcol table fits the shared memory (RC_ERR_SLOTS,
// no device work), pair_nlogn fills its N log N table.  sample_K: the K of S device samples on the host and their largest.
// partition_dists_run: dist (nref x S fp64) and pairs (NULL or nref x S int64, exact Binder counts) of the references
// against S device samples (bytes 1..K, device K) into device buffers.
struct PartitionRefs {
  uint8_t* L;
  int* K;
  int kmax;
  int64_t nref;
  int loss;
};
struct PairLaunch {
  int wide, tabwords, stride;
  size_t smem;
  double* nlogn;
};
int partition_refs(const int64_t* refs, int64_t nref, int64_t n, int32_t loss, const void* dist_out, const char* who, Bufs& B,
                   PartitionRefs& r);
int pair_geometry(int64_t n, int krow, int kcol, const char* who, PairLaunch& p);
int pair_nlogn(int64_t n, Bufs& B, PairLaunch& p);
int sample_K(const int* Kd, int64_t S, std::vector<int>& Kh, int* kmax);
int partition_dists_run(const PartitionRefs& r, const PairLaunch& p, const uint8_t* L, const int* Kd, int64_t S, int64_t n, double* dist,
                        long long* pairs);

// allocation probabilities to the clusters of an estimate (rc_align.cu).  AlignEstimate: the estimate relabelled and uploaded
// (bytes 1..K, n points), after align_estimate's checks (more than 255 clusters: RC_ERR_SLOTS).  align_check: 1 <= S < 2^31
// pooled samples (RC_ERR_ARG) and the table of the estimate against the samples' largest K (pair_geometry).  AlignDev: the
// device results of R samples (counts n x (K + 1) int32, maps R x 256 bytes with sigma_t(l) at [t][l - 1], matched R
// int64); align_alloc refuses them, plus extra_bytes of the caller's own buffers (named extra_what), when they do not fit
// the free device memory, with their sizes.  align_run: zeroes the counts, then k_align_match and k_align_count over R
// device samples L (bytes 1..K, K on the device in Kd).
struct AlignEstimate {
  uint8_t* L;
  int K;
  int64_t n;
};
struct AlignDev {
  int* counts;
  uint8_t* maps;
  long long* matched;
};
int align_estimate(const int64_t* estimate, int64_t n, const char* who, Bufs& B, AlignEstimate& e);
int align_check(const AlignEstimate& e, int64_t S, int kmax, const char* who, PairLaunch& p);
int align_alloc(const AlignEstimate& e, int64_t R, double extra_bytes, const char* extra_what, const char* who, Bufs& B, AlignDev& d);
int align_run(const AlignEstimate& e, const PairLaunch& p, const uint8_t* L, const int* Kd, int64_t R, AlignDev& d);

// split-R-hat of the co-clustering indicators (rc_rhat.cu).  The limits on chains, samples per chain and n; the device
// buffers of one call (N the pooled counts, Q = sum of squared group counts, Na / Nb one chain's halves, dev = {sum d,
// max d} per local chain, R the matrix or NULL); pass 1 (N), pass 2 (Q and dev against the N of m groups in all), the
// finish (summary, matrix) and the deviations from the host copy of dev.  RhatTimes: CUDA-event times with RCB200_VERBOSE.
struct RhatDev {
  int *N, *Na, *Nb;
  long long* Q;
  unsigned long long* dev;
  double* R;
};
struct RhatTimes { float pass1_ms = 0, pass2_counts_ms = 0, acc_ms = 0, finish_ms = 0; };
int rhat_check_args(int64_t C, int64_t S, int64_t n, const char* who);
int rhat_alloc(int64_t Cl, int64_t S, int64_t n, bool matrix, Bufs& B, RhatDev& d, const char* who);
int rhat_pass1(const uint8_t* L, int64_t Cl, int64_t S, int64_t n, RhatDev& d, RhatTimes& t);
int rhat_pass2(const uint8_t* L, int64_t Cl, int64_t S, int64_t n, int64_t m, RhatDev& d, RhatTimes& t);
int rhat_finish(const RhatDev& d, int64_t S, int64_t n, int64_t m, rc_rhat_summary* sum, double* rhat_out, RhatTimes& t);
void rhat_deviations(const unsigned long long* dev, int64_t C, int64_t S, int64_t n, int64_t m, double* meandev, double* maxdev);
void rhat_report(const RhatTimes& t, int64_t C, int64_t S, int64_t n);

// ---- 128-bit two's complement accumulators (block totals of the fixed-point images) ------------
struct rc_i128 {
  unsigned long long lo;
  long long hi;
};
__host__ __device__ __forceinline__ void rc_add128(rc_i128& a, long long s) {
  unsigned long long lo = a.lo + (unsigned long long)s;
  a.hi += (s < 0 ? -1LL : 0LL) + (lo < a.lo ? 1LL : 0LL);
  a.lo = lo;
}
__host__ __device__ __forceinline__ void rc_add128(rc_i128& a, const rc_i128& b) {
  unsigned long long lo = a.lo + b.lo;
  a.hi += b.hi + (lo < a.lo ? 1LL : 0LL);
  a.lo = lo;
}
__host__ __device__ __forceinline__ void rc_sub128(rc_i128& a, const rc_i128& b) {
  unsigned long long lo = a.lo - b.lo;
  a.hi -= b.hi + (a.lo < b.lo ? 1LL : 0LL);
  a.lo = lo;
}
__host__ __device__ __forceinline__ rc_i128 rc_make128(long long s) {
  rc_i128 r; r.lo = (unsigned long long)s; r.hi = s < 0 ? -1LL : 0LL; return r;
}
__host__ __device__ __forceinline__ double rc_deq128(const rc_i128& a, int q) { return rc_dequant128(a.hi, a.lo, q); }

// ---- MCMCData on the device (src/types.jl:145-157) ----------------------------------------------
// D   : n x n fp64 (as given / as built by the distance kernel)
// DL  : n x n interleaved fixed-point images {Dq, Lq} = {round(D * 2^qD), round(logD * 2^qL)}; the
//       sampler streams ONLY this array (16 B per matrix entry = the same bytes as fp64 D + fp64 logD).
struct rc_data {
  int64_t n;
  int device;
  double* D;
  longlong2* DL;
  int qD, qL;
  double mD, mL;        // max |D| over every entry and max |log D| (the diagonal's log is 0): qD, qL are chosen from them
};

// the domain error of MCMCData(D) and of new-point dissimilarities (their log must be finite for the fixed-point image)
#define RC_DOMAIN_MSG                                                                                                  \
  "D must have finite entries and strictly positive off-diagonal dissimilarities: log D must be finite for the "      \
  "fixed-point image the sampler streams (the reference accepts a zero and carries log D = -Inf, src/types.jl:155). " \
  "Remove duplicate observations or add a small jitter to them."

#define RC_MAXCAP 128                // default live cluster slots per chain (slot_cap = 0)
#define RC_MAXCAP_INC 255            // largest slot_cap: labels are bytes, recorded labels are 1-based bytes
#define RC_NSI ((RC_MAXCAP_INC + 31) / 32)
#define RC_DETACHED 0xFF
