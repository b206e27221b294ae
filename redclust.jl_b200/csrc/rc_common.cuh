// rc_common.cuh -- shared declarations of the sm_100a implementation (internal, not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
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

// pairwise Euclidean distances on the FP64 tensor cores (rc_gram.cu): X_dev n x dim row-major -> rows [row0, row0 + nrows) in D_dev (nrows x n)
int rc_distm_dmma(const double* X_dev, int64_t dim, int64_t n, int64_t row0, int64_t nrows, double* D_dev);
// int32 co-clustering counts on the device -> host fp64 counts / denom (rc_post.cu)
int rc_counts_to_host_psm(const int* counts, size_t total, double denom, double* out);
// posterior expected Binder loss from the counts (rc_post.cu): the sampler-range checks, W and P of a chain range against
// counts of at most nmax samples, and the exact totals T_s = S P_s + sum_t P_t - 2 W_s with their first argmin
int rc_sampler_binder_check(const rc_sampler* s, int64_t chain0, int64_t nch, const char* who);
int rc_sampler_binder_wp(const rc_sampler* s, int64_t chain0, int64_t nch, const int* counts, int64_t nmax, unsigned long long* W,
                         unsigned long long* P);
int rc_binder_finish(const unsigned long long* W, const unsigned long long* P, int64_t S, int64_t n, double* loss_sums,
                     int64_t* best, int64_t* totals);

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
