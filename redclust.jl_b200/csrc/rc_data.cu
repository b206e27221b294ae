// rc_data.cu -- MCMCData on the device: validation, log D, fixed-point images, Euclidean distance
// matrix.  Replaces /root/reference/src/types.jl:145-162 and the pairwise(Euclidean(), X, dims=2)
// call sites (src/types.jl:160, src/utils.jl:144-145, src/prior.jl:51,180).
#include <stdlib.h>
#include <string.h>
#include <chrono>
#include <cstdio>
#include "rc_common.cuh"

namespace {

// any(D .!= D') (types.jl:149) + domain scan.  flags[0]: asymmetric, flags[1]: bad off-diagonal entry
// (non-finite or <= 0, whose log cannot be represented), maxbits[0/1]: bit patterns of max|D|, max|logD|.
__global__ void k_scan(const double* __restrict__ D, int64_t n, int* flags, unsigned long long* maxbits) {
  const int64_t total = n * n;
  double mD = 0.0, mL = 0.0;
  int asym = 0, bad = 0;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / n, j = t - i * n;
    const double v = D[t];
    if (i != j) {
      if (v != D[j * n + i]) asym = 1;
      if (!(v > 0.0) || !(v < RC_INF)) { bad = 1; continue; }
      const double l = rc_log(v - 0.0 + 0.0);
      mL = fmax(mL, fabs(l));
    } else if (!(fabs(v) < RC_INF)) { bad = 1; continue; }
    mD = fmax(mD, fabs(v));
  }
  for (int off = 16; off; off >>= 1) {
    mD = fmax(mD, __shfl_xor_sync(0xffffffffu, mD, off));
    mL = fmax(mL, __shfl_xor_sync(0xffffffffu, mL, off));
    asym |= __shfl_xor_sync(0xffffffffu, asym, off);
    bad |= __shfl_xor_sync(0xffffffffu, bad, off);
  }
  if ((threadIdx.x & 31) == 0) {
    if (asym) atomicOr(&flags[0], 1);
    if (bad) atomicOr(&flags[1], 1);
    atomicMax(&maxbits[0], (unsigned long long)__double_as_longlong(mD));   // non-negative doubles order like their bits
    atomicMax(&maxbits[1], (unsigned long long)__double_as_longlong(mL));
  }
}

// logD = log.(D .- Diagonal(D) .+ I) (types.jl:155) and the fixed-point images the sampler streams.
__global__ void k_build_dl(const double* __restrict__ D, int64_t n, int qD, int qL, longlong2* __restrict__ DL) {
  const int64_t total = n * n;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / n, j = t - i * n;
    const double v = D[t];
    const double arg = (i == j) ? (v - v + 1.0) : (v - 0.0 + 0.0);
    longlong2 o;
    o.x = rc_quantize(v, qD);
    o.y = rc_quantize(rc_log(arg), qL);
    DL[t] = o;
  }
}

__global__ void k_logd(const double* __restrict__ D, int64_t n, double* __restrict__ out) {
  const int64_t total = n * n;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / n, j = t - i * n;
    const double v = D[t];
    out[t] = rc_log((i == j) ? (v - v + 1.0) : (v - 0.0 + 0.0));
  }
}

// |x_i|^2, ascending-coordinate summation (no FMA: the file is compiled with -fmad=false).
__global__ void k_sqnorm(const double* __restrict__ X, int64_t dim, int64_t n, double* __restrict__ sq) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a = 0.0;
  for (int64_t t = 0; t < dim; ++t) { const double x = X[i * dim + t]; a += x * x; }
  sq[i] = a;
}

// Gram-form Euclidean distances, upper triangle mirrored, exact zero diagonal:
// D_ij = sqrt(max(|x_i|^2 + |x_j|^2 - 2 x_i.x_j, 0)).  32x32 output tile per CTA, operands staged
// through shared memory; each dot product is accumulated in ascending coordinate order, so the result
// is independent of the tiling (and identical to the CPU oracle's).
#define DT 32
__global__ void __launch_bounds__(256) k_distm(const double* __restrict__ X, const double* __restrict__ sq, int64_t dim,
                                                int64_t n, double* __restrict__ D) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ double Xi[DT][DT + 1], Xj[DT][DT + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int64_t i0 = (int64_t)bi * DT, j0 = (int64_t)bj * DT;
  for (int64_t t0 = 0; t0 < dim; t0 += DT) {
    for (int r = ty; r < DT; r += 8) {
      const int64_t t = t0 + tx;
      Xi[r][tx] = (i0 + r < n && t < dim) ? X[(i0 + r) * dim + t] : 0.0;
      Xj[r][tx] = (j0 + r < n && t < dim) ? X[(j0 + r) * dim + t] : 0.0;
    }
    __syncthreads();
    const int tmax = (int)((dim - t0) < DT ? (dim - t0) : DT);
    for (int t = 0; t < tmax; ++t) {
      const double xj = Xj[tx][t];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] += Xi[ty + 8 * q][t] * xj;
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int64_t i = i0 + ty + 8 * q, j = j0 + tx;
    if (i >= n || j >= n || j < i) continue;    // diagonal tile: lower half comes from the mirror
    double r = 0.0;
    if (i != j) {
      double v = sq[i] + sq[j] - 2 * acc[q];
      if (rc_dist_unresolved(v, sq[i] + sq[j])) v = rc_dist_direct2(X + i * dim, X + j * dim, dim);
      r = sqrt(v > 0.0 ? v : 0.0);
    }
    D[i * n + j] = r;
    D[j * n + i] = r;
  }
}

// FP64 tensor-core variant (RCB200_DISTM=dmma): the Gram block X_i X_j^T is accumulated with
// mma.sync.aligned.m8n8k4.row.col.f64 (DMMA; tcgen05 has no f64 kind).  32x32 output tile per CTA of 4 warps, warp w
// owns rows 8w..8w+7 and the four 8-column blocks; operands are staged through shared memory in chunks of 32
// coordinates.  The summation order differs from the sequential kernel above (k-blocks of 4, fused multiply-add inside
// the tensor core), so this path is checked against the error bound instead of bit-exactly; symmetry and the zero diagonal
// stay exact (upper triangle mirrored).
__global__ void __launch_bounds__(128) k_distm_dmma(const double* __restrict__ X, const double* __restrict__ sq, int64_t dim,
                                                     int64_t n, double* __restrict__ D) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ double Xi[DT][DT + 1], Xj[DT][DT + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fr = lane >> 2, fk = lane & 3;       // fragment row (A) / column (B), k index
  double c0[4] = {0, 0, 0, 0}, c1[4] = {0, 0, 0, 0};
  const int64_t i0 = (int64_t)bi * DT, j0 = (int64_t)bj * DT;
  for (int64_t t0 = 0; t0 < dim; t0 += DT) {
    for (int e = threadIdx.x; e < DT * DT; e += 128) {
      const int r = e / DT, t = e % DT;
      Xi[r][t] = (i0 + r < n && t0 + t < dim) ? X[(i0 + r) * dim + t0 + t] : 0.0;
      Xj[r][t] = (j0 + r < n && t0 + t < dim) ? X[(j0 + r) * dim + t0 + t] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < DT; k += 4) {
      const double a = Xi[8 * warp + fr][k + fk];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const double b = Xj[8 * nt + fr][k + fk];
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                     : "+d"(c0[nt]), "+d"(c1[nt]) : "d"(a), "d"(b));
      }
    }
    __syncthreads();
  }
  // C fragment: lane holds C[row = lane / 4][col = 2 * (lane % 4) + {0, 1}]
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t i = i0 + 8 * warp + fr, j = j0 + 8 * nt + 2 * fk + h;
      if (i >= n || j >= n) continue;
      if (i == j) { D[i * n + i] = 0.0; continue; }
      if (j < i) continue;
      double v = sq[i] + sq[j] - 2 * (h ? c1[nt] : c0[nt]);
      if (rc_dist_unresolved(v, sq[i] + sq[j])) v = rc_dist_direct2(X + i * dim, X + j * dim, dim);
      const double r = sqrt(v > 0.0 ? v : 0.0);
      D[i * n + j] = r;
      D[j * n + i] = r;
    }
}

int finish_data(rc_data* d) {
  const int64_t n = d->n;
  int* flags = nullptr; unsigned long long* maxbits = nullptr;
  RC_CUDA(rc_dev_malloc((void**)&flags, 2 * sizeof(int)));
  RC_CUDA(rc_dev_malloc((void**)&maxbits, 2 * sizeof(unsigned long long)));
  RC_CUDA(cudaMemset(flags, 0, 2 * sizeof(int)));
  RC_CUDA(cudaMemset(maxbits, 0, 2 * sizeof(unsigned long long)));
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, d->device);
  const int grid = nsm * 8;
  (void)cudaGetLastError();   // drop any stale error of an unrelated earlier call
  k_scan<<<grid, 256>>>(d->D, n, flags, maxbits);
  RC_CUDA(cudaGetLastError());
  int hflags[2]; unsigned long long hbits[2];
  RC_CUDA(cudaMemcpy(hflags, flags, sizeof(hflags), cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(hbits, maxbits, sizeof(hbits), cudaMemcpyDeviceToHost));
  rc_dev_free(flags); rc_dev_free(maxbits);
  if (hflags[0]) { rc_set_error("D must be symmetric."); return RC_ERR_NOTSYM; }
  if (hflags[1]) {
    rc_set_error(RC_DOMAIN_MSG);
    return RC_ERR_DOMAIN;
  }
  double mD, mL;
  memcpy(&mD, &hbits[0], 8); memcpy(&mL, &hbits[1], 8);
  d->mD = mD; d->mL = mL;
  d->qD = rc_choose_q(mD, n);
  d->qL = rc_choose_q(mL, n);
  if (d->qD < 0 || d->qL < 0) { rc_set_error("dissimilarities too large for the fixed-point image."); return RC_ERR_DOMAIN; }
  RC_CUDA(rc_dev_malloc((void**)&d->DL, sizeof(longlong2) * (size_t)n * n));
  k_build_dl<<<grid, 256>>>(d->D, n, d->qD, d->qL, d->DL);
  RC_CUDA(cudaGetLastError());
  RC_CUDA(cudaDeviceSynchronize());
  return RC_OK;
}

// Rows [row0, row0 + nrows) of the distance matrix, every entry computed (no mirroring) with the operation order of
// k_distm: products and sums commute pairwise, so the block equals the same rows of the single-GPU matrix bit for bit.
__global__ void __launch_bounds__(256) k_distm_rows(const double* __restrict__ X, const double* __restrict__ sq, int64_t dim, int64_t n,
                                                    int64_t row0, int64_t nrows, double* __restrict__ Drows) {
  __shared__ double Xi[DT][DT + 1], Xj[DT][DT + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int64_t i0 = row0 + (int64_t)blockIdx.y * DT, j0 = (int64_t)blockIdx.x * DT, iend = row0 + nrows;
  for (int64_t t0 = 0; t0 < dim; t0 += DT) {
    for (int r = ty; r < DT; r += 8) {
      const int64_t t = t0 + tx;
      Xi[r][tx] = (i0 + r < iend && t < dim) ? X[(i0 + r) * dim + t] : 0.0;
      Xj[r][tx] = (j0 + r < n && t < dim) ? X[(j0 + r) * dim + t] : 0.0;
    }
    __syncthreads();
    const int tmax = (int)((dim - t0) < DT ? (dim - t0) : DT);
    for (int t = 0; t < tmax; ++t) {
      const double xj = Xj[tx][t];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] += Xi[ty + 8 * q][t] * xj;
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int64_t i = i0 + ty + 8 * q, j = j0 + tx;
    if (i >= iend || j >= n) continue;
    double r = 0.0;
    if (i != j) {
      double v = sq[i] + sq[j] - 2 * acc[q];
      if (rc_dist_unresolved(v, sq[i] + sq[j])) v = rc_dist_direct2(X + i * dim, X + j * dim, dim);
      r = sqrt(v > 0.0 ? v : 0.0);
    }
    Drows[(i - row0) * n + j] = r;
  }
}

}  // namespace

// the device of an entry point: fails with RC_ERR_CUDA without one and RC_ERR_ARG out of range
int rc_select_device(int32_t device) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
    rc_set_error("no CUDA device available (librcb200 has no CPU fallback)");
    return RC_ERR_CUDA;
  }
  if (device < 0 || device >= cnt) { rc_set_error("device %d out of range (0..%d)", device, cnt - 1); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(device));
  return RC_OK;
}

extern "C" {

int32_t rc_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) return 0;
  return cnt;
}

int32_t rc_data_from_dist(const double* D, int64_t n, int32_t device, rc_data** out) {
  if (!D || !out || n < 1) { rc_set_error("rc_data_from_dist: null pointer or n < 1"); return RC_ERR_ARG; }
  int st = rc_select_device(device);
  if (st) return st;
  rc_data* d = new rc_data();
  d->n = n; d->device = device; d->D = nullptr; d->DL = nullptr;
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  if (rc_dev_malloc((void**)&d->D, sizeof(double) * (size_t)n * n) != cudaSuccess) {
    rc_set_error("out of device memory for D (%lld x %lld)", (long long)n, (long long)n); delete d; return RC_ERR_CUDA;
  }
  const double t1 = now();
  if (cudaMemcpy(d->D, D, sizeof(double) * (size_t)n * n, cudaMemcpyHostToDevice) != cudaSuccess) {
    rc_set_error("upload of D failed"); rc_data_destroy(d); return RC_ERR_CUDA;
  }
  const double t2 = now();
  st = finish_data(d);
  if (verbose) fprintf(stderr, "[rcb200] rc_data_from_dist n=%lld: alloc %.4f s, upload %.4f s, checks + images %.4f s\n", (long long)n, t1 - t0, t2 - t1, now() - t2);
  if (st) { rc_data_destroy(d); return st; }
  *out = d;
  return RC_OK;
}

int32_t rc_data_from_points(const double* X, int64_t dim, int64_t n, int32_t device, rc_data** out) {
  if (!X || !out || n < 1 || dim < 1) { rc_set_error("rc_data_from_points: null pointer or empty input"); return RC_ERR_ARG; }
  int st = rc_select_device(device);
  if (st) return st;
  rc_data* d = new rc_data();
  d->n = n; d->device = device; d->D = nullptr; d->DL = nullptr;
  double *dX = nullptr, *sq = nullptr;
  if (rc_dev_malloc((void**)&d->D, sizeof(double) * (size_t)n * n) != cudaSuccess || cudaMalloc(&dX, sizeof(double) * (size_t)n * dim) != cudaSuccess ||
      cudaMalloc(&sq, sizeof(double) * (size_t)n) != cudaSuccess) {
    rc_set_error("out of device memory for the distance matrix"); cudaFree(dX); cudaFree(sq); rc_data_destroy(d); return RC_ERR_CUDA;
  }
  cudaMemcpy(dX, X, sizeof(double) * (size_t)n * dim, cudaMemcpyHostToDevice);
  k_sqnorm<<<(unsigned)((n + 255) / 256), 256>>>(dX, dim, n, sq);
  const unsigned nb = (unsigned)((n + DT - 1) / DT);
  // Default: the Gram blocks on the FP64 tensor cores (rc_gram.cu).  Every path is within (dim + 4) u / tau relative of the
  // exact distance (rc_dist_unresolved, rc_math.h).
  // RCB200_DISTM=exact: the ascending-coordinate kernel whose operation order is the oracle's (bit-equal to it);
  // RCB200_DISTM=dmma32: round 1's 32 x 32-tile DMMA kernel (kept for comparison).
  const char* mode = getenv("RCB200_DISTM");
  if (mode && !strcmp(mode, "exact")) k_distm<<<dim3(nb, nb), 256>>>(dX, sq, dim, n, d->D);
  else if (mode && !strcmp(mode, "dmma32")) k_distm_dmma<<<dim3(nb, nb), 128>>>(dX, sq, dim, n, d->D);
  else if (rc_distm_dmma(dX, dim, n, 0, n, d->D) != RC_OK) { cudaFree(dX); cudaFree(sq); rc_data_destroy(d); return RC_ERR_CUDA; }
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(dX); cudaFree(sq);
  if (e != cudaSuccess) { rc_set_error("distance kernel failed: %s", cudaGetErrorString(e)); rc_data_destroy(d); return RC_ERR_CUDA; }
  st = finish_data(d);
  if (st) { rc_data_destroy(d); return st; }
  *out = d;
  return RC_OK;
}

// Multi-GPU distance build (SURVEY 8e): this rank's block of rows into a caller device buffer (nrows x n fp64); the
// caller all-gathers the blocks and hands the complete matrix to rc_data_from_dist_dev.
int32_t rc_distm_rows_dev(const double* X, int64_t dim, int64_t n, int64_t row0, int64_t nrows, int32_t device, void* D_rows_dev) {
  if (!X || !D_rows_dev || n < 1 || dim < 1 || row0 < 0 || nrows < 0 || row0 + nrows > n) { rc_set_error("rc_distm_rows_dev: bad arguments"); return RC_ERR_ARG; }
  int st = rc_select_device(device);
  if (st) return st;
  if (nrows == 0) return RC_OK;
  double *dX = nullptr, *sq = nullptr;
  if (cudaMalloc(&dX, sizeof(double) * (size_t)n * dim) != cudaSuccess || cudaMalloc(&sq, sizeof(double) * (size_t)n) != cudaSuccess) {
    rc_set_error("out of device memory for the points"); cudaFree(dX); cudaFree(sq); return RC_ERR_CUDA;
  }
  cudaMemcpy(dX, X, sizeof(double) * (size_t)n * dim, cudaMemcpyHostToDevice);
  const char* mode = getenv("RCB200_DISTM");            // default / exact: the row block equals the same rows of rc_data_from_points bit
                                                        // for bit (dmma32 has no row kernel: its blocks are the exact kernel's rows)
  if (mode && (!strcmp(mode, "exact") || !strcmp(mode, "dmma32"))) {
    k_sqnorm<<<(unsigned)((n + 255) / 256), 256>>>(dX, dim, n, sq);
    k_distm_rows<<<dim3((unsigned)((n + DT - 1) / DT), (unsigned)((nrows + DT - 1) / DT)), 256>>>(dX, sq, dim, n, row0, nrows, (double*)D_rows_dev);
  } else if (rc_distm_dmma(dX, dim, n, row0, nrows, (double*)D_rows_dev) != RC_OK) { cudaFree(dX); cudaFree(sq); return RC_ERR_CUDA; }
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(dX); cudaFree(sq);
  if (e != cudaSuccess) { rc_set_error("distance kernel failed: %s", cudaGetErrorString(e)); return RC_ERR_CUDA; }
  return RC_OK;
}

// MCMCData(D) from a matrix that already lives on the device (same checks and images as rc_data_from_dist).
int32_t rc_data_from_dist_dev(const void* D_dev, int64_t n, int32_t device, rc_data** out) {
  if (!D_dev || !out || n < 1) { rc_set_error("rc_data_from_dist_dev: null pointer or n < 1"); return RC_ERR_ARG; }
  int st = rc_select_device(device);
  if (st) return st;
  rc_data* d = new rc_data();
  d->n = n; d->device = device; d->D = nullptr; d->DL = nullptr;
  if (rc_dev_malloc((void**)&d->D, sizeof(double) * (size_t)n * n) != cudaSuccess) {
    rc_set_error("out of device memory for D (%lld x %lld)", (long long)n, (long long)n); delete d; return RC_ERR_CUDA;
  }
  if (cudaMemcpy(d->D, D_dev, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice) != cudaSuccess) {
    rc_set_error("copy of D failed"); rc_data_destroy(d); return RC_ERR_CUDA;
  }
  st = finish_data(d);
  if (st) { rc_data_destroy(d); return st; }
  *out = d;
  return RC_OK;
}

int64_t rc_data_n(const rc_data* d) { return d ? d->n : 0; }

int32_t rc_data_copy_dist(const rc_data* d, double* D_out) {
  if (!d || !D_out) { rc_set_error("rc_data_copy_dist: null pointer"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(d->device));
  RC_CUDA(cudaMemcpy(D_out, d->D, sizeof(double) * (size_t)d->n * d->n, cudaMemcpyDeviceToHost));
  return RC_OK;
}

int32_t rc_data_copy_logdist(const rc_data* d, double* logD_out) {
  if (!d || !logD_out) { rc_set_error("rc_data_copy_logdist: null pointer"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(d->device));
  double* tmp = nullptr;
  RC_CUDA(cudaMalloc(&tmp, sizeof(double) * (size_t)d->n * d->n));
  k_logd<<<148 * 8, 256>>>(d->D, d->n, tmp);
  cudaError_t e = cudaMemcpy(logD_out, tmp, sizeof(double) * (size_t)d->n * d->n, cudaMemcpyDeviceToHost);
  cudaFree(tmp);
  RC_CUDA(e);
  return RC_OK;
}

int32_t rc_data_scales(const rc_data* d, int32_t* qD, int32_t* qL) {
  if (!d) { rc_set_error("rc_data_scales: null pointer"); return RC_ERR_ARG; }
  if (qD) *qD = d->qD;
  if (qL) *qL = d->qL;
  return RC_OK;
}

void rc_data_destroy(rc_data* d) {
  if (!d) return;
  cudaSetDevice(d->device);
  rc_dev_free(d->D);
  rc_dev_free(d->DL);
  delete d;
}

}  // extern "C"
