// rc_post.cu -- posterior similarity matrix and the minimum-posterior-expected-loss search.
//   PSM   sum(adjacencymatrix.(clusts)) ./ numsamples      /root/reference/src/mcmc.jl:560, src/utils.jl:59-63
//   MPEL  lossmatrix[i,j] = lossfn(c_i, c_j), argmin of column sums   /root/reference/src/pointestimate.jl:34-59
//         binder = randindex[3] (Mirkin), omARI = 1 - randindex[1], VI = varinfo, ID = max(H) - I
//         (Clustering.jl randindex / varinfo / mutualinfo, restated from their contingency-table definitions)
//   Binder MPEL over pooled samples   the same argmin for binderloss (pointestimate.jl:68-76) from the counts alone:
//         O(S n^2) compares, no S x S matrix (k_binder_w, k_binder_pairs, rc_binder_finish)
// The reference materialises S dense n x n Bool matrices; here the label matrix is transposed once
// (point-major, samples contiguous) and co-clustering counts are byte-compare popcounts -- exact integers.
#include <vector>
#include <thread>
#include <chrono>
#include <atomic>
#include <algorithm>
#include <cstring>
#include <cstdio>
#include <cstdlib>
#include "rc_common.cuh"
#include "rc_labels.h"

int rc_psm_counts_tc(const uint8_t* Lt, int64_t n, int64_t Rpad, int64_t R, int kmax, int* counts, cudaStream_t st);
double rc_psm_tc_macs(int64_t n, int64_t R, int kmax);

extern "C" const uint8_t* rc_sampler_dev_labels(const rc_sampler* s, int64_t* S, int64_t* n, int64_t* nchains, int* device);
extern "C" const rc_data* rc_sampler_dev_traces(const rc_sampler* s, rc_params* par, int64_t* iters_done, int64_t* numiters, const int** K,
                                                const double** r, const double** p);

namespace {

// Lt[i][r] = L[r][i]; rows r >= R are filled with 0 (every pair then "matches" Rpad - R extra times,
// which the count kernel subtracts).
__global__ void k_transpose(const uint8_t* __restrict__ L, int64_t R, int64_t n, int64_t Rpad, uint8_t* __restrict__ Lt) {
  __shared__ uint8_t t[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, i0 = (int64_t)blockIdx.x * 32;
  for (int q = threadIdx.y; q < 32; q += blockDim.y) {
    const int64_t r = r0 + q, i = i0 + threadIdx.x;
    t[q][threadIdx.x] = (r < R && i < n) ? L[r * n + i] : 0;
  }
  __syncthreads();
  for (int q = threadIdx.y; q < 32; q += blockDim.y) {
    const int64_t i = i0 + q, r = r0 + threadIdx.x;
    if (i < n && r < Rpad) Lt[i * Rpad + r] = t[threadIdx.x][q];
  }
}

__device__ __forceinline__ unsigned eq_bytes(unsigned a, unsigned b) {   // number of equal bytes (0..4)
  const unsigned x = a ^ b;
  const unsigned t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;
  return __popc(~(t | x | 0x7f7f7f7fu));
}

// counts[i][j] = #{r < R : Lt[i][r] == Lt[j][r]}; 64 x 64 tile of pairs per CTA, upper triangle mirrored.
#define PT 64
#define PW 16   // 32-bit words (64 samples) per smem stage
__global__ void __launch_bounds__(256) k_psm_counts(const uint8_t* __restrict__ Lt, int64_t n, int64_t Rpad, int64_t R,
                                                    int* __restrict__ counts) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ unsigned A[PT][PW + 1], B[PT][PW + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  unsigned acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0;
  const int64_t i0 = (int64_t)bi * PT, j0 = (int64_t)bj * PT;
  const int64_t words = Rpad / 4;
  const unsigned* Lw = reinterpret_cast<const unsigned*>(Lt);
  for (int64_t w0 = 0; w0 < words; w0 += PW) {
    for (int t = threadIdx.x; t < PT * PW; t += 256) {
      const int row = t / PW, w = t % PW;
      const bool okw = w0 + w < words;
      A[row][w] = (okw && i0 + row < n) ? Lw[(i0 + row) * words + w0 + w] : 0u;
      B[row][w] = (okw && j0 + row < n) ? Lw[(j0 + row) * words + w0 + w] : 0x01010101u * 0xffu;   // never equal to A's filler
    }
    __syncthreads();
#pragma unroll 4
    for (int w = 0; w < PW; ++w) {
      unsigned a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = A[ty + 16 * q][w]; b[q] = B[tx + 16 * q][w]; }
#pragma unroll
      for (int qa = 0; qa < 4; ++qa)
#pragma unroll
        for (int qb = 0; qb < 4; ++qb) acc[qa][qb] += eq_bytes(a[qa], b[qb]);
    }
    __syncthreads();
  }
  const int pad = (int)(Rpad - R);
#pragma unroll
  for (int qa = 0; qa < 4; ++qa)
#pragma unroll
    for (int qb = 0; qb < 4; ++qb) {
      const int64_t i = i0 + ty + 16 * qa, j = j0 + tx + 16 * qb;
      if (i >= n || j >= n) continue;
      // words beyond `words` were filled with non-matching patterns; rows R..Rpad match for every pair
      const int v = (int)acc[qa][qb] - pad;
      counts[i * n + j] = v;
      counts[j * n + i] = v;
    }
}

__global__ void k_maxlabel(const uint8_t* __restrict__ L, size_t total, int* __restrict__ out) {
  unsigned m = 0;
  const uint4* L4 = reinterpret_cast<const uint4*>(L);
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total / 16; t += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = L4[t];
    m = __vmaxu4(m, __vmaxu4(__vmaxu4(v.x, v.y), __vmaxu4(v.z, v.w)));
  }
  m = max(max(m & 0xffu, (m >> 8) & 0xffu), max((m >> 16) & 0xffu, m >> 24));
  for (int off = 16; off; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, (int)m);
}

// ---- Binder MPEL over pooled samples ---------------------------------------------------------------
// W_s = sum_{a<b} N_ab [c_s(a) == c_s(b)] for every sample s, N the co-clustering counts.  One CTA per 64 x 64 tile
// (i, j >= i) of point pairs stages its N tile in shared memory (zero where a pair is not counted: a >= b, or outside n),
// then walks 128-sample chunks of the transposed labels: lane l holds the 32-bit word of samples 4l..4l+3, warp g the
// tile's points a = 8g..8g+7 against every b.  A byte-equality mask of the a- and b-words selects which of the four
// per-sample accumulators N_ab goes to.
//
// Exactness: every N_ab <= nmax (the samples behind the counts).  Per chunk a thread adds at most 8 x 64 = 512 values
// into each accumulator, so Acc = uint32 is exact for nmax < 2^23 (512 * nmax < 2^32); beyond that Acc = uint64
// (512 * 2^31 = 2^40).  A CTA's sum over its 8 warps is at most 4096 * nmax < 2^43 and is added once per (CTA, chunk,
// sample) into the uint64 W_s, which never exceeds C(n, 2) * nmax < 2^31 * 2^31 = 2^62 for n <= 65 535 and nmax < 2^31.
// Integer adds commute, so W does not depend on the tiling, the grid or the order of the atomics.
#define BT 64   // points per tile side
#define BW 32   // label words (128 samples) per chunk, one per lane

__device__ __forceinline__ unsigned eq_mask(unsigned a, unsigned b) {   // 0x80 in every byte where a and b agree
  const unsigned x = a ^ b;
  return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
}

template <typename Acc>
__global__ void __launch_bounds__(256) k_binder_w(const uint8_t* __restrict__ Lt, int64_t n, int64_t Rpad, int64_t R,
                                                  const int* __restrict__ counts, unsigned long long* __restrict__ W) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ __align__(16) int Ns[BT][BT];                 // Ns[b][a] = N(i0 + a, j0 + b) or 0
  __shared__ unsigned A[BT][BW], B[BT][BW];
  __shared__ unsigned long long red[8][4 * BW];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int64_t i0 = (int64_t)bi * BT, j0 = (int64_t)bj * BT;
  for (int q = threadIdx.x; q < BT * BT; q += 256) {
    const int b = q / BT, a = q % BT;
    const int64_t i = i0 + a, j = j0 + b;
    Ns[b][a] = (i < j && j < n) ? counts[j * n + i] : 0;
  }
  const int64_t words = Rpad / 4, nchunk = (words + BW - 1) / BW;
  const unsigned* Lw = reinterpret_cast<const unsigned*>(Lt);
  for (int64_t c = blockIdx.z; c < nchunk; c += gridDim.z) {
    const int64_t w0 = c * BW;
    __syncthreads();                                       // Ns written; the previous chunk is done with A, B, red
    for (int q = threadIdx.x; q < BT * BW; q += 256) {
      const int row = q / BW, w = q % BW;
      const bool okw = w0 + w < words;
      A[row][w] = (okw && i0 + row < n) ? Lw[(i0 + row) * words + w0 + w] : 0u;
      B[row][w] = (okw && j0 + row < n) ? Lw[(j0 + row) * words + w0 + w] : 0u;
    }
    __syncthreads();
    unsigned la[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) la[q] = A[8 * g + q][lane];
    Acc acc[4] = {0, 0, 0, 0};
#pragma unroll 2
    for (int b = 0; b < BT; ++b) {
      const unsigned lb = B[b][lane];
      const int4 n0 = *reinterpret_cast<const int4*>(&Ns[b][8 * g]), n1 = *reinterpret_cast<const int4*>(&Ns[b][8 * g + 4]);
      const unsigned nv[8] = {(unsigned)n0.x, (unsigned)n0.y, (unsigned)n0.z, (unsigned)n0.w,
                              (unsigned)n1.x, (unsigned)n1.y, (unsigned)n1.z, (unsigned)n1.w};
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const unsigned m = eq_mask(la[q], lb) >> 7;        // 1 in every byte where the labels agree
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] += (Acc)nv[q] * __byte_perm(m, 0u, 0x4440u + k);   // byte k of m, as 0 or 1
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) red[g][4 * lane + k] = acc[k];
    __syncthreads();
    if (threadIdx.x < 4 * BW) {
      const int64_t s = 4 * w0 + threadIdx.x;              // byte k of word w holds sample 4w + k
      unsigned long long v = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) v += red[q][threadIdx.x];
      if (s < R && v) atomicAdd(&W[s], v);
    }
  }
}

// P_s = sum_k C(n_k, 2) from the label histogram of sample s (L sample-major, any byte labels); one CTA per sample.
__global__ void __launch_bounds__(256) k_binder_pairs(const uint8_t* __restrict__ L, int64_t n, unsigned long long* __restrict__ P) {
  __shared__ unsigned h[256];
  __shared__ unsigned long long part[8];
  const uint8_t* l = L + (int64_t)blockIdx.x * n;
  h[threadIdx.x] = 0;
  __syncthreads();
  for (int64_t x = threadIdx.x; x < n; x += 256) atomicAdd(&h[l[x]], 1u);
  __syncthreads();
  const unsigned long long c = h[threadIdx.x];
  unsigned long long v = c ? c * (c - 1) / 2 : 0;
  for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int q = 0; q < 8; ++q) t += part[q];
    P[blockIdx.x] = t;
  }
}

// Co-clustering counts of R label vectors (device, sample-major).  Default: the tensor-core kernel of
// rc_psm_tc.cu (labels up to 128); RCB200_PSM=compare or more labels: the byte-compare kernel.  Both are exact.
// Lt_keep (may be NULL) receives the transposed labels (n x Rpad, Rpad = R rounded up to 64, filler 0), which the
// caller then frees.
int psm_counts_device(const uint8_t* L, int64_t R, int64_t n, int* counts, uint8_t** Lt_keep = nullptr) {
  const int64_t Rpad = (R + 63) & ~63LL;
  uint8_t* Lt = nullptr; int* dmax = nullptr;
  RC_CUDA(cudaMalloc(&Lt, (size_t)n * Rpad));
  if (cudaMalloc(&dmax, sizeof(int)) != cudaSuccess) { cudaFree(Lt); rc_set_error("out of device memory"); return RC_ERR_CUDA; }
  cudaMemset(dmax, 0, sizeof(int));
  dim3 tb(32, 8), tg((unsigned)((n + 31) / 32), (unsigned)((Rpad + 31) / 32));
  k_transpose<<<tg, tb>>>(L, R, n, Rpad, Lt);
  k_maxlabel<<<148 * 4, 256>>>(Lt, (size_t)n * Rpad, dmax);     // n * Rpad is a multiple of 64
  int kmax = 0;
  cudaError_t e = cudaMemcpy(&kmax, dmax, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(dmax);
  if (e != cudaSuccess) { cudaFree(Lt); RC_CUDA(e); }
  const char* mode = getenv("RCB200_PSM");
  const bool tc = kmax <= 128 && !(mode && !strcmp(mode, "compare"));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  if (verbose) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, 0); }
  int st = RC_OK;
  if (tc) st = rc_psm_counts_tc(Lt, n, Rpad, R, kmax, counts, 0);
  else {
    const unsigned nb = (unsigned)((n + PT - 1) / PT);
    k_psm_counts<<<dim3(nb, nb), 256>>>(Lt, n, Rpad, R, counts);
  }
  if (verbose) cudaEventRecord(e1, 0);
  e = cudaDeviceSynchronize();
  if (verbose) {
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    const double macs = tc ? rc_psm_tc_macs(n, R, kmax) : 0.0;
    fprintf(stderr, "[rcb200] psm counts: n=%lld samples=%lld kmax=%d kernel=%s %.3f ms  %.3e label compares/s  tensor %.1f TOP/s\n",
            (long long)n, (long long)R, kmax, tc ? "tcgen05-i8" : "byte-compare", ms, (double)n * n * R / (ms * 1e-3), 2 * macs / (ms * 1e-3) * 1e-12);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (Lt_keep && !st && e == cudaSuccess) *Lt_keep = Lt;
  else cudaFree(Lt);
  if (st) return st;
  RC_CUDA(e);
  return RC_OK;
}

// Binder totals of R device label vectors (sample-major L, transposed Lt as psm_counts_device keeps it, or NULL to
// transpose here) against co-clustering counts of at most nmax samples: W (uint64 per sample) and P (C(n_k, 2) summed
// per sample) to the host.  w_ms (may be NULL): the W kernel's time, CUDA events.
static int binder_wp(const uint8_t* L, const uint8_t* Lt, int64_t R, int64_t n, const int* counts, int64_t nmax,
                     unsigned long long* W_out, unsigned long long* P_out, float* w_ms) {
  const int64_t Rpad = (R + 63) & ~63LL;
  uint8_t* own = nullptr;
  unsigned long long *W = nullptr, *P = nullptr;
  if (!Lt) {
    RC_CUDA(cudaMalloc(&own, (size_t)n * Rpad));
    dim3 tb(32, 8), tg((unsigned)((n + 31) / 32), (unsigned)((Rpad + 31) / 32));
    k_transpose<<<tg, tb>>>(L, R, n, Rpad, own);
    Lt = own;
  }
  cudaError_t e = cudaMalloc(&W, sizeof(unsigned long long) * (size_t)R);
  if (e == cudaSuccess) e = cudaMalloc(&P, sizeof(unsigned long long) * (size_t)R);
  if (e == cudaSuccess) e = cudaMemset(W, 0, sizeof(unsigned long long) * (size_t)R);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (e == cudaSuccess && w_ms) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, 0); }
  if (e == cudaSuccess) {
    const unsigned nb = (unsigned)((n + BT - 1) / BT);
    const int64_t tiles = (int64_t)nb * (nb + 1) / 2, nchunk = (Rpad / 4 + BW - 1) / BW;
    // enough CTAs to fill the device several times; beyond that a CTA walks more chunks and reuses its N tile
    const unsigned gz = (unsigned)std::min<int64_t>({nchunk, 65535, std::max<int64_t>(1, (148 * 16 + tiles - 1) / tiles)});
    const dim3 grid(nb, nb, gz);
    if (nmax < ((int64_t)1 << 23)) k_binder_w<unsigned><<<grid, 256>>>(Lt, n, Rpad, R, counts, W);
    else k_binder_w<unsigned long long><<<grid, 256>>>(Lt, n, Rpad, R, counts, W);
    if (w_ms) cudaEventRecord(e1, 0);
    k_binder_pairs<<<(unsigned)R, 256>>>(L, n, P);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess && w_ms) cudaEventElapsedTime(w_ms, e0, e1);
  if (e0) { cudaEventDestroy(e0); cudaEventDestroy(e1); }
  if (e == cudaSuccess) e = cudaMemcpy(W_out, W, sizeof(unsigned long long) * (size_t)R, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(P_out, P, sizeof(unsigned long long) * (size_t)R, cudaMemcpyDeviceToHost);
  cudaFree(W); cudaFree(P); cudaFree(own);
  RC_CUDA(e);
  return RC_OK;
}

// ---- MPEL ----------------------------------------------------------------------------------------
// One CTA per (i, block of PJ columns j > i): sample i's labels are staged once, then for every j the
// contingency table is built in shared memory (packed 16-bit counters, shared-memory atomics) and reduced to the
// loss.  Points are visited lane-spread (lane l walks segment l of the label vector), so the 32 lanes of an
// atomic hit different table cells even when cluster members are contiguous; N log N comes from a table.
#define PJ 8
__global__ void k_nlogn(int64_t n, double* __restrict__ out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t <= n) out[t] = t ? (double)t * log((double)t) : 0.0;
}
__device__ __forceinline__ unsigned tab_get(const unsigned* tab, int t, int wide) {
  return wide ? tab[t] : ((tab[t >> 1] >> ((t & 1) * 16)) & 0xffffu);
}
__global__ void __launch_bounds__(256) k_pair_loss(const uint8_t* __restrict__ L, const int* __restrict__ Kc, int64_t S,
                                                   int64_t n, int loss, int wide, int tabwords, int stride,
                                                   const double* __restrict__ nlogn, double* __restrict__ M, int64_t row_first,
                                                   int64_t row_stride, int mirror) {
  const int64_t i = row_first + (int64_t)blockIdx.y * row_stride;       // sharded: this rank's rows are row_first, + stride, ...
  if (i >= S) return;
  const int64_t jlo = max((long long)(i + 1), (long long)blockIdx.x * PJ), jhi = min((long long)S, (long long)(blockIdx.x + 1) * PJ);
  if (jlo >= jhi) return;
  extern __shared__ __align__(16) unsigned tab[];
  const int64_t nv = (n + 15) / 16;                       // 16-byte vectors per label vector
  uint8_t* la = reinterpret_cast<uint8_t*>(tab + tabwords);
  uint8_t* lb = la + nv * 16;
  __shared__ double red[6][8];
  const bool vec = (n % 16) == 0;                          // rows of L are 16-byte aligned only then
  auto stage = [&](uint8_t* dst, const uint8_t* src) {
    if (vec) for (int64_t t = threadIdx.x; t < nv; t += blockDim.x) reinterpret_cast<uint4*>(dst)[t] = reinterpret_cast<const uint4*>(src)[t];
    else for (int64_t t = threadIdx.x; t < n; t += blockDim.x) dst[t] = src[t];
  };
  stage(la, L + i * n);
  const int Ki = Kc[i];
  const double dn = (double)n;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int64_t j = jlo; j < jhi; ++j) {
    const int Kj = Kc[j];
    const int cells = Ki * Kj;
    const int nwords = wide ? cells : (cells + 1) / 2;
    __syncthreads();                                       // previous j has finished with tab / lb / red
    for (int t = threadIdx.x; t < nwords; t += blockDim.x) tab[t] = 0;
    stage(lb, L + j * n);
    __syncthreads();
    for (int w = wid; w < stride; w += 8) {
      const int64_t x = (int64_t)lane * stride + w;
      if (x < n) {
        const int cell = (int)(la[x] - 1) * Kj + (int)(lb[x] - 1);
        if (wide) atomicAdd(&tab[cell], 1u);
        else atomicAdd(&tab[cell >> 1], (cell & 1) ? 0x10000u : 1u);
      }
    }
    __syncthreads();
    // sums over the table: t2 = sum N^2, snl = sum N log N; margins via row / column passes
    double t2 = 0, snl = 0, nis = 0, njs = 0, hA = 0, hB = 0;
    for (int t = threadIdx.x; t < cells; t += blockDim.x) {
      const unsigned c = tab_get(tab, t, wide);
      const double d = (double)c; t2 += d * d; snl += nlogn[c];
    }
    for (int r = threadIdx.x; r < Ki + Kj; r += blockDim.x) {
      unsigned sm = 0;
      if (r < Ki) { for (int q = 0; q < Kj; ++q) sm += tab_get(tab, r * Kj + q, wide); }
      else { const int q = r - Ki; for (int pp = 0; pp < Ki; ++pp) sm += tab_get(tab, pp * Kj + q, wide); }
      const double d = (double)sm;
      if (r < Ki) { nis += d * d; hA += nlogn[sm]; } else { njs += d * d; hB += nlogn[sm]; }
    }
  double v[6] = {t2, snl, nis, njs, hA, hB};
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    for (int off = 16; off; off >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], off);
    if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v[q];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 0; q < 6; ++q) { double s = 0; for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[q][w]; v[q] = s; }
    t2 = v[0]; snl = v[1]; nis = v[2]; njs = v[3]; hA = v[4]; hB = v[5];
    double out;
    if (loss <= 1) {                                   // Clustering.randindex
      const double t1 = dn * (dn - 1) / 2, t3 = 0.5 * (nis + njs);
      const double nc = (dn * (dn * dn + 1) - (dn + 1) * nis - (dn + 1) * njs + 2 * (nis * njs) / dn) / (2 * (dn - 1));
      const double A = t1 + t2 - t3, Dg = -t2 + t3;
      if (loss == 0) out = Dg / t1;                    // Mirkin
      else out = 1 - ((t1 == nc) ? 0.0 : (A - nc) / (t1 - nc));
    } else {
      // H(A) = log n - (1/n) sum a log a;  I = (1/n) sum N log N - (1/n) sum a log a - (1/n) sum b log b + log n
      const double HA = log(dn) - hA / dn, HB = log(dn) - hB / dn;
      const double I = snl / dn - hA / dn - hB / dn + log(dn);
      out = loss == 2 ? (HA + HB - 2 * I) : ((HA > HB ? HA : HB) - I);
    }
    if (mirror) { M[i * S + j] = out; M[j * S + i] = out; }
    else M[(int64_t)blockIdx.y * S + j] = out;                         // row block of the upper triangle
  }
  }
}

__global__ void k_colsum(const double* __restrict__ M, int64_t S, double* __restrict__ sums) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= S) return;
  double s = 0;
  for (int64_t i = 0; i < S; ++i) s += M[i * S + j];   // ascending-row order, as sum(lossmatrix, dims = 1)
  sums[j] = s;
}

// column sums of the symmetric loss matrix given its strict upper triangle U, rows in ascending order (= k_colsum on
// the mirrored matrix: the diagonal contributes +0.0)
__global__ void k_colsum_upper(const double* __restrict__ U, int64_t S, double* __restrict__ sums) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= S) return;
  double s = 0;
  for (int64_t i = 0; i < S; ++i) s += i < j ? U[i * S + j] : (i > j ? U[j * S + i] : 0.0);
  sums[j] = s;
}

}  // namespace

// D2H of the counts as int32 through two pinned staging buffers; host threads turn each chunk into counts / denom
// (fp64) while the next chunk is in flight -- half the PCIe bytes of an fp64 copy and no pageable-memory bounce.
int rc_counts_to_host_psm(const int* counts, size_t total, double denom, double* out) {
  const size_t CH = (size_t)8 << 20;                       // entries per chunk (32 MB)
  int* stage[2] = {nullptr, nullptr};
  cudaStream_t st; cudaEvent_t ev[2];
  RC_CUDA(cudaStreamCreate(&st));
  for (int b = 0; b < 2; ++b) { RC_CUDA(cudaMallocHost(&stage[b], sizeof(int) * std::min(CH, total))); RC_CUDA(cudaEventCreate(&ev[b])); }
  const size_t nch = (total + CH - 1) / CH;
  const int nthr = (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency()));
  cudaError_t e = cudaSuccess;
  for (size_t c = 0; c <= nch && e == cudaSuccess; ++c) {
    if (c < nch) {
      const size_t off = c * CH, len = std::min(CH, total - off);
      e = cudaMemcpyAsync(stage[c & 1], counts + off, sizeof(int) * len, cudaMemcpyDeviceToHost, st);
      cudaEventRecord(ev[c & 1], st);
    }
    if (c > 0) {
      const size_t off = (c - 1) * CH, len = std::min(CH, total - off);
      cudaError_t e2 = cudaEventSynchronize(ev[(c - 1) & 1]);
      if (e2 != cudaSuccess) { e = e2; break; }
      const int* src = stage[(c - 1) & 1];
      auto body = [&](int w) {
        const size_t lo = len * w / nthr, hi = len * (w + 1) / nthr;
        for (size_t t = lo; t < hi; ++t) out[off + t] = (double)src[t] / denom;
      };
      std::vector<std::thread> pool;
      for (int w = 1; w < nthr; ++w) pool.emplace_back(body, w);
      body(0);
      for (auto& t : pool) t.join();
    }
  }
  for (int b = 0; b < 2; ++b) { cudaFreeHost(stage[b]); cudaEventDestroy(ev[b]); }
  cudaStreamDestroy(st);
  RC_CUDA(e);
  return RC_OK;
}

extern "C" {

int32_t rc_sampler_psm_counts_dev(const rc_sampler* s, int64_t chain0, int64_t nch, void* counts_dev) {
  if (!s || !counts_dev) { rc_set_error("rc_sampler_psm_counts_dev: null pointer"); return RC_ERR_ARG; }
  int64_t S, n, nchains; int device;
  const uint8_t* L = rc_sampler_dev_labels(s, &S, &n, &nchains, &device);
  if (chain0 < 0 || nch < 1 || chain0 + nch > nchains) { rc_set_error("rc_sampler_psm_counts_dev: bad chain range"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(device));
  if (S == 0) { RC_CUDA(cudaMemset(counts_dev, 0, sizeof(int) * (size_t)n * n)); return RC_OK; }
  return psm_counts_device(L + (size_t)chain0 * S * n, nch * S, n, (int*)counts_dev);
}

int32_t rc_sampler_psm(const rc_sampler* s, int64_t chain0, int64_t nch, double* psm_out) {
  if (!s || !psm_out) { rc_set_error("rc_sampler_psm: null pointer"); return RC_ERR_ARG; }
  int64_t S, n, nchains; int device;
  rc_sampler_dev_labels(s, &S, &n, &nchains, &device);
  RC_CUDA(cudaSetDevice(device));
  int* counts = nullptr;
  RC_CUDA(cudaMalloc(&counts, sizeof(int) * (size_t)n * n));
  int st = rc_sampler_psm_counts_dev(s, chain0, nch, counts);
  if (!st) st = rc_counts_to_host_psm(counts, (size_t)n * n, (double)(nch * S), psm_out);   // ./ numsamples (0/0 = NaN if no samples)
  cudaFree(counts);
  return st;
}

// Exact co-clustering counts of S host label vectors into a caller DEVICE buffer (n x n int32): the per-rank half of
// a PSM whose samples are sharded over GPUs (the caller all-reduces the counts and divides by the global S).
int32_t rc_psm_counts_dev(const int64_t* labels, int64_t S, int64_t n, int32_t device, void* counts_dev) {
  if (!labels || !counts_dev || S < 0 || n < 1) { rc_set_error("rc_psm_counts_dev: bad arguments"); return RC_ERR_ARG; }
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { rc_set_error("no CUDA device available (librcb200 has no CPU fallback)"); return RC_ERR_CUDA; }
  RC_CUDA(cudaSetDevice(device));
  if (S == 0) { RC_CUDA(cudaMemset(counts_dev, 0, sizeof(int) * (size_t)n * n)); return RC_OK; }
  std::vector<uint8_t> L; std::vector<int> K;
  int st = compact_labels(labels, S, n, L, K);
  if (st) return st;
  uint8_t* dL = nullptr;
  RC_CUDA(cudaMalloc(&dL, L.size()));
  cudaError_t e = cudaMemcpy(dL, L.data(), L.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) st = psm_counts_device(dL, S, n, (int*)counts_dev);
  cudaFree(dL);
  RC_CUDA(e);
  return st;
}

int32_t rc_psm(const int64_t* labels, int64_t S, int64_t n, int32_t device, double* psm_out) {
  if (!labels || !psm_out || S < 1 || n < 1) { rc_set_error("rc_psm: null pointer or empty input"); return RC_ERR_ARG; }
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { rc_set_error("no CUDA device available (librcb200 has no CPU fallback)"); return RC_ERR_CUDA; }
  RC_CUDA(cudaSetDevice(device));
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  std::vector<uint8_t> L; std::vector<int> K;
  int st = compact_labels(labels, S, n, L, K);
  if (st) return st;
  const double t1 = now();
  uint8_t* dL = nullptr; int* counts = nullptr;
  RC_CUDA(cudaMalloc(&dL, L.size()));
  RC_CUDA(cudaMemcpy(dL, L.data(), L.size(), cudaMemcpyHostToDevice));
  if (cudaMalloc(&counts, sizeof(int) * (size_t)n * n) != cudaSuccess) { cudaFree(dL); rc_set_error("out of device memory"); return RC_ERR_CUDA; }
  st = psm_counts_device(dL, S, n, counts);
  const double t2 = now();
  if (!st) st = rc_counts_to_host_psm(counts, (size_t)n * n, (double)S, psm_out);
  cudaFree(dL); cudaFree(counts);
  if (verbose) fprintf(stderr, "[rcb200] rc_psm: relabel %.3f s, upload + counts %.3f s, download + divide %.3f s\n", t1 - t0, t2 - t1, now() - t2);
  return st;
}

}  // extern "C"

// ---- posterior expected Binder loss of every sample from the co-clustering counts -------------------------------------
// The reference's MPEL (src/pointestimate.jl:34-59) with binderloss (:68-76, the Mirkin count of disagreeing pairs over
// C(n, 2)) sums, for candidate s, the disagreeing pairs of s and every sample t.  With P_s = sum_k C(n_k, 2) and
// W_s = sum_{a<b} N_ab [c_s(a) == c_s(b)] (N the counts of src/mcmc.jl:560), that sum is exactly
//   T_s = S * P_s + sum_t P_t - 2 W_s
// (a pair together in s and apart in t, or apart in s and together in t).  Everything is an integer: T_s < 2^63 for
// S < 2^31 and n <= 65 535.  loss_sums[s] = T_s / C(n, 2) (one rounding), best = first argmin of T.

int rc_binder_finish(const unsigned long long* W, const unsigned long long* P, int64_t S, int64_t n, double* loss_sums,
                     int64_t* best, int64_t* totals) {
  unsigned long long sumP = 0;
  for (int64_t s = 0; s < S; ++s) sumP += P[s];
  const double pairs = (double)(n * (n - 1) / 2);
  int64_t b = 0;
  unsigned long long tb = 0;
  for (int64_t s = 0; s < S; ++s) {
    const unsigned long long t = (unsigned long long)S * P[s] + sumP - 2 * W[s];
    if (s == 0 || t < tb) { tb = t; b = s; }
    if (loss_sums) loss_sums[s] = (double)t / pairs;
    if (totals) totals[s] = (int64_t)t;
  }
  if (best) *best = b;
  return RC_OK;
}

int rc_binder_check_args(int64_t S, int64_t n, const char* who) {
  if (S < 1 || S >= ((int64_t)1 << 31) || n < 1 || n > 65535) {
    rc_set_error("%s: needs 1 <= samples < 2^31 and 1 <= n <= 65535 (S = %lld, n = %lld)", who, (long long)S, (long long)n);
    return RC_ERR_ARG;
  }
  return RC_OK;
}

// The sampler's samples of chains [chain0, chain0 + nch) exist only after a run to numiters, and not for a chain that
// stopped at the slot capacity (the rules of rc_sampler_predict).
int rc_sampler_binder_check(const rc_sampler* s, int64_t chain0, int64_t nch, const char* who) {
  int64_t S, n, nchains; int device;
  rc_sampler_dev_labels(s, &S, &n, &nchains, &device);
  if (chain0 < 0 || nch < 1 || chain0 + nch > nchains) { rc_set_error("%s: bad chain range", who); return RC_ERR_ARG; }
  rc_params par; const int* K; const double *r, *p; int64_t done, numiters;
  rc_sampler_dev_traces(s, &par, &done, &numiters, &K, &r, &p);
  if (done < numiters) {
    rc_set_error("%s: the sampler ran %lld of %lld iterations; its samples are recorded only by a complete run", who, (long long)done,
                 (long long)numiters);
    return RC_ERR_STATE;
  }
  for (int64_t c = chain0; c < chain0 + nch; ++c)
    if (rc_sampler_chain_status(s, c) != 0) {
      rc_set_error("%s: chain %lld stopped at the slot capacity; its samples are incomplete", who, (long long)c);
      return RC_ERR_SLOTS;
    }
  return rc_binder_check_args(nch * S, n, who);
}

// W and P of the device-resident samples of chains [chain0, chain0 + nch) against counts of at most nmax samples.
int rc_sampler_binder_wp(const rc_sampler* s, int64_t chain0, int64_t nch, const int* counts, int64_t nmax, unsigned long long* W,
                         unsigned long long* P) {
  int64_t S, n, nchains; int device;
  const uint8_t* L = rc_sampler_dev_labels(s, &S, &n, &nchains, &device);
  RC_CUDA(cudaSetDevice(device));
  return binder_wp(L + (size_t)chain0 * S * n, nullptr, nch * S, n, counts, nmax, W, P, nullptr);
}

// counts, W, P and the totals of R device label vectors (sample-major, bytes)
static int binder_device(const uint8_t* L, int64_t R, int64_t n, double* loss_sums, int64_t* best, int64_t* totals) {
  int* counts = nullptr; uint8_t* Lt = nullptr;
  RC_CUDA(cudaMalloc(&counts, sizeof(int) * (size_t)n * n));
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  int st = psm_counts_device(L, R, n, counts, &Lt);
  const double t1 = now();
  std::vector<unsigned long long> W((size_t)R), P((size_t)R);
  float w_ms = 0;
  if (!st) st = binder_wp(L, Lt, R, n, counts, R, W.data(), P.data(), &w_ms);
  cudaFree(Lt); cudaFree(counts);
  if (st) return st;
  if (verbose)
    fprintf(stderr, "[rcb200] binder mpel: n=%lld samples=%lld counts %.3f ms, W kernel %.3f ms (CUDA events), %.3e pair-samples/s\n",
            (long long)n, (long long)R, (t1 - t0) * 1e3, w_ms, 0.5 * (double)n * (double)(n - 1) * (double)R / (w_ms * 1e-3));
  return rc_binder_finish(W.data(), P.data(), R, n, loss_sums, best, totals);
}

extern "C" {

int32_t rc_binder_mpel(const int64_t* labels, int64_t S, int64_t n, int32_t device, double* loss_sums, int64_t* best, int64_t* totals) {
  if (!labels) { rc_set_error("rc_binder_mpel: null pointer"); return RC_ERR_ARG; }
  int st = rc_binder_check_args(S, n, "rc_binder_mpel");
  if (st) return st;
  st = rc_select_device(device);
  if (st) return st;
  std::vector<uint8_t> L; std::vector<int> K;
  st = compact_labels(labels, S, n, L, K);
  if (st) return st;
  uint8_t* dL = nullptr;
  RC_CUDA(cudaMalloc(&dL, L.size()));
  cudaError_t e = cudaMemcpy(dL, L.data(), L.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) st = binder_device(dL, S, n, loss_sums, best, totals);
  cudaFree(dL);
  RC_CUDA(e);
  return st;
}

int32_t rc_sampler_binder_mpel(const rc_sampler* s, int64_t chain0, int64_t nch, double* loss_sums, int64_t* best, int64_t* totals) {
  if (!s) { rc_set_error("rc_sampler_binder_mpel: null handle"); return RC_ERR_ARG; }
  int st = rc_sampler_binder_check(s, chain0, nch, "rc_sampler_binder_mpel");
  if (st) return st;
  int64_t S, n, nchains; int device;
  const uint8_t* L = rc_sampler_dev_labels(s, &S, &n, &nchains, &device);
  RC_CUDA(cudaSetDevice(device));
  return binder_device(L + (size_t)chain0 * S * n, nch * S, n, loss_sums, best, totals);   // chain-major, sample-minor
}

}  // extern "C"

// Device buffers that are released when the call returns, whatever the path.
struct DevScratch {
  std::vector<void*> p;
  ~DevScratch() { for (void* q : p) cudaFree(q); }
  template <class T> cudaError_t get(T** out, size_t count) {
    cudaError_t e = cudaMalloc((void**)out, sizeof(T) * (count ? count : 1));
    if (e == cudaSuccess) p.push_back(*out);
    return e;
  }
};

// Shared front end of the MPEL entry points: relabel, upload, size the contingency table, and launch the pair-loss
// kernel for the rows row_first, row_first + row_stride, ... (nrows of them).  mirror = 1 writes the full symmetric
// S x S matrix M; mirror = 0 writes the rows' strict upper triangle into an nrows x S block.
static int mpel_pairs(const int64_t* labels, int64_t S, int64_t n, int32_t loss, int64_t row_first, int64_t row_stride,
                      int64_t nrows, int mirror, double* M, DevScratch& scr, int* kmax_out) {
  std::vector<uint8_t> L; std::vector<int> K;
  int st = compact_labels(labels, S, n, L, K);
  if (st) return st;
  int kmax = 0;
  for (int k : K) kmax = std::max(kmax, k);
  if (kmax_out) *kmax_out = kmax;
  const int wide = n > 65535;
  const int tabwords = ((wide ? kmax * kmax : (kmax * kmax + 1) / 2) + 3) & ~3;
  const size_t smem = (size_t)tabwords * 4 + 2 * (size_t)((n + 15) / 16) * 16;
  if (smem > 220 * 1024) { rc_set_error("rc_mpel: n = %lld with %d x %d clusters does not fit shared memory", (long long)n, kmax, kmax); return RC_ERR_SLOTS; }
  int stride = (int)((n + 31) / 32);
  while ((stride & 3) || !((stride >> 2) & 1)) ++stride;      // multiple of 4 with an odd quotient: lane segments start in different banks
  uint8_t* dL = nullptr; int* dK = nullptr; double* nlogn = nullptr;
  if (scr.get(&dL, L.size()) || scr.get(&dK, (size_t)S) || scr.get(&nlogn, (size_t)(n + 1))) { rc_set_error("rc_mpel: out of device memory"); return RC_ERR_CUDA; }
  RC_CUDA(cudaMemcpy(dL, L.data(), L.size(), cudaMemcpyHostToDevice));
  RC_CUDA(cudaMemcpy(dK, K.data(), sizeof(int) * S, cudaMemcpyHostToDevice));
  k_nlogn<<<(unsigned)((n + 256) / 256), 256>>>(n, nlogn);
  RC_CUDA(cudaFuncSetAttribute(k_pair_loss, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (nrows > 0)
    k_pair_loss<<<dim3((unsigned)((S + PJ - 1) / PJ), (unsigned)nrows), 256, smem>>>(dL, dK, S, n, loss, wide, tabwords, stride, nlogn, M,
                                                                                  row_first, row_stride, mirror);
  RC_CUDA(cudaGetLastError());
  return RC_OK;
}

static int mpel_argmin(const double* sums_dev, int64_t S, double* loss_sums, int64_t* best) {
  std::vector<double> hs((size_t)S);
  RC_CUDA(cudaMemcpy(hs.data(), sums_dev, sizeof(double) * S, cudaMemcpyDeviceToHost));
  int64_t b = 0;
  for (int64_t i = 1; i < S; ++i) if (hs[i] < hs[b]) b = i;     // argmin: first minimum
  if (loss_sums) memcpy(loss_sums, hs.data(), sizeof(double) * S);
  if (best) *best = b;
  return RC_OK;
}

static int mpel_device_ready(int32_t device) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { rc_set_error("no CUDA device available (librcb200 has no CPU fallback)"); return RC_ERR_CUDA; }
  RC_CUDA(cudaSetDevice(device));
  return RC_OK;
}

extern "C" {

// Multi-GPU MPEL (SURVEY 8e): the candidate rows row_first, row_first + row_stride, ... (nrows of them) of the strict
// upper triangle of the pairwise loss matrix into a caller DEVICE buffer (nrows x S fp64, zero where j <= i); the
// caller all-gathers the row blocks into the S x S upper triangle and calls rc_mpel_finish_dev, which sums the columns
// in ascending row order -- the result is bit-equal to rc_mpel on one GPU.
int32_t rc_mpel_rows_dev(const int64_t* labels, int64_t S, int64_t n, int32_t loss, int32_t device, int64_t row_first,
                         int64_t row_stride, int64_t nrows, void* M_rows_dev) {
  if (!labels || !M_rows_dev || S < 1 || n < 1 || loss < 0 || loss > 3 || row_first < 0 || row_stride < 1 || nrows < 0) {
    rc_set_error("rc_mpel_rows_dev: bad arguments"); return RC_ERR_ARG;
  }
  int st = mpel_device_ready(device);
  if (st) return st;
  DevScratch scr;
  RC_CUDA(cudaMemset(M_rows_dev, 0, sizeof(double) * (size_t)nrows * S));
  st = mpel_pairs(labels, S, n, loss, row_first, row_stride, nrows, 0, (double*)M_rows_dev, scr, nullptr);
  if (st) return st;
  RC_CUDA(cudaDeviceSynchronize());
  return RC_OK;
}

int32_t rc_mpel_finish_dev(const void* M_upper_dev, int64_t S, int32_t device, double* loss_sums, int64_t* best) {
  if (!M_upper_dev || S < 1) { rc_set_error("rc_mpel_finish_dev: bad arguments"); return RC_ERR_ARG; }
  int st = mpel_device_ready(device);
  if (st) return st;
  DevScratch scr;
  double* sums = nullptr;
  if (scr.get(&sums, (size_t)S)) { rc_set_error("rc_mpel: out of device memory"); return RC_ERR_CUDA; }
  k_colsum_upper<<<(unsigned)((S + 127) / 128), 128>>>((const double*)M_upper_dev, S, sums);
  return mpel_argmin(sums, S, loss_sums, best);
}

int32_t rc_mpel(const int64_t* labels, int64_t S, int64_t n, int32_t loss, int32_t device, double* loss_sums, int64_t* best) {
  if (!labels || S < 1 || n < 1 || loss < 0 || loss > 3) { rc_set_error("rc_mpel: bad arguments"); return RC_ERR_ARG; }
  int st = mpel_device_ready(device);
  if (st) return st;
  DevScratch scr;
  double *M = nullptr, *sums = nullptr;
  if (scr.get(&M, (size_t)S * S) || scr.get(&sums, (size_t)S)) { rc_set_error("rc_mpel: out of device memory"); return RC_ERR_CUDA; }
  RC_CUDA(cudaMemset(M, 0, sizeof(double) * (size_t)S * S));
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  int kmax = 0;
  st = mpel_pairs(labels, S, n, loss, 0, 1, S, 1, M, scr, &kmax);
  if (st) return st;
  const double tk = now();
  k_colsum<<<(unsigned)((S + 127) / 128), 128>>>(M, S, sums);
  st = mpel_argmin(sums, S, loss_sums, best);
  if (verbose) {
    const double dt = now() - tk;
    fprintf(stderr, "[rcb200] rc_mpel: S=%lld n=%lld kmax=%d loss=%d pair kernel + column sums %.3f s (%.3e pairs/s)\n", (long long)S, (long long)n, kmax,
            loss, dt, 0.5 * S * (S - 1) / dt);
  }
  return st;
}

}  // extern "C"
