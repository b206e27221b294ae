// rc_align.cu -- allocation probabilities of every point to the clusters of a point estimate (no reference call; the pivot
// method of the ECR algorithm, Papastamoulis & Iliopoulos 2010, JCGS 19(2); R package label.switching::ecr).
//   k_align_match   per sample: the K^ x K_t contingency table with the estimate in shared memory (as k_pair_loss<true>
//                   builds it), then the assignment of the sample's clusters to the estimate's that maximises the number of
//                   agreeing points, solved on one warp by the canonical Hungarian method below -> sigma_t, matched[t]
//   k_align_count   per point: counts[i][k] = #{t : sigma_t(c_t(i)) = k}, column K^ = "unmatched"
// Canonical assignment (the tie rule decides which optimum is returned, so the algorithm is part of the definition): the
// shortest-augmenting-path Hungarian method with int64 dual potentials in its O(N^3) "e-maxx" form on the square
// N = max(K^, K_t) cost a[k][l] = -n_kl (0 in the padding); rows k = 1..N are added in ascending order; in each Dijkstra
// step over the unused columns, `cur < minv[j]` (strict) updates minv[j] / way[j] and `minv[j] < delta` (strict) takes j,
// so ties go to the smallest column.  sigma_t(l) = k when column l is assigned to row k <= K^ and n_kl > 0, else 0.
// Everything is an integer: the results do not depend on the grid or the order.
#include <vector>
#include "rc_common.cuh"
#include "rc_labels.h"

namespace {

#define AQ 8                                  // columns per lane: N <= 255 < 32 * AQ
#define ACT 256                               // threads of k_align_count, one point each
#define ACH 64                                // samples whose sigma k_align_count holds in shared memory at a time
#define ALD 16                                // labels a k_align_count thread loads before it counts them
#define ASLICE 65535                          // samples per k_align_count CTA: its 16-bit bins cannot overflow

__device__ __forceinline__ unsigned cell(const unsigned* tab, int t, int wide) {
  return wide ? tab[t] : ((tab[t >> 1] >> ((t & 1) * 16)) & 0xffffu);
}

// One CTA per sample at a time (grid-stride over the samples).  The estimate E (bytes 1..Kh) is staged once per CTA; every
// sample's table is built with lane-spread shared-memory atomics (lane l walks segment l of the label vector, so the lanes
// of one atomic hit different cells even when cluster members are contiguous), then warp 0 solves the assignment while the
// other warps wait.  Warp 0: lane owns columns j = 1 + lane + 32 q (q < AQ) with minv, way and used in registers; u, v and
// p (the row assigned to each column) in shared memory; the argmin of a Dijkstra step returns the smallest column among
// the minima, as the sequential scan does.  KEY64 = true takes the 64-bit reduction on every step.
template <bool KEY64>
__global__ void __launch_bounds__(256, 4) k_align_match(const uint8_t* __restrict__ L, const int* __restrict__ Kc, int64_t S,
                                                        int64_t n, const uint8_t* __restrict__ E, int Kh, int wide, int tabwords,
                                                        int stride, uint8_t* __restrict__ maps, long long* __restrict__ matched) {
  extern __shared__ __align__(16) unsigned tab[];
  const int64_t nv = (n + 15) / 16;
  uint8_t* la = reinterpret_cast<uint8_t*>(tab + tabwords);
  uint8_t* lb = la + nv * 16;
  __shared__ long long u[256], v[256];
  __shared__ int p[256];
  const bool vec = (n % 16) == 0;                          // rows of L are 16-byte aligned only then
  auto stage = [&](uint8_t* dst, const uint8_t* src) {
    if (vec) for (int64_t t = threadIdx.x; t < nv; t += blockDim.x) reinterpret_cast<uint4*>(dst)[t] = reinterpret_cast<const uint4*>(src)[t];
    else for (int64_t t = threadIdx.x; t < n; t += blockDim.x) dst[t] = src[t];
  };
  stage(la, E);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long INF = 0x1fffffffffffffffLL;
  for (int64_t s = blockIdx.x; s < S; s += gridDim.x) {
    const int Kt = Kc[s], cells = Kh * Kt, N = max(Kh, Kt);
    const int nwords = wide ? cells : (cells + 1) / 2;
    __syncthreads();                                       // the previous sample has finished with tab / lb
    for (int t = threadIdx.x; t < nwords; t += blockDim.x) tab[t] = 0;
    stage(lb, L + s * n);
    __syncthreads();
    for (int w = wid; w < stride; w += 8) {
      const int64_t x = (int64_t)lane * stride + w;
      if (x < n) {
        const int c = (int)(la[x] - 1) * Kt + (int)(lb[x] - 1);
        if (wide) atomicAdd(&tab[c], 1u);
        else atomicAdd(&tab[c >> 1], (c & 1) ? 0x10000u : 1u);
      }
    }
    __syncthreads();
    if (wid != 0) continue;
    for (int j = lane; j <= N; j += 32) { u[j] = 0; v[j] = 0; p[j] = 0; }
    __syncwarp();
    for (int i = 1; i <= N; ++i) {
      long long minv[AQ];
      int way[AQ];
      unsigned used = 0;                                   // bit q: column 1 + lane + 32 q is used
#pragma unroll
      for (int q = 0; q < AQ; ++q) { minv[q] = INF; way[q] = 0; }
      if (lane == 0) p[0] = i;
      __syncwarp();
      int j0 = 0;
      for (;;) {                                           // Dijkstra from row i until a free column is reached
        if (j0 && ((j0 - 1) & 31) == lane) used |= 1u << ((j0 - 1) >> 5);
        const int i0 = p[j0];
        const long long ui0 = u[i0];
        long long best = INF;
        int bj = 0x7fffffff;
#pragma unroll
        for (int q = 0; q < AQ; ++q) {
          const int j = 1 + lane + 32 * q;
          if (j <= N && !((used >> q) & 1)) {
            const long long a = (i0 <= Kh && j <= Kt) ? -(long long)cell(tab, (i0 - 1) * Kt + (j - 1), wide) : 0;
            const long long cur = a - ui0 - v[j];
            if (cur < minv[q]) { minv[q] = cur; way[q] = j0; }
            if (minv[q] < best) { best = minv[q]; bj = j; }
          }
        }
        // with |minv| < 2^23 the 32-bit key (minv + 2^23) * 256 + (j - 1) orders by minv, then by column, and one warp
        // min-reduction finds it; a larger |minv| takes the (value, column) 64-bit shuffle reduction.  Nothing bounds the
        // potentials below 2^23 under pair_geometry's limits (N n reaches 255 x 112 640), so the fallback stays.
        const long long OFF = 1LL << 23;
        if (KEY64 || __any_sync(0xffffffffu, best != INF && (best < -OFF || best >= OFF))) {
          for (int off = 16; off; off >>= 1) {
            const long long ob = __shfl_xor_sync(0xffffffffu, best, off);
            const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
            if (ob < best || (ob == best && oj < bj)) { best = ob; bj = oj; }
          }
        } else {
          const unsigned key = __reduce_min_sync(0xffffffffu, best == INF ? 0xffffffffu : ((unsigned)(best + OFF) << 8) | (unsigned)(bj - 1));
          best = (long long)(key >> 8) - OFF;
          bj = (int)(key & 255u) + 1;
        }
        const long long delta = best;
        __syncwarp();                                      // every lane has read u / v / p of this step
        if (lane == 0) u[i] += delta;                      // column 0 is used: p[0] = i
#pragma unroll
        for (int q = 0; q < AQ; ++q) {
          const int j = 1 + lane + 32 * q;
          if (j <= N) {
            if ((used >> q) & 1) { u[p[j]] += delta; v[j] -= delta; }
            else minv[q] -= delta;
          }
        }
        __syncwarp();
        j0 = bj;
        if (p[j0] == 0) break;
      }
      for (;;) {                                           // augment along way[] back to column 0
        int w = 0;
#pragma unroll
        for (int q = 0; q < AQ; ++q) if (q == ((j0 - 1) >> 5)) w = way[q];
        const int j1 = __shfl_sync(0xffffffffu, w, (j0 - 1) & 31);
        if (lane == 0) p[j0] = p[j1];
        __syncwarp();
        j0 = j1;
        if (!j0) break;
      }
    }
    long long m = 0;
    for (int l = 1 + lane; l <= 256; l += 32) {
      int k = 0;
      if (l <= Kt) {                                       // byte 255 of the 256-byte row stays 0
        const int r = p[l];
        const unsigned c = r <= Kh ? cell(tab, (r - 1) * Kt + (l - 1), wide) : 0;
        if (c) { k = r; m += c; }
      }
      maps[s * 256 + (l - 1)] = (uint8_t)k;
    }
    for (int off = 16; off; off >>= 1) m += __shfl_xor_sync(0xffffffffu, m, off);
    if (lane == 0) matched[s] = m;
  }
}

// counts (n x (Kh + 1) int32, zeroed) += the allocations of points [blockIdx.x * ACT, + ACT) in samples
// [blockIdx.y * slice, + slice).  Thread i reads L[t][i] (a row of samples is coalesced across the threads) and the sigma of
// ACH samples at a time from shared memory (256-byte rows, 16-byte copies); it keeps its current sigma value and run length
// in registers and adds the run to its own 16-bit shared bin only when the value changes.  Bin v counts sigma = v, which is
// column v - 1, and bin 0 the unmatched column Kh.  slice <= ASLICE, so no bin overflows before the final flush.
__global__ void __launch_bounds__(ACT) k_align_count(const uint8_t* __restrict__ L, const uint8_t* __restrict__ maps, int64_t S,
                                                     int64_t n, int Kh, int64_t slice, int* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned short bins[];   // [Kh + 1][ACT]
  __shared__ __align__(16) uint8_t sig[ACH][256];          // sigma of label l of a sample at [l - 1]
  const int64_t i = (int64_t)blockIdx.x * ACT + threadIdx.x;
  const int64_t t0 = (int64_t)blockIdx.y * slice, t1 = min((long long)S, (long long)(t0 + slice));
  for (int b = threadIdx.x; b < (Kh + 1) * ACT; b += ACT) bins[b] = 0;
  int cur = 0, run = 0;
  for (int64_t c0 = t0; c0 < t1; c0 += ACH) {
    const int nc = (int)min((long long)ACH, (long long)(t1 - c0));
    __syncthreads();                                       // the previous chunk's sigma is no longer read
    for (int e = threadIdx.x; e < nc * 16; e += ACT)
      reinterpret_cast<uint4*>(&sig[0][0])[e] = reinterpret_cast<const uint4*>(maps + c0 * 256)[e];
    __syncthreads();
    if (i < n)
      for (int r0 = 0; r0 < nc; r0 += ALD) {
        uint8_t lab[ALD];                                  // ALD loads in flight per thread
#pragma unroll
        for (int q = 0; q < ALD; ++q) lab[q] = r0 + q < nc ? L[(c0 + r0 + q) * n + i] : 0;
#pragma unroll
        for (int q = 0; q < ALD; ++q)
          if (r0 + q < nc) {
            const int k = sig[r0 + q][lab[q] - 1];
            if (k == cur) ++run;
            else { if (run) bins[cur * ACT + threadIdx.x] += (unsigned short)run; cur = k; run = 1; }
          }
      }
  }
  if (i >= n) return;
  if (run) bins[cur * ACT + threadIdx.x] += (unsigned short)run;
  for (int k = 0; k <= Kh; ++k) {
    const unsigned c = bins[k * ACT + threadIdx.x];
    if (c) atomicAdd(&counts[i * (Kh + 1) + (k ? k - 1 : Kh)], (int)c);
  }
}

}  // namespace

// ---- host side -----------------------------------------------------------------------------------------------------------
int align_estimate(const int64_t* estimate, int64_t n, const char* who, Bufs& B, AlignEstimate& e) {
  if (!estimate || n < 1) { rc_set_error("%s: needs an estimate of n >= 1 points (n = %lld)", who, (long long)n); return RC_ERR_ARG; }
  std::vector<int> K;
  const int st = upload_labels(estimate, 1, n, B, &e.L, K);
  if (st == RC_ERR_SLOTS) rc_set_error("%s: the estimate has more than 255 clusters", who);
  TRYP(st);
  e.K = K[0];
  e.n = n;
  return RC_OK;
}

int align_check(const AlignEstimate& e, int64_t S, int kmax, const char* who, PairLaunch& p) {
  if (S < 1 || S >= ((int64_t)1 << 31)) {
    rc_set_error("%s: needs 1 <= S < 2^31 pooled samples (the counts are int32; S = %lld)", who, (long long)S);
    return RC_ERR_ARG;
  }
  return pair_geometry(e.n, e.K, kmax, who, p);
}

int align_alloc(const AlignEstimate& e, int64_t R, double extra_bytes, const char* extra_what, const char* who, Bufs& B, AlignDev& d) {
  const double GB = 1e9, cC = 4.0 * e.n * (e.K + 1), cM = 256.0 * R + 8.0 * R;
  size_t free_b = 0, total_b = 0;
  RC_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (cC + cM + extra_bytes > (double)free_b) {
    rc_set_error("%s: needs %.2f GB of device memory (counts %.2f GB, per-sample maps and matched %.2f GB, %s %.2f GB); "
                 "%.2f GB are free", who, (cC + cM + extra_bytes) / GB, cC / GB, cM / GB, extra_what, extra_bytes / GB,
                 (double)free_b / GB);
    return RC_ERR_CUDA;
  }
  TRYP(B.get(&d.counts, (size_t)(e.n * (e.K + 1))));
  TRYP(B.get(&d.maps, (size_t)R * 256));
  TRYP(B.get(&d.matched, (size_t)R));
  return RC_OK;
}

// counts (zeroed first), maps and matched of R device samples L (bytes 1..K, K on the device in Kd) against the estimate.
int align_run(const AlignEstimate& e, const PairLaunch& p, const uint8_t* L, const int* Kd, int64_t R, AlignDev& d) {
  RC_CUDA(cudaMemset(d.counts, 0, sizeof(int) * (size_t)(e.n * (e.K + 1))));
  if (R == 0) return RC_OK;
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  if (verbose) { for (auto& x : ev) cudaEventCreate(&x); cudaEventRecord(ev[0], 0); }
  // RCB200_ALIGN_KEY64=1: every argmin by the 64-bit reduction (the same results; it keeps the fallback exercised)
  const auto match = getenv("RCB200_ALIGN_KEY64") ? k_align_match<true> : k_align_match<false>;
  RC_CUDA(cudaFuncSetAttribute(match, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  int dev = 0, sms = 0, per_sm = 0;
  RC_CUDA(cudaGetDevice(&dev));
  RC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  RC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, match, 256, p.smem));
  const int64_t grid = std::min<int64_t>(R, (int64_t)sms * std::max(per_sm, 1));
  match<<<(unsigned)grid, 256, p.smem>>>(L, Kd, R, e.n, e.L, e.K, p.wide, p.tabwords, p.stride, d.maps, d.matched);
  RC_CUDA(cudaGetLastError());
  if (verbose) cudaEventRecord(ev[1], 0);
  // enough sample slices for about 8 CTAs per SM, each at most ASLICE samples
  const int64_t gx = (e.n + ACT - 1) / ACT;
  int64_t gy = std::max<int64_t>((R + ASLICE - 1) / ASLICE, std::min<int64_t>(R, (8LL * sms + gx - 1) / gx));
  const int64_t slice = (R + gy - 1) / gy;
  gy = (R + slice - 1) / slice;
  const size_t smem = sizeof(unsigned short) * (size_t)(e.K + 1) * ACT;
  RC_CUDA(cudaFuncSetAttribute(k_align_count, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_align_count<<<dim3((unsigned)gx, (unsigned)gy), ACT, smem>>>(L, d.maps, R, e.n, e.K, slice, d.counts);
  RC_CUDA(cudaGetLastError());
  if (verbose) cudaEventRecord(ev[2], 0);
  const cudaError_t err = cudaDeviceSynchronize();
  if (verbose) {
    float m1 = 0, m2 = 0;
    cudaEventElapsedTime(&m1, ev[0], ev[1]); cudaEventElapsedTime(&m2, ev[1], ev[2]);
    fprintf(stderr, "[rcb200] aligned allocation: samples=%lld n=%lld Kh=%d k_align_match %.3f ms (grid %lld, %d per SM) "
            "k_align_count %.3f ms (grid %lld x %lld) (CUDA events)\n", (long long)R, (long long)e.n, e.K, m1, (long long)grid,
            per_sm, m2, (long long)gx, (long long)gy);
    for (auto& x : ev) cudaEventDestroy(x);
  }
  RC_CUDA(err);
  return RC_OK;
}

// the single-GPU entry points, after align_check and align_alloc: run over R device samples L (K on the device in Kd and on
// the host in Kh) and copy the results to the caller's host outputs
static int aligned_out(const AlignEstimate& e, const PairLaunch& p, AlignDev& d, const uint8_t* L, const int* Kd, int64_t R,
                       const std::vector<int>& Kh, int32_t* counts_out, int64_t* matched_out, int32_t* K_out, uint8_t* maps_out) {
  TRYP(align_run(e, p, L, Kd, R, d));
  RC_CUDA(cudaMemcpy(counts_out, d.counts, sizeof(int) * (size_t)(e.n * (e.K + 1)), cudaMemcpyDeviceToHost));
  if (matched_out) RC_CUDA(cudaMemcpy(matched_out, d.matched, sizeof(long long) * (size_t)R, cudaMemcpyDeviceToHost));
  if (maps_out) RC_CUDA(cudaMemcpy2D(maps_out, 255, d.maps, 256, 255, (size_t)R, cudaMemcpyDeviceToHost));
  if (K_out) std::copy(Kh.begin(), Kh.end(), K_out);
  return RC_OK;
}

extern "C" {

// The sample labels are relabelled on the host first, so that the free-memory check counts their device copy too.
int32_t rc_aligned_alloc(const int64_t* estimate, const int64_t* labels, int64_t S, int64_t n, int32_t device, int32_t* counts_out,
                         int64_t* matched_out, int32_t* K_out, uint8_t* maps_out) {
  const char* who = "rc_aligned_alloc";
  if (!labels || !counts_out || S < 1 || S >= ((int64_t)1 << 31)) {
    rc_set_error("%s: needs 1 <= S < 2^31 sample label vectors and counts_out (S = %lld)", who, (long long)S);
    return RC_ERR_ARG;
  }
  TRYP(rc_select_device(device));
  Bufs B;
  AlignEstimate e;
  TRYP(align_estimate(estimate, n, who, B, e));
  std::vector<uint8_t> Lh;
  std::vector<int> K;
  TRYP(compact_labels(labels, S, n, Lh, K));
  PairLaunch p;
  AlignDev d;
  TRYP(align_check(e, S, *std::max_element(K.begin(), K.end()), who, p));
  TRYP(align_alloc(e, S, (double)Lh.size() + 4.0 * S, "sample labels", who, B, d));
  uint8_t* dL; int* dK;
  TRYP(B.get(&dL, Lh.size())); TRYP(B.get(&dK, (size_t)S));
  RC_CUDA(cudaMemcpy(dL, Lh.data(), Lh.size(), cudaMemcpyHostToDevice));
  RC_CUDA(cudaMemcpy(dK, K.data(), sizeof(int) * S, cudaMemcpyHostToDevice));
  return aligned_out(e, p, d, dL, dK, S, K, counts_out, matched_out, K_out, maps_out);
}

int32_t rc_sampler_aligned_alloc(const rc_sampler* s, const int64_t* estimate, int64_t chain0, int64_t nch, int32_t* counts_out,
                                 int64_t* matched_out, int32_t* K_out, uint8_t* maps_out) {
  const char* who = "rc_sampler_aligned_alloc";
  if (!s || !counts_out) { rc_set_error("%s: needs a sampler and counts_out", who); return RC_ERR_ARG; }
  rc_sample_range v;
  TRYP(rc_sampler_range(s, chain0, nch, who, v));
  Bufs B;
  AlignEstimate e;
  TRYP(align_estimate(estimate, v.n, who, B, e));
  std::vector<int> Kh;
  int kmax = 0;
  PairLaunch p;
  AlignDev d;
  TRYP(sample_K(v.K, v.R, Kh, &kmax));
  TRYP(align_check(e, v.R, kmax, who, p));
  TRYP(align_alloc(e, v.R, 0, "", who, B, d));
  return aligned_out(e, p, d, v.labels, v.K, v.R, Kh, counts_out, matched_out, K_out, maps_out);   // chain-major, sample-minor
}

}  // extern "C"
