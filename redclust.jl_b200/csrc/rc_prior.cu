// rc_prior.cu -- the O(n^2) pieces of fitprior on the device-resident dissimilarity matrix.
//   k-medoids      Clustering.kmedoids(dissM, k; maxiter) as called by fitprior  /root/reference/src/prior.jl:55-71
//                  and by runsampler's default initialisation                     /root/reference/src/mcmc.jl:519-527
//   pair statistics  A = uppertriangle(dissM)[adjacency], B = the rest; fit_mle(Gamma, .) needs count, sum and
//                  sum of logs of each                                            /root/reference/src/prior.jl:73-110
// Sums run over the exact fixed-point images (Dq, Lq), so every comparison and every statistic is independent of the
// order of summation: a host restatement with the same integers reproduces the medoids bit for bit.
#include <vector>
#include <cstring>
#include "rc_common.cuh"

namespace {

// assignment step: nearest medoid (first minimum, as argmin over the medoid rows)
__global__ void k_km_assign(const double* __restrict__ D, int64_t n, const int* __restrict__ med, int k, int* __restrict__ assign,
                            int* __restrict__ changed) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double best = D[(size_t)med[0] * n + i];
  int arg = 0;
  for (int c = 1; c < k; ++c) {
    const double v = D[(size_t)med[c] * n + i];      // row of the medoid: consecutive threads, consecutive addresses
    if (v < best) { best = v; arg = c; }
  }
  if (assign[i] != arg) { assign[i] = arg; *changed = 1; }
}

// member lists: perm = the points ordered by cluster (index order inside a cluster), start[c] .. start[c + 1] = cluster c's
// range.  One CTA; k and n are small next to the matrix.
__global__ void __launch_bounds__(1024) k_km_members(const int* __restrict__ assign, int64_t n, int k, int* __restrict__ start, int* __restrict__ perm) {
  extern __shared__ int cnt[];                       // k + 1 counters, then a running cursor per cluster
  for (int c = threadIdx.x; c <= k; c += blockDim.x) cnt[c] = 0;
  __syncthreads();
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) atomicAdd(&cnt[assign[j] + 1], 1);
  __syncthreads();
  if (threadIdx.x == 0) for (int c = 1; c <= k; ++c) cnt[c] += cnt[c - 1];
  __syncthreads();
  for (int c = threadIdx.x; c <= k; c += blockDim.x) start[c] = cnt[c];
  // stable placement: cluster c's members in index order (warp w takes clusters w, w + nwarps, ...; ballot-compacted sweeps)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int c = warp; c < k; c += nw) {
    int at = cnt[c];
    for (int64_t j0 = 0; j0 < n; j0 += 32) {
      const int64_t j = j0 + lane;
      const bool in = j < n && assign[j] == c;
      const unsigned m = __ballot_sync(0xffffffffu, in);
      if (in) perm[at + __popc(m & ((1u << lane) - 1))] = (int)j;
      at += __popc(m);
    }
  }
}
// s[i] = sum of Dq[i][j] over the members j of i's cluster: one warp per row, a gather over the cluster's member list
// (n / k entries of the row instead of all n)
__global__ void __launch_bounds__(256) k_km_rowsum(const longlong2* __restrict__ DL, int64_t n, const int* __restrict__ assign,
                                                   const int* __restrict__ start, const int* __restrict__ perm, long long* __restrict__ s) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = w0; i < n; i += nw) {
    const longlong2* row = DL + (size_t)i * n;
    const int c = assign[i], lo = start[c], hi = start[c + 1];
    long long acc = 0;
    for (int m = lo + lane; m < hi; m += 32) acc += row[perm[m]].x;
    for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) s[i] = acc;
  }
}
// medoid update: the member with the smallest sum, lowest index on ties (two passes of integer atomics)
__global__ void k_km_min1(const long long* __restrict__ s, const int* __restrict__ assign, int64_t n, long long* __restrict__ mins) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) atomicMin(&mins[assign[i]], s[i]);
}
__global__ void k_km_min2(const long long* __restrict__ s, const int* __restrict__ assign, int64_t n, const long long* __restrict__ mins,
                          int* __restrict__ newmed) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n && s[i] == mins[assign[i]]) atomicMin(&newmed[assign[i]], (int)i);
}
__global__ void k_km_finish(const int* __restrict__ med, int k, int* __restrict__ newmed, int* __restrict__ changed) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= k) return;
  if (newmed[c] == 0x7f7f7f7f) newmed[c] = med[c];          // empty cluster keeps its medoid
  if (newmed[c] != med[c]) *changed = 1;
}
// total cost as an exact integer: per-block partial sums of Dq[medoid(i)][i]
__global__ void __launch_bounds__(256) k_km_cost(const longlong2* __restrict__ DL, int64_t n, const int* __restrict__ med,
                                                 const int* __restrict__ assign, long long* __restrict__ partial) {
  long long acc = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += DL[(size_t)med[assign[i]] * n + i].x;
  __shared__ long long red[8];
  for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { long long t = 0; for (int w = 0; w < 8; ++w) t += red[w]; partial[blockIdx.x] = t; }
}

// row i: sums over j > i of (Dq, Lq) within i's cluster and over all j > i, and the within count
__global__ void __launch_bounds__(256) k_pair_rows(const longlong2* __restrict__ DL, int64_t n, const int* __restrict__ lab,
                                                   long long* __restrict__ out) {
  __shared__ long long red[5][8];
  for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
    const longlong2* row = DL + (size_t)i * n;
    const int li = lab[i];
    long long v[5] = {0, 0, 0, 0, 0};          // within D, within L, all D, all L, within count
    for (int64_t j = i + 1 + threadIdx.x; j < n; j += blockDim.x) {
      const longlong2 e = row[j];
      v[2] += e.x; v[3] += e.y;
      if (lab[j] == li) { v[0] += e.x; v[1] += e.y; v[4] += 1; }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      for (int off = 16; off; off >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], off);
      if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = v[q];
    }
    __syncthreads();
    if (threadIdx.x < 5) {
      long long t = 0;
      for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
      out[(size_t)i * 5 + threadIdx.x] = t;
    }
    __syncthreads();
  }
}


// ---- k-means on the points (Clustering.kmeans(x, k; maxiter), src/prior.jl:63-69 with algo = "k-means") --------------
// Xt: dim x n (a point per column: consecutive threads read consecutive addresses), Xr: n x dim (a point per row: the
// centre update reads whole points), C: k x dim.
__global__ void k_kmn_transpose(const double* __restrict__ Xr, int64_t n, int64_t dim, double* __restrict__ Xt) {
  __shared__ double t[32][33];
  const int64_t j0 = (int64_t)blockIdx.x * 32, d0 = (int64_t)blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t j = j0 + r, d = d0 + threadIdx.x;
    t[r][threadIdx.x] = (j < n && d < dim) ? Xr[(size_t)j * dim + d] : 0.0;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t d = d0 + r, j = j0 + threadIdx.x;
    if (j < n && d < dim) Xt[(size_t)d * n + j] = t[threadIdx.x][r];
  }
}
// block total of one value per thread in a fixed order (128 threads)
__device__ __forceinline__ double kmn_block_sum(double v, double* red) {
  for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}
// k-means++ seeding, one step: squared distance of every point to the newest centre (point *pick), running minimum,
// per-block totals of the minima (the weights of the next draw)
__global__ void __launch_bounds__(128) k_kmn_seed_dist(const double* __restrict__ Xt, const double* __restrict__ Xr, int64_t n, int64_t dim,
                                                      const int* __restrict__ pick, int first, double* __restrict__ mind,
                                                      double* __restrict__ partial) {
  __shared__ double red[4];
  const int64_t j = (int64_t)blockIdx.x * 128 + threadIdx.x;
  const double* c = Xr + (size_t)(*pick) * dim;
  double v = 0.0;
  if (j < n) {
    for (int64_t d = 0; d < dim; ++d) { const double e = Xt[(size_t)d * n + j] - __ldg(c + d); v += e * e; }
    if (!first) v = fmin(v, mind[j]);
    mind[j] = v;
  }
  const double tot = kmn_block_sum(j < n ? v : 0.0, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
// ... and the draw: the first point whose cumulative weight exceeds u * total (u * n-th point when every weight is 0);
// the chosen point becomes centre t
__global__ void __launch_bounds__(128) k_kmn_seed_pick(const double* __restrict__ mind, const double* __restrict__ partial, int nb, int64_t n,
                                                      double u, int fixed, const double* __restrict__ Xr, int64_t dim, double* __restrict__ C, int t,
                                                      int* __restrict__ pick, int* __restrict__ picks) {
  __shared__ int sel;
  if (threadIdx.x == 0) {
    int64_t j = fixed;
    if (fixed < 0) {
      double tot = 0.0;
      for (int b = 0; b < nb; ++b) tot += partial[b];
      if (!(tot > 0.0)) j = (int64_t)(u * (double)n);
      else {
        const double target = u * tot;
        double cum = 0.0;
        int b = 0;
        for (; b < nb - 1 && cum + partial[b] <= target; ++b) cum += partial[b];
        const int64_t lo = (int64_t)b * 128, hi = lo + 128 < n ? lo + 128 : n;
        for (j = lo; j < hi - 1; ++j) { cum += mind[j]; if (cum > target) break; }
      }
      if (j >= n) j = n - 1;
    }
    sel = (int)j; *pick = (int)j;
    if (picks) picks[t] = (int)j;
  }
  __syncthreads();
  for (int64_t d = threadIdx.x; d < dim; d += blockDim.x) C[(size_t)t * dim + d] = Xr[(size_t)sel * dim + d];
}
// k-medoids++ seeding step on the resident matrix: dissimilarity to the newest medoid (its row of D), running minimum,
// per-block totals (Clustering.jl's kmpp on costs: a point is drawn in proportion to its cost itself)
__global__ void __launch_bounds__(128) k_km_seed_dist(const double* __restrict__ D, int64_t n, const int* __restrict__ pick, int first,
                                                     double* __restrict__ mind, double* __restrict__ partial) {
  __shared__ double red[4];
  const int64_t j = (int64_t)blockIdx.x * 128 + threadIdx.x;
  double v = 0.0;
  if (j < n) {
    v = D[(size_t)(*pick) * n + j];
    if (!first) v = fmin(v, mind[j]);
    mind[j] = v;
  }
  const double tot = kmn_block_sum(j < n ? v : 0.0, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
// assignment: nearest centre (first minimum), the point's cost, per-block totals of the costs; out[nb] != 0 when a label
// changed.  Block = 32 points x 8 centre groups: thread (x, y) scans the centres 8 y .. 8 y + 7, 8 (y + 8) .. for point x
// (8 accumulators per read of the point's coordinate), the groups' minima are merged through shared memory.
__global__ void __launch_bounds__(256) k_kmn_assign(const double* __restrict__ Xt, int64_t n, int64_t dim, const double* __restrict__ C, int k,
                                                   int* __restrict__ assign, double* __restrict__ out, int nb) {
  __shared__ double sb[8][32];
  __shared__ int sa[8][32];
  const int x = threadIdx.x, y = threadIdx.y;
  const int64_t j = (int64_t)blockIdx.x * 32 + x;
  double best = 0.0;
  int arg = -1;
  if (j < n) {
    for (int c0 = 8 * y; c0 < k; c0 += 64) {
      double a[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] = 0.0;
      const int kc = k - c0 < 8 ? k - c0 : 8;
      for (int64_t d = 0; d < dim; ++d) {
        const double xv = Xt[(size_t)d * n + j];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (q < kc) { const double e = xv - __ldg(C + (size_t)(c0 + q) * dim + d); a[q] += e * e; }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (q < kc && (arg < 0 || a[q] < best)) { best = a[q]; arg = c0 + q; }
    }
  }
  sb[y][x] = best; sa[y][x] = arg;
  __syncthreads();
  if (y == 0) {
    double cost = 0.0;
    if (j < n) {
      for (int g = 1; g < 8; ++g) {
        const double b = sb[g][x]; const int a = sa[g][x];
        if (a >= 0 && (b < best || (b == best && a < arg))) { best = b; arg = a; }
      }
      if (assign[j] != arg) { assign[j] = arg; out[nb] = 1.0; }
      cost = best;
    }
    for (int off = 16; off; off >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, off);
    if (x == 0) out[blockIdx.x] = cost;
  }
}
// centre update, part 1: block (c, p) adds the members of cluster c among points [p * chunk, (p + 1) * chunk) in index order
__global__ void k_kmn_update_partial(const double* __restrict__ Xr, int64_t n, int64_t dim, const int* __restrict__ assign, int64_t chunk,
                                     double* __restrict__ psum, int* __restrict__ pcnt) {
  const int c = blockIdx.x, p = blockIdx.y, P = gridDim.y;
  const int64_t lo = (int64_t)p * chunk, hi = lo + chunk < n ? lo + chunk : n;
  for (int64_t d0 = 0; d0 < dim; d0 += blockDim.x) {
    const int64_t d = d0 + threadIdx.x;
    double acc = 0.0;
    int cnt = 0;
    for (int64_t j = lo; j < hi; ++j)
      if (assign[j] == c) { ++cnt; if (d < dim) acc += Xr[(size_t)j * dim + d]; }
    if (d < dim) psum[((size_t)c * P + p) * dim + d] = acc;
    if (d0 == 0 && threadIdx.x == 0) pcnt[c * P + p] = cnt;
  }
}
// ... part 2: the mean; an empty cluster keeps its centre
__global__ void k_kmn_update_final(const double* __restrict__ psum, const int* __restrict__ pcnt, int k, int P, int64_t dim, double* __restrict__ C) {
  const int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (int64_t)k * dim) return;
  const int c = (int)(id / dim); const int64_t d = id % dim;
  double s = 0.0; int cnt = 0;
  for (int p = 0; p < P; ++p) { s += psum[((size_t)c * P + p) * dim + d]; cnt += pcnt[c * P + p]; }
  if (cnt > 0) C[id] = s / (double)cnt;
}

struct Scratch {      // frees everything on scope exit
  std::vector<void*> p;
  ~Scratch() { for (void* q : p) rc_dev_free(q); }
  template <class T> cudaError_t get(T** out, size_t count) {
    cudaError_t e = rc_dev_malloc((void**)out, sizeof(T) * (count ? count : 1));
    if (e == cudaSuccess) p.push_back(*out);
    return e;
  }
};

}  // namespace

extern "C" {

int32_t rc_data_copy_row(const rc_data* d, int64_t i, double* row_out) {
  if (!d || !row_out || i < 0 || i >= d->n) { rc_set_error("rc_data_copy_row: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(d->device));
  RC_CUDA(cudaMemcpy(row_out, d->D + (size_t)i * d->n, sizeof(double) * d->n, cudaMemcpyDeviceToHost));
  return RC_OK;
}

int32_t rc_kmedoids_seed(const rc_data* d, int64_t k, const double* u01, int64_t* medoids_out) {
  if (!d || !u01 || !medoids_out || k < 1 || k > d->n) { rc_set_error("rc_kmedoids_seed: bad arguments (need 1 <= k <= n)"); return RC_ERR_ARG; }
  const int64_t n = d->n;
  RC_CUDA(cudaSetDevice(d->device));
  const int nb = (int)((n + 127) / 128);
  Scratch S;
  double *mind, *partial; int *pick, *picks;
  if (S.get(&mind, n) || S.get(&partial, nb) || S.get(&pick, 1) || S.get(&picks, k)) { rc_set_error("rc_kmedoids_seed: out of device memory"); return RC_ERR_CUDA; }
  for (int64_t t = 0; t < k; ++t) {
    const int fixed = t == 0 ? (int)fmin((double)(n - 1), u01[0] * (double)n) : -1;
    k_kmn_seed_pick<<<1, 128>>>(mind, partial, nb, n, u01[t], fixed, nullptr, 0, nullptr, (int)t, pick, picks);
    if (t + 1 < k) k_km_seed_dist<<<nb, 128>>>(d->D, n, pick, t == 0, mind, partial);
  }
  std::vector<int> h((size_t)k);
  RC_CUDA(cudaMemcpy(h.data(), picks, sizeof(int) * k, cudaMemcpyDeviceToHost));
  for (int64_t t = 0; t < k; ++t) medoids_out[t] = h[t];
  return RC_OK;
}

int32_t rc_kmedoids(const rc_data* d, int64_t k, const int64_t* init_medoids, int64_t maxiter, int64_t* assignments,
                    int64_t* medoids, double* totalcost, int32_t* converged, int64_t* iterations) {
  if (!d || !init_medoids || !assignments || !medoids || k < 1 || k > d->n || maxiter < 0) {
    rc_set_error("rc_kmedoids: bad arguments (need 1 <= k <= n)"); return RC_ERR_ARG;
  }
  const int64_t n = d->n;
  RC_CUDA(cudaSetDevice(d->device));
  std::vector<int> hmed((size_t)k);
  for (int64_t c = 0; c < k; ++c) {
    if (init_medoids[c] < 0 || init_medoids[c] >= n) { rc_set_error("rc_kmedoids: initial medoid out of range"); return RC_ERR_ARG; }
    hmed[c] = (int)init_medoids[c];
  }
  Scratch S;
  int *med, *newmed, *assign, *flag, *start, *perm; long long *s, *mins, *partial;
  const int nb = 148 * 4;
  if ((size_t)(k + 1) * sizeof(int) > 200 * 1024) { rc_set_error("rc_kmedoids: k = %lld is beyond the member-list kernel (k <= 51199)", (long long)k); return RC_ERR_ARG; }
  if (S.get(&med, k) || S.get(&newmed, k) || S.get(&assign, n) || S.get(&flag, 2) || S.get(&s, n) || S.get(&mins, k) || S.get(&partial, nb) ||
      S.get(&start, k + 1) || S.get(&perm, n)) {
    rc_set_error("rc_kmedoids: out of device memory"); return RC_ERR_CUDA;
  }
  RC_CUDA(cudaMemcpy(med, hmed.data(), sizeof(int) * k, cudaMemcpyHostToDevice));
  RC_CUDA(cudaMemset(assign, 0xff, sizeof(int) * n));
  if ((size_t)(k + 1) * sizeof(int) > 48 * 1024)
    RC_CUDA(cudaFuncSetAttribute(k_km_members, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) * (k + 1))));
  const unsigned gn = (unsigned)((n + 255) / 256), gk = (unsigned)((k + 255) / 256);
  k_km_assign<<<gn, 256>>>(d->D, n, med, (int)k, assign, flag);
  bool conv = false;
  int64_t it = 0;
  for (; it < maxiter; ++it) {
    RC_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(int)));
    RC_CUDA(cudaMemsetAsync(mins, 0x7f, sizeof(long long) * k));          // 0x7f7f... > any row sum (< 2^61)
    RC_CUDA(cudaMemsetAsync(newmed, 0x7f, sizeof(int) * k));              // 0x7f7f7f7f > any index: start value of the atomicMin
    k_km_members<<<1, 1024, sizeof(int) * (k + 1)>>>(assign, n, (int)k, start, perm);
    k_km_rowsum<<<148 * 8, 256>>>(d->DL, n, assign, start, perm, s);
    k_km_min1<<<gn, 256>>>(s, assign, n, mins);
    k_km_min2<<<gn, 256>>>(s, assign, n, mins, newmed);
    k_km_finish<<<gk, 256>>>(med, (int)k, newmed, flag);
    k_km_assign<<<gn, 256>>>(d->D, n, newmed, (int)k, assign, flag + 1);
    int h[2] = {0, 0};
    RC_CUDA(cudaMemcpy(h, flag, sizeof(h), cudaMemcpyDeviceToHost));
    std::swap(med, newmed);
    if (!h[0] && !h[1]) { conv = true; break; }
  }
  k_km_cost<<<nb, 256>>>(d->DL, n, med, assign, partial);
  std::vector<long long> hp((size_t)nb);
  std::vector<int> ha((size_t)n);
  RC_CUDA(cudaMemcpy(hp.data(), partial, sizeof(long long) * nb, cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(ha.data(), assign, sizeof(int) * n, cudaMemcpyDeviceToHost));
  RC_CUDA(cudaMemcpy(hmed.data(), med, sizeof(int) * k, cudaMemcpyDeviceToHost));
  rc_i128 tot = {0ull, 0ll};
  for (long long v : hp) rc_add128(tot, v);
  for (int64_t i = 0; i < n; ++i) assignments[i] = (int64_t)ha[i] + 1;
  for (int64_t c = 0; c < k; ++c) medoids[c] = hmed[c];
  if (totalcost) *totalcost = rc_deq128(tot, d->qD);
  if (converged) *converged = conv ? 1 : 0;
  if (iterations) *iterations = it + (conv ? 1 : 0);
  return RC_OK;
}

int32_t rc_kmeans(const double* X, int64_t n, int64_t dim, int64_t k, const int64_t* init_idx, const double* u01, int64_t maxiter,
                  double tol, int32_t device, int64_t* assignments, double* centers, double* totalcost, int32_t* converged,
                  int64_t* iterations) {
  if (!X || !assignments || n < 1 || dim < 1 || k < 1 || k > n || maxiter < 0 || (!init_idx && !u01) || n > 0x7fffff00LL || k > 0x7fffffLL) {
    rc_set_error("rc_kmeans: bad arguments (need 1 <= k <= n, dim >= 1 and either init_idx or u01)"); return RC_ERR_ARG;
  }
  const int st = rc_select_device(device);
  if (st) return st;
  if (init_idx)
    for (int64_t c = 0; c < k; ++c)
      if (init_idx[c] < 0 || init_idx[c] >= n) { rc_set_error("rc_kmeans: initial centre index out of range"); return RC_ERR_ARG; }
  const int nb = (int)((n + 127) / 128), nba = (int)((n + 31) / 32);          // blocks of the seeding / of the assignment
  int P = (int)(592 / k); if (P < 1) P = 1; if (P > 64) P = 64;
  while (P > 1 && (n + P - 1) / P < 64) --P;
  const int64_t chunk = (n + P - 1) / P;
  Scratch S;
  double *Xr, *Xt, *C, *mind, *out, *psum; int *assign, *pick, *pcnt;
  if (S.get(&Xr, (size_t)n * dim) || S.get(&Xt, (size_t)n * dim) || S.get(&C, (size_t)k * dim) || S.get(&mind, n) || S.get(&out, (size_t)nba + 1) ||
      S.get(&psum, (size_t)k * P * dim) || S.get(&assign, n) || S.get(&pick, 1) || S.get(&pcnt, (size_t)k * P)) {
    rc_set_error("rc_kmeans: out of device memory"); return RC_ERR_CUDA;
  }
  RC_CUDA(cudaMemcpy(Xr, X, sizeof(double) * n * dim, cudaMemcpyHostToDevice));
  k_kmn_transpose<<<dim3((unsigned)((n + 31) / 32), (unsigned)((dim + 31) / 32)), dim3(32, 8)>>>(Xr, n, dim, Xt);
  // seeding: the given points, or k-means++ (first centre uniform, then proportional to the squared distance to the nearest centre)
  for (int64_t t = 0; t < k; ++t) {
    const int fixed = init_idx ? (int)init_idx[t] : (t == 0 ? (int)fmin((double)(n - 1), u01[0] * (double)n) : -1);
    k_kmn_seed_pick<<<1, 128>>>(mind, out, nb, n, init_idx ? 0.0 : u01[t], fixed, Xr, dim, C, (int)t, pick, nullptr);
    if (!init_idx && t + 1 < k) k_kmn_seed_dist<<<nb, 128>>>(Xt, Xr, n, dim, pick, t == 0, mind, out);
  }
  RC_CUDA(cudaMemset(assign, 0xff, sizeof(int) * n));
  std::vector<double> h((size_t)nba + 1);
  auto assign_pass = [&](double* objv, bool* changed) -> cudaError_t {
    cudaError_t e = cudaMemsetAsync(out + nba, 0, sizeof(double));
    if (e != cudaSuccess) return e;
    k_kmn_assign<<<nba, dim3(32, 8)>>>(Xt, n, dim, C, (int)k, assign, out, nba);
    e = cudaMemcpy(h.data(), out, sizeof(double) * (nba + 1), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return e;
    double s = 0.0;
    for (int b = 0; b < nba; ++b) s += h[b];
    *objv = s; *changed = h[nba] != 0.0;
    return cudaSuccess;
  };
  double objv = 0.0; bool changed = true, conv = false;
  RC_CUDA(assign_pass(&objv, &changed));
  int64_t it = 0;
  while (!conv && it < maxiter) {
    ++it;
    const unsigned tu = (unsigned)(dim < 256 ? ((dim + 31) / 32) * 32 : 256);
    k_kmn_update_partial<<<dim3((unsigned)k, (unsigned)P), tu>>>(Xr, n, dim, assign, chunk, psum, pcnt);
    k_kmn_update_final<<<(unsigned)((k * dim + 255) / 256), 256>>>(psum, pcnt, (int)k, P, dim, C);
    double prev = objv;
    RC_CUDA(assign_pass(&objv, &changed));
    if (k == 1 || !changed || fabs(objv - prev) < tol) conv = true;          // Clustering.jl: |change of the objective| < tol
  }
  std::vector<int> ha((size_t)n);
  RC_CUDA(cudaMemcpy(ha.data(), assign, sizeof(int) * n, cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < n; ++i) assignments[i] = (int64_t)ha[i] + 1;
  if (centers) RC_CUDA(cudaMemcpy(centers, C, sizeof(double) * k * dim, cudaMemcpyDeviceToHost));
  if (totalcost) *totalcost = objv;
  if (converged) *converged = conv ? 1 : 0;
  if (iterations) *iterations = it;
  return RC_OK;
}

int32_t rc_pair_stats(const rc_data* d, const int64_t* labels, int64_t* rows_out) {
  if (!d || !labels || !rows_out) { rc_set_error("rc_pair_stats: null pointer"); return RC_ERR_ARG; }
  const int64_t n = d->n;
  RC_CUDA(cudaSetDevice(d->device));
  std::vector<int> hl((size_t)n);
  for (int64_t i = 0; i < n; ++i) hl[i] = (int)labels[i];
  Scratch S;
  int* lab; long long* out;
  if (S.get(&lab, n) || S.get(&out, 5 * n)) { rc_set_error("rc_pair_stats: out of device memory"); return RC_ERR_CUDA; }
  RC_CUDA(cudaMemcpy(lab, hl.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
  k_pair_rows<<<148 * 8, 256>>>(d->DL, n, lab, out);
  RC_CUDA(cudaMemcpy(rows_out, out, sizeof(long long) * 5 * n, cudaMemcpyDeviceToHost));
  return RC_OK;
}

}  // extern "C"
