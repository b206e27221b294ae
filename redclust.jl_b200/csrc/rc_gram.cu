// rc_gram.cu -- the two dense contractions of the path on the FP64 tensor cores (DMMA; tcgen05 has no f64 kind, so on
// sm_100a fp64 matrix math is the warp-level mma.sync.m8n8k4 -- SASS DMMA.8x8x4; the larger PTX shapes lower to the same
// instruction):
//   * pairwise(Euclidean(), X, dims=2) (src/types.jl:160, src/utils.jl:144-145, src/prior.jl:51,180): the Gram block
//     X_i X_j^T, epilogue sqrt(max(|x_i|^2 + |x_j|^2 - 2 g, 0)) (an entry it cannot resolve recomputed from the
//     differences, rc_math.h), exact zero diagonal, upper-triangle tiles mirrored;
//   * the oracle co-clustering matrix of generatemixture (src/utils.jl:130-143): sum over 5000 Dirichlet draws of P'P --
//     a Gram matrix of the stacked posterior rows, accumulated chunk by chunk.
// One kernel serves both: C tile 128 x 128 per CTA, 8 warps as 2 x 4 (warp tile 64 x 32 = 8 x 4 DMMA tiles, 64 fp64
// accumulators per thread), operands K-contiguous ("TN"), staged in 16-coordinate chunks by cp.async into a double-
// buffered shared-memory ring whose row pitch (20 doubles) makes the fragment loads conflict-free.  The finished tile
// goes through shared memory so that both the tile and its mirror image are written with coalesced rows.
#include <vector>
#include "rc_common.cuh"

namespace {

constexpr int GT = 128;        // C tile edge
constexpr int GK = 16;         // coordinates per staged chunk
constexpr int GP = GK + 4;     // shared-memory row pitch in doubles (160 B: the 8 rows of a fragment hit 8 bank groups)
constexpr int GTP = GT + 1;    // pitch of the staged C tile
constexpr int GS = 3;          // stages of the operand ring (two chunks in flight while one is multiplied)

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct EpiDist {          // Euclidean distances from the Gram block
  const double* sq;       // |x_i|^2
  double* D;              // n x n
  int64_t n;
  int* flags;             // unused here (the checks run in finish_data)
};
struct EpiAccum {         // C += G on the upper-triangle tiles (mirrored and scaled afterwards)
  double* C;
  int64_t n;
};

// A: M x Kd, Bm: N x Kd, both row-major (K contiguous), Kd a multiple of GK, 16-byte aligned rows; C = A Bm^T.
// SYM: Bm == A and only the tiles with bj >= bi are computed (the epilogue mirrors them); otherwise the grid is
// (column tiles, row tiles).  An entry's value does not depend on which tile computes it or on the operand order
// (same coordinates in the same order, products commute), so a row block equals the same rows of the symmetric build.
template <class Epi, bool SYM>
__global__ void __launch_bounds__(256, 1) k_gram128(const double* __restrict__ A, int64_t M, const double* __restrict__ Bm, int64_t N,
                                                    int64_t Kd, Epi epi) {
  int bi, bj;
  if (SYM) {                                 // tile index -> (bi, bj) of the upper triangle, row by row
    const int nb = (int)((M + GT - 1) / GT);
    int rem = blockIdx.x;
    bi = 0;
    while (rem >= nb - bi) { rem -= nb - bi; ++bi; }
    bj = bi + rem;
  } else { bi = blockIdx.y; bj = blockIdx.x; }
  extern __shared__ __align__(16) double gsm[];
  double* As = gsm;                          // [GS][GT][GP]
  double* Bs = gsm + GS * GT * GP;           // [GS][GT][GP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 2, wn = warp & 3;   // 2 x 4 warps: rows wm*64.., columns wn*32..
  const int fr = lane >> 2, fk = lane & 3;   // fragment row (A) / column (B), k index
  const int64_t i0 = (int64_t)bi * GT, j0 = (int64_t)bj * GT;
  double acc[8][4][2];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }

  auto stage = [&](int buf, int64_t k0) {
    // 128 rows x 8 16-byte pieces per operand; thread t moves pieces t, t + 256, ... (a row's pieces are consecutive)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + q * 256, r = e >> 3, c = e & 7;
      const int64_t ra = min(i0 + r, M - 1), rb = min(j0 + r, N - 1);       // rows beyond the end repeat the last one (discarded later)
      cp_async16(As + ((size_t)buf * GT + r) * GP + 2 * c, A + ra * Kd + k0 + 2 * c);
      cp_async16(Bs + ((size_t)buf * GT + r) * GP + 2 * c, Bm + rb * Kd + k0 + 2 * c);
    }
    cp_async_commit();
  };
  const int nchunk = (int)(Kd / GK);
  stage(0, 0);
  if (nchunk > 1) stage(1, GK);
  for (int ch = 0; ch < nchunk; ++ch) {
    const int buf = ch % GS;
    if (ch + 2 < nchunk) { stage((ch + 2) % GS, (int64_t)(ch + 2) * GK); cp_async_wait<2>(); }   // (its slot was released by the barrier that ended chunk ch - 1)
    else if (ch + 1 < nchunk) cp_async_wait<1>();
    else cp_async_wait<0>();
    __syncthreads();
    const double* as = As + (size_t)buf * GT * GP + (size_t)(wm * 64 + fr) * GP + fk;
    const double* bs = Bs + (size_t)buf * GT * GP + (size_t)(wn * 32 + fr) * GP + fk;
#pragma unroll
    for (int k = 0; k < GK; k += 4) {
      double af[8], bf[4];
#pragma unroll
      for (int a = 0; a < 8; ++a) af[a] = as[(size_t)a * 8 * GP + k];
#pragma unroll
      for (int b = 0; b < 4; ++b) bf[b] = bs[(size_t)b * 8 * GP + k];
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                       : "+d"(acc[a][b][0]), "+d"(acc[a][b][1]) : "d"(af[a]), "d"(bf[b]));
    }
    __syncthreads();
  }
  // the finished tile through shared memory: T[r][c], pitch GTP (the operand ring is dead now)
  double* T = gsm;
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int r = wm * 64 + a * 8 + fr, c = wn * 32 + b * 8 + 2 * fk;     // C fragment: row lane / 4, columns 2 (lane % 4) + {0, 1}
      T[(size_t)r * GTP + c] = acc[a][b][0];
      T[(size_t)r * GTP + c + 1] = acc[a][b][1];
    }
  __syncthreads();
  epi.store(T, i0, j0, SYM && bi == bj, SYM, tid);
}

// ---- epilogues -------------------------------------------------------------------------------------------------------
struct EpiDistImpl : EpiDist {
  int64_t row0, nrows;     // row block [row0, row0 + nrows) of the matrix held by D (row0 = 0, nrows = n for the whole matrix)
  const double* Xp;        // the padded points (n x Kd): an entry the Gram form cannot resolve is recomputed from them
  int64_t Kd;              // (the padding adds exact zeros to the direct sum)
  __device__ __forceinline__ void store(double* T, int64_t i0, int64_t j0, bool diag, bool sym, int tid) const {
    // rows of the tile: thread t handles column t % 128 of rows t / 128, t / 128 + 2, ...
    const int c = tid & (GT - 1);
    bool redo = false;
#pragma unroll 8
    for (int r = tid >> 7; r < GT; r += 2) {                                // (unrolled: the fp64 square roots of several rows overlap)
      const int64_t il = i0 + r, i = row0 + il, j = j0 + c;                 // il: row within the block
      if (il >= nrows || j >= n) continue;
      double v = 0.0;
      if (i != j) {
        const double s = sq[i] + sq[j], w = s - 2 * T[(size_t)r * GTP + c];
        v = sqrt(w > 0.0 ? w : 0.0);
        if (rc_dist_unresolved(w, s)) { v = -1.0; redo = true; }            // marked for the loop below
      }
      D[il * n + j] = v;
      T[(size_t)r * GTP + c] = v;                                            // the mirror image below copies it (one square root per pair)
    }
    // the unresolved entries, out of the unrolled loop, so that tiles without any pay only the test (with the direct sum
    // inside it the kernel took 9 % longer on the bench points, where no entry is recomputed; B200 at 1000 W)
    if (redo)
      for (int r = tid >> 7; r < GT; r += 2) {
        const int64_t il = i0 + r, i = row0 + il, j = j0 + c;
        if (il >= nrows || j >= n || !(T[(size_t)r * GTP + c] < 0.0)) continue;
        const double v = sqrt(rc_dist_direct2(Xp + i * Kd, Xp + j * Kd, Kd));
        D[il * n + j] = v;
        T[(size_t)r * GTP + c] = v;
      }
    if (diag || !sym) return;
    __syncthreads();
    // the mirror image: row j0 + c of D, columns i0 + r (r fastest across the threads: column reads of T, pitch 129)
    const int r = tid & (GT - 1);
#pragma unroll 8
    for (int cc = tid >> 7; cc < GT; cc += 2) {
      const int64_t i = i0 + r, j = j0 + cc;
      if (i >= n || j >= n) continue;
      D[j * n + i] = T[(size_t)r * GTP + cc];
    }
  }
};
struct EpiAccumImpl : EpiAccum {
  __device__ __forceinline__ void store(double* T, int64_t i0, int64_t j0, bool diag, bool sym, int tid) const {
    const int c = tid & (GT - 1);
    for (int r = tid >> 7; r < GT; r += 2) {
      const int64_t i = i0 + r, j = j0 + c;
      if (i >= n || j >= n) continue;
      C[i * n + j] += T[(size_t)r * GTP + c];
    }
  }
};

// |x_i|^2 of padded rows (ascending coordinates)
__global__ void k_sqnorm_pad(const double* __restrict__ X, int64_t Kd, int64_t n, double* __restrict__ sq) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a = 0.0;
  for (int64_t t = 0; t < Kd; ++t) { const double x = X[i * Kd + t]; a += x * x; }
  sq[i] = a;
}
// rows of X (n x dim) into zero-padded rows of Kd coordinates
__global__ void k_pad_rows(const double* __restrict__ X, int64_t dim, int64_t Kd, int64_t n, double* __restrict__ out) {
  const int64_t total = n * Kd;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / Kd, k = t - i * Kd;
    out[t] = k < dim ? X[i * dim + k] : 0.0;
  }
}

// posterior responsibilities of generatemixture's oracle (src/utils.jl:134-140) for draws t0 .. t0 + B - 1:
// Q[i][(t - t0) K + j] = w_tj N(x_i; c_j, sigma^2 I) / sum_j', c_j = radius e_j, evaluated as a softmax of
// log w_tj - |x_i - c_j|^2 / (2 sigma^2) (the common factor of the densities cancels).  Columns beyond B K are zero.
__global__ void k_posterior(const double* __restrict__ X, int64_t dim, int64_t n, int K, double radius, double inv2s2,
                            const double* __restrict__ logW, int64_t t0, int B, int64_t Kd, double* __restrict__ Q) {
  const int64_t total = n * (int64_t)B;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / B; const int t = (int)(e - i * B);
    const double* x = X + i * dim;
    double x2 = 0.0;
    for (int64_t d = 0; d < dim; ++d) x2 += x[d] * x[d];
    const double* lw = logW + (t0 + t) * K;
    double mx = -RC_INF;
    for (int j = 0; j < K; ++j) {
      const double d2 = x2 - 2.0 * radius * x[j] + radius * radius;
      const double l = lw[j] - d2 * inv2s2;
      mx = l > mx ? l : mx;
    }
    double s = 0.0;
    for (int j = 0; j < K; ++j) {
      const double d2 = x2 - 2.0 * radius * x[j] + radius * radius;
      s += exp(lw[j] - d2 * inv2s2 - mx);
    }
    double* q = Q + i * Kd + (int64_t)t * K;
    for (int j = 0; j < K; ++j) {
      const double d2 = x2 - 2.0 * radius * x[j] + radius * radius;
      q[j] = exp(lw[j] - d2 * inv2s2 - mx) / s;
    }
  }
}
__global__ void k_zero_tail(double* __restrict__ Q, int64_t n, int64_t Kd, int64_t used) {
  const int64_t w = Kd - used, total = n * w;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / w, k = used + (e - i * w);
    Q[i * Kd + k] = 0.0;
  }
}
// upper triangle (tile-wise complete: every entry of the tiles bj >= bi) scaled and mirrored into the lower one
__global__ void k_scale_mirror(double* __restrict__ C, int64_t n, double scale) {
  const int64_t total = n * n;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / n, j = e - i * n;
    if (j >= i) { const double v = C[e] * scale; C[e] = v; if (j > i) C[j * n + i] = v; }
  }
}

size_t gram_smem() { return sizeof(double) * (size_t)std::max(2 * GS * GT * GP, GT * GTP); }

}  // namespace

// Rows [row0, row0 + nrows) of the distance matrix of n points (rows of X, dim coordinates) on the FP64 tensor cores into
// D_dev (nrows x n).  The whole matrix (row0 = 0, nrows = n) computes the upper-triangle tiles and mirrors them.
int rc_distm_dmma(const double* X_dev, int64_t dim, int64_t n, int64_t row0, int64_t nrows, double* D_dev) {
  const int64_t Kd = (dim + GK - 1) / GK * GK;
  double *Xp = nullptr, *sq = nullptr;
  if (cudaMalloc(&Xp, sizeof(double) * (size_t)n * Kd) != cudaSuccess || cudaMalloc(&sq, sizeof(double) * (size_t)n) != cudaSuccess) {
    cudaFree(Xp); cudaFree(sq); rc_set_error("out of device memory for the padded points"); return RC_ERR_CUDA;
  }
  k_pad_rows<<<1024, 256>>>(X_dev, dim, Kd, n, Xp);
  k_sqnorm_pad<<<(unsigned)((n + 255) / 256), 256>>>(Xp, Kd, n, sq);
  const int nb = (int)((n + GT - 1) / GT);
  EpiDistImpl epi; epi.sq = sq; epi.D = D_dev; epi.n = n; epi.flags = nullptr; epi.row0 = row0; epi.nrows = nrows; epi.Xp = Xp; epi.Kd = Kd;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
  if (verbose) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0); }
  if (row0 == 0 && nrows == n) {
    cudaFuncSetAttribute(k_gram128<EpiDistImpl, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gram_smem());
    k_gram128<EpiDistImpl, true><<<nb * (nb + 1) / 2, 256, gram_smem()>>>(Xp, n, Xp, n, Kd, epi);
  } else if (nrows > 0) {
    cudaFuncSetAttribute(k_gram128<EpiDistImpl, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gram_smem());
    k_gram128<EpiDistImpl, false><<<dim3(nb, (unsigned)((nrows + GT - 1) / GT)), 256, gram_smem()>>>(Xp + row0 * Kd, nrows, Xp, n, Kd, epi);
  }
  if (verbose) cudaEventRecord(e1);
  cudaError_t e = cudaDeviceSynchronize();
  if (verbose && e == cudaSuccess) {
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    const double tiles = (row0 == 0 && nrows == n) ? 0.5 * nb * (nb + 1) : (double)nb * ((nrows + GT - 1) / GT);
    const double flop = tiles * 2.0 * GT * GT * (double)Kd;      // executed DMMA work (padded tiles and coordinates included)
    fprintf(stderr, "[rcb200] k_gram128 (distances) n=%lld dim=%lld rows=%lld: %.3f ms, %.2f TFLOP/s executed on the fp64 tensor pipe (%.2f algorithmic 2 n^2 dim)\n",
            (long long)n, (long long)dim, (long long)nrows, ms, flop / ms / 1e9, 2.0 * (double)nrows * n * dim / ms / 1e9);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  cudaFree(Xp); cudaFree(sq);
  if (e != cudaSuccess) { rc_set_error("distance kernel failed: %s", cudaGetErrorString(e)); return RC_ERR_CUDA; }
  return RC_OK;
}

extern "C" {

// generatemixture's oracle co-clustering matrix (src/utils.jl:130-143) for given points and Dirichlet draws:
// out[i][j] = (1 / numiters) sum_t sum_k P_t[k][i] P_t[k][j].  X: n x dim row-major (host), W: numiters x K (host).
int32_t rc_oracle_coclustering(const double* X, int64_t dim, int64_t n, int64_t K, double radius, double sigma, const double* W,
                               int64_t numiters, int32_t device, double* out) {
  if (!X || !W || !out || n < 1 || dim < 1 || K < 1 || K > dim || numiters < 1 || !(sigma > 0)) {
    rc_set_error("rc_oracle_coclustering: bad arguments"); return RC_ERR_ARG;
  }
  const int st = rc_select_device(device);
  if (st) return st;
  // draws per chunk: the stacked posterior rows of a chunk are one n x (B K) operand of at most ~1 GB
  int64_t B = std::max<int64_t>(1, std::min<int64_t>(numiters, ((int64_t)1 << 27) / std::max<int64_t>(1, n * K)));
  const int64_t Kd = (B * K + GK - 1) / GK * GK;
  std::vector<double> logW((size_t)numiters * K);
  for (size_t t = 0; t < logW.size(); ++t) logW[t] = log(W[t]);
  double *dX = nullptr, *dlw = nullptr, *Q = nullptr, *C = nullptr;
  cudaError_t e = cudaMalloc(&dX, sizeof(double) * (size_t)n * dim);
  if (e == cudaSuccess) e = cudaMalloc(&dlw, sizeof(double) * logW.size());
  if (e == cudaSuccess) e = cudaMalloc(&Q, sizeof(double) * (size_t)n * Kd);
  if (e == cudaSuccess) e = cudaMalloc(&C, sizeof(double) * (size_t)n * n);
  if (e == cudaSuccess) e = cudaMemcpy(dX, X, sizeof(double) * (size_t)n * dim, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dlw, logW.data(), sizeof(double) * logW.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(C, 0, sizeof(double) * (size_t)n * n);
  if (e == cudaSuccess) {
    const int nb = (int)((n + GT - 1) / GT);
    EpiAccumImpl epi; epi.C = C; epi.n = n;
    cudaFuncSetAttribute(k_gram128<EpiAccumImpl, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gram_smem());
    const bool verbose = getenv("RCB200_VERBOSE") != nullptr;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float gram_ms = 0; double gram_flop = 0;
    for (int64_t t0 = 0; t0 < numiters; t0 += B) {
      const int b = (int)std::min<int64_t>(B, numiters - t0);
      k_posterior<<<2048, 256>>>(dX, dim, n, (int)K, radius, 1.0 / (2.0 * sigma * sigma), dlw, t0, b, Kd, Q);
      if ((int64_t)b * K < Kd) k_zero_tail<<<512, 256>>>(Q, n, Kd, (int64_t)b * K);
      if (verbose) cudaEventRecord(e0);
      k_gram128<EpiAccumImpl, true><<<nb * (nb + 1) / 2, 256, gram_smem()>>>(Q, n, Q, n, Kd, epi);
      if (verbose) { cudaEventRecord(e1); cudaEventSynchronize(e1); float ms = 0; cudaEventElapsedTime(&ms, e0, e1); gram_ms += ms; gram_flop += 0.5 * nb * (nb + 1) * 2.0 * GT * GT * (double)Kd; }
    }
    k_scale_mirror<<<2048, 256>>>(C, n, 1.0 / (double)numiters);
    e = cudaDeviceSynchronize();
    if (verbose) fprintf(stderr, "[rcb200] k_gram128 (oracle co-clustering) n=%lld inner=%lld x %lld draws: %.1f ms in the Gram launches, %.2f TFLOP/s executed on the fp64 tensor pipe\n",
                         (long long)n, (long long)K, (long long)numiters, gram_ms, gram_flop / gram_ms / 1e9);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, C, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToHost);
  cudaFree(dX); cudaFree(dlw); cudaFree(Q); cudaFree(C);
  RC_CUDA(e);
  return RC_OK;
}

}  // extern "C"
