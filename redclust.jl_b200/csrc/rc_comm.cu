// rc_comm.cu -- the three exchange steps of the path behind the C ABI (SURVEY.md 8b / 8e): one NCCL communicator per
// handle, created from a unique id that the launcher distributes (torch.distributed, MPI, Julia's Distributed -- the
// library does not care).  NCCL is resolved at run time (dlopen of libnccl.so.2: whichever copy the process already
// holds, e.g. PyTorch's), so librcb200.so itself loads on a machine without NCCL.
//
//   distance build   row blocks                  -> ncclAllGather of the n x n fp64 matrix (src/types.jl:159-162)
//   PSM              sample shards (chains are)  -> ncclAllReduce(sum) of the n x n int32 counts (src/mcmc.jl:560)
//   MPEL             candidate rows, cyclic deal -> ncclAllGather of the S x S loss rows (src/pointestimate.jl:49-57)
// The sampler itself has no collective: chains are independent (chain_offset of rc_sampler_create).
#include <dlfcn.h>
#include <string.h>
#include <vector>
#include "rc_common.cuh"

namespace {

// the slice of nccl.h this file needs (ABI-stable since NCCL 2.0)
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclSuccess = 0 };
enum { ncclInt32 = 2, ncclInt64 = 4, ncclFloat64 = 8 };   // ncclDataType_t
enum { ncclSum = 0 };                                     // ncclRedOp_t

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

NcclApi* nccl() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {getenv("RCB200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      if (!nm) continue;
      api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (api.handle) {
      api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
      api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
      api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
      api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
      api.AllGather = (decltype(api.AllGather))dlsym(api.handle, "ncclAllGather");
      api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
      if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.AllGather) api.handle = nullptr;
    }
  }
  return api.handle ? &api : nullptr;
}

#define RC_NCCL(call)                                                                                          \
  do {                                                                                                         \
    ncclResult_t r_ = (call);                                                                                  \
    if (r_ != ncclSuccess) {                                                                                   \
      rc_set_error("NCCL error %d at %s:%d: %s", (int)r_, __FILE__, __LINE__,                                  \
                   nccl()->GetErrorString ? nccl()->GetErrorString(r_) : "?");                                 \
      return RC_ERR_CUDA;                                                                                      \
    }                                                                                                          \
  } while (0)

// all-gathered cyclic deal (rank-major blocks of `per` rows) -> rows in natural order: out[r + k * world] = in[r][k]
__global__ void k_uncycle(const double* __restrict__ in, double* __restrict__ out, int64_t S, int world, int64_t per) {
  const int64_t total = S * S;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = t / S, col = t - row * S;
    out[t] = in[((row % world) * per + row / world) * S + col];
  }
}

}  // namespace

struct rc_comm {
  ncclComm_t comm;
  int rank, world, device;
  cudaStream_t stream;
};

extern "C" {

int32_t rc_comm_unique_id(uint8_t* id128) {
  if (!id128) { rc_set_error("rc_comm_unique_id: null pointer"); return RC_ERR_ARG; }
  NcclApi* a = nccl();
  if (!a) { rc_set_error("NCCL is not available (libnccl.so.2 could not be loaded)"); return RC_ERR_CUDA; }
  ncclUniqueId id;
  RC_NCCL(a->GetUniqueId(&id));
  memcpy(id128, id.internal, 128);
  return RC_OK;
}

int32_t rc_comm_init(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, rc_comm** out) {
  if (!id128 || !out || world < 1 || rank < 0 || rank >= world) { rc_set_error("rc_comm_init: bad arguments"); return RC_ERR_ARG; }
  NcclApi* a = nccl();
  if (!a) { rc_set_error("NCCL is not available (libnccl.so.2 could not be loaded)"); return RC_ERR_CUDA; }
  RC_CUDA(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(id.internal, id128, 128);
  rc_comm* c = new rc_comm();
  c->rank = rank; c->world = world; c->device = device; c->comm = nullptr; c->stream = nullptr;
  ncclResult_t r = a->CommInitRank(&c->comm, world, id, rank);
  if (r != ncclSuccess) { rc_set_error("ncclCommInitRank failed: %s", a->GetErrorString ? a->GetErrorString(r) : "?"); delete c; return RC_ERR_CUDA; }
  if (cudaStreamCreate(&c->stream) != cudaSuccess) { a->CommDestroy(c->comm); delete c; rc_set_error("cudaStreamCreate failed"); return RC_ERR_CUDA; }
  // NCCL connects its channels lazily on the first collective (tens of milliseconds): pay that here, not in the first
  // PSM exchange (round 1 timed a 64 MB all-reduce at 118 ms because it was the communicator's first)
  {
    int* w = nullptr;
    if (cudaMalloc(&w, 256 * sizeof(int)) == cudaSuccess) {
      cudaMemset(w, 0, 256 * sizeof(int));
      a->AllReduce(w, w, 256, ncclInt32, ncclSum, c->comm, c->stream);
      a->AllGather(w, w, 256 / world, ncclInt32, c->comm, c->stream);
      cudaStreamSynchronize(c->stream);
      cudaFree(w);
    }
  }
  *out = c;
  return RC_OK;
}

int32_t rc_comm_info(const rc_comm* c, int32_t* rank, int32_t* world) {
  if (!c) { rc_set_error("rc_comm_info: null handle"); return RC_ERR_ARG; }
  if (rank) *rank = c->rank;
  if (world) *world = c->world;
  return RC_OK;
}

void rc_comm_destroy(rc_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->comm && nccl()) nccl()->CommDestroy(c->comm);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// sum of an int32 device matrix over the ranks, in place (the PSM exchange step).
int32_t rc_comm_allreduce_i32(rc_comm* c, void* buf_dev, int64_t count) {
  if (!c || !buf_dev || count < 0) { rc_set_error("rc_comm_allreduce_i32: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  RC_CUDA(cudaDeviceSynchronize());                       // producers of the buffer ran on other streams
  RC_NCCL(nccl()->AllReduce(buf_dev, buf_dev, (size_t)count, ncclInt32, ncclSum, c->comm, c->stream));
  RC_CUDA(cudaStreamSynchronize(c->stream));
  return RC_OK;
}

// MCMCData(points) with the distance build split into row blocks (src/types.jl:159-162 across GPUs): this rank's rows,
// one all-gather, then the checks / logD / fixed-point images on the complete device-resident matrix.  Bit-equal to
// rc_data_from_points on one GPU.
int32_t rc_comm_data_from_points(rc_comm* c, const double* X, int64_t dim, int64_t n, rc_data** out) {
  if (!c || !X || !out || n < 1 || dim < 1) { rc_set_error("rc_comm_data_from_points: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const int64_t per = (n + c->world - 1) / c->world;                  // equal blocks, the last one padded
  double* full = nullptr;
  RC_CUDA(cudaMalloc(&full, sizeof(double) * (size_t)per * c->world * n));
  const int64_t row0 = std::min<int64_t>((int64_t)c->rank * per, n), nrows = std::min<int64_t>(per, n - row0);
  double* mine = full + (size_t)c->rank * per * n;
  int st = RC_OK;
  if (nrows < per) st = cudaMemset(mine, 0, sizeof(double) * (size_t)per * n) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!st) st = rc_distm_rows_dev(X, dim, n, row0, nrows, c->device, mine);
  if (!st && c->world > 1) {
    ncclResult_t r = nccl()->AllGather(mine, full, (size_t)per * n, ncclFloat64, c->comm, c->stream);
    if (r != ncclSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) { rc_set_error("all-gather of the distance rows failed"); st = RC_ERR_CUDA; }
  }
  if (!st) st = rc_data_from_dist_dev(full, n, c->device, out);
  cudaFree(full);
  return st;
}

// PSM over the samples of every rank (src/mcmc.jl:560 across chain shards): exact int32 counts per rank, ONE all-reduce
// of the n x n matrix, one divide by the global number of samples.  psm_out (host n x n fp64) may be NULL when only
// counts_dev_out (device n x n int32, may be NULL too) is wanted.
static int32_t finish_psm(rc_comm* c, int* counts, int64_t n, long long local_samples, double* psm_out) {
  long long* tot = nullptr;
  RC_CUDA(cudaMalloc(&tot, sizeof(long long)));
  RC_CUDA(cudaMemcpy(tot, &local_samples, sizeof(long long), cudaMemcpyHostToDevice));
  RC_CUDA(cudaDeviceSynchronize());
  if (c->world > 1) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->stream);
    RC_NCCL(nccl()->AllReduce(counts, counts, (size_t)n * n, ncclInt32, ncclSum, c->comm, c->stream));
    cudaEventRecord(e1, c->stream);
    RC_NCCL(nccl()->AllReduce(tot, tot, 1, ncclInt64, ncclSum, c->comm, c->stream));
    RC_CUDA(cudaStreamSynchronize(c->stream));
    if (getenv("RCB200_VERBOSE")) {
      float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
      const double bytes = 4.0 * (double)n * (double)n;
      fprintf(stderr, "[rcb200] rank %d: ncclAllReduce of the %lld x %lld int32 counts (%.2f GB): %.2f ms, algorithm bandwidth %.1f GB/s, bus bandwidth %.1f GB/s\n",
              c->rank, (long long)n, (long long)n, bytes / 1e9, ms, bytes / ms / 1e6, bytes / ms / 1e6 * 2.0 * (c->world - 1) / c->world);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  long long total = 0;
  RC_CUDA(cudaMemcpy(&total, tot, sizeof(long long), cudaMemcpyDeviceToHost));
  cudaFree(tot);
  if (psm_out) return rc_counts_to_host_psm(counts, (size_t)n * n, (double)total, psm_out);
  return RC_OK;
}

int32_t rc_comm_sampler_psm(rc_comm* c, const rc_sampler* s, double* psm_out, void* counts_dev_out) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_psm: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const int64_t n = rc_sampler_n(s), nch = rc_sampler_nchains(s), S = rc_sampler_numsamples(s);
  int* counts = (int*)counts_dev_out;
  if (!counts) RC_CUDA(cudaMalloc(&counts, sizeof(int) * (size_t)n * n));
  int st = rc_sampler_psm_counts_dev(s, 0, nch, counts);
  if (!st) st = finish_psm(c, counts, n, (long long)(nch * S), psm_out);
  if (!counts_dev_out) cudaFree(counts);
  return st;
}

int32_t rc_comm_psm(rc_comm* c, const int64_t* labels, int64_t S_local, int64_t n, double* psm_out, void* counts_dev_out) {
  if (!c || (!labels && S_local > 0) || n < 1 || S_local < 0) { rc_set_error("rc_comm_psm: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  int* counts = (int*)counts_dev_out;
  if (!counts) RC_CUDA(cudaMalloc(&counts, sizeof(int) * (size_t)n * n));
  int st = RC_OK;
  if (S_local > 0) st = rc_psm_counts_dev(labels, S_local, n, c->device, counts);
  else st = cudaMemset(counts, 0, sizeof(int) * (size_t)n * n) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!st) st = finish_psm(c, counts, n, (long long)S_local, psm_out);
  if (!counts_dev_out) cudaFree(counts);
  return st;
}

// Binder MPEL over the samples of every rank (src/pointestimate.jl:34-59,68-76 with the counts of src/mcmc.jl:560): the
// all-reduced counts of rc_comm_sampler_psm, W and P of this rank's samples, ONE all-gather of the per-rank int64 vectors
// (padded to the largest rank), and the totals over all samples in rank order.  Integers throughout: identical to one
// GPU over the same chains.  Every rank first learns whether any rank refuses, so none is left waiting in a collective.
int32_t rc_comm_sampler_binder_mpel(rc_comm* c, const rc_sampler* s, double* loss_sums, int64_t* best, int64_t* totals) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_binder_mpel: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const int64_t n = rc_sampler_n(s), nch = rc_sampler_nchains(s), R = nch * rc_sampler_numsamples(s);
  const int local = rc_sampler_binder_check(s, 0, nch, "rc_comm_sampler_binder_mpel");
  const std::string why = local ? rc_last_error() : "";
  long long* info = nullptr;                                   // per rank: {status, samples}
  RC_CUDA(cudaMalloc(&info, sizeof(long long) * 2 * (c->world + 1)));
  const long long mine[2] = {local, (long long)R};
  std::vector<long long> all(2 * (size_t)c->world);
  cudaError_t e = cudaMemcpy(info, mine, sizeof(mine), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && nccl()->AllGather(info, info + 2, 2, ncclInt64, c->comm, c->stream) != ncclSuccess) e = cudaErrorUnknown;
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaMemcpy(all.data(), info + 2, sizeof(long long) * 2 * c->world, cudaMemcpyDeviceToHost);
  cudaFree(info);
  if (e != cudaSuccess) { rc_set_error("rc_comm_sampler_binder_mpel: exchange of the sample counts failed"); return RC_ERR_CUDA; }
  int64_t total = 0, per = 0;
  for (int r = 0; r < c->world; ++r) {
    if (all[2 * r] != 0) {
      if (local) { rc_set_error("%s", why.c_str()); return local; }
      rc_set_error("rc_comm_sampler_binder_mpel: rank %d refused (status %lld)", r, all[2 * r]);
      return (int32_t)all[2 * r];
    }
    total += all[2 * r + 1];
    per = std::max<int64_t>(per, all[2 * r + 1]);
  }
  if (total >= ((int64_t)1 << 31)) { rc_set_error("rc_comm_sampler_binder_mpel: %lld samples in all; needs < 2^31", (long long)total); return RC_ERR_ARG; }
  int* counts = nullptr;
  unsigned long long* buf = nullptr;                           // [world + 1][2 per]: this rank's {W, P}, then the gathered ranks
  RC_CUDA(cudaMalloc(&counts, sizeof(int) * (size_t)n * n));
  if (cudaMalloc(&buf, sizeof(unsigned long long) * 2 * (size_t)per * (c->world + 1)) != cudaSuccess) {
    cudaFree(counts); rc_set_error("rc_comm_sampler_binder_mpel: out of device memory"); return RC_ERR_CUDA;
  }
  std::vector<unsigned long long> wp(2 * (size_t)per, 0ull), gathered(2 * (size_t)per * c->world);
  int st = rc_comm_sampler_psm(c, s, nullptr, counts);
  if (!st) st = rc_sampler_binder_wp(s, 0, nch, counts, total, wp.data(), wp.data() + per);
  if (!st && cudaMemcpy(buf, wp.data(), sizeof(unsigned long long) * 2 * per, cudaMemcpyHostToDevice) != cudaSuccess) st = RC_ERR_CUDA;
  if (!st && (nccl()->AllGather(buf, buf + 2 * per, 2 * (size_t)per, ncclInt64, c->comm, c->stream) != ncclSuccess ||
              cudaStreamSynchronize(c->stream) != cudaSuccess ||
              cudaMemcpy(gathered.data(), buf + 2 * per, sizeof(unsigned long long) * gathered.size(), cudaMemcpyDeviceToHost) != cudaSuccess)) {
    rc_set_error("rc_comm_sampler_binder_mpel: all-gather of the per-rank totals failed"); st = RC_ERR_CUDA;
  }
  cudaFree(counts); cudaFree(buf);
  if (st) return st;
  std::vector<unsigned long long> W, P;                        // rank order = global chain order
  for (int r = 0; r < c->world; ++r) {
    const unsigned long long* g = gathered.data() + 2 * (size_t)per * r;
    W.insert(W.end(), g, g + all[2 * r + 1]);
    P.insert(P.end(), g + per, g + per + all[2 * r + 1]);
  }
  return rc_binder_finish(W.data(), P.data(), total, n, loss_sums, best, totals);
}

// MPEL search with the candidate samples dealt cyclically over the ranks (src/pointestimate.jl:49-57): every rank holds
// all S label vectors, evaluates rows rank, rank + world, ... of the upper triangle of the loss matrix, one all-gather
// assembles it, the column sums run in ascending row order -- bit-equal to rc_mpel on one GPU.
int32_t rc_comm_mpel(rc_comm* c, const int64_t* labels, int64_t S, int64_t n, int32_t loss, double* loss_sums, int64_t* best) {
  if (!c || !labels || !loss_sums || !best || S < 1 || n < 1) { rc_set_error("rc_comm_mpel: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  if (c->world == 1) return rc_mpel(labels, S, n, loss, c->device, loss_sums, best);
  const int64_t per = (S + c->world - 1) / c->world;
  double *flat = nullptr, *upper = nullptr;
  RC_CUDA(cudaMalloc(&flat, sizeof(double) * (size_t)per * c->world * S));
  if (cudaMalloc(&upper, sizeof(double) * (size_t)S * S) != cudaSuccess) { cudaFree(flat); rc_set_error("out of device memory for the loss matrix"); return RC_ERR_CUDA; }
  double* mine = flat + (size_t)c->rank * per * S;
  int st = cudaMemset(mine, 0, sizeof(double) * (size_t)per * S) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!st) st = rc_mpel_rows_dev(labels, S, n, loss, c->device, c->rank, c->world, per, mine);
  if (!st) {
    cudaDeviceSynchronize();
    ncclResult_t r = nccl()->AllGather(mine, flat, (size_t)per * S, ncclFloat64, c->comm, c->stream);
    if (r != ncclSuccess) { rc_set_error("all-gather of the loss rows failed"); st = RC_ERR_CUDA; }
  }
  if (!st) {
    k_uncycle<<<1024, 256, 0, c->stream>>>(flat, upper, S, c->world, per);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) { rc_set_error("assembling the loss matrix failed"); st = RC_ERR_CUDA; }
  }
  if (!st) st = rc_mpel_finish_dev(upper, S, c->device, loss_sums, best);
  cudaFree(flat); cudaFree(upper);
  return st;
}

}  // extern "C"
