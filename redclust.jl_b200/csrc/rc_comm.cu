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
  TRYP(rc_select_device(device));
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
    Bufs B;
    int* w;
    if (B.get(&w, 256) == RC_OK) {
      cudaMemset(w, 0, 256 * sizeof(int));
      a->AllReduce(w, w, 256, ncclInt32, ncclSum, c->comm, c->stream);
      a->AllGather(w, w, 256 / world, ncclInt32, c->comm, c->stream);
      cudaStreamSynchronize(c->stream);
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
  Bufs B;
  double* full;
  TRYP(B.get(&full, (size_t)per * c->world * n));
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
  return st;
}

// PSM over the samples of every rank (src/mcmc.jl:560 across chain shards): exact int32 counts per rank, ONE all-reduce
// of the n x n matrix, one divide by the global number of samples.  psm_out (host n x n fp64) may be NULL when only
// counts_dev_out (device n x n int32, may be NULL too) is wanted.
static int32_t finish_psm(rc_comm* c, int* counts, int64_t n, long long local_samples, double* psm_out) {
  Bufs B;
  long long* tot;
  TRYP(B.get(&tot, 1));
  RC_CUDA(cudaMemcpy(tot, &local_samples, sizeof(long long), cudaMemcpyHostToDevice));
  RC_CUDA(cudaDeviceSynchronize());
  if (c->world > 1) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->stream);
    ncclResult_t r = nccl()->AllReduce(counts, counts, (size_t)n * n, ncclInt32, ncclSum, c->comm, c->stream);
    cudaEventRecord(e1, c->stream);
    if (r == ncclSuccess) r = nccl()->AllReduce(tot, tot, 1, ncclInt64, ncclSum, c->comm, c->stream);
    const cudaError_t e = r == ncclSuccess ? cudaStreamSynchronize(c->stream) : cudaSuccess;
    if (r == ncclSuccess && e == cudaSuccess && getenv("RCB200_VERBOSE")) {
      float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
      const double bytes = 4.0 * (double)n * (double)n;
      fprintf(stderr, "[rcb200] rank %d: ncclAllReduce of the %lld x %lld int32 counts (%.2f GB): %.2f ms, algorithm bandwidth %.1f GB/s, bus bandwidth %.1f GB/s\n",
              c->rank, (long long)n, (long long)n, bytes / 1e9, ms, bytes / ms / 1e6, bytes / ms / 1e6 * 2.0 * (c->world - 1) / c->world);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    RC_NCCL(r);
    RC_CUDA(e);
  }
  long long total = 0;
  RC_CUDA(cudaMemcpy(&total, tot, sizeof(long long), cudaMemcpyDeviceToHost));
  if (psm_out) return rc_counts_to_host_psm(counts, (size_t)n * n, (double)total, psm_out);
  return RC_OK;
}

// The {status, vals...} of every rank, exchanged before the collectives of a call that a rank may refuse: a refusing rank
// returns its own error and the others "rank r refused", instead of leaving them waiting in the next collective.
// all (out): world x {status, vals...}.
static int agree_vals(rc_comm* c, int local, const std::vector<long long>& vals, const char* who, std::vector<long long>& all) {
  const std::string why = local ? rc_last_error() : "";
  const size_t w = 1 + vals.size();
  Bufs B;
  long long* info;                                             // this rank's values, then the gathered ranks
  TRYP(B.get(&info, w * (size_t)(c->world + 1)));
  std::vector<long long> mine(1, (long long)local);
  mine.insert(mine.end(), vals.begin(), vals.end());
  all.assign(w * (size_t)c->world, 0);
  cudaError_t e = cudaMemcpy(info, mine.data(), sizeof(long long) * w, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && nccl()->AllGather(info, info + w, w, ncclInt64, c->comm, c->stream) != ncclSuccess) e = cudaErrorUnknown;
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaMemcpy(all.data(), info + w, sizeof(long long) * w * c->world, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { rc_set_error("%s: exchange of the sample counts failed", who); return RC_ERR_CUDA; }
  for (int r = 0; r < c->world; ++r)
    if (all[w * r] != 0) {
      if (local) { rc_set_error("%s", why.c_str()); return local; }
      rc_set_error("%s: rank %d refused (status %lld)", who, r, all[w * r]);
      return (int32_t)all[w * r];
    }
  return RC_OK;
}
// the {status, samples} form: all = world x {status, samples}
static int agree(rc_comm* c, int local, int64_t samples, const char* who, std::vector<long long>& all) {
  return agree_vals(c, local, {(long long)samples}, who, all);
}

int32_t rc_comm_sampler_psm(rc_comm* c, const rc_sampler* s, double* psm_out, void* counts_dev_out) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_psm: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  rc_sample_range v;
  const int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), "rc_comm_sampler_psm", v);
  std::vector<long long> all;
  TRYP(agree(c, local, local ? 0 : v.R, "rc_comm_sampler_psm", all));
  Bufs B;
  int* counts = (int*)counts_dev_out;
  if (!counts) TRYP(B.get(&counts, (size_t)v.n * v.n));
  TRYP(psm_counts_device(v.labels, v.R, v.n, counts, B));
  return finish_psm(c, counts, v.n, (long long)v.R, psm_out);
}

int32_t rc_comm_psm(rc_comm* c, const int64_t* labels, int64_t S_local, int64_t n, double* psm_out, void* counts_dev_out) {
  if (!c || (!labels && S_local > 0) || n < 1 || S_local < 0) { rc_set_error("rc_comm_psm: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  Bufs B;
  int* counts = (int*)counts_dev_out;
  if (!counts) TRYP(B.get(&counts, (size_t)n * n));
  int st = RC_OK;
  if (S_local > 0) st = rc_psm_counts_dev(labels, S_local, n, c->device, counts);
  else st = cudaMemset(counts, 0, sizeof(int) * (size_t)n * n) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!st) st = finish_psm(c, counts, n, (long long)S_local, psm_out);
  return st;
}

// Binder MPEL over the samples of every rank (src/pointestimate.jl:34-59,68-76 with the counts of src/mcmc.jl:560): this
// rank's counts, all-reduced as rc_comm_sampler_psm does, W and P of this rank's samples against them (from the transposed
// labels the counts were built from), ONE all-gather of the per-rank int64 vectors (padded to the largest rank), and the
// totals over all samples in rank order.  Integers throughout: identical to one GPU over the same chains.
int32_t rc_comm_sampler_binder_mpel(rc_comm* c, const rc_sampler* s, double* loss_sums, int64_t* best, int64_t* totals) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_binder_mpel: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_binder_mpel";
  rc_sample_range v;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = rc_binder_check_args(v.R, v.n, who);
  std::vector<long long> all;
  TRYP(agree(c, local, local ? 0 : v.R, who, all));
  const int64_t n = v.n;
  int64_t total = 0, per = 0;
  for (int r = 0; r < c->world; ++r) {
    total += all[2 * r + 1];
    per = std::max<int64_t>(per, all[2 * r + 1]);
  }
  if (total >= ((int64_t)1 << 31)) { rc_set_error("%s: %lld samples in all; needs < 2^31", who, (long long)total); return RC_ERR_ARG; }
  Bufs B;
  int* counts;
  unsigned long long* buf;                                     // [world + 1][2 per]: this rank's {W, P}, then the gathered ranks
  const uint8_t* Lt;
  TRYP(B.get(&counts, (size_t)n * n));
  TRYP(B.get(&buf, 2 * (size_t)per * (c->world + 1)));
  std::vector<unsigned long long> wp(2 * (size_t)per, 0ull), gathered(2 * (size_t)per * c->world);
  TRYP(psm_counts_device(v.labels, v.R, n, counts, B, &Lt));
  TRYP(finish_psm(c, counts, n, (long long)v.R, nullptr));
  TRYP(binder_wp(v.labels, Lt, v.R, n, counts, total, wp.data(), wp.data() + per, nullptr));
  RC_CUDA(cudaMemcpy(buf, wp.data(), sizeof(unsigned long long) * 2 * per, cudaMemcpyHostToDevice));
  if (nccl()->AllGather(buf, buf + 2 * per, 2 * (size_t)per, ncclInt64, c->comm, c->stream) != ncclSuccess ||
      cudaStreamSynchronize(c->stream) != cudaSuccess ||
      cudaMemcpy(gathered.data(), buf + 2 * per, sizeof(unsigned long long) * gathered.size(), cudaMemcpyDeviceToHost) != cudaSuccess) {
    rc_set_error("%s: all-gather of the per-rank totals failed", who); return RC_ERR_CUDA;
  }
  std::vector<unsigned long long> W, P;                        // rank order = global chain order
  for (int r = 0; r < c->world; ++r) {
    const unsigned long long* g = gathered.data() + 2 * (size_t)per * r;
    W.insert(W.end(), g, g + all[2 * r + 1]);
    P.insert(P.end(), g + per, g + per + all[2 * r + 1]);
  }
  return rc_binder_finish(W.data(), P.data(), total, n, loss_sums, best, totals);
}

// Split-R-hat of the co-clustering indicators over the chains of every rank (rc_rhat.cu): this rank's pooled counts,
// all-reduced as rc_comm_sampler_psm does; pass 2 over the rank's own chains against them with m = 2 x all chains; ONE
// all-reduce of Q (int64) and ONE all-gather of the chains' {sum d, max d} padded to the largest rank; every rank then
// finishes.  Integers throughout: identical to one GPU over the same chains.  The buffers are sized before the status
// exchange, so a rank that cannot hold them refuses with the others.
int32_t rc_comm_sampler_cocl_rhat(rc_comm* c, const rc_sampler* s, rc_rhat_summary* sum, double* rhat_out, double* meandev,
                                  double* maxdev) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_cocl_rhat: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_cocl_rhat";
  const int64_t Cl = rc_sampler_nchains(s), S = rc_sampler_numsamples(s);
  rc_sample_range v;
  Bufs B;
  RhatDev d;
  RhatTimes t;
  int local = rc_sampler_range(s, 0, Cl, who, v);
  if (!local) local = rhat_check_args(Cl, S, v.n, who);
  if (!local) local = rhat_alloc(Cl, S, v.n, rhat_out != nullptr, B, d, who);
  std::vector<long long> all;
  TRYP(agree(c, local, local ? 0 : Cl, who, all));
  const int64_t n = v.n;
  int64_t C = 0, per = 0;
  for (int r = 0; r < c->world; ++r) {
    C += all[2 * r + 1];
    per = std::max<int64_t>(per, all[2 * r + 1]);
  }
  TRYP(rhat_check_args(C, S, n, who));                          // the same on every rank
  unsigned long long* buf;                                     // [world + 1][2 per]: this rank's chains, then the gathered ranks
  TRYP(B.get(&buf, 2 * (size_t)per * (c->world + 1)));
  RC_CUDA(cudaMemset(buf, 0, sizeof(unsigned long long) * 2 * (size_t)per));
  TRYP(rhat_pass1(v.labels, Cl, S, n, d, t));
  TRYP(finish_psm(c, d.N, n, (long long)(Cl * S), nullptr));
  TRYP(rhat_pass2(v.labels, Cl, S, n, 2 * C, d, t));
  RC_CUDA(cudaMemcpy(buf, d.dev, sizeof(unsigned long long) * 2 * (size_t)Cl, cudaMemcpyDeviceToDevice));
  if (c->world > 1) {
    if (nccl()->AllReduce(d.Q, d.Q, (size_t)(n * n), ncclInt64, ncclSum, c->comm, c->stream) != ncclSuccess ||
        nccl()->AllGather(buf, buf + 2 * per, 2 * (size_t)per, ncclInt64, c->comm, c->stream) != ncclSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) {
      rc_set_error("%s: all-reduce of Q or all-gather of the chain deviations failed", who); return RC_ERR_CUDA;
    }
  } else {
    RC_CUDA(cudaMemcpy(buf + 2 * per, buf, sizeof(unsigned long long) * 2 * (size_t)per, cudaMemcpyDeviceToDevice));
  }
  std::vector<unsigned long long> gathered(2 * (size_t)per * c->world), dev;   // rank order = global chain order
  RC_CUDA(cudaMemcpy(gathered.data(), buf + 2 * per, sizeof(unsigned long long) * gathered.size(), cudaMemcpyDeviceToHost));
  for (int r = 0; r < c->world; ++r) {
    const unsigned long long* g = gathered.data() + 2 * (size_t)per * r;
    dev.insert(dev.end(), g, g + 2 * all[2 * r + 1]);
  }
  TRYP(rhat_finish(d, S, n, 2 * C, sum, rhat_out, t));
  rhat_deviations(dev.data(), C, S, n, 2 * C, meandev, maxdev);
  rhat_report(t, Cl, S, n);
  return RC_OK;
}

// Distances from reference partitions to the samples of every rank (rc_sampler_partition_dists over chains sharded over
// GPUs): every rank holds the references and computes its own samples; ONE all-gather of the per-rank {dist, pairs, K}
// blocks (8-byte words, padded to the largest rank) gives every rank all samples in rank order (= global chain order).
// Each distance comes from the same kernel and the same table as on one GPU: identical to one GPU over the same chains.
// Nothing a rank can refuse happens after a collective it might leave the others waiting in.  The first exchange carries
// {samples, their largest K, nref, a hash of the references, pairs wanted}: every rank then applies the same checks to the
// same values (equal nref, references and pairs on every rank; the table of the references against the largest K of ALL
// samples fits the shared memory, so the call refuses exactly when one GPU over the same chains would).  The buffers are
// allocated before a second exchange of the status.
int32_t rc_comm_sampler_partition_dists(rc_comm* c, const rc_sampler* s, const int64_t* refs, int64_t nref, int32_t loss,
                                        double* dist_out, int64_t* pairs_out, int32_t* K_out) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_partition_dists: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_partition_dists";
  rc_sample_range v;
  Bufs B;
  PartitionRefs r;
  std::vector<int> Kh;
  int kmax = 0;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = partition_refs(refs, nref, v.n, loss, dist_out, who, B, r);
  if (!local) local = sample_K(v.K, v.R, Kh, &kmax);
  const long long want_pairs = pairs_out != nullptr;
  unsigned long long h = 14695981039346656037ull;             // FNV-1a of the references as given
  if (!local)
    for (int64_t t = 0; t < nref * v.n; ++t) h = (h ^ (unsigned long long)refs[t]) * 1099511628211ull;
  std::vector<long long> all, ok;
  TRYP(agree_vals(c, local, {local ? 0 : (long long)v.R, kmax, (long long)nref, (long long)h, want_pairs}, who, all));
  int64_t total = 0, per = 0;
  int kall = 0;
  for (int q = 0; q < c->world; ++q) {
    const long long* a = all.data() + 6 * q;
    total += a[1];
    per = std::max<int64_t>(per, a[1]);
    kall = std::max<int>(kall, (int)a[2]);
    if (a[3] != nref || a[4] != (long long)h || a[5] != want_pairs) {
      rc_set_error("%s: rank %d holds other references or another pairs_out (nref %lld, pairs %lld)", who, q, a[3], a[5]);
      return RC_ERR_ARG;
    }
  }
  if (total < 1) { rc_set_error("%s: no samples on any rank", who); return RC_ERR_ARG; }
  PairLaunch p;
  TRYP(pair_geometry(v.n, r.kmax, kall, who, p));
  // one rank's block: dist (nref x R_rank fp64 bits), then from word nref * per the pairs (nref x R_rank) when wanted, then K
  const int64_t kw = (want_pairs ? 2 : 1) * nref * per, words = kw + per;
  long long* buf = nullptr;                                    // [world + 1][words]: this rank's block, then the gathered ranks
  local = B.get(&buf, (size_t)words * (c->world + 1));
  if (!local) local = pair_nlogn(v.n, B, p);
  TRYP(agree(c, local, 0, who, ok));
  RC_CUDA(cudaMemset(buf, 0, sizeof(long long) * words));
  if (v.R > 0) {
    TRYP(partition_dists_run(r, p, v.labels, v.K, v.R, v.n, (double*)buf, want_pairs ? buf + nref * per : nullptr));
    const std::vector<long long> K64(Kh.begin(), Kh.end());
    RC_CUDA(cudaMemcpy(buf + kw, K64.data(), sizeof(long long) * v.R, cudaMemcpyHostToDevice));
  }
  const long long* gathered = buf;
  if (c->world > 1) {
    if (nccl()->AllGather(buf, buf + words, (size_t)words, ncclInt64, c->comm, c->stream) != ncclSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) {
      rc_set_error("%s: all-gather of the per-rank distances failed", who); return RC_ERR_CUDA;
    }
    gathered = buf + words;
  }
  std::vector<long long> hv((size_t)words * c->world);
  RC_CUDA(cudaMemcpy(hv.data(), gathered, sizeof(long long) * hv.size(), cudaMemcpyDeviceToHost));
  int64_t off = 0;                                             // rank order = global chain order
  for (int q = 0; q < c->world; ++q) {
    const int64_t Rq = all[6 * q + 1];
    const long long* g = hv.data() + (size_t)words * q;
    for (int64_t k = 0; k < nref; ++k) {
      memcpy(dist_out + k * total + off, g + k * Rq, sizeof(double) * Rq);
      if (pairs_out) memcpy(pairs_out + k * total + off, g + nref * per + k * Rq, sizeof(int64_t) * Rq);
    }
    if (K_out) for (int64_t t = 0; t < Rq; ++t) K_out[off + t] = (int32_t)g[kw + t];
    off += Rq;
  }
  return RC_OK;
}

// Allocation probabilities to the clusters of an estimate over the samples of every rank (rc_sampler_aligned_alloc over
// chains sharded over GPUs): every rank holds the estimate and aligns its own samples; ONE all-reduce of the int32 counts
// and ONE all-gather of the per-rank {matched, K, maps} blocks (8-byte words, padded to the largest rank) give every rank
// the results of all samples in rank order (= global chain order).  Each sample's assignment comes from the same kernel and
// the same table as on one GPU, and the counts are integer sums: identical to one GPU over the same chains.  The first
// exchange carries {samples, their largest K, a hash of the estimate}: every rank then applies the same checks to the same
// values (the same estimate on every rank, fewer than 2^31 samples in all, the table of the estimate against the largest K
// of ALL samples fits the shared memory).  The buffers are allocated before a second exchange of the status.
int32_t rc_comm_sampler_aligned_alloc(rc_comm* c, const rc_sampler* s, const int64_t* estimate, int32_t* counts_out,
                                      int64_t* matched_out, int32_t* K_out, uint8_t* maps_out) {
  if (!c || !s || !counts_out) { rc_set_error("rc_comm_sampler_aligned_alloc: needs the handles and counts_out"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_aligned_alloc";
  rc_sample_range v;
  Bufs B;
  AlignEstimate e;
  std::vector<int> Kh;
  int kmax = 0;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = align_estimate(estimate, v.n, who, B, e);
  if (!local) local = sample_K(v.K, v.R, Kh, &kmax);
  unsigned long long h = 14695981039346656037ull;             // FNV-1a of the estimate as given
  if (!local)
    for (int64_t t = 0; t < v.n; ++t) h = (h ^ (unsigned long long)estimate[t]) * 1099511628211ull;
  std::vector<long long> all, ok;
  TRYP(agree_vals(c, local, {local ? 0 : (long long)v.R, kmax, (long long)h}, who, all));
  int64_t total = 0, per = 0;
  int kall = 0;
  for (int q = 0; q < c->world; ++q) {
    const long long* a = all.data() + 4 * q;
    total += a[1];
    per = std::max<int64_t>(per, a[1]);
    kall = std::max<int>(kall, (int)a[2]);
    if (a[3] != (long long)h) { rc_set_error("%s: rank %d holds another estimate", who, q); return RC_ERR_ARG; }
  }
  PairLaunch p;
  TRYP(align_check(e, total, kall, who, p));
  // one rank's block: matched (per words), K (per words), then the maps (per x 255 bytes)
  const int64_t words = 2 * per + (per * 255 + 7) / 8;
  AlignDev d;
  long long* buf = nullptr;                                    // [world + 1][words]: this rank's block, then the gathered ranks
  local = align_alloc(e, v.R, 8.0 * words * (c->world + 1), "exchange buffers", who, B, d);
  if (!local) local = B.get(&buf, (size_t)words * (c->world + 1));
  TRYP(agree(c, local, 0, who, ok));
  TRYP(align_run(e, p, v.labels, v.K, v.R, d));
  RC_CUDA(cudaMemset(buf, 0, sizeof(long long) * words));
  if (v.R > 0) {
    const std::vector<long long> K64(Kh.begin(), Kh.end());
    RC_CUDA(cudaMemcpy(buf, d.matched, sizeof(long long) * v.R, cudaMemcpyDeviceToDevice));
    RC_CUDA(cudaMemcpy(buf + per, K64.data(), sizeof(long long) * v.R, cudaMemcpyHostToDevice));
    RC_CUDA(cudaMemcpy2D(buf + 2 * per, 255, d.maps, 256, 255, (size_t)v.R, cudaMemcpyDeviceToDevice));
  }
  const size_t ncount = (size_t)(e.n * (e.K + 1));
  const long long* gathered = buf;
  if (c->world > 1) {
    if (nccl()->AllReduce(d.counts, d.counts, ncount, ncclInt32, ncclSum, c->comm, c->stream) != ncclSuccess ||
        nccl()->AllGather(buf, buf + words, (size_t)words, ncclInt64, c->comm, c->stream) != ncclSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) {
      rc_set_error("%s: all-reduce of the counts or all-gather of the per-rank alignments failed", who); return RC_ERR_CUDA;
    }
    gathered = buf + words;
  }
  RC_CUDA(cudaMemcpy(counts_out, d.counts, sizeof(int) * ncount, cudaMemcpyDeviceToHost));
  std::vector<long long> hv((size_t)words * c->world);
  RC_CUDA(cudaMemcpy(hv.data(), gathered, sizeof(long long) * hv.size(), cudaMemcpyDeviceToHost));
  int64_t off = 0;                                             // rank order = global chain order
  for (int q = 0; q < c->world; ++q) {
    const int64_t Rq = all[4 * q + 1];
    const long long* g = hv.data() + (size_t)words * q;
    if (matched_out) memcpy(matched_out + off, g, sizeof(long long) * Rq);
    if (K_out) for (int64_t t = 0; t < Rq; ++t) K_out[off + t] = (int32_t)g[per + t];
    if (maps_out) memcpy(maps_out + off * 255, g + 2 * per, (size_t)Rq * 255);
    off += Rq;
  }
  return RC_OK;
}

// MPEL search with the candidate samples dealt cyclically over the ranks (src/pointestimate.jl:49-57): every rank holds
// all S label vectors, evaluates rows rank, rank + world, ... of the upper triangle of the loss matrix, one all-gather
// assembles it, the column sums run in ascending row order -- bit-equal to rc_mpel on one GPU.
int32_t rc_comm_mpel(rc_comm* c, const int64_t* labels, int64_t S, int64_t n, int32_t loss, double* loss_sums, int64_t* best) {
  if (!c || !labels || !loss_sums || !best || S < 1 || n < 1) { rc_set_error("rc_comm_mpel: bad arguments"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  if (c->world == 1) return rc_mpel(labels, S, n, loss, c->device, loss_sums, best);
  const int64_t per = (S + c->world - 1) / c->world;
  Bufs B;
  double *flat, *upper;
  TRYP(B.get(&flat, (size_t)per * c->world * S)); TRYP(B.get(&upper, (size_t)S * S));
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
  return st;
}

}  // extern "C"
