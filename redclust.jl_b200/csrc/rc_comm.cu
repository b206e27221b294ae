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

namespace {

// A value that must be the same on every rank, named for the message when it is not.
struct Same {
  const char* name;
  long long v;
};

// What the status exchange tells every rank: the items (samples, chains or label vectors) of every rank in rank order,
// their total and the largest rank's, and the largest kmax of any rank.
struct Shards {
  std::vector<int64_t> items;
  int64_t total = 0, per = 0;
  int kmax = 0;
};

// FNV-1a over the 8-byte words of a host array, for the inputs every rank must hold alike.
long long hash_words(const void* p, int64_t count) {
  unsigned long long h = 14695981039346656037ull;
  for (int64_t t = 0; t < count; ++t) {
    unsigned long long w;
    memcpy(&w, (const char*)p + 8 * t, 8);
    h = (h ^ w) * 1099511628211ull;
  }
  return (long long)h;
}

// The status exchange every rc_comm_* call with a collective makes before its first one: one all-gather of each rank's
// {status, items, kmax, values that must be the same}.  A refusing rank returns its own error and the others "rank r
// refused" with its status, instead of leaving them waiting in the next collective; when ranks disagree on a value, every
// rank returns RC_ERR_ARG naming it.  sh (may be NULL) receives the item counts.
int exchange(rc_comm* c, int local, const char* who, Shards* sh = nullptr, int64_t items = 0, int kmax = 0,
             std::initializer_list<Same> same = {}) {
  const std::string why = local ? rc_last_error() : "";
  std::vector<long long> mine = {(long long)local, (long long)items, (long long)kmax};
  for (const Same& s : same) mine.push_back(s.v);
  const size_t w = mine.size();
  std::vector<long long> all(w * c->world);
  Bufs B;
  long long* info;                                             // this rank's words, then the gathered ranks
  TRYP(B.get(&info, w * (size_t)(c->world + 1)));
  cudaError_t e = cudaMemcpy(info, mine.data(), sizeof(long long) * w, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && nccl()->AllGather(info, info + w, w, ncclInt64, c->comm, c->stream) != ncclSuccess) e = cudaErrorUnknown;
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaMemcpy(all.data(), info + w, sizeof(long long) * all.size(), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { rc_set_error("%s: the status exchange failed", who); return RC_ERR_CUDA; }
  for (int r = 0; r < c->world; ++r)
    if (all[w * r] != 0) {
      if (local) { rc_set_error("%s", why.c_str()); return local; }
      rc_set_error("%s: rank %d refused (status %lld)", who, r, all[w * r]);
      return (int32_t)all[w * r];
    }
  Shards s;
  for (int r = 0; r < c->world; ++r) {
    const long long* a = all.data() + w * r;
    for (size_t k = 3; k < w; ++k)
      if (a[k] != mine[k]) {
        rc_set_error("%s: the ranks disagree on %s (%lld on rank %d, %lld on rank %d)", who, same.begin()[k - 3].name, mine[k],
                     c->rank, a[k], r);
        return RC_ERR_ARG;
      }
    s.items.push_back(a[1]);
    s.total += a[1];
    s.per = std::max<int64_t>(s.per, a[1]);
    s.kmax = std::max<int>(s.kmax, (int)a[2]);
  }
  if (sh) *sh = s;
  return RC_OK;
}

// The rank-ordered gather of the sampler paths.  buf (device, (world + 1) x words 8-byte words) starts with this rank's
// block, laid out for the largest rank's items; one all-gather puts every rank's block behind it and g receives them on
// the host in rank order.  NCCL with one rank copies, so one GPU runs the same code as several.
int gather(rc_comm* c, long long* buf, int64_t words, const char* who, std::vector<long long>& g) {
  g.resize((size_t)words * c->world);
  if (nccl()->AllGather(buf, buf + words, (size_t)words, ncclInt64, c->comm, c->stream) != ncclSuccess ||
      cudaStreamSynchronize(c->stream) != cudaSuccess ||
      cudaMemcpy(g.data(), buf + words, sizeof(long long) * g.size(), cudaMemcpyDeviceToHost) != cudaSuccess) {
    rc_set_error("%s: all-gather of the per-rank results failed", who);
    return RC_ERR_CUDA;
  }
  return RC_OK;
}

// One field of every rank's gathered block into out (NULL: not wanted) in global chain order.  The field starts at byte
// `at` of a block and holds `rows` rows of the rank's items, `size` bytes each, one row after the other; row k of rank q
// lands at item k * total + (the items of the ranks before q).
void unpack(const std::vector<long long>& g, int64_t words, const Shards& sh, size_t at, int64_t rows, size_t size, void* out) {
  if (!out) return;
  int64_t off = 0;
  for (size_t q = 0; q < sh.items.size(); ++q) {
    const char* b = (const char*)(g.data() + (size_t)words * q) + at;
    for (int64_t k = 0; k < rows; ++k)
      memcpy((char*)out + (k * sh.total + off) * size, b + k * sh.items[q] * size, sh.items[q] * size);
    off += sh.items[q];
  }
}

}  // namespace

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
  if (!c) { rc_set_error("rc_comm_data_from_points: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  int local = RC_OK;
  if (!X || !out || n < 1 || dim < 1) { rc_set_error("rc_comm_data_from_points: bad arguments"); local = RC_ERR_ARG; }
  const int64_t per = (n + c->world - 1) / c->world;                  // equal blocks, the last one padded
  const int64_t row0 = std::min<int64_t>((int64_t)c->rank * per, n), nrows = std::min<int64_t>(per, n - row0);
  Bufs B;
  double* full = nullptr;
  if (!local) local = B.get(&full, (size_t)per * c->world * n);
  double* mine = local ? nullptr : full + (size_t)c->rank * per * n;
  if (!local && nrows < per) local = cudaMemset(mine, 0, sizeof(double) * (size_t)per * n) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!local) local = rc_distm_rows_dev(X, dim, n, row0, nrows, c->device, mine);
  TRYP(exchange(c, local, "rc_comm_data_from_points", nullptr, 0, 0,
                {{"n", n}, {"dim", dim}, {"the points", local ? 0 : hash_words(X, n * dim)}}));
  if (c->world > 1) {
    ncclResult_t r = nccl()->AllGather(mine, full, (size_t)per * n, ncclFloat64, c->comm, c->stream);
    if (r != ncclSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) { rc_set_error("all-gather of the distance rows failed"); return RC_ERR_CUDA; }
  }
  return rc_data_from_dist_dev(full, n, c->device, out);
}

// PSM over the samples of every rank (src/mcmc.jl:560 across chain shards): exact int32 counts per rank, ONE all-reduce
// of the n x n matrix, one divide by the global number of samples.  psm_out (host n x n fp64) may be NULL when only
// counts_dev_out (device n x n int32, may be NULL too) is wanted.
static int32_t finish_psm(rc_comm* c, int* counts, int64_t n, int64_t total, double* psm_out) {
  RC_CUDA(cudaDeviceSynchronize());
  if (c->world > 1) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->stream);
    ncclResult_t r = nccl()->AllReduce(counts, counts, (size_t)n * n, ncclInt32, ncclSum, c->comm, c->stream);
    cudaEventRecord(e1, c->stream);
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
  if (psm_out) return rc_counts_to_host_psm(counts, (size_t)n * n, (double)total, psm_out);
  return RC_OK;
}

int32_t rc_comm_sampler_psm(rc_comm* c, const rc_sampler* s, double* psm_out, void* counts_dev_out) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_psm: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  rc_sample_range v{};
  Bufs B;
  int* counts = (int*)counts_dev_out;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), "rc_comm_sampler_psm", v);
  if (!local && !counts) local = B.get(&counts, (size_t)v.n * v.n);
  Shards sh;
  TRYP(exchange(c, local, "rc_comm_sampler_psm", &sh, v.R, 0, {{"n", v.n}}));
  TRYP(psm_counts_device(v.labels, v.R, v.n, counts, B));
  return finish_psm(c, counts, v.n, sh.total, psm_out);
}

int32_t rc_comm_psm(rc_comm* c, const int64_t* labels, int64_t S_local, int64_t n, double* psm_out, void* counts_dev_out) {
  if (!c) { rc_set_error("rc_comm_psm: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  int local = RC_OK;
  if ((!labels && S_local > 0) || n < 1 || S_local < 0) { rc_set_error("rc_comm_psm: bad arguments"); local = RC_ERR_ARG; }
  Bufs B;
  int* counts = (int*)counts_dev_out;
  if (!local && !counts) local = B.get(&counts, (size_t)n * n);
  if (!local && S_local > 0) local = rc_psm_counts_dev(labels, S_local, n, c->device, counts);
  else if (!local) local = cudaMemset(counts, 0, sizeof(int) * (size_t)n * n) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  Shards sh;
  TRYP(exchange(c, local, "rc_comm_psm", &sh, S_local, 0, {{"n", n}}));
  return finish_psm(c, counts, n, sh.total, psm_out);
}

// Binder MPEL over the samples of every rank (src/pointestimate.jl:34-59,68-76 with the counts of src/mcmc.jl:560): this
// rank's counts, all-reduced as rc_comm_sampler_psm does, W and P of this rank's samples against them (from the transposed
// labels the counts were built from), the gather of the per-rank int64 vectors, and the totals over all samples in rank
// order.  Integers throughout: identical to one GPU over the same chains.
int32_t rc_comm_sampler_binder_mpel(rc_comm* c, const rc_sampler* s, double* loss_sums, int64_t* best, int64_t* totals) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_binder_mpel: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_binder_mpel";
  rc_sample_range v{};
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = rc_binder_check_args(v.R, v.n, who);
  Shards sh;
  TRYP(exchange(c, local, who, &sh, v.R, 0, {{"n", v.n}}));
  const int64_t n = v.n, total = sh.total, per = sh.per;
  if (total >= ((int64_t)1 << 31)) { rc_set_error("%s: %lld samples in all; needs < 2^31", who, (long long)total); return RC_ERR_ARG; }
  Bufs B;
  int* counts;
  long long* buf;                                              // [world + 1][2 per]: this rank's {W, P}, then the gathered ranks
  const uint8_t* Lt;
  TRYP(B.get(&counts, (size_t)n * n));
  TRYP(B.get(&buf, 2 * (size_t)per * (c->world + 1)));
  std::vector<unsigned long long> wp(2 * (size_t)per, 0ull), W(total), P(total);
  TRYP(psm_counts_device(v.labels, v.R, n, counts, B, &Lt));
  TRYP(finish_psm(c, counts, n, total, nullptr));
  TRYP(binder_wp(v.labels, Lt, v.R, n, counts, total, wp.data(), wp.data() + per, nullptr));
  RC_CUDA(cudaMemcpy(buf, wp.data(), sizeof(unsigned long long) * 2 * per, cudaMemcpyHostToDevice));
  std::vector<long long> g;
  TRYP(gather(c, buf, 2 * per, who, g));
  unpack(g, 2 * per, sh, 0, 1, 8, W.data());
  unpack(g, 2 * per, sh, 8 * per, 1, 8, P.data());
  return rc_binder_finish(W.data(), P.data(), total, n, loss_sums, best, totals);
}

// Split-R-hat of the co-clustering indicators over the chains of every rank (rc_rhat.cu): this rank's pooled counts,
// all-reduced as rc_comm_sampler_psm does; pass 2 over the rank's own chains against them with m = 2 x all chains; ONE
// all-reduce of Q (int64) and the gather of the chains' {sum d, max d}; every rank then finishes.  Integers throughout:
// identical to one GPU over the same chains.  The buffers are sized before the status exchange, so a rank that cannot
// hold them refuses with the others.
int32_t rc_comm_sampler_cocl_rhat(rc_comm* c, const rc_sampler* s, rc_rhat_summary* sum, double* rhat_out, double* meandev,
                                  double* maxdev) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_cocl_rhat: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_cocl_rhat";
  const int64_t Cl = rc_sampler_nchains(s), S = rc_sampler_numsamples(s);
  rc_sample_range v{};
  Bufs B;
  RhatDev d;
  RhatTimes t;
  int local = rc_sampler_range(s, 0, Cl, who, v);
  if (!local) local = rhat_check_args(Cl, S, v.n, who);
  if (!local) local = rhat_alloc(Cl, S, v.n, rhat_out != nullptr, B, d, who);
  Shards sh;
  TRYP(exchange(c, local, who, &sh, Cl, 0, {{"n", v.n}, {"samples per chain", S}}));
  const int64_t n = v.n, C = sh.total, per = sh.per;
  TRYP(rhat_check_args(C, S, n, who));                          // the same on every rank
  long long* buf;                                              // [world + 1][2 per]: this rank's chains, then the gathered ranks
  TRYP(B.get(&buf, 2 * (size_t)per * (c->world + 1)));
  RC_CUDA(cudaMemset(buf, 0, sizeof(long long) * 2 * (size_t)per));
  TRYP(rhat_pass1(v.labels, Cl, S, n, d, t));
  TRYP(finish_psm(c, d.N, n, C * S, nullptr));
  TRYP(rhat_pass2(v.labels, Cl, S, n, 2 * C, d, t));
  RC_CUDA(cudaMemcpy(buf, d.dev, sizeof(unsigned long long) * 2 * (size_t)Cl, cudaMemcpyDeviceToDevice));
  RC_NCCL(nccl()->AllReduce(d.Q, d.Q, (size_t)(n * n), ncclInt64, ncclSum, c->comm, c->stream));
  std::vector<long long> g;
  TRYP(gather(c, buf, 2 * per, who, g));
  std::vector<unsigned long long> dev(2 * (size_t)C);          // rank order = global chain order
  unpack(g, 2 * per, sh, 0, 1, 16, dev.data());
  TRYP(rhat_finish(d, S, n, 2 * C, sum, rhat_out, t));
  rhat_deviations(dev.data(), C, S, n, 2 * C, meandev, maxdev);
  rhat_report(t, Cl, S, n);
  return RC_OK;
}

// Distances from reference partitions to the samples of every rank (rc_sampler_partition_dists over chains sharded over
// GPUs): every rank holds the references and computes its own samples; the gather of the per-rank {dist, pairs, K} blocks
// gives every rank all samples in rank order (= global chain order).  Each distance comes from the same kernel and the
// same table as on one GPU: identical to one GPU over the same chains.  Nothing a rank can refuse happens after a
// collective it might leave the others waiting in: the status exchange carries the samples' largest K, so every rank
// checks that the table of the references against the largest K of ALL samples fits the shared memory (the call refuses
// exactly when one GPU over the same chains would), and the buffers are allocated before a second exchange of the status.
int32_t rc_comm_sampler_partition_dists(rc_comm* c, const rc_sampler* s, const int64_t* refs, int64_t nref, int32_t loss,
                                        double* dist_out, int64_t* pairs_out, int32_t* K_out) {
  if (!c || !s) { rc_set_error("rc_comm_sampler_partition_dists: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_partition_dists";
  rc_sample_range v{};
  Bufs B;
  PartitionRefs r;
  std::vector<int> Kh;
  int kmax = 0;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = partition_refs(refs, nref, v.n, loss, dist_out, who, B, r);
  if (!local) local = sample_K(v.K, v.R, Kh, &kmax);
  Shards sh;
  TRYP(exchange(c, local, who, &sh, v.R, kmax, {{"n", v.n}, {"nref", nref}, {"pairs_out", pairs_out != nullptr},
                                               {"the references", local ? 0 : hash_words(refs, nref * v.n)}}));
  if (sh.total < 1) { rc_set_error("%s: no samples on any rank", who); return RC_ERR_ARG; }
  PairLaunch p;
  TRYP(pair_geometry(v.n, r.kmax, sh.kmax, who, p));
  // one rank's block: dist (nref x R_rank fp64), then from word nref * per the pairs (nref x R_rank int64) when wanted,
  // then from word kw the K (R_rank int32)
  const int64_t per = sh.per, kw = (pairs_out ? 2 : 1) * nref * per, words = kw + (per + 1) / 2;
  long long* buf = nullptr;                                    // [world + 1][words]: this rank's block, then the gathered ranks
  local = B.get(&buf, (size_t)words * (c->world + 1));
  if (!local) local = pair_nlogn(v.n, B, p);
  TRYP(exchange(c, local, who));
  RC_CUDA(cudaMemset(buf, 0, sizeof(long long) * words));
  if (v.R > 0) {
    TRYP(partition_dists_run(r, p, v.labels, v.K, v.R, v.n, (double*)buf, pairs_out ? buf + nref * per : nullptr));
    RC_CUDA(cudaMemcpy(buf + kw, Kh.data(), sizeof(int) * v.R, cudaMemcpyHostToDevice));
  }
  std::vector<long long> g;
  TRYP(gather(c, buf, words, who, g));
  unpack(g, words, sh, 0, nref, 8, dist_out);
  unpack(g, words, sh, 8 * nref * per, nref, 8, pairs_out);
  unpack(g, words, sh, 8 * kw, 1, 4, K_out);
  return RC_OK;
}

// Allocation probabilities to the clusters of an estimate over the samples of every rank (rc_sampler_aligned_alloc over
// chains sharded over GPUs): every rank holds the estimate and aligns its own samples; ONE all-reduce of the int32 counts
// and the gather of the per-rank {matched, K, maps} blocks give every rank the results of all samples in rank order (=
// global chain order).  Each sample's assignment comes from the same kernel and the same table as on one GPU, and the
// counts are integer sums: identical to one GPU over the same chains.  The status exchange carries the samples' largest K:
// every rank then applies the same checks to the same values (fewer than 2^31 samples in all, the table of the estimate
// against the largest K of ALL samples fits the shared memory).  The buffers are allocated before a second exchange of the
// status.
int32_t rc_comm_sampler_aligned_alloc(rc_comm* c, const rc_sampler* s, const int64_t* estimate, int32_t* counts_out,
                                      int64_t* matched_out, int32_t* K_out, uint8_t* maps_out) {
  if (!c || !s || !counts_out) { rc_set_error("rc_comm_sampler_aligned_alloc: needs the handles and counts_out"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  const char* who = "rc_comm_sampler_aligned_alloc";
  rc_sample_range v{};
  Bufs B;
  AlignEstimate e;
  std::vector<int> Kh;
  int kmax = 0;
  int local = rc_sampler_range(s, 0, rc_sampler_nchains(s), who, v);
  if (!local) local = align_estimate(estimate, v.n, who, B, e);
  if (!local) local = sample_K(v.K, v.R, Kh, &kmax);
  Shards sh;
  TRYP(exchange(c, local, who, &sh, v.R, kmax, {{"n", v.n}, {"the estimate", local ? 0 : hash_words(estimate, v.n)}}));
  PairLaunch p;
  TRYP(align_check(e, sh.total, sh.kmax, who, p));
  // one rank's block: matched (per int64), K (per int32), then the maps (per x 255 bytes)
  const int64_t per = sh.per, words = (267 * per + 7) / 8;
  AlignDev d;
  long long* buf = nullptr;                                    // [world + 1][words]: this rank's block, then the gathered ranks
  local = align_alloc(e, v.R, 8.0 * words * (c->world + 1), "exchange buffers", who, B, d);
  if (!local) local = B.get(&buf, (size_t)words * (c->world + 1));
  TRYP(exchange(c, local, who));
  TRYP(align_run(e, p, v.labels, v.K, v.R, d));
  char* blk = (char*)buf;
  RC_CUDA(cudaMemset(buf, 0, sizeof(long long) * words));
  if (v.R > 0) {
    RC_CUDA(cudaMemcpy(blk, d.matched, sizeof(long long) * v.R, cudaMemcpyDeviceToDevice));
    RC_CUDA(cudaMemcpy(blk + 8 * per, Kh.data(), sizeof(int) * v.R, cudaMemcpyHostToDevice));
    RC_CUDA(cudaMemcpy2D(blk + 12 * per, 255, d.maps, 256, 255, (size_t)v.R, cudaMemcpyDeviceToDevice));
  }
  const size_t ncount = (size_t)(e.n * (e.K + 1));
  RC_NCCL(nccl()->AllReduce(d.counts, d.counts, ncount, ncclInt32, ncclSum, c->comm, c->stream));
  std::vector<long long> g;
  TRYP(gather(c, buf, words, who, g));
  RC_CUDA(cudaMemcpy(counts_out, d.counts, sizeof(int) * ncount, cudaMemcpyDeviceToHost));
  unpack(g, words, sh, 0, 1, 8, matched_out);
  unpack(g, words, sh, 8 * per, 1, 4, K_out);
  unpack(g, words, sh, 12 * per, 1, 255, maps_out);
  return RC_OK;
}

// MPEL search with the candidate samples dealt cyclically over the ranks (src/pointestimate.jl:49-57): every rank holds
// all S label vectors, evaluates rows rank, rank + world, ... of the upper triangle of the loss matrix, one all-gather
// assembles it, the column sums run in ascending row order -- bit-equal to rc_mpel on one GPU.
int32_t rc_comm_mpel(rc_comm* c, const int64_t* labels, int64_t S, int64_t n, int32_t loss, double* loss_sums, int64_t* best) {
  if (!c) { rc_set_error("rc_comm_mpel: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(c->device));
  int local = RC_OK;
  if (!labels || !loss_sums || !best || S < 1 || n < 1) { rc_set_error("rc_comm_mpel: bad arguments"); local = RC_ERR_ARG; }
  if (c->world == 1) return local ? local : rc_mpel(labels, S, n, loss, c->device, loss_sums, best);
  const int64_t per = (S + c->world - 1) / c->world;
  Bufs B;
  double *flat = nullptr, *upper = nullptr;
  if (!local) local = B.get(&flat, (size_t)per * c->world * S);
  if (!local) local = B.get(&upper, (size_t)S * S);
  double* mine = local ? nullptr : flat + (size_t)c->rank * per * S;
  if (!local) local = cudaMemset(mine, 0, sizeof(double) * (size_t)per * S) == cudaSuccess ? RC_OK : RC_ERR_CUDA;
  if (!local) local = rc_mpel_rows_dev(labels, S, n, loss, c->device, c->rank, c->world, per, mine);
  TRYP(exchange(c, local, "rc_comm_mpel", nullptr, 0, 0,
                {{"n", n}, {"S", S}, {"loss", loss}, {"the labels", local ? 0 : hash_words(labels, S * n)}}));
  cudaDeviceSynchronize();
  if (nccl()->AllGather(mine, flat, (size_t)per * S, ncclFloat64, c->comm, c->stream) != ncclSuccess) {
    rc_set_error("all-gather of the loss rows failed");
    return RC_ERR_CUDA;
  }
  k_uncycle<<<1024, 256, 0, c->stream>>>(flat, upper, S, c->world, per);
  if (cudaStreamSynchronize(c->stream) != cudaSuccess) { rc_set_error("assembling the loss matrix failed"); return RC_ERR_CUDA; }
  return rc_mpel_finish_dev(upper, S, c->device, loss_sums, best);
}

}  // extern "C"
