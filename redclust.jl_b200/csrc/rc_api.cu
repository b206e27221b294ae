// rc_api.cu -- C ABI of librcb200.so (include/rcb200.h): handles, validation, launches.
// There is NO CPU fallback: every compute entry point needs a CUDA device.
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <vector>
#include <algorithm>
#include <thread>
#include <chrono>
#include "rc_sampler.cuh"

static thread_local char g_err[512] = "";

void rc_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Host copy of every chain's recorded outputs, filled by ONE set of device-to-host copies on the first read after a
// run (reading C chains one by one would otherwise cost 9 C small synchronous copies).
struct rc_host_mirror {
  bool valid = false;
  std::vector<uint8_t> labels, r_acc, sm_acc, sm_split;
  std::vector<int> K;
  std::vector<double> r, p, ll, lp;
};

struct rc_sampler {
  const rc_data* d;
  rc_options opt;
  rc_params par;
  int64_t nchains, chain_offset, numsamples;
  uint64_t seed;
  int cap;
  int device;                  // copied from the data handle: the sampler may be destroyed after it
  int64_t n;
  // device
  double *LGA, *LGZ, *LOGN;
  uint8_t* labels; int* sizes; double *r, *p; int* status;
  rc_i128 *WD, *WL, *WDbak, *WLbak; uint8_t* labbak; int* szbak; unsigned short* Slist;
  uint8_t* origM; longlong4* AB; double2* L2s; double2* NZ; longlong2* DG; double* terms;
  long long* stats;
  // Group state: what k_chain_inc keeps per chain that can be rebuilt from the labels at any launch, allocated for `group`
  // chains.  group == nchains (resident): it persists across runs.  group < nchains (grouped): the chains run in launch
  // groups of `group` that share it, each launch rebuilding S and W and starting with every cache stale.
  longlong2* S;                // [group][cap][n] row sums by slot
  double2* Cc; unsigned *Vv, *epochs;   // cached per-slot terms, per-point / per-slot change counts that validate them
  void* Rs;                    // row summaries of the scan (group x n x 32 B)
  double* LLF; unsigned* LLFs; // merged-state log-likelihoods per ordered slot pair and their change counts
  double4* Cm; unsigned* Cms;  // per-slot margins of the row summaries, the change count they were built at and whether the build succeeded
  int64_t group;               // chains per launch
  int64_t last_g0;             // first chain of the group launched last (its S is the one that exists)
  int tw_smem, shortcuts;
  int inc_nthr;                // threads per chain (= per CTA) of k_chain_inc
  size_t inc_smem, terms_stride;
  int inc_mcap;                // split-merge members whose running sums fit the chain's shared memory
  int ovl_min_thr, rs_team;    // scan beside the restricted scans: from this many threads per chain on, with this many on the restricted scans
  uint8_t* out_labels; int* out_K; double *out_r, *out_p, *out_ll, *out_lp;
  uint8_t *r_acc, *sm_acc, *sm_split;
  // progress
  int64_t iters_done;
  int64_t overflowed;          // chains stopped by the slot capacity so far
  double dev_seconds;
  bool W_ready;                // S and W have been built (by the first run)
  bool shared_init;            // every chain starts from the same labels: the row sums are built once and copied
  cudaStream_t stream;
  cudaEvent_t e0, e1;
  mutable rc_host_mirror mirror;
};

static bool pool_enabled() { static const bool on = getenv("RCB200_NO_POOL") == nullptr; return on; }
cudaError_t rc_dev_malloc(void** p, size_t bytes) {
  if (!pool_enabled()) return cudaMalloc(p, bytes);
  static bool configured[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      // The device's default pool is process-global: freed handle memory is kept for the next handle up to this bound
      // (RCB200_POOL_KEEP_GB, default 32) and handed back to the driver beyond it, so that other allocators in the
      // process (PyTorch's cudaMalloc cache) are not starved by a destroyed sampler's tens of gigabytes.
      unsigned long long keep = 32ull << 30;
      if (const char* e = getenv("RCB200_POOL_KEEP_GB")) keep = (unsigned long long)atoll(e) << 30;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    configured[dev] = true;
  }
  cudaError_t e = cudaMallocAsync(p, bytes, 0);      // legacy default stream: ordered against every blocking stream
  if (e != cudaSuccess) { (void)cudaGetLastError(); e = cudaMalloc(p, bytes); }
  return e;
}
void rc_dev_free(void* p) {
  if (!p) return;
  if (!pool_enabled() || cudaFreeAsync(p, 0) != cudaSuccess) { (void)cudaGetLastError(); cudaFree(p); }
}

namespace {

int validate_options(const rc_options* o) {
  // messages of MCMCOptionsList's constructor, src/types.jl:40-54
  if (o->numiters < 1) { rc_set_error("numiters must be \xe2\x89\xa5 1."); return RC_ERR_ARG; }
  if (o->burnin > o->numiters) { rc_set_error("burnin must be < numiters"); return RC_ERR_ARG; }
  if (o->burnin < 0) { rc_set_error("burnin must be non-negative."); return RC_ERR_ARG; }
  if (o->thin < 1) { rc_set_error("thin must be positive."); return RC_ERR_ARG; }
  if (o->numGibbs < 0) { rc_set_error("numGibbs must be non-negative."); return RC_ERR_ARG; }
  if (o->numMH < 0) { rc_set_error("numMH must be non-negative."); return RC_ERR_ARG; }
  return RC_OK;
}

template <class T>
int dalloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = rc_dev_malloc((void**)p, sizeof(T) * count);
  if (e != cudaSuccess) { rc_set_error("cudaMalloc of %zu bytes failed: %s", sizeof(T) * count, cudaGetErrorString(e)); return RC_ERR_CUDA; }
  return RC_OK;
}

// Kernel parameters of the launch of chains [g0, g0 + m), m = min(group, nchains - g0): every per-chain pointer starts at
// chain g0 and chain_offset is advanced by g0 (the chains keep their Philox keys); the group state is not offset.
void fill_kparams(const rc_sampler* s, rc_kparams& kp, int64_t g0 = 0) {
  memset(&kp, 0, sizeof(kp));
  const size_t n = (size_t)s->n, cap = (size_t)s->cap, g = (size_t)g0;
  const size_t NS = (size_t)s->numsamples, ni = (size_t)s->opt.numiters, nm = ni * (size_t)s->opt.numMH;
  kp.n = (int)n; kp.cap = s->cap;
  kp.qD = s->d->qD; kp.qL = s->d->qL; kp.DL = s->d->DL;
  kp.S = s->S; kp.terms_stride = s->terms_stride; kp.inc_mcap = s->inc_mcap; kp.ovl_min_thr = s->ovl_min_thr; kp.rs_team = s->rs_team; kp.Cc = s->Cc; kp.Vv = s->Vv; kp.epochs = s->epochs; kp.tw_smem = s->tw_smem; kp.shortcuts = s->shortcuts; kp.Rs = (RowSum*)s->Rs; kp.LLF = s->LLF; kp.LLFs = s->LLFs; kp.Cm = s->Cm; kp.Cms = s->Cms;
  kp.P = s->par;
  kp.abratio = rc_gamma_lognorm(s->par.alpha, s->par.beta);    // mcmc.jl:17,186,293
  kp.zgratio = rc_gamma_lognorm(s->par.zeta, s->par.gamma);     // mcmc.jl:18,187,294
  kp.lgd1 = rc_lgamma(s->par.delta1);
  kp.lgd2 = rc_lgamma(s->par.delta2);
  kp.LGA = s->LGA; kp.LGZ = s->LGZ; kp.LOGN = s->LOGN;
  kp.burnin = s->opt.burnin; kp.thin = s->opt.thin; kp.numGibbs = s->opt.numGibbs; kp.numMH = s->opt.numMH;
  kp.numiters = s->opt.numiters; kp.numsamples = s->numsamples;
  kp.seed = s->seed; kp.chain_offset = s->chain_offset + g0; kp.nchains = (int)std::min<int64_t>(s->group, s->nchains - g0);
  kp.labels = s->labels + g * n; kp.sizes = s->sizes + g * cap; kp.r = s->r + g; kp.p = s->p + g; kp.status = s->status + g;
  kp.WD = s->WD + g * cap * cap; kp.WL = s->WL + g * cap * cap;
  if (s->WDbak) { kp.WDbak = s->WDbak + g * cap * cap; kp.WLbak = s->WLbak + g * cap * cap; kp.labbak = s->labbak + g * n; kp.szbak = s->szbak + g * (cap + 1); }
  kp.Slist = s->Slist + g * (n + 2); kp.origM = s->origM + g * (n + 2); kp.AB = s->AB + g * (n + 2); kp.L2s = s->L2s + g * n;
  kp.NZ = s->NZ + g * (size_t)(s->opt.numGibbs + 1) * n;
  kp.DG = s->DG + g * (n + 2); kp.terms = s->terms + g * s->terms_stride; kp.stats = s->stats + g * 16;
  kp.out_labels = s->out_labels + g * NS * n; kp.out_K = s->out_K + g * NS; kp.out_r = s->out_r + g * NS; kp.out_p = s->out_p + g * NS;
  kp.out_ll = s->out_ll + g * NS; kp.out_lp = s->out_lp + g * NS;
  kp.r_acc = s->r_acc + g * ni; kp.sm_acc = s->sm_acc + g * nm; kp.sm_split = s->sm_split + g * nm;
}

__global__ void k_fill_u32(unsigned* __restrict__ p, size_t count, unsigned v) {
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < count; t += (size_t)gridDim.x * blockDim.x) p[t] = v;
}

// Every cache of the group state stale: no point's cached terms (Vv = 0), row summary (stamp 0), per-slot margin (change
// count 0) or merged-state log-likelihood (change count 0) is valid at the chains' change count 1 (epochs).
int reset_caches(const rc_sampler* s) {
  const size_t m = (size_t)s->group, n = (size_t)s->n, cap = (size_t)s->cap;
  RC_CUDA(cudaMemsetAsync(s->Vv, 0, sizeof(unsigned) * m * n, s->stream));
  RC_CUDA(cudaMemsetAsync(s->Rs, 0, m * n * 32, s->stream));
  RC_CUDA(cudaMemsetAsync(s->LLFs, 0, sizeof(unsigned) * m * cap * cap, s->stream));
  RC_CUDA(cudaMemsetAsync(s->Cms, 0, sizeof(unsigned) * m * 2, s->stream));
  k_fill_u32<<<256, 256, 0, s->stream>>>(s->epochs, m * (cap + 1), 1u);
  RC_CUDA(cudaGetLastError());
  return RC_OK;
}

}  // namespace

extern "C" {

int32_t rc_version(void) { return RCB200_VERSION; }
const char* rc_last_error(void) { return g_err; }

int32_t rc_init_rp(const rc_params* params, uint64_t seed, int64_t chain_id, double* r, double* p) {
  if (!params || !r || !p) { rc_set_error("rc_init_rp: null pointer"); return RC_ERR_ARG; }
  rc_init_rp_draw(params->eta, params->sigma, params->u, params->v, seed, (uint64_t)chain_id, r, p);
  return RC_OK;
}

void rc_sampler_destroy(rc_sampler* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  rc_dev_free(s->LGA); rc_dev_free(s->LGZ); rc_dev_free(s->LOGN);
  rc_dev_free(s->labels); rc_dev_free(s->sizes); rc_dev_free(s->r); rc_dev_free(s->p); rc_dev_free(s->status);
  rc_dev_free(s->WD); rc_dev_free(s->WL); rc_dev_free(s->WDbak); rc_dev_free(s->WLbak); rc_dev_free(s->labbak);
  rc_dev_free(s->szbak); rc_dev_free(s->Slist); rc_dev_free(s->origM); rc_dev_free(s->AB);
  rc_dev_free(s->L2s); rc_dev_free(s->NZ); rc_dev_free(s->DG); rc_dev_free(s->terms);
  rc_dev_free(s->stats);
  rc_dev_free(s->out_labels); rc_dev_free(s->out_K); rc_dev_free(s->out_r); rc_dev_free(s->out_p); rc_dev_free(s->out_ll); rc_dev_free(s->out_lp);
  rc_dev_free(s->r_acc); rc_dev_free(s->sm_acc); rc_dev_free(s->sm_split);
  rc_dev_free(s->S); rc_dev_free(s->Cc); rc_dev_free(s->Vv); rc_dev_free(s->epochs); rc_dev_free(s->Rs); rc_dev_free(s->LLF); rc_dev_free(s->LLFs); rc_dev_free(s->Cm); rc_dev_free(s->Cms);
  if (s->e0) cudaEventDestroy(s->e0);
  if (s->e1) cudaEventDestroy(s->e1);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int32_t rc_sampler_create(const rc_data* d, const rc_options* opt, const rc_params* par, int64_t nchains,
                          int64_t chain_offset, const int64_t* init_labels, const double* init_r,
                          const double* init_p, uint64_t seed, int32_t slot_cap, rc_sampler** out) {
  if (!d || !opt || !par || !init_labels || !init_r || !init_p || !out || nchains < 1) {
    rc_set_error("rc_sampler_create: null pointer or nchains < 1"); return RC_ERR_ARG;
  }
  int st = validate_options(opt);
  if (st) return st;
  const int64_t n = d->n;
  if (opt->numMH > 0 && n < 2) { rc_set_error("split-merge needs at least 2 observations."); return RC_ERR_ARG; }
  // slot capacity: 128 by default, up to 255 (byte labels)
  int cap = slot_cap == 0 ? RC_MAXCAP : slot_cap;
  if (cap < 2 || cap > RC_MAXCAP_INC) { rc_set_error("slot_cap must be in 2..%d", RC_MAXCAP_INC); return RC_ERR_ARG; }
  if (par->maxK < 0 || !(par->proposalsd_r > 0)) { rc_set_error("invalid hyperparameters (maxK < 0 or proposalsd_r <= 0)"); return RC_ERR_ARG; }
  if (n > 65535) { rc_set_error("n = %lld: the sampler indexes points with 16 bits (n <= 65535)", (long long)n); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(d->device));
  int maxsmem = 0, nsm = 0;
  RC_CUDA(cudaDeviceGetAttribute(&maxsmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, d->device));
  RC_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, d->device));
  const bool vb_ = getenv("RCB200_VERBOSE") != nullptr;
  auto tnow_ = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double tc0_ = tnow_();
  // host-side state: 0-based slots and sizes (MCMCState, src/types.jl:131-137)
  std::vector<uint8_t> lab((size_t)nchains * n);
  std::vector<int> sizes((size_t)nchains * cap, 0);
  for (int64_t c = 0; c < nchains; ++c) {
    if (c > 0 && memcmp(init_labels + c * n, init_labels + (c - 1) * n, sizeof(int64_t) * (size_t)n) == 0) {   // same as the chain before: copy
      memcpy(lab.data() + c * n, lab.data() + (c - 1) * n, (size_t)n);
      memcpy(sizes.data() + c * cap, sizes.data() + (c - 1) * cap, sizeof(int) * (size_t)cap);
      continue;
    }
    for (int64_t j = 0; j < n; ++j) {
      const int64_t l = init_labels[c * n + j];
      if (l < 1 || l > cap) {
        rc_set_error("initial label %lld of chain %lld is outside 1..slot_cap (%d); relabel with sortlabels first",
                     (long long)l, (long long)c, cap);
        return RC_ERR_SLOTS;
      }
      lab[c * n + j] = (uint8_t)(l - 1);
      sizes[c * cap + (l - 1)] += 1;
    }
  }
  for (int64_t c = 0; c < nchains; ++c)
    if (!(init_r[c] > 0) || !(init_p[c] > 0 && init_p[c] < 1)) {
      rc_set_error("initial r must be > 0 and p in (0, 1) (chain %lld)", (long long)c); return RC_ERR_ARG;
    }
  const double tc1_ = tnow_();
  rc_sampler* s = new rc_sampler();     // value-initialised: every scalar member starts at zero
  s->shared_init = nchains > 1;
  for (int64_t c = 1; c < nchains && s->shared_init; ++c) s->shared_init = memcmp(lab.data(), lab.data() + c * n, (size_t)n) == 0;
  s->d = d; s->device = d->device; s->n = d->n; s->opt = *opt; s->par = *par; s->nchains = nchains; s->chain_offset = chain_offset; s->seed = seed;
  s->cap = cap;
  s->numsamples = (opt->numiters - opt->burnin) / opt->thin;   // floor((numiters - burnin) / thin), types.jl:55
  const size_t NS = (size_t)std::max<int64_t>(s->numsamples, 1);
#define TRY(x) do { st = (x); if (st) { rc_sampler_destroy(s); return st; } } while (0)
  TRY(dalloc(&s->LGA, n + 2)); TRY(dalloc(&s->LGZ, n + 2)); TRY(dalloc(&s->LOGN, n + 2));
  TRY(dalloc(&s->labels, (size_t)nchains * n)); TRY(dalloc(&s->sizes, (size_t)nchains * cap));
  TRY(dalloc(&s->r, nchains)); TRY(dalloc(&s->p, nchains)); TRY(dalloc(&s->status, nchains));
  TRY(dalloc(&s->WD, (size_t)nchains * cap * cap)); TRY(dalloc(&s->WL, (size_t)nchains * cap * cap));
  // Group size: as many chains per launch as have their group state (S and Cc, cap x n entries each, row summaries,
  // change counts, merged-state log-likelihoods, per-slot margins) in 60 % of the free memory.
  {
    const size_t per = (sizeof(longlong2) + sizeof(double2)) * (size_t)cap * n + (32 + sizeof(unsigned)) * (size_t)n +
                       sizeof(unsigned) * (size_t)(cap + 1) + (sizeof(double) + sizeof(unsigned)) * (size_t)cap * cap +
                       sizeof(double4) * (size_t)cap + sizeof(unsigned) * 2;
    size_t freeb = 0, totalb = 0;
    cudaMemGetInfo(&freeb, &totalb);
    s->group = std::min<int64_t>(nchains, (int64_t)(freeb / 10 * 6 / per));
    if (const char* e = getenv("RCB200_CHAINS_PER_GROUP")) s->group = std::min<int64_t>(s->group, atoll(e));   // test hook
    if (s->group < 1) {
      rc_set_error("n = %lld, slot_cap = %d: one chain's row sums and caches (%.2f GB) do not fit 60 %% of the free device memory (%.2f GB)",
                   (long long)n, cap, per / 1e9, freeb / 1e9);
      rc_sampler_destroy(s); return RC_ERR_ARG;
    }
    const int64_t L = s->group;                // chains per launch
    int nthr = L <= nsm ? 512 : 256;
    if (const char* e = getenv("RCB200_INC_THREADS")) nthr = std::max(32, std::min(512, atoi(e) / 32 * 32));
    s->inc_nthr = nthr;
    s->shortcuts = 1;
    if (const char* e = getenv("RCB200_SHORTCUTS")) s->shortcuts = atoi(e) != 0;
    // The scan runs beside the restricted scans (dry, on a copy of the labels) when there is one proposal per iteration:
    // measured at n = 10^4 / 50 clusters, 256 threads with 64 on the restricted scans +12 % (256 chains), 512 with 128 +11 %.
    s->ovl_min_thr = 256; s->rs_team = nthr >= 512 ? 128 : 64;
    if (const char* e = getenv("RCB200_OVERLAP_MIN_THREADS")) s->ovl_min_thr = atoi(e);
    if (const char* e = getenv("RCB200_RS_TEAM")) s->rs_team = std::max(32, atoi(e) / 32 * 32);
    // shared memory per chain: the fixed part plus as many split-merge members (64 B each) as fit next to the other
    // CTAs of the SM (two chains per SM when there are more chains than SMs)
    const size_t budget = L <= nsm ? (size_t)maxsmem : ((size_t)maxsmem + 1024) / 2 - 1024;
    // the per-point validity counts of the cached terms (4 B per point) go to shared memory when at least 512 split-merge
    // members still fit beside them: the row evaluation then knows which entries are valid without a trip to memory
    s->tw_smem = rc_sampler_inc_smem_bytes((int)n, cap, 512, 1) <= budget ? 1 : 0;
    if (const char* e = getenv("RCB200_TW_SMEM")) s->tw_smem = atoi(e) != 0 && rc_sampler_inc_smem_bytes((int)n, cap, 0, 1) <= budget;
    const size_t base = rc_sampler_inc_smem_bytes((int)n, cap, 0, s->tw_smem);
    int mcap = base < budget ? (int)((budget - base) / 64) : 0;
    mcap = std::min<int>(mcap, (int)n + 2) / 8 * 8;
    s->inc_mcap = std::max(mcap, 0);
    s->inc_smem = rc_sampler_inc_smem_bytes((int)n, cap, s->inc_mcap, s->tw_smem);
    if (s->inc_smem > (size_t)maxsmem) { s->inc_mcap = 0; s->inc_smem = base; }
    // (the largest case, n = 65535 and slot_cap = 255 with no member scratch and the counts in global memory, needs about
    // 177 KB: below the 227 KB a CTA can have on sm_100)
    if (s->inc_smem > (size_t)maxsmem) {
      rc_set_error("n = %lld, slot_cap = %d: the chain kernel needs %zu B of shared memory per chain, the device allows %d",
                   (long long)n, cap, s->inc_smem, maxsmem);
      rc_sampler_destroy(s); return RC_ERR_ARG;
    }
    if (vb_) fprintf(stderr, "[rcb200] %lld of %lld chains per launch (%.2f GB of row sums and caches per chain, %.2f GB free), %d threads per chain, %zu B shared memory (%d split-merge members)\n",
                     (long long)L, (long long)nchains, per / 1e9, freeb / 1e9, nthr, s->inc_smem, s->inc_mcap);
  }
  s->terms_stride = (size_t)std::max(cap * cap, 8192);
  {
    const size_t G = (size_t)s->group;
    TRY(dalloc(&s->S, G * cap * n)); TRY(dalloc(&s->Cc, G * cap * n)); TRY(dalloc(&s->Vv, G * n));
    TRY(dalloc(&s->epochs, G * (cap + 1)));
    { char* rs = nullptr; TRY(dalloc(&rs, G * n * 32)); s->Rs = rs; }
    TRY(dalloc(&s->LLF, G * cap * cap)); TRY(dalloc(&s->LLFs, G * cap * cap));
    TRY(dalloc(&s->Cm, G * cap)); TRY(dalloc(&s->Cms, G * 2));
  }
  if (opt->numMH > 1) {
    TRY(dalloc(&s->WDbak, (size_t)nchains * cap * cap)); TRY(dalloc(&s->WLbak, (size_t)nchains * cap * cap));
    TRY(dalloc(&s->labbak, (size_t)nchains * n)); TRY(dalloc(&s->szbak, (size_t)nchains * (cap + 1)));
  }
  TRY(dalloc(&s->Slist, (size_t)nchains * (n + 2))); TRY(dalloc(&s->origM, (size_t)nchains * (n + 2)));
  TRY(dalloc(&s->AB, (size_t)nchains * (n + 2))); TRY(dalloc(&s->L2s, (size_t)nchains * n));
  TRY(dalloc(&s->NZ, opt->numMH > 0 ? (size_t)nchains * (opt->numGibbs + 1) * n : 1));
  TRY(dalloc(&s->DG, (size_t)nchains * (n + 2)));
  TRY(dalloc(&s->stats, (size_t)nchains * 16)); TRY(dalloc(&s->terms, (size_t)nchains * s->terms_stride));
  TRY(dalloc(&s->out_labels, (size_t)nchains * NS * n)); TRY(dalloc(&s->out_K, (size_t)nchains * NS));
  TRY(dalloc(&s->out_r, (size_t)nchains * NS)); TRY(dalloc(&s->out_p, (size_t)nchains * NS));
  TRY(dalloc(&s->out_ll, (size_t)nchains * NS)); TRY(dalloc(&s->out_lp, (size_t)nchains * NS));
  TRY(dalloc(&s->r_acc, (size_t)nchains * opt->numiters));
  TRY(dalloc(&s->sm_acc, (size_t)nchains * opt->numiters * std::max<int64_t>(opt->numMH, 1)));
  TRY(dalloc(&s->sm_split, (size_t)nchains * opt->numiters * std::max<int64_t>(opt->numMH, 1)));
  const double tc2_ = tnow_();
#undef TRY
#define TRYC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc_set_error("sampler setup: CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); rc_sampler_destroy(s); return RC_ERR_CUDA; } } while (0)
  TRYC(cudaMemcpy(s->labels, lab.data(), lab.size(), cudaMemcpyHostToDevice));
  TRYC(cudaMemcpy(s->sizes, sizes.data(), sizes.size() * sizeof(int), cudaMemcpyHostToDevice));
  TRYC(cudaMemcpy(s->r, init_r, sizeof(double) * nchains, cudaMemcpyHostToDevice));
  TRYC(cudaMemcpy(s->p, init_p, sizeof(double) * nchains, cudaMemcpyHostToDevice));
  TRYC(cudaMemset(s->status, 0, sizeof(int) * nchains));
  TRYC(cudaMemset(s->stats, 0, sizeof(long long) * 16 * nchains));
  TRYC(cudaMemset(s->r_acc, 0, (size_t)nchains * opt->numiters));
  TRYC(cudaMemset(s->sm_acc, 0, (size_t)nchains * opt->numiters * std::max<int64_t>(opt->numMH, 1)));
  TRYC(cudaMemset(s->sm_split, 0, (size_t)nchains * opt->numiters * std::max<int64_t>(opt->numMH, 1)));
  TRYC(cudaStreamCreate(&s->stream));
  TRYC(cudaEventCreate(&s->e0)); TRYC(cudaEventCreate(&s->e1));
#undef TRYC
  if ((st = reset_caches(s))) { rc_sampler_destroy(s); return st; }
  rc_launch_tables(s->par, (int)n, s->LGA, s->LGZ, s->LOGN, s->stream);
  cudaError_t e = cudaStreamSynchronize(s->stream);
  if (e != cudaSuccess) { rc_set_error("sampler setup failed: %s", cudaGetErrorString(e)); rc_sampler_destroy(s); return RC_ERR_CUDA; }
  if (vb_) fprintf(stderr, "[rcb200] sampler create: host labels %.1f ms, allocations %.1f ms, uploads / memsets / tables %.1f ms\n", (tc1_ - tc0_) * 1e3, (tc2_ - tc1_) * 1e3, (tnow_() - tc2_) * 1e3);
  *out = s;
  return RC_OK;
}

int32_t rc_sampler_run(rc_sampler* s, int64_t iters) {
  if (!s) { rc_set_error("rc_sampler_run: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  int64_t it1 = iters < 0 ? s->opt.numiters : std::min<int64_t>(s->opt.numiters, s->iters_done + iters);
  if (it1 <= s->iters_done && s->W_ready) return RC_OK;
  // Resident (one group): S and W are built before the first launch and maintained from then on.  Grouped: every launch
  // rebuilds them from its chains' labels with every cache stale; S and W are exact integers and every cache is validated
  // by change counts, so the chains compute the same bits as resident ones.
  const bool resident = s->group == s->nchains;
  RC_CUDA(cudaEventRecord(s->e0, s->stream));
  for (int64_t g0 = 0; g0 < s->nchains; g0 += s->group) {
    rc_kparams kp;
    fill_kparams(s, kp, g0);
    kp.it0 = s->iters_done; kp.it1 = it1;
    if (!resident) { int st = reset_caches(s); if (st) return st; }
    if (!resident || !s->W_ready)
      if (rc_launch_inc_init(kp, resident && s->shared_init, s->stream)) { rc_set_error("chain state initialisation failed: %s", cudaGetErrorString(cudaGetLastError())); return RC_ERR_CUDA; }
    if (kp.it1 > kp.it0) rc_launch_chain_inc(kp, s->inc_smem, s->inc_nthr, s->stream);
    s->last_g0 = g0;
  }
  RC_CUDA(cudaGetLastError());
  RC_CUDA(cudaEventRecord(s->e1, s->stream));
  RC_CUDA(cudaStreamSynchronize(s->stream));
  float ms = 0;
  RC_CUDA(cudaEventElapsedTime(&ms, s->e0, s->e1));
  s->dev_seconds += ms * 1e-3;
  s->iters_done = it1;
  s->W_ready = true;
  s->mirror.valid = false;
  // A chain that needed more than slot_cap live clusters has stopped (rc_sampler_chain_status reports it); the other
  // chains are unaffected and their results stay readable.  The call fails only when no healthy chain is left.
  std::vector<int> status((size_t)s->nchains);
  RC_CUDA(cudaMemcpy(status.data(), s->status, sizeof(int) * s->nchains, cudaMemcpyDeviceToHost));
  int64_t bad = 0, firstbad = -1;
  for (int64_t c = 0; c < s->nchains; ++c)
    if (status[c]) { if (firstbad < 0) firstbad = c; ++bad; }
  s->overflowed = bad;
  if (bad == s->nchains) {
    rc_set_error("chain %lld needed more than slot_cap = %d simultaneously live clusters (%lld of %lld chains stopped)", (long long)firstbad,
                 s->cap, (long long)bad, (long long)s->nchains);
    return RC_ERR_SLOTS;
  }
  return RC_OK;
}

int32_t rc_sampler_progress(const rc_sampler* s, int64_t* iters_done, double* device_seconds) {
  if (!s) { rc_set_error("rc_sampler_progress: null handle"); return RC_ERR_ARG; }
  if (iters_done) *iters_done = s->iters_done;
  if (device_seconds) *device_seconds = s->dev_seconds;
  return RC_OK;
}

int64_t rc_sampler_numsamples(const rc_sampler* s) { return s ? s->numsamples : 0; }

// Fills the host mirror when the whole set of recorded outputs is small enough to be worth one bulk download.
static int mirror_fill(const rc_sampler* s) {
  rc_host_mirror& m = s->mirror;
  if (m.valid) return RC_OK;
  const size_t C = (size_t)s->nchains, S = (size_t)s->numsamples, n = (size_t)s->n;
  const size_t ni = (size_t)s->opt.numiters, nm = ni * (size_t)s->opt.numMH;
  m.labels.resize(C * S * n); m.K.resize(C * S); m.r.resize(C * S); m.p.resize(C * S); m.ll.resize(C * S); m.lp.resize(C * S);
  m.r_acc.resize(C * ni); m.sm_acc.resize(C * nm); m.sm_split.resize(C * nm);
  if (S) {
    RC_CUDA(cudaMemcpy(m.labels.data(), s->out_labels, m.labels.size(), cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.K.data(), s->out_K, sizeof(int) * C * S, cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.r.data(), s->out_r, sizeof(double) * C * S, cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.p.data(), s->out_p, sizeof(double) * C * S, cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.ll.data(), s->out_ll, sizeof(double) * C * S, cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.lp.data(), s->out_lp, sizeof(double) * C * S, cudaMemcpyDeviceToHost));
  }
  if (ni) RC_CUDA(cudaMemcpy(m.r_acc.data(), s->r_acc, C * ni, cudaMemcpyDeviceToHost));
  if (nm) {
    RC_CUDA(cudaMemcpy(m.sm_acc.data(), s->sm_acc, C * nm, cudaMemcpyDeviceToHost));
    RC_CUDA(cudaMemcpy(m.sm_split.data(), s->sm_split, C * nm, cudaMemcpyDeviceToHost));
  }
  m.valid = true;
  return RC_OK;
}
static bool mirror_wanted(const rc_sampler* s) {
  return s->nchains > 1 && (size_t)s->nchains * (size_t)s->numsamples * (size_t)s->n <= ((size_t)256 << 20);
}

int32_t rc_sampler_copy_samples(const rc_sampler* s, int64_t chain, int64_t* labels, int64_t* K, double* r, double* p,
                                double* loglik, double* logposterior) {
  if (!s || chain < 0 || chain >= s->nchains) { rc_set_error("rc_sampler_copy_samples: bad handle or chain"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  const int64_t n = s->n, S = s->numsamples;
  if (S == 0) return RC_OK;
  if (mirror_wanted(s)) {
    int st = mirror_fill(s);
    if (st) return st;
    const rc_host_mirror& m = s->mirror;
    const size_t o = (size_t)chain * S;
    if (labels) { const uint8_t* src = m.labels.data() + o * n; for (size_t t = 0; t < (size_t)S * n; ++t) labels[t] = src[t]; }
    if (K) for (int64_t t = 0; t < S; ++t) K[t] = m.K[o + t];
    if (r) memcpy(r, m.r.data() + o, sizeof(double) * S);
    if (p) memcpy(p, m.p.data() + o, sizeof(double) * S);
    if (loglik) memcpy(loglik, m.ll.data() + o, sizeof(double) * S);
    if (logposterior) memcpy(logposterior, m.lp.data() + o, sizeof(double) * S);
    return RC_OK;
  }
  if (labels) {
    std::vector<uint8_t> tmp((size_t)S * n);
    RC_CUDA(cudaMemcpy(tmp.data(), s->out_labels + (size_t)chain * S * n, tmp.size(), cudaMemcpyDeviceToHost));
    for (size_t t = 0; t < tmp.size(); ++t) labels[t] = tmp[t];
  }
  if (K) {
    std::vector<int> tmp((size_t)S);
    RC_CUDA(cudaMemcpy(tmp.data(), s->out_K + (size_t)chain * S, sizeof(int) * S, cudaMemcpyDeviceToHost));
    for (int64_t t = 0; t < S; ++t) K[t] = tmp[t];
  }
  if (r) RC_CUDA(cudaMemcpy(r, s->out_r + (size_t)chain * S, sizeof(double) * S, cudaMemcpyDeviceToHost));
  if (p) RC_CUDA(cudaMemcpy(p, s->out_p + (size_t)chain * S, sizeof(double) * S, cudaMemcpyDeviceToHost));
  if (loglik) RC_CUDA(cudaMemcpy(loglik, s->out_ll + (size_t)chain * S, sizeof(double) * S, cudaMemcpyDeviceToHost));
  if (logposterior) RC_CUDA(cudaMemcpy(logposterior, s->out_lp + (size_t)chain * S, sizeof(double) * S, cudaMemcpyDeviceToHost));
  return RC_OK;
}

// Every chain's recorded outputs at once: ONE device-to-host copy per array into a pinned staging buffer, then the label
// bytes are widened to the int64 the reference's API returns (Vector{Int}) by all host threads.  Layouts: labels
// nchains x numsamples x n; K, r, p, loglik, logposterior nchains x numsamples; r_acc nchains x numiters; sm_* nchains x
// numiters*numMH.  Any pointer may be NULL.
static void* pinned_staging(size_t bytes) {
  static void* buf = nullptr; static size_t cap = 0;     // grow-only, process lifetime (one reader at a time per process)
  if (bytes > cap) {
    if (buf) cudaFreeHost(buf);
    buf = nullptr; cap = 0;
    if (cudaMallocHost(&buf, bytes) != cudaSuccess) { (void)cudaGetLastError(); buf = nullptr; return nullptr; }
    cap = bytes;
  }
  return buf;
}
int32_t rc_sampler_copy_all(const rc_sampler* s, int64_t* labels, int64_t* K, double* r, double* p, double* loglik,
                            double* logposterior, uint8_t* r_acc, uint8_t* sm_acc, uint8_t* sm_split) {
  if (!s) { rc_set_error("rc_sampler_copy_all: null handle"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  const size_t Cn = (size_t)s->nchains, S = (size_t)s->numsamples, n = (size_t)s->n;
  const size_t ni = (size_t)s->opt.numiters, nm = ni * (size_t)s->opt.numMH;
  if (S) {
    if (labels) {
      const size_t total = Cn * S * n;
      uint8_t* st = (uint8_t*)pinned_staging(total);
      std::vector<uint8_t> fallback;
      if (!st) { fallback.resize(total); st = fallback.data(); }
      RC_CUDA(cudaMemcpy(st, s->out_labels, total, cudaMemcpyDeviceToHost));
      const unsigned nth = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
      std::vector<std::thread> th;
      for (unsigned t = 0; t < nth; ++t)
        th.emplace_back([=]() {
          const size_t b = total * t / nth, e = total * (t + 1) / nth;
          for (size_t i = b; i < e; ++i) labels[i] = st[i];
        });
      for (auto& x : th) x.join();
    }
    if (K) {
      std::vector<int> tmp(Cn * S);
      RC_CUDA(cudaMemcpy(tmp.data(), s->out_K, sizeof(int) * Cn * S, cudaMemcpyDeviceToHost));
      for (size_t t = 0; t < Cn * S; ++t) K[t] = tmp[t];
    }
    if (r) RC_CUDA(cudaMemcpy(r, s->out_r, sizeof(double) * Cn * S, cudaMemcpyDeviceToHost));
    if (p) RC_CUDA(cudaMemcpy(p, s->out_p, sizeof(double) * Cn * S, cudaMemcpyDeviceToHost));
    if (loglik) RC_CUDA(cudaMemcpy(loglik, s->out_ll, sizeof(double) * Cn * S, cudaMemcpyDeviceToHost));
    if (logposterior) RC_CUDA(cudaMemcpy(logposterior, s->out_lp, sizeof(double) * Cn * S, cudaMemcpyDeviceToHost));
  }
  if (r_acc && ni) RC_CUDA(cudaMemcpy(r_acc, s->r_acc, Cn * ni, cudaMemcpyDeviceToHost));
  if (sm_acc && nm) RC_CUDA(cudaMemcpy(sm_acc, s->sm_acc, Cn * nm, cudaMemcpyDeviceToHost));
  if (sm_split && nm) RC_CUDA(cudaMemcpy(sm_split, s->sm_split, Cn * nm, cudaMemcpyDeviceToHost));
  return RC_OK;
}

int32_t rc_sampler_copy_acceptances(const rc_sampler* s, int64_t chain, uint8_t* r_acc, uint8_t* sm_acc, uint8_t* sm_split) {
  if (!s || chain < 0 || chain >= s->nchains) { rc_set_error("rc_sampler_copy_acceptances: bad handle or chain"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  const size_t ni = (size_t)s->opt.numiters, nm = ni * (size_t)s->opt.numMH;
  if (mirror_wanted(s)) {
    int st = mirror_fill(s);
    if (st) return st;
    if (r_acc && ni) memcpy(r_acc, s->mirror.r_acc.data() + chain * ni, ni);
    if (sm_acc && nm) memcpy(sm_acc, s->mirror.sm_acc.data() + chain * nm, nm);
    if (sm_split && nm) memcpy(sm_split, s->mirror.sm_split.data() + chain * nm, nm);
    return RC_OK;
  }
  if (r_acc) RC_CUDA(cudaMemcpy(r_acc, s->r_acc + chain * ni, ni, cudaMemcpyDeviceToHost));
  if (sm_acc && nm) RC_CUDA(cudaMemcpy(sm_acc, s->sm_acc + chain * nm, nm, cudaMemcpyDeviceToHost));
  if (sm_split && nm) RC_CUDA(cudaMemcpy(sm_split, s->sm_split + chain * nm, nm, cudaMemcpyDeviceToHost));
  return RC_OK;
}

int32_t rc_sampler_copy_state(const rc_sampler* s, int64_t chain, int64_t* labels, double* r, double* p) {
  if (!s || chain < 0 || chain >= s->nchains) { rc_set_error("rc_sampler_copy_state: bad handle or chain"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  const int64_t n = s->n;
  if (labels) {
    std::vector<uint8_t> tmp((size_t)n);
    RC_CUDA(cudaMemcpy(tmp.data(), s->labels + (size_t)chain * n, n, cudaMemcpyDeviceToHost));
    for (int64_t j = 0; j < n; ++j) labels[j] = (int64_t)tmp[j] + 1;
  }
  if (r) RC_CUDA(cudaMemcpy(r, s->r + chain, sizeof(double), cudaMemcpyDeviceToHost));
  if (p) RC_CUDA(cudaMemcpy(p, s->p + chain, sizeof(double), cudaMemcpyDeviceToHost));
  return RC_OK;
}

// Debug / profiling aid: 16 SM-cycle counters per chain accumulated by the chain kernel (decision wait / work,
// bulk waits, split-merge phases, ...; slot names in rc_sampler.cu).  out: nchains x 16 int64.
int32_t rc_sampler_copy_stats(const rc_sampler* s, int64_t* out) {
  if (!s || !out) { rc_set_error("rc_sampler_copy_stats: null pointer"); return RC_ERR_ARG; }
  RC_CUDA(cudaSetDevice(s->device));
  RC_CUDA(cudaMemcpy(out, s->stats, sizeof(long long) * 16 * s->nchains, cudaMemcpyDeviceToHost));
  return RC_OK;
}

int64_t rc_sampler_overflowed(const rc_sampler* s) { return s ? s->overflowed : 0; }

// Invariant check of the maintained sums: rebuilds the row sums S and block sums W of the chains launched last (every
// chain in resident mode, the last group in grouped mode: only its S still exists) from their current labels and counts
// the 64-bit words that differ from the incrementally maintained ones (both must be 0).  Before the first run there is
// nothing to compare: both counts are returned as -1.
int32_t rc_sampler_check_sums(const rc_sampler* s, int64_t* mismatches_S, int64_t* mismatches_W) {
  if (!s || !mismatches_S || !mismatches_W) { rc_set_error("rc_sampler_check_sums: null pointer"); return RC_ERR_ARG; }
  *mismatches_S = -1; *mismatches_W = -1;
  if (!s->W_ready) return RC_OK;
  RC_CUDA(cudaSetDevice(s->device));
  rc_kparams kp;
  fill_kparams(s, kp, s->last_g0);
  long long a = 0, b = 0;
  if (rc_inc_check(kp, &a, &b, s->stream)) { rc_set_error("rc_sampler_check_sums: rebuild failed (out of memory?)"); return RC_ERR_CUDA; }
  *mismatches_S = a; *mismatches_W = b;
  return RC_OK;
}

int32_t rc_sampler_chain_status(const rc_sampler* s, int64_t chain) {
  if (!s || chain < 0 || chain >= s->nchains) { rc_set_error("rc_sampler_chain_status: bad handle or chain"); return RC_ERR_ARG; }
  cudaSetDevice(s->device);
  int st = 0;
  if (cudaMemcpy(&st, s->status + chain, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return RC_ERR_CUDA;
  return st;
}

// loglik(data, state, params) for one host label vector (src/mcmc.jl:1-56): a one-chain sampler builds the block sums
// from scratch, then the chain kernel evaluates the log-likelihood once, as the sampler does.
int32_t rc_loglik(const rc_data* d, const rc_params* par, const int64_t* labels, double* out) {
  if (!d || !par || !labels || !out) { rc_set_error("rc_loglik: null pointer"); return RC_ERR_ARG; }
  rc_options opt = {1, 0, 1, 0, 0};
  const int64_t n = d->n;
  // compact arbitrary positive labels order-preservingly (loglik visits clusters in ascending slot order)
  std::vector<int64_t> uniq(labels, labels + n);
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  if ((int64_t)uniq.size() > RC_MAXCAP) { rc_set_error("rc_loglik: more than %d clusters", RC_MAXCAP); return RC_ERR_SLOTS; }
  std::vector<int64_t> lab((size_t)n);
  for (int64_t j = 0; j < n; ++j) lab[j] = (std::lower_bound(uniq.begin(), uniq.end(), labels[j]) - uniq.begin()) + 1;
  double r0 = 1.0, p0 = 0.5;
  rc_sampler* s = nullptr;
  int st = rc_sampler_create(d, &opt, par, 1, 0, lab.data(), &r0, &p0, 0, 0, &s);
  if (st) return st;
  rc_kparams kp;
  fill_kparams(s, kp);
  kp.loglik_only = 1;
  if (rc_launch_inc_init(kp, false, s->stream)) { rc_set_error("rc_loglik: block sums failed: %s", cudaGetErrorString(cudaGetLastError())); rc_sampler_destroy(s); return RC_ERR_CUDA; }
  rc_launch_chain_inc(kp, s->inc_smem, s->inc_nthr, s->stream);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
  if (e == cudaSuccess) e = cudaMemcpy(out, s->out_ll, sizeof(double), cudaMemcpyDeviceToHost);
  rc_sampler_destroy(s);
  RC_CUDA(e);
  return RC_OK;
}

int64_t rc_sampler_n(const rc_sampler* s) { return s ? s->n : 0; }
int64_t rc_sampler_nchains(const rc_sampler* s) { return s ? s->nchains : 0; }

// sample_rp(clustsizes, options, params) (mcmc.jl:592-636): the (r, p)-only chain of fitprior (prior.jl:80) on the device.
int32_t rc_sample_rp(const int64_t* clustsizes, int64_t nsizes, const rc_options* opt, const rc_params* par, uint64_t seed, int32_t device,
                     double* r_out, double* p_out, uint8_t* r_acc_out) {
  if (!clustsizes || !opt || !par || !r_out || !p_out || nsizes < 1) { rc_set_error("rc_sample_rp: null pointer or no cluster sizes"); return RC_ERR_ARG; }
  int st = validate_options(opt);
  if (st) return st;
  if (!(par->proposalsd_r > 0)) { rc_set_error("invalid hyperparameters (proposalsd_r <= 0)"); return RC_ERR_ARG; }
  st = rc_select_device(device);
  if (st) return st;
  std::vector<int> C;                                  // C = clustsizes[findall(clustsizes .> 0)]  (:613)
  long long n = 0;
  for (int64_t k = 0; k < nsizes; ++k) if (clustsizes[k] > 0) { C.push_back((int)clustsizes[k]); n += clustsizes[k]; }
  if (C.empty()) { rc_set_error("rc_sample_rp: every cluster is empty"); return RC_ERR_ARG; }
  const int K = (int)C.size();
  const int64_t S = (opt->numiters - opt->burnin) / opt->thin;
  int* dsz = nullptr; double *terms = nullptr, *dr = nullptr, *dp = nullptr; uint8_t* dacc = nullptr;
  cudaError_t e = cudaMalloc(&dsz, sizeof(int) * K);
  if (e == cudaSuccess) e = cudaMalloc(&terms, sizeof(double) * 2 * K);
  if (e == cudaSuccess) e = cudaMalloc(&dr, sizeof(double) * std::max<int64_t>(S, 1));
  if (e == cudaSuccess) e = cudaMalloc(&dp, sizeof(double) * std::max<int64_t>(S, 1));
  if (e == cudaSuccess) e = cudaMalloc(&dacc, (size_t)opt->numiters);
  if (e == cudaSuccess) e = cudaMemcpy(dsz, C.data(), sizeof(int) * K, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    rc_kparams kp;
    memset(&kp, 0, sizeof(kp));
    kp.n = (int)n; kp.P = *par; kp.numiters = opt->numiters; kp.burnin = opt->burnin; kp.thin = opt->thin; kp.numsamples = S;
    kp.seed = seed; kp.chain_offset = 0;
    rc_launch_sample_rp(kp, dsz, K, terms, dr, dp, dacc, 0);
    e = cudaDeviceSynchronize();
  }
  if (e == cudaSuccess && S > 0) e = cudaMemcpy(r_out, dr, sizeof(double) * S, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && S > 0) e = cudaMemcpy(p_out, dp, sizeof(double) * S, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && r_acc_out) e = cudaMemcpy(r_acc_out, dacc, (size_t)opt->numiters, cudaMemcpyDeviceToHost);
  cudaFree(dsz); cudaFree(terms); cudaFree(dr); cudaFree(dp); cudaFree(dacc);
  RC_CUDA(e);
  return RC_OK;
}

}  // extern "C"

// The samples of a chain range for the post-processing entry points: only a run to numiters has recorded every sample,
// and a chain stopped by the slot capacity has not (its out_labels were never written).
int rc_sampler_range(const rc_sampler* s, int64_t chain0, int64_t nch, const char* who, rc_sample_range& v) {
  if (chain0 < 0 || nch < 1 || chain0 + nch > s->nchains) { rc_set_error("%s: bad chain range", who); return RC_ERR_ARG; }
  if (s->iters_done < s->opt.numiters) {
    rc_set_error("%s: the sampler ran %lld of %lld iterations; its samples are recorded only by a complete run", who,
                 (long long)s->iters_done, (long long)s->opt.numiters);
    return RC_ERR_STATE;
  }
  TRYP(rc_select_device(s->device));
  std::vector<int> status((size_t)nch);
  RC_CUDA(cudaMemcpy(status.data(), s->status + chain0, sizeof(int) * (size_t)nch, cudaMemcpyDeviceToHost));
  for (int64_t c = 0; c < nch; ++c)
    if (status[c] != 0) {
      rc_set_error("%s: chain %lld stopped at the slot capacity; its samples are incomplete", who, (long long)(chain0 + c));
      return RC_ERR_SLOTS;
    }
  const size_t first = (size_t)chain0 * s->numsamples;
  v.d = s->d; v.par = s->par; v.n = s->n; v.R = nch * s->numsamples;
  v.labels = s->out_labels + first * s->n; v.K = s->out_K + first; v.r = s->out_r + first; v.p = s->out_p + first;
  return RC_OK;
}
