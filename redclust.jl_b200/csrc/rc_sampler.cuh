// rc_sampler.cuh -- kernel-side parameter block of the persistent chain kernel (internal).
#pragma once
#include "rc_common.cuh"

struct RowSum { double cT, c2, L2i; int T; unsigned stamp; };   // row summary of the incremental scan, see rc_sampler.cu
struct rc_kparams {
  int n, cap;
  int qD, qL;
  const longlong2* DL;  // rc_data::DL
  rc_params P;
  double abratio, zgratio, lgd1, lgd2;
  const double* LGA;    // lgamma(alpha + delta1 * s), s = 0..n+1
  const double* LGZ;    // lgamma(zeta + delta2 * s)
  const double* LOGN;   // log(s)
  long long it0, it1;   // run iterations it0+1 .. it1 (1-based, as in mcmc.jl:537)
  long long burnin, thin, numGibbs, numMH, numiters, numsamples;
  unsigned long long seed;
  long long chain_offset;
  int nchains;
  // per-chain state (global memory)
  uint8_t* labels;      // [nchains][n]   0-based slot ids
  int* sizes;           // [nchains][cap]
  double* r;            // [nchains]
  double* p;            // [nchains]
  int* status;          // [nchains]
  rc_i128* WD;          // [nchains][cap*cap]  block sums of Dq, entry (min(k,t), max(k,t))
  rc_i128* WL;          // [nchains][cap*cap]  block sums of Lq
  rc_i128 *WDbak, *WLbak; // [nchains][cap*cap]  numMH > 1 only: the chain's own block sums while a proposal is committed
  uint8_t* labbak;      // [nchains][n]
  int* szbak;           // [nchains][cap+1]
  longlong2* S;         // [nchains][cap][n]   row sums by slot of EVERY point, S[k][x] = sum_{j in k} DL[x][j]
  unsigned short* Slist;// [nchains][n+2]  members of ci u cj of the current split-merge step
  uint8_t* origM;       // [nchains][n+2]  their labels in the chain's state
  longlong4* AB;        // [nchains][n+2]  running candidate sums of the members (restricted scans)
  double2* L2s;         // [nchains][n]    static repulsion terms per item
  double2* NZ;          // [nchains][(numGibbs+1)*n] Gumbel noise of the free restricted scans
  longlong2* DG;        // [nchains][n+2]  diagonal entries DL[x][x] of the split-merge members
  double* terms;        // [nchains][terms_stride]  log-likelihood terms / reduction scratch
  size_t terms_stride;  // max(cap*cap, 8192) doubles
  double2* Cc;          // [nchains][cap][n]  cached per-slot terms (L1, L2') of every (slot, point)
  unsigned* Vv;         // [nchains][n]       change count at which each point's cached entries were last all valid (0: never)
  unsigned* epochs;     // [nchains][cap + 1] change count at which each slot last changed (>= 1), then the chain's change count
  int tw_smem;          // the per-point counts of a chain live in shared memory during a launch
  int shortcuts;        // 1: rows decided by their summaries and merge proposals rejected by their bound skip the work (same results; RCB200_SHORTCUTS=0 turns both off)
  double* LLF; unsigned* LLFs;   // [nchains][cap][cap] merged-state log-likelihoods per ordered slot pair and their change counts
  RowSum* Rs;           // [nchains][n]       row summaries of the incremental scan (32 B each, see rc_sampler.cu)
  double4* Cm;          // [nchains][cap]     per-slot margins of the row summaries (see inc_margins_build)
  unsigned* Cms;        // [nchains][2]       the change count they were built at (0: never) and whether that build succeeded
  int inc_mcap;         // split-merge members that fit the shared-memory scratch (64 B each)
  int ovl_min_thr;      // the scan runs beside the restricted scans when the chain has at least this many threads (0: never)
  int rs_team;          // ... and this many of them run the restricted scans
  // outputs
  uint8_t* out_labels;  // [nchains][numsamples][n]  sortlabels'd, 1-based
  int* out_K;           // [nchains][numsamples]
  double *out_r, *out_p, *out_ll, *out_lp;
  uint8_t *r_acc, *sm_acc, *sm_split;
  long long* stats;     // [nchains][16] cycle counters (debug / profiling aid)
  // standalone log-likelihood mode (rc_loglik): skip iterations, write loglik to out_ll[chain]
  int loglik_only;
};

size_t rc_sampler_inc_smem_bytes(int n, int cap, int mcap, int tw_smem);
int rc_launch_inc_init(const rc_kparams& kp, bool shared_labels, cudaStream_t st);
int rc_inc_check(const rc_kparams& kp, long long* mismatches_S, long long* mismatches_W, cudaStream_t st);
void rc_launch_chain_inc(const rc_kparams& kp, size_t smem, int nthr, cudaStream_t st);
void rc_launch_sample_rp(const rc_kparams& kp, int* sizes, int K, double* terms, double* out_r, double* out_p, uint8_t* out_acc, cudaStream_t st);
void rc_launch_tables(const rc_params& P, int n, double* LGA, double* LGZ, double* LOGN, cudaStream_t st);
