// rc_sampler.cu -- the persistent chain kernel: one launch runs every iteration of runsampler's loop
// (/root/reference/src/mcmc.jl:537-555) for every chain on the device.
//
//   sample_r!  (mcmc.jl:80-136)      -> update_r()
//   sample_p!  (mcmc.jl:138-155)     -> update_p()
//   sample_labels! (mcmc.jl:356-479) -> splitmerge_step() x numMH, then inc_full_scan()
//   sample_labels_Gibbs! (:158-256)  -> inc_full_scan(): inc_eval_row()
//   sample_labels_Gibbs_restricted! (:259-354) -> restricted_scans_team()
//   loglik (:1-56), logprior (:58-78), record step (:546-554), sortlabels (utils.jl:69-74)
//
// The kernel works on DL[i][j] = {Dq, Lq}, the 64-bit fixed-point images of D and log D (DESIGN.md section 2): every cluster
// sum is an exact integer, so results do not depend on lane count or reduction order -- or on whether a sum is recomputed
// or maintained -- and are bit-identical to the CPU oracle.
//
// k_chain_inc: one CTA = one chain, all iterations of a launch inside the kernel.
//   * S[slot][x] = sum of row x over the members of slot is kept in HBM; a Gibbs step reads one entry per live slot
//     (inc_eval_row: G lanes per row, the lane's slots in registers), only a move streams a row (inc_update_S).
//   * Rows are evaluated speculatively in batches and committed up to the first one that moves (inc_full_scan).
//   * Per-slot terms are cached (Cc) and validated by change counts (tw / tchg); a row whose stored summary (RowSum) proves
//     the Gumbel-max outcome is decided without being evaluated.
//   * Split-merge by the whole team: member sums gathered once (member_sums_inc), restricted scans with the moves of eight
//     steps resolved inside a warp (restricted_scans_team), merge proposals that cannot be accepted rejected by their bound
//     (splitmerge_step); the scan runs dry beside the restricted scans while it is long.
//   * W (K x K block sums, 128-bit) is maintained from the row sums of every move, so loglik() never reads D.
// S, W and every cache can be rebuilt from the labels at any launch (k_init_S / k_initw_from_S, caches reset): chains that
// do not all fit the device run in launch groups that share this state (rc_api.cu).
#include <algorithm>
#include "rc_sampler.cuh"

namespace {

struct Scal {
  double r, p, logp, log1mp;
  double ltp;
  double dtmp[4];
  rc_i128 aaD, aaL, abD, abL, bbD, bbL;   // block sums of the proposed state (rows a, b)
  int K;
  int status;
  int forked;                             // numMH > 1: an accepted proposal replaced the local state this iteration
  int fslotA, fslotB;                     // slots whose W rows come from the scratch rows (-1: none)
  int itmp[8];
  double llcur; unsigned llclk;           // incremental kernel: loglik of the chain's own state at change count llclk (0: none)
};

// cycle counters of rc_sampler_copy_stats: compile with -DRC_NO_STATS to drop the clock reads from the hot loops
#ifdef RC_NO_STATS
#define RC_CLOCK() 0LL
#else
#define RC_CLOCK() clock64()
#endif

// Incremental mode (k_chain_inc): hand-off block of the chain's team.
#define RC_INC_MAXW 16               // warps per chain, at most
#define RC_RS_MAXW 8                 // warps that evaluate a batch of the restricted scans, at most
struct IncShared {
  int first[3];      // lowest warp / step of a batch that needs a commit (three rotating slots, see inc_scan_rows)
  int ev;            // what that warp found: 1 move, 2 a slot beyond this instantiation is needed, 3 slot capacity exhausted
  int mv_i, mv_a, mv_b;
  int nmoves;
  unsigned clk;      // number of changes of the chain's state so far (moves of the scan, committed proposals): the clock of the cached terms
  int nlive, e0;     // live slots of the chain's state and its first empty slot (-1: none), see inc_build_tables
  int sfirst[3];     // the scan's own rotating slots (the restricted scans use first[] and may run beside it)
  int dry_stop;      // row at which the scan that ran beside the restricted scans stopped (first row that moves; n: none)
  int hint;          // rows per batch the previous scan ended with (0: none yet)
  int narrow;        // lanes per row of the scan (4 / 8 / 16: every live slot and the first empty slot lie below 64 / 128 / 256)
  int fa[3], fm[3];  // row summaries (see RowSum): first row of a batch its summary does not decide / first decided row that moves
  int mksum;         // the last committed scan moved at most two points: rows keep summaries and are tried against them first
  int nfast_dry;     // rows the dry part of the current pass decided by their summaries
  int scanfast;      // at least half the rows of the last complete pass were: the scan is short, nothing is gained by running it beside the restricted scans
  int tabs_ok;       // every live slot's size-dependent prior term is finite ...
  double maxtab;     // ... and this is their maximum (at the slot's size and at size - 1)
  unsigned cm_clk;   // change count the per-slot margins (Cm) were built at (0: never) ...
  int cm_ok;         // ... and whether that build succeeded (see inc_margins_build)
  int rs_mv[RC_INC_MAXW][8];            // restricted scans: per warp the moves of its eight steps, in step order: item << 1 | (1: ca -> cb)
  int rs_nm[RC_INC_MAXW];               // ... and how many
  double rs_win[RC_RS_MAXW][6][16];     // ... per evaluating warp: LGA / LGZ / LPR at the sixteen sizes its steps can see ({A, B} x 3 tables)
  double ltbuf[2][RC_INC_MAXW * 8];     // restricted scans: log transition probabilities of a batch's steps (last scan)
};
#define RC_INC_NONE 0x7fffffff

// Summary of a row's last full evaluation (incremental mode, one per point and chain): the leading slot T, its term c_T and
// the largest term c_2 among the other live slots, where the log-probability of slot k is tab_k + c_k with tab_k the only part
// that depends on (r, p), and the repulsion total L2i (the new-cluster candidate is A(r, p) + L2i).  While the chain's state
// has not changed (stamp == clk) every c_k is bit for bit what a fresh evaluation would compute, so
//   tab_T + c_T - (max_k tab_k + c_2) > 41   and   tab_T + c_T - (A + L2i) > 41
// prove that slot T wins the Gumbel-max whatever the noise is (noise lies in [-3.61, 36.74] for every 53-bit uniform > 0;
// the leader's own uniform is drawn and checked to be > 0): the row is decided without being evaluated.
// (struct RowSum { double cT, c2, L2i; int T; unsigned stamp; } is declared in rc_sampler.cuh)
#define RC_SUM_MARGIN 41.0

struct Ctx {
  int n, cap;
  int qD, qL;
  int ctid, cwarp, lane, barid;           // thread / warp index within the chain, named barrier of the chain
  int nthr, nwarp;                        // threads / warps of the chain's team (the whole CTA, or part of it beside the restricted scans)
  const longlong2* DL;
  const rc_kparams* kp;
  // shared memory
  uint8_t* lab;
  uint8_t* labL;          // the labels a split-merge step works on in place (launch state): the chain's own array, or -- with one
                          // proposal per iteration -- a copy, so that the scan can run beside the restricted scans
  rc_i128* prows;         // [4][cap] rows A_D, A_L, B_D, B_L of the block sums of a split-merge step's proposed state
  int* sizes;
  int* szL;
  int* itmp;              // [cap]
  uint8_t* clist;         // [cap]
  Scal* sc;
  // per-chain global memory
  rc_i128* WD;
  rc_i128* WL;
  rc_i128* WDbak;         // numMH > 1: the chain's own block sums / labels / sizes while an accepted proposal is the local state
  rc_i128* WLbak;
  uint8_t* labbak;
  int* szbak;
  longlong2* S;           // [cap][n] row sums by slot, S[k][x] = sum_{j in k} DL[x][j]
  struct IncShared* inc;  // hand-off block of the scan
  int mcap;               // members of a split-merge step whose AB / DG / L2s fit the shared-memory scratch
  longlong4* mAB; longlong2* mDG; double2* mL2s;   // that scratch
  uint8_t* live;          // (shared memory) live slots, ascending
  uint8_t* rank;          // (shared memory) [cap] number of live slots below each slot
  double* tabs;           // (shared memory) [6][cap] lgamma(alpha + delta1 s), lgamma(zeta + delta2 s), prior term at the slot's size / at size - 1
  int* res;               // (shared memory) [nthr] slot chosen by each row of a batch
  double2* Cc;            // (global) [cap][n] cached per-slot terms, see inc_eval_row
  RowSum* Rs;             // (global) [n] row summaries
  double4* Cm; unsigned* Cms;    // (global) [cap] per-slot margins of the row summaries, [2] their change count and build result
  double* LLF; unsigned* LLFs;   // (global) [cap][cap] loglik of the state with slot ci merged into cj, and the change count it was computed at (0: never)
  unsigned* tw;           // (shared memory when it fits, else global) [n] change count at which point x's cached entries were last made valid
  unsigned* tchg;         // (shared memory) [cap] change count at which each slot last gained or lost a point
  unsigned short* Slist;  // members of ci u cj: S ascending, then i, then j
  uint8_t* origM;         // their labels in the chain's state
  longlong4* AB;          // [n+2] running sums of each member's row over the two candidate clusters {aD, aL, bD, bL}
  double2* L2s;           // [n]   static repulsion terms of the first two live slots, per item
  double2* NZ;            // [(numGibbs+1) * n] Gumbel noise of the free restricted scans
  longlong2* DG;          // [n+2] DL[x][x] of the members
  double* terms;
  long long* stats;       // [16] cycle counters of this chain (see rc_sampler_copy_stats)
  unsigned long long key;
};
// Incremental mode: point y moved from slot a to slot b.  Every x's sums over a and b follow from row y (D is symmetric:
// DL[x][y] == DL[y][x]); exact integers, so S stays what a from-scratch build would give.  Thread t always owns the same
// x's for a given t0, so successive moves with the same t0 need no barrier between them (one before the sums are read again).
__device__ __forceinline__ void inc_update_S(const Ctx& c, int y, int a, int b, int skip = -1, int t0 = 0) {
  const longlong2* __restrict__ row = c.DL + (size_t)y * c.n;
  longlong2* Sa = c.S + (size_t)a * c.n;
  longlong2* Sb = c.S + (size_t)b * c.n;
  // threads t0 .. nthr-1 share the work (the scan keeps warp 0 busy with the block sums meanwhile)
  const int n = c.n, nt = c.nthr - t0;
  int x = c.ctid - t0;
  if (x < 0) return;
  for (; x + 3 * nt < n; x += 4 * nt) {
    longlong2 v[4], sa[4], sb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { v[u] = __ldg(row + x + u * nt); sa[u] = Sa[x + u * nt]; sb[u] = Sb[x + u * nt]; }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (x + u * nt == skip) continue;                  // (the caller updates this entry itself)
      sa[u].x -= v[u].x; sa[u].y -= v[u].y; sb[u].x += v[u].x; sb[u].y += v[u].y;
      Sa[x + u * nt] = sa[u]; Sb[x + u * nt] = sb[u];
    }
  }
  for (; x < n; x += nt) {
    if (x == skip) continue;
    const longlong2 v = __ldg(row + x);
    longlong2 sa = Sa[x], sb = Sb[x];
    sa.x -= v.x; sa.y -= v.y; sb.x += v.x; sb.y += v.y;
    Sa[x] = sa; Sb[x] = sb;
  }
}
// stats slots (in the default library, -DRC_NO_STATS, the timing slots stay 0 and a few count events instead: dec_wait the
// merge proposals rejected by their bound, bulk_rows the rows decided by their summaries, bulk_reduce the scans decided by
// the per-slot margins)
enum { ST_DEC_WAIT = 0, ST_DEC_WORK, ST_BULK_WAIT_CONSUMED, ST_BULK_WAIT_FULL, ST_BULK_ROWS, ST_BULK_PATCH, ST_MOVES, ST_REBUILDS,
       ST_MH_SETUP, ST_MH_RSCAN, ST_MH_LOGLIK, ST_SCAN_TOTAL, ST_RECORD, ST_ITER_TOTAL, ST_RP, ST_BULK_REDUCE };
__device__ __forceinline__ void st_add(const Ctx& c, int slot, long long v) { c.stats[slot] += v; }

__device__ __forceinline__ void csync(const Ctx& c) { asm volatile("bar.sync %0, %1;" ::"r"(c.barid), "r"(c.nthr) : "memory"); }

// sum of a 128-bit value over the lanes of a warp (every lane gets the total)
__device__ __forceinline__ rc_i128 warp_sum128(rc_i128 v) {
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    rc_i128 o;
    o.lo = __shfl_xor_sync(0xffffffffu, v.lo, off);
    o.hi = __shfl_xor_sync(0xffffffffu, v.hi, off);
    rc_add128(v, o);
  }
  return v;
}
__device__ __forceinline__ int tri(int k, int t, int cap) { return k < t ? k * cap + t : t * cap + k; }

// ------------------------------------------------------------------------------------------------
// loglik (mcmc.jl:1-56) from the block sums.  `sz` are the cluster sizes of the evaluated state; rows of
// slots fslotA / fslotB (proposed state of a split-merge step) come from the scratch rows c.prows,
// everything else from the chain's W.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ rc_i128 getW(const Ctx& c, bool logm, int k, int t) {
  const Scal& s = *c.sc;
  const int A = s.fslotA, B = s.fslotB;
  if (k == A || t == A || k == B || t == B) {
    if (A >= 0 && B >= 0 && ((k == A && t == B) || (k == B && t == A))) return logm ? s.abL : s.abD;
    if (k == A && t == A) return logm ? s.aaL : s.aaD;
    if (k == B && t == B) return logm ? s.bbL : s.bbD;
    const rc_i128* rows = c.prows;    // [rowA_D | rowA_L | rowB_D | rowB_L] x cap
    const bool isA = (k == A || t == A);
    const int other = isA ? (k == A ? t : k) : (k == B ? t : k);
    return rows[((isA ? 0 : 2) + (logm ? 1 : 0)) * c.cap + other];
  }
  return (logm ? c.WL : c.WD)[tri(k, t, c.cap)];
}

__device__ double loglik_eval(const Ctx& c, const int* sz) {
  const rc_kparams& kp = *c.kp;
  const rc_params& P = kp.P;
  csync(c);
  if (c.ctid < 32) {                                                        // C = findall(clustsizes .> 0)  (:22)
    int base = 0;
    for (int w = 0; w * 32 < c.cap; ++w) {
      const int s = w * 32 + c.ctid;
      const bool live = s < c.cap && sz[s] > 0;
      const unsigned m = __ballot_sync(0xffffffffu, live);
      if (live) c.clist[base + __popc(m & ((1u << c.ctid) - 1u))] = (uint8_t)s;
      base += __popc(m);
    }
    if (c.ctid == 0) c.sc->itmp[0] = base;
  }
  csync(c);
  const int K = c.sc->itmp[0];
  // The terms are added by one thread in the reference's order (:54), which is a chain of dependent additions: when they fit,
  // they are staged in shared memory (the split-merge member scratch, dead whenever a log-likelihood is evaluated) in exactly
  // that order -- K diagonal terms, then the pairs (k, t > k) row by row -- instead of being read back from global memory.
  const int nT = K + K * (K - 1) / 2;
  double* st = (c.mAB && (size_t)nT * sizeof(double) <= (size_t)c.mcap * sizeof(longlong4)) ? reinterpret_cast<double*>(c.mAB) : nullptr;
  for (int idx = c.ctid; idx < K * K; idx += c.nthr) {
    const int ki = idx / K, ti = idx - ki * K;
    if (ti < ki) continue;
    const int k = c.clist[ki], t = c.clist[ti];
    const double msD = rc_deq128(getW(c, false, k, t), c.qD);
    const double msL = rc_deq128(getW(c, true, k, t), c.qL);
    double term;
    if (ki == ti) {                                                          // :26-36
      const long long szk = sz[k];
      const double pairs = (double)(szk * (szk - 1) / 2);
      const double a = P.alpha + P.delta1 * pairs;
      const double b = P.beta + msD / 2;
      term = (P.delta1 - 1) * msL / 2 - pairs * kp.lgd1 + kp.abratio + rc_lgamma(a) - a * rc_log(b);
    } else {                                                                 // :40-53
      const double pairs = (double)((long long)sz[k] * (long long)sz[t]);
      const double z = P.zeta + P.delta2 * pairs;
      const double g = P.gamma + msD;
      term = (P.delta2 - 1) * msL - pairs * kp.lgd2 + kp.zgratio + rc_lgamma(z) - z * rc_log(g);
    }
    if (st) st[ki == ti ? ki : K + ki * K - ki * (ki + 1) / 2 + (ti - ki - 1)] = term;
    else c.terms[idx] = term;
  }
  csync(c);
  if (c.ctid == 0) {
    double L1 = 0, L2 = 0;
    if (st) {
      for (int q = 0; q < K; ++q) L1 += st[q];
      for (int q = K; q < nT; ++q) L2 += st[q];
    } else {
      for (int ki = 0; ki < K; ++ki) L1 += c.terms[ki * K + ki];
      for (int ki = 0; ki < K; ++ki)
        for (int ti = ki + 1; ti < K; ++ti) L2 += c.terms[ki * K + ti];
    }
    c.sc->dtmp[0] = P.repulsion ? (L1 + L2) : (L1 + copysign(0.0, L2));      // :54
  }
  csync(c);
  return c.sc->dtmp[0];
}

// loglik of the chain's own state (fslotA / fslotB must be -1).  The value only changes when the state does, so it is kept
// with the chain's change count -- a stationary chain evaluates it once, not twice per iteration.
__device__ double loglik_cur(const Ctx& c) {
  if (c.sc->llclk == c.inc->clk) return c.sc->llcur;                        // (uniform: both were written before the last barrier)
  const double v = loglik_eval(c, c.sizes);
  if (c.ctid == 0) { c.sc->llcur = v; c.sc->llclk = c.inc->clk; }
  csync(c);
  return v;
}

__device__ __forceinline__ double xlogy(double a, double b) { return (a == 0.0 && !rc_isnan(b)) ? 0.0 : a * rc_log(b); }
__device__ __forceinline__ double xlog1py(double a, double b) { return (a == 0.0 && !rc_isnan(b)) ? 0.0 : a * rc_log1p(b); }

// logprior (mcmc.jl:58-78); warp 0 of the chain.
__device__ double logprior_eval(const Ctx& c) {
  const rc_params& P = c.kp->P;
  const int lane = c.lane;
  const double r = c.sc->r, p = c.sc->p;
  double* tv = c.terms;   // scratch: per-slot terms
  for (int s = lane; s < c.cap; s += 32)
    if (c.sizes[s] > 0) { const double nj = (double)c.sizes[s]; tv[s] = rc_log(nj) + rc_lgamma(nj + r - 1); }
  __syncwarp();
  double L = 0.0;
  if (lane == 0) {
    const double K = (double)c.sc->K;
    const double theta = 1 / P.sigma;
    const double xt = (r > 0 ? r : 0.0) / theta;
    double gl = -rc_lgamma(P.eta) - rc_log(theta) - xt;
    if (xt < RC_INF && xt > -RC_INF) gl += xlogy(P.eta - 1, xt);
    if (r < 0) gl = -RC_INF;
    const double y = p < 0 ? 0.0 : (p > 1 ? 1.0 : p);
    double bl = xlogy(P.u - 1, y) + xlog1py(P.v - 1, -y) - (rc_lgamma(P.u) + rc_lgamma(P.v) - rc_lgamma(P.u + P.v));
    if (p < 0 || p > 1) bl = -RC_INF;
    L = rc_lgamma(K + 1) + ((double)c.n - K) * rc_log(p) + (r * K) * rc_log(1 - p) - K * rc_lgamma(r) + gl + bl;
    for (int s = 0; s < c.cap; ++s)
      if (c.sizes[s] > 0) L += tv[s];
  }
  return __shfl_sync(0xffffffffu, L, 0);
}

// sample_r! (mcmc.jl:80-136); warp 0 of the chain.  Returns accept.
__device__ bool update_r(const Ctx& c, unsigned it) {
  const rc_params& P = c.kp->P;
  const int lane = c.lane;
  const double r = c.sc->r, p = c.sc->p, sd = P.proposalsd_r;
  double cand = r;
  if (lane == 0) {
    const double lb = (0.0 - r) / sd;
    double z = 0;
    for (uint32_t att = 0; att < 100000u; ++att) {
      z = rc_norminv(rc_open01(rc_draw1(c.key, it, RC_SITE_R_NORMAL, 0, att, 0)));
      if (z >= lb) break;
    }
    cand = r + sd * z;
  }
  cand = __shfl_sync(0xffffffffu, cand, 0);
  double* tc = c.terms;            // per-slot lgamma terms (candidate / current)
  double* tr = c.terms + c.cap;
  for (int s = lane; s < c.cap; s += 32)
    if (c.sizes[s] > 0) {
      const double nk1 = (double)(c.sizes[s] - 1);
      tc[s] = rc_lgamma(nk1 + cand);
      tr[s] = rc_lgamma(nk1 + r);
    }
  __syncwarp();
  int accept = 0;
  if (lane == 0) {
    const double K = (double)c.sc->K;
    const double l1mp = rc_log(1 - p);
    double lpc = (P.eta - 1) * rc_log(cand) + K * (cand * l1mp - rc_lgamma(cand)) - cand * P.sigma;
    double lpr = (P.eta - 1) * rc_log(r) + K * (r * l1mp - rc_lgamma(r)) - r * P.sigma;
    for (int s = 0; s < c.cap; ++s)
      if (c.sizes[s] > 0) { lpc = lpc + tc[s]; lpr = lpr + tr[s]; }
    const double log2pi = 1.8378770664093454836;
    double lq[2];   // logpdf(truncated(Normal(mu, sd), 0, Inf), x)
    for (int q = 0; q < 2; ++q) {
      const double mu = q == 0 ? r : cand, x = q == 0 ? cand : r;
      const double zz = (x - mu) / sd;
      const double lcdf = rc_normcdf((0.0 - mu) / sd);
      const double logtp = rc_log(1.0 - lcdf);
      lq[q] = -(zz * zz + log2pi) / 2 - rc_log(sd) - logtp;
    }
    const double lratio = lq[0] - lq[1];
    const double lu = rc_log(rc_draw1(c.key, it, RC_SITE_R_ACCEPT, 0, 0, 0));
    accept = lu < rc_min0(lpc - lpr - lratio);
    if (accept) c.sc->r = cand;
  }
  return __shfl_sync(0xffffffffu, accept, 0) != 0;
}

// sample_p! (mcmc.jl:138-155); one thread.
__device__ void update_p(const Ctx& c, unsigned it) {
  const rc_params& P = c.kp->P;
  const double a = (double)(c.n - c.sc->K) + P.u;
  const double b = c.sc->r * (double)c.sc->K + P.v;
  const double p = rc_beta(a, b, c.key, it);
  c.sc->p = p;
  c.sc->logp = rc_log(p);
  c.sc->log1mp = rc_log(1 - p);
}

// ------------------------------------------------------------------------------------------------
// Prior term of joining an existing cluster of size s (mcmc.jl:226, 324) for this iteration's (r, p):
// log(s+1) + log p + log(s-1+r) - log(s), evaluated in the reference's order, on demand (only a few sizes are ever needed
// per iteration, so no table is built).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double lpr_at(const Ctx& c, int s) {
  return c.kp->LOGN[s + 1] + c.sc->logp + rc_log((double)(s - 1) + c.sc->r) - c.kp->LOGN[s];
}

// ------------------------------------------------------------------------------------------------
// Split-merge setup and restricted Gibbs scans (mcmc.jl:259-354), run by the whole team of the chain.
// member_sums_inc: thread t owns the members q = t, t + nthr, ...; it walks ALL members y and adds DL[y][x_q]
// (= DL[x_q][y], D is symmetric; reading row y makes the threads of a warp hit neighbouring columns) to the sum of
// y's launch label.  No reductions; the sums over the first two live slots, clusters the launch did not touch, are
// single entries of S.
// ------------------------------------------------------------------------------------------------
__device__ void member_sums_inc(const Ctx& c, int nS, int ca, int cb, int c1, int c2) {
  const rc_kparams& kp = *c.kp;
  const rc_params& P = kp.P;
  const int mt = nS + 2, n = c.n;
  // Only the smaller launch side is gathered: the members are exactly the clusters ca and cb of the chain's state (a split's
  // new slot ca is empty there), so both sides together are S[ca][x] + S[cb][x] and the other side is the difference.
  const bool gA = c.szL[ca] <= c.szL[cb];
  const int side = gA ? ca : cb;
  for (int q0 = 0; q0 < mt; q0 += 2 * c.nthr) {
    const int qa = q0 + c.ctid, qb = q0 + c.nthr + c.ctid;
    const bool oa = qa < mt, ob = qb < mt;
    const int xa = oa ? (int)c.Slist[qa] : 0, xb = ob ? (int)c.Slist[qb] : 0;
    long long va[2] = {0, 0}, vb[2] = {0, 0};
#pragma unroll 4
    for (int q2 = 0; q2 < mt; ++q2) {
      const int y = c.Slist[q2];                               // uniform over the team
      if (c.labL[y] != side) continue;
      const longlong2* row = c.DL + (size_t)y * n;
      const longlong2 ea = oa ? __ldg(row + xa) : make_longlong2(0, 0);
      const longlong2 eb = ob ? __ldg(row + xb) : make_longlong2(0, 0);
      va[0] += ea.x; va[1] += ea.y; vb[0] += eb.x; vb[1] += eb.y;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = h ? qb : qa;
      if (!(h ? ob : oa)) continue;
      const int x = h ? xb : xa;
      const long long* v = h ? vb : va;
      const longlong2 ta = c.S[(size_t)ca * n + x], tb = c.S[(size_t)cb * n + x];
      const long long od = ta.x + tb.x - v[0], ol = ta.y + tb.y - v[1];
      longlong4 ab;
      if (gA) { ab.x = v[0]; ab.y = v[1]; ab.z = od; ab.w = ol; } else { ab.x = od; ab.y = ol; ab.z = v[0]; ab.w = v[1]; }
      c.AB[q] = ab;
      c.DG[q] = __ldg(c.DL + (size_t)x * n + x);
      if (q < nS) {
        double val[2] = {0.0, 0.0};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int t = e == 0 ? c1 : c2;
          if (t != ca && t != cb) {
            const longlong2 sv = c.S[(size_t)t * n + x];
            const int szs = c.szL[t];
            const double szd = (double)szs;
            const double sD = rc_dequant(sv.x, c.qD), sL = rc_dequant(sv.y, c.qL);
            const double z_i = P.zeta + P.delta2 * szd, g_i = P.gamma + sD;
            val[e] = kp.LGZ[szs] - z_i * rc_log(g_i) + kp.zgratio + (P.delta2 - 1) * sL - szd * kp.lgd2;
          }
        }
        c.L2s[q] = make_double2(val[0], val[1]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// All restricted Gibbs scans of one split-merge step (mcmc.jl:259-354, called at :411-414, :419, :454) over the items
// Slist[0..nS) on the launch state, which lives IN PLACE in c.labL / c.szL (the chain's own labels of the members are kept
// in origM and restored by the caller).
//   * AB[q] holds the sums of member q's row over the current members of the two candidate clusters; a move of item y
//     updates all of them from row y (exact integers), so a step that does not move reads nothing but its own entry.
//   * the Gumbel noise and the repulsion terms of non-candidate slots do not depend on the evolving state and are
//     precomputed (NZ, L2s).
//   * the transition probability (:347-351) is only evaluated in the last scan -- the reference discards the return value
//     of the intermediate scans (:411-414).
// Every warp evaluates eight consecutive steps (a quad of lanes per step, one logarithm per lane) and resolves them among
// themselves -- each quad holds the matrix entries between its item and the items of the warp's earlier steps, so when an
// earlier step moves its item the later quads correct their sums in registers and decide again, in step order.  A warp's
// eight steps are therefore final given the state at the start of the batch.  A batch covers 8 * nwact steps: the warps up
// to and including the first one with a move are committed, that warp's moves (up to eight) are applied to the running
// candidate sums of all members by all threads with one round of gathers, and the scan continues behind them.  Every
// committed step sees exactly the inputs of the sequential scan, so the results are the same bits.
// Returns the log transition probability of the last scan in c.sc->ltp.
// ------------------------------------------------------------------------------------------------
#define RC_RS_B 8       // steps per warp
#define RC_RS_PF 4      // steps of a short batch whose rows the idle warps pull towards L2
__device__ void restricted_scans_team(const Ctx& c, int nS, int ca, int cb, int c1, int c2, bool split) {
  const rc_kparams& kp = *c.kp;
  const rc_params& P = kp.P;
  const int lane = c.lane, warp = c.cwarp, NW = c.nwarp;
  const int mt = nS + 2;
  const int numGibbs = (int)kp.numGibbs;
  IncShared* sh = c.inc;
  if (nS == 0) { if (c.ctid == 0) c.sc->ltp = 0.0; csync(c); return; }
  if (c.ctid == 0) { sh->first[0] = RC_INC_NONE; sh->first[1] = RC_INC_NONE; sh->first[2] = RC_INC_NONE; }
  csync(c);
  const bool c1dyn = (c1 == ca || c1 == cb), c2dyn = (c2 == ca || c2 == cb);
  const int st = lane >> 2, role = lane & 3, quad = lane & ~3;
  const bool isA = (role & 1) == 0;
  const unsigned qm = 0xfu << quad;
  double ltp = 0.0;                                   // accumulated by thread 0 in step order
  int batch = 0;
  const int NWE = min(NW, RC_RS_MAXW);
  int nwact = NWE;                                    // warps that evaluate a batch: follows the observed run length between moves
  for (int g = 0; g <= numGibbs; ++g) {
    const bool last = g == numGibbs;
    const bool forced = last && !split;
    int pos0 = 0;
    while (pos0 < nS) {
      const int slot3 = batch % 3, par = batch & 1;
      if (c.ctid == 0) sh->first[(batch + 1) % 3] = RC_INC_NONE;
      ++batch;
      const long long tr0 = RC_CLOCK();
      const int nb = min(RC_RS_B * nwact, nS - pos0);
      const int stepi = warp * RC_RS_B + st;           // step within the batch
      const int pos = pos0 + stepi;
      const bool on = stepi < nb;
      if (nwact <= 2 && warp >= nwact && mt <= 1024) {
        // Short runs: moves are likely within the next few steps, and their update gathers the movers' rows at every
        // member column (DRAM latency on the critical path).  The warps that sit this batch out pull those entries
        // towards L2 for the first steps of the batch while the evaluating warps are busy.
        const int npf = min(nb, RC_RS_PF);
        const int nidle = (NW - nwact) * 32, me = (warp - nwact) * 32 + lane;
        for (int q = me; q < mt; q += nidle) {
          const int xq = c.Slist[q];
          for (int u = 0; u < npf; ++u) {
            const longlong2* pr = c.DL + (size_t)c.Slist[pos0 + u] * c.n + xq;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pr));
          }
        }
      }
      int y = 0, cur = 0, cnew = 0, k = 0;
      double lt = 0.0;
      long long trx = tr0;
      if (warp < nwact) {                                // (uniform per warp)
        // the size-indexed tables at the sizes this warp's steps can see (start-of-batch size - 8 .. + 7), into shared memory:
        // a step that is decided again after an earlier step moved must not wait for global memory
        double (*win)[16] = sh->rs_win[warp];
        const int loA = c.szL[ca] - 8, loB = c.szL[cb] - 8;
        double wv[3];
#pragma unroll
        for (int u = 0; u < 3; ++u) {
          const int idx = lane + 32 * u, tb = idx >> 4, off = idx & 15;
          const int sz = min(max(((tb & 1) ? loB : loA) + off, 0), c.n);
          wv[u] = tb < 2 ? kp.LGA[sz] : (tb < 4 ? kp.LGZ[sz] : lpr_at(c, sz > 0 ? sz : 1));
        }
        long long sAd = 0, sAl = 0, sBd = 0, sBl = 0;
        int szA = 0, szB = 0, forcedto = 0;
        double2 l2s = make_double2(0.0, 0.0), nz = make_double2(0.0, 0.0);
        longlong2 e0 = make_longlong2(0, 0), e1 = make_longlong2(0, 0);
        if (on) {
          y = c.Slist[pos];
          // entries between this step's item and the items of the warp's earlier steps (role r holds steps r and r + 4)
          const longlong2* row = c.DL + (size_t)y * c.n;
          if (role < st) e0 = __ldg(row + c.Slist[pos - st + role]);
          if (role + 4 < st) e1 = __ldg(row + c.Slist[pos - st + role + 4]);
          const longlong2 self = c.DG[pos];
          const longlong4 ab = c.AB[pos];
          l2s = c.L2s[pos];
          if (!forced) nz = c.NZ[(size_t)g * nS + pos]; else forcedto = c.origM[pos];
          cur = c.labL[y];
          // sums over the candidates with y detached (:303-304)
          sAd = ab.x - (cur == ca ? self.x : 0); sAl = ab.y - (cur == ca ? self.y : 0);
          sBd = ab.z - (cur == cb ? self.x : 0); sBl = ab.w - (cur == cb ? self.y : 0);
          szA = c.szL[ca] - (cur == ca ? 1 : 0); szB = c.szL[cb] - (cur == cb ? 1 : 0);
        }
#pragma unroll
        for (int u = 0; u < 3; ++u) { const int idx = lane + 32 * u; win[idx >> 4][idx & 15] = wv[u]; }     // (after every load of the step is in flight)
        __syncwarp();
        // one step's decision from its current sums (the four lanes of the quad: one logarithm each)
        auto decide = [&]() {
          // roles 0..3: {L2'(ca), L2'(cb), L1(ca), L1(cb)}
          double X;
          {
            const int szs = isA ? szA : szB;
            const double szd = (double)szs;
            const double sD = rc_dequant(isA ? sAd : sBd, c.qD), sL = rc_dequant(isA ? sAl : sBl, c.qL);
            if ((role & 2) == 0) {                                                                    // :313-319, 327-330
              const double z_i = P.zeta + P.delta2 * szd, g_i = P.gamma + sD;
              X = win[2 + (isA ? 0 : 1)][szs - (isA ? loA : loB)] - z_i * rc_log(g_i) + kp.zgratio + (P.delta2 - 1) * sL - szd * kp.lgd2;
            } else {                                                                                  // :307-312, 321-326
              const double a_i = P.alpha + P.delta1 * szd, b_i = P.beta + sD;
              X = win[isA ? 0 : 1][szs - (isA ? loA : loB)] + kp.abratio - a_i * rc_log(b_i) + (P.delta1 - 1) * sL - szd * kp.lgd1;
            }
          }
          const double L2pA = __shfl_sync(qm, X, quad), L2pB = __shfl_sync(qm, X, quad + 1);
          const double L1A = __shfl_sync(qm, X, quad + 2), L1B = __shfl_sync(qm, X, quad + 3);
          const double L2p1 = c1dyn ? (c1 == ca ? L2pA : L2pB) : l2s.x;
          const double L2p2 = c2dyn ? (c2 == ca ? L2pA : L2pB) : l2s.y;
          const double L2i = L2p1 + L2p2;                                                             // :331 (quirk Q2)
          const double L2a = L2i - L2pA, L2b = L2i - L2pB;                                            // :332-334
          double lp0 = win[4][szA - loA] + (L1A + (P.repulsion ? L2a : copysign(0.0, L2a)));          // :335
          double lp1 = win[5][szB - loB] + (L1B + (P.repulsion ? L2b : copysign(0.0, L2b)));
          if (!forced) {                                                                              // :336-338
            double mn = lp0;
            if (!rc_isnan(mn)) { if (rc_isnan(lp1) || lp1 < mn) mn = lp1; }
            lp0 -= mn; lp1 -= mn;
            const double g0 = nz.x + lp0, g1 = nz.y + lp1;
            k = 0;
            if (!rc_isnan(g0)) { if (rc_isnan(g1) || g1 > g0) k = 1; }
            cnew = k == 0 ? ca : cb;
          } else {                                                                                    // :339-342
            cnew = forcedto;
            k = (ca == cnew) ? 0 : 1;
          }
          if (last) {                                                                                 // :347-351
            double mn = lp0;                                                                          // quirk Q3
            if (!rc_isnan(mn)) { if (rc_isnan(lp1) || lp1 < mn) mn = lp1; }
            lp0 += mn; lp1 += mn;
            double p0 = rc_exp(lp0), p1 = rc_exp(lp1);
            const double den = p0 + p1;
            p0 /= den; p1 /= den;
            lt = rc_log(k == 0 ? p0 : p1);
          }
        };
        if (on) decide();
        trx = RC_CLOCK();
        // resolve the warp's steps in order: a step that moves its item changes the sums of the steps behind it (:344-345)
        unsigned pend = __ballot_sync(0xffffffffu, on && role == 0 && cnew != cur);     // steps that move their item, as decided so far
        while (pend) {
          const int l0 = __ffs(pend) - 1, s2 = l0 >> 2;                                  // the earliest one is final
          const int a2b = __shfl_sync(0xffffffffu, cur == ca ? 1 : 0, l0);
          if (on && st > s2) {
            const longlong2 mine = (s2 >> 2) ? e1 : e0;
            const int src = quad + (s2 & 3);
            const long long ex = __shfl_sync(qm, mine.x, src), ey = __shfl_sync(qm, mine.y, src);
            if (a2b) { sAd -= ex; sAl -= ey; sBd += ex; sBl += ey; szA -= 1; szB += 1; }
            else { sAd += ex; sAl += ey; sBd -= ex; sBl -= ey; szA += 1; szB -= 1; }
            decide();
          }
          pend = __ballot_sync(0xffffffffu, on && role == 0 && cnew != cur && st > s2);
        }
        if (last && on && role == 0) sh->ltbuf[par][stepi] = lt;
        // the warp's moves, in step order
        const unsigned mv = __ballot_sync(0xffffffffu, on && role == 0 && cnew != cur);
        if (mv) {
          if (on && role == 0 && cnew != cur) sh->rs_mv[warp][__popc(mv & ((1u << lane) - 1))] = (y << 1) | (cur == ca ? 1 : 0);
          if (lane == 0) { sh->rs_nm[warp] = __popc(mv); atomicMin(&sh->first[slot3], warp); }
        }
      }
      const long long trb = RC_CLOCK();
      csync(c);
      const long long tr1 = RC_CLOCK();
      const int F = sh->first[slot3];                                                               // first warp with moves
      const int nvalid = F == RC_INC_NONE ? nb : min(nb, (F + 1) * RC_RS_B);
      nwact = F == RC_INC_NONE ? min(NWE, nwact * 2) : max(1, min(NWE, F + 1));
      if (last && c.ctid == 0)
        for (int q = 0; q < nvalid; ++q) ltp += sh->ltbuf[par][q];                                  // in step order, as the scan adds them
      if (F != RC_INC_NONE) {
        const int nm = sh->rs_nm[F];
        if (c.ctid == 0)
          for (int m = 0; m < nm; ++m) {
            const int v = sh->rs_mv[F][m];
            const bool a2b = v & 1;
            c.labL[v >> 1] = (uint8_t)(a2b ? cb : ca);
            c.szL[ca] += a2b ? -1 : 1; c.szL[cb] += a2b ? 1 : -1;
          }
        // every member's candidate sums follow the moves (D is symmetric: DL[q][y] == DL[y][q]); four rows in flight
        for (int m0 = 0; m0 < nm; m0 += 4) {
          int mvv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) mvv[u] = m0 + u < nm ? sh->rs_mv[F][m0 + u] : -1;
          for (int q = c.ctid; q < mt; q += 2 * c.nthr) {
            const int q1 = q + c.nthr;
            const bool o1 = q1 < mt;
            const int xq = c.Slist[q], xq1 = o1 ? (int)c.Slist[q1] : 0;
            longlong2 e[4], f[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const longlong2* row = c.DL + (size_t)(mvv[u] >> 1) * c.n;
              e[u] = mvv[u] >= 0 ? __ldg(row + xq) : make_longlong2(0, 0);
              f[u] = (mvv[u] >= 0 && o1) ? __ldg(row + xq1) : make_longlong2(0, 0);
            }
            longlong4 t = c.AB[q], t1 = o1 ? c.AB[q1] : longlong4{0, 0, 0, 0};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (mvv[u] & 1) {                                                                       // (an absent move has zero entries)
                t.x -= e[u].x; t.y -= e[u].y; t.z += e[u].x; t.w += e[u].y;
                t1.x -= f[u].x; t1.y -= f[u].y; t1.z += f[u].x; t1.w += f[u].y;
              } else {
                t.x += e[u].x; t.y += e[u].y; t.z -= e[u].x; t.w -= e[u].y;
                t1.x += f[u].x; t1.y += f[u].y; t1.z -= f[u].x; t1.w -= f[u].y;
              }
            }
            c.AB[q] = t;
            if (o1) c.AB[q1] = t1;
          }
        }
        csync(c);
      }
      if (c.ctid == 0) { st_add(c, ST_BULK_ROWS, trx - tr0); st_add(c, ST_BULK_REDUCE, trb - trx); st_add(c, ST_DEC_WAIT, tr1 - tr0); st_add(c, ST_DEC_WORK, RC_CLOCK() - tr1); st_add(c, ST_BULK_WAIT_CONSUMED, 1); st_add(c, ST_BULK_WAIT_FULL, F != RC_INC_NONE); }
      pos0 += nvalid;
    }
  }
  if (c.ctid == 0) c.sc->ltp = ltp;
  csync(c);
}

__device__ void inc_full_scan(const Ctx& c, unsigned it, int istart, bool dry);

// One split-merge proposal (mcmc.jl:372-474) on the current LOCAL state of sample_labels!.  Returns accept through
// c.sc->itmp[1], split through itmp[2].  With commit == false the state is unchanged on return.  With commit == true
// (more proposals follow in this iteration, numMH > 1) an accepted proposal becomes the local state (:470): labels,
// sizes, K and the block sums W are replaced -- the caller backs the chain's own state up first and restores it
// after the last proposal (quirk Q1: the accepted state never reaches runsampler's state).
__device__ void splitmerge_step(Ctx& c, unsigned it, unsigned mh, bool commit) {
  const rc_kparams& kp = *c.kp;
  const rc_params& P = kp.P;
  const int tid = c.ctid, lane = c.lane, warp = c.cwarp;
  const int n = c.n, cap = c.cap;
  const double r = c.sc->r, p = c.sc->p;
  const int K = c.sc->K;
  const long long tm0 = RC_CLOCK();
  // (i, j) = sample(1:n, 2, replace = false)  (:379)
  const rc_draw dr = rc_draw2(c.key, it, RC_SITE_SM_PAIR, mh, 0, 0);
  long long i1 = rc_randint(dr.u0, n), i2 = rc_randint(dr.u1, n - 1);
  if (i2 == i1) i2 = n;
  const int pi = (int)i1 - 1, pj = (int)i2 - 1;
  if (c.labL != c.lab) {                       // the proposal lives in its own copy of the labels (see the restricted scans below)
    for (int k = tid; k < n; k += c.nthr) c.labL[k] = c.lab[k];
    csync(c);
  }
  const int ci = c.labL[pi], cj = c.labL[pj];
  csync(c);
  if (tid == 0) { c.sc->itmp[1] = 0; c.sc->itmp[2] = 0; }
  if (P.maxK > 0 && ci == cj && K >= P.maxK) { csync(c); return; }          // :384-386
  if (ci != cj && kp.shortcuts) {
    // Merge proposals that cannot be accepted.  The acceptance ratio of a merge (:435-468) is
    //   prior ratio + likelihood ratio - log proposal ratio,   log proposal ratio = -(sum of the final scan's log transition
    // probabilities) >= 0,
    // and neither the prior ratio nor the likelihood ratio depends on the restricted scans: the merged state is known (sizes,
    // block sums W[ci] + W[cj]).  So x = prior ratio + likelihood ratio bounds the ratio from above (every log transition
    // probability is <= 0 and floating-point addition is monotone), and when log U >= min(0, x) the proposal is rejected
    // whatever the restricted scans would have produced -- they are not run.  (A NaN x fails the test and takes the long way.)
    // The uniforms are counter-based, so skipping the scans' draws changes nothing else.
    const int szf = c.sizes[ci] + c.sizes[cj];
    // (the merged state's log-likelihood only changes when the chain's state does: kept per ordered pair with the change count)
    const size_t pidx = (size_t)ci * cap + cj;
    const bool have = c.LLFs[pidx] == c.inc->clk;                            // (written before the last barrier: uniform)
    double ll_fin;
    if (have) ll_fin = c.LLF[pidx];
    else {
      rc_i128* rows = c.prows;
      for (int t = tid; t < cap; t += c.nthr) {                             // row cj of the merged state
        rc_i128 bD = c.WD[tri(ci, t, cap)], bL = c.WL[tri(ci, t, cap)];
        rc_add128(bD, c.WD[tri(cj, t, cap)]); rc_add128(bL, c.WL[tri(cj, t, cap)]);
        rows[2 * cap + t] = bD; rows[3 * cap + t] = bL;
        rc_i128 z; z.lo = 0; z.hi = 0;
        rows[0 * cap + t] = z; rows[1 * cap + t] = z;
      }
      if (tid == 0) {
        rc_i128 bbD = c.WD[tri(ci, ci, cap)], bbL = c.WL[tri(ci, ci, cap)];
        rc_add128(bbD, c.WD[tri(cj, cj, cap)]); rc_add128(bbL, c.WL[tri(cj, cj, cap)]);
        rc_add128(bbD, c.WD[tri(ci, cj, cap)]); rc_add128(bbD, c.WD[tri(ci, cj, cap)]);
        rc_add128(bbL, c.WL[tri(ci, cj, cap)]); rc_add128(bbL, c.WL[tri(ci, cj, cap)]);
        rc_i128 z; z.lo = 0; z.hi = 0;
        c.sc->aaD = z; c.sc->aaL = z; c.sc->abD = z; c.sc->abL = z; c.sc->bbD = bbD; c.sc->bbL = bbL;
        c.sc->fslotA = ci; c.sc->fslotB = cj;
      }
      for (int s = tid; s < cap; s += c.nthr) c.szL[s] = (s == ci) ? 0 : (s == cj ? szf : c.sizes[s]);   // sizes of the merged state
      csync(c);
      ll_fin = loglik_eval(c, c.szL);
      if (tid == 0) { c.sc->fslotA = -1; c.sc->fslotB = -1; c.LLF[pidx] = ll_fin; c.LLFs[pidx] = c.inc->clk; }
    }
    const double ll_cur = loglik_cur(c);
    if (tid == 0) {
      const double log_prior_ratio = -(rc_log((double)K) + r * rc_log(1 - p) - rc_log(p) - rc_lgamma(r)) +
                                     rc_lgamma((double)(szf - 1) + r) + rc_log((double)szf) +
                                     -(rc_lgamma((double)(c.sizes[ci] - 1) + r) + rc_lgamma((double)(c.sizes[cj] - 1) + r) +
                                       rc_log((double)c.sizes[ci]) + rc_log((double)c.sizes[cj]));
      const double x = log_prior_ratio + (ll_fin - ll_cur);
      const double lu = rc_log(rc_draw1(c.key, it, RC_SITE_SM_ACCEPT, mh, 0, 0));
      c.sc->itmp[7] = (lu >= rc_min0(x) + 1e-6) ? 1 : 0;                     // (1e-6: slack for a log transition probability that rounds above 0)
#ifdef RC_NO_STATS
      st_add(c, ST_DEC_WAIT, c.sc->itmp[7]);                                 // (default library: merge proposals rejected by the bound)
#endif
    }
    csync(c);
    if (c.sc->itmp[7]) return;                                               // itmp[1] (accept) and itmp[2] (split) are 0
  }
  // S = members of ci or cj except i, j, ascending (:389-390): ordered compaction
  {
    const int chunk = (n + c.nthr - 1) / c.nthr;
    const int b = tid * chunk, e = min(n, b + chunk);
    int cntm = 0;
    for (int k = b; k < e; ++k) cntm += ((c.labL[k] == ci || c.labL[k] == cj) && k != pi && k != pj);
    int incl = cntm;
    for (int off = 1; off < 32; off <<= 1) { const int o = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += o; }
    if (lane == 31) c.itmp[warp] = incl;
    csync(c);
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += c.itmp[w];
    int o = woff + incl - cntm;
    for (int k = b; k < e; ++k)
      if ((c.labL[k] == ci || c.labL[k] == cj) && k != pi && k != pj) { c.Slist[o] = (unsigned short)k; c.origM[o] = c.labL[k]; ++o; }
    if (tid == c.nthr - 1) c.sc->itmp[3] = woff + incl;
    csync(c);
  }
  const int nS = c.sc->itmp[3];
  // the per-member running sums live in shared memory when the members fit (the restricted scans are a chain of dependent
  // reads and writes of exactly these arrays)
  longlong4* const gAB = c.AB; longlong2* const gDG = c.DG; double2* const gL2s = c.L2s;
  if (nS + 2 <= c.mcap) { c.AB = c.mAB; c.DG = c.mDG; c.L2s = c.mL2s; }
  auto unswap = [&]() { c.AB = gAB; c.DG = gDG; c.L2s = gL2s; };
  if (tid == 0) { c.Slist[nS] = (unsigned short)pi; c.origM[nS] = (uint8_t)ci; c.Slist[nS + 1] = (unsigned short)pj; c.origM[nS + 1] = (uint8_t)cj; }
  // launch state (:393-408), in place in c.labL / c.szL
  for (int s = tid; s < cap; s += c.nthr) c.szL[s] = c.sizes[s];
  const bool split = ci == cj;
  int ca = ci;
  if (split) {
    if (tid < 32) {
      int e = -1;
      for (int w = 0; w * 32 < cap && e < 0; ++w) {
        const int s = w * 32 + lane;
        const unsigned m = __ballot_sync(0xffffffffu, s < cap && c.sizes[s] == 0);
        if (m) e = w * 32 + __ffs(m) - 1;
      }
      if (lane == 0) c.sc->itmp[4] = e;
    }
    csync(c);
    ca = c.sc->itmp[4];
    if (ca < 0) { if (tid == 0) c.sc->status = RC_ERR_SLOTS; csync(c); unswap(); return; }
    if (tid == 0) c.labL[pi] = (uint8_t)ca;
  }
  const int cb = cj;
  csync(c);
  {
    int na = 0, nb = 0;   // launch allocation of S (:402-407)
    for (int pos = tid; pos < nS; pos += c.nthr) {
      const int k = c.Slist[pos];
      const double u = rc_draw1(c.key, it, RC_SITE_SM_LAUNCH, mh, (uint32_t)pos, 0);
      const int cn = rc_randint(u, 2) == 1 ? ca : cb;
      c.labL[k] = (uint8_t)cn;
      na += cn == ca; nb += cn == cb;
    }
    for (int off = 16; off; off >>= 1) { na += __shfl_xor_sync(0xffffffffu, na, off); nb += __shfl_xor_sync(0xffffffffu, nb, off); }
    if (lane == 0) { c.itmp[warp * 2] = na; c.itmp[warp * 2 + 1] = nb; }
    csync(c);
    if (tid == 0) {
      int ta = 0, tb = 0;
      for (int w = 0; w < c.nwarp; ++w) { ta += c.itmp[w * 2]; tb += c.itmp[w * 2 + 1]; }
      if (split) c.szL[ci] = 0;
      c.szL[ca] = 1 + ta;
      c.szL[cb] = 1 + tb;
      int c1 = -1, c2 = -1;                   // first two live slots of the launch state (C[1], C[2] of :273, :331)
      for (int s = 0; s < cap && c2 < 0; ++s)
        if (c.szL[s] > 0) { if (c1 < 0) c1 = s; else c2 = s; }
      c.sc->itmp[5] = c1; c.sc->itmp[6] = c2;
    }
    csync(c);
  }
  const int c1 = c.sc->itmp[5], c2 = c.sc->itmp[6];
  // member x member entries by launch label; the sums over the first two live slots, when they are not candidates, are
  // clusters the launch did not touch and come straight from S
  member_sums_inc(c, nS, ca, cb, c1, c2);
  {
    const int nfree = (int)kp.numGibbs + (split ? 1 : 0);
    for (int e = tid; e < nfree * nS; e += c.nthr) {
      const int g = e / nS, pos = e - g * nS;
      const rc_draw dr = rc_draw2(c.key, it, RC_SITE_SM_RGIBBS, mh, (uint32_t)g, (uint32_t)pos);
      c.NZ[e] = make_double2(-rc_log(-rc_log(dr.u0)), -rc_log(-rc_log(dr.u1)));
    }
  }
  csync(c);
  const long long tm1 = RC_CLOCK();
  if (c.labL != c.lab && nS + 2 <= 1024 && !c.inc->scanfast) {   // (large member sets need every thread; a scan decided by its row summaries is too short to matter)
    // The restricted scans are a chain of dependent steps that keeps one or two warps busy.  With one proposal per
    // iteration the full scan that follows does not depend on them unless the proposal is accepted (quirk Q1: then the
    // scan is discarded), so the rest of the CTA runs it now, DRY: it commits nothing and stops at the first row that
    // would move its point.  Labels, sizes, S and W are only read by both sides (the proposal's labels are a copy).
    // The restricted scans resolve the moves of eight steps inside one warp, so a small team (kp.rs_team: 64 of 256 threads,
    // 128 of 512) runs them as fast as the whole CTA would.  Measured at n = 10^4, 50 clusters: +12 % chain-sweeps/s with two
    // chains per SM (256 threads each), +11 % with one (512 threads).
    const int TA = min(kp.rs_team, c.nthr / 2);
    if (tid < TA) {
      Ctx cA = c;
      cA.nthr = TA; cA.nwarp = TA / 32; cA.barid = 2;
      restricted_scans_team(cA, nS, ca, cb, c1, c2, split);                  // :411-414, :419 / :454-455
    } else {
      Ctx cB = c;
      cB.ctid = tid - TA; cB.cwarp = cB.ctid >> 5; cB.nthr = c.nthr - TA; cB.nwarp = cB.nthr / 32; cB.barid = 3;
      inc_full_scan(cB, it, 0, true);
    }
  } else restricted_scans_team(c, nS, ca, cb, c1, c2, split);
  csync(c);
  const long long tm2 = RC_CLOCK();
  if (tid == 0) { st_add(c, ST_MH_SETUP, tm1 - tm0); st_add(c, ST_MH_RSCAN, tm2 - tm1); }
  double log_prior_ratio = 0.0, log_proposal_ratio = 0.0;
  if (split) {                                                              // :416-434
    const int sza = c.szL[ca], szb = c.szL[cb];   // szfinal[cfinal[i]], szfinal[cfinal[j]]
    if (tid == 0) {
      log_prior_ratio = rc_log((double)(K + 1)) + r * rc_log(1 - p) - rc_log(p) - rc_lgamma(r) +
                        rc_lgamma((double)(sza - 1) + r) + rc_lgamma((double)(szb - 1) + r) +
                        rc_log((double)sza) + rc_log((double)szb) +
                        -(rc_lgamma((double)(c.sizes[ci] - 1) + r) + rc_log((double)c.sizes[ci]));
      log_proposal_ratio = c.sc->ltp;
    }
    // block sums of the proposed state: rows a (= new slot ca) and b (= cb)
    rc_i128* rows = c.prows;   // [rowA_D | rowA_L | rowB_D | rowB_L] x cap
    // the slots other than ca / cb are untouched clusters: their sums over the members that ended in ca are entries of S.
    // A warp per slot, the members over its lanes.
    for (int t = warp; t < cap; t += c.nwarp) {
      rc_i128 sd, sl; sd.lo = 0; sd.hi = 0; sl.lo = 0; sl.hi = 0;
      if (t != ca && t != cb && c.sizes[t] > 0) {
        for (int q = lane; q < nS + 2; q += 32) {
          const int x = c.Slist[q];
          if (c.labL[x] == ca) { const longlong2 v = c.S[(size_t)t * n + x]; rc_add128(sd, v.x); rc_add128(sl, v.y); }
        }
        sd = warp_sum128(sd); sl = warp_sum128(sl);
      }
      if (lane == 0) { rows[0 * cap + t] = sd; rows[1 * cap + t] = sl; }
    }
    // within / cross sums from the running candidate sums of the final state:
    //   aa = sum_{x in a_F} sum_{y in a_F} DL[x][y],  ab = sum_{x in a_F} sum_{y in b_F} DL[x][y]
    rc_i128 acc[4];
    for (int h = 0; h < 4; ++h) { acc[h].lo = 0; acc[h].hi = 0; }
    for (int q = tid; q < nS + 2; q += c.nthr)
      if (c.labL[c.Slist[q]] == ca) {
        const longlong4 ab = c.AB[q];
        rc_add128(acc[0], ab.x); rc_add128(acc[1], ab.y); rc_add128(acc[2], ab.z); rc_add128(acc[3], ab.w);
      }
    rc_i128* red128 = reinterpret_cast<rc_i128*>(c.terms);    // scratch [c.nwarp][4]
    for (int h = 0; h < 4; ++h) {
      const rc_i128 w = warp_sum128(acc[h]);
      if (lane == 0) red128[warp * 4 + h] = w;
    }
    csync(c);
    if (tid == 0) {
      rc_i128 tot[4];
      for (int h = 0; h < 4; ++h) { tot[h].lo = 0; tot[h].hi = 0; }
      for (int w = 0; w < c.nwarp; ++w)
        for (int h = 0; h < 4; ++h) rc_add128(tot[h], red128[w * 4 + h]);
      const rc_i128 aaD = tot[0], aaL = tot[1], xD = tot[2], xL = tot[3];
      rc_i128 bbD = c.WD[tri(ci, ci, cap)], bbL = c.WL[tri(ci, ci, cap)];
      rc_sub128(bbD, aaD); rc_sub128(bbD, xD); rc_sub128(bbD, xD);
      rc_sub128(bbL, aaL); rc_sub128(bbL, xL); rc_sub128(bbL, xL);
      c.sc->aaD = aaD; c.sc->aaL = aaL; c.sc->abD = xD; c.sc->abL = xL; c.sc->bbD = bbD; c.sc->bbL = bbL;
    }
    csync(c);
    for (int t = tid; t < cap; t += c.nthr) {                               // row b = row ci of the current state - row a
      rc_i128 bD = c.WD[tri(ci, t, cap)], bL = c.WL[tri(ci, t, cap)];
      rc_sub128(bD, rows[0 * cap + t]); rc_sub128(bL, rows[1 * cap + t]);
      rows[2 * cap + t] = bD; rows[3 * cap + t] = bL;
    }
    if (tid == 0) { c.sc->fslotA = ca; c.sc->fslotB = cb; c.sc->itmp[2] = 1; }
    csync(c);
  } else {                                                                  // merge (:435-459)
    const int szf = c.sizes[ci] + c.sizes[cj];
    if (tid == 0) {
      log_prior_ratio = -(rc_log((double)K) + r * rc_log(1 - p) - rc_log(p) - rc_lgamma(r)) +
                        rc_lgamma((double)(szf - 1) + r) + rc_log((double)szf) +
                        -(rc_lgamma((double)(c.sizes[ci] - 1) + r) + rc_lgamma((double)(c.sizes[cj] - 1) + r) +
                          rc_log((double)c.sizes[ci]) + rc_log((double)c.sizes[cj]));
      log_proposal_ratio = -c.sc->ltp;
    }
    rc_i128* rows = c.prows;
    for (int t = tid; t < cap; t += c.nthr) {                               // row cj of the merged state
      rc_i128 bD = c.WD[tri(ci, t, cap)], bL = c.WL[tri(ci, t, cap)];
      rc_add128(bD, c.WD[tri(cj, t, cap)]); rc_add128(bL, c.WL[tri(cj, t, cap)]);
      rows[2 * cap + t] = bD; rows[3 * cap + t] = bL;
      rc_i128 z; z.lo = 0; z.hi = 0;
      rows[0 * cap + t] = z; rows[1 * cap + t] = z;
    }
    if (tid == 0) {
      rc_i128 bbD = c.WD[tri(ci, ci, cap)], bbL = c.WL[tri(ci, ci, cap)];
      rc_add128(bbD, c.WD[tri(cj, cj, cap)]); rc_add128(bbL, c.WL[tri(cj, cj, cap)]);
      rc_add128(bbD, c.WD[tri(ci, cj, cap)]); rc_add128(bbD, c.WD[tri(ci, cj, cap)]);
      rc_add128(bbL, c.WL[tri(ci, cj, cap)]); rc_add128(bbL, c.WL[tri(ci, cj, cap)]);
      rc_i128 z; z.lo = 0; z.hi = 0;
      c.sc->aaD = z; c.sc->aaL = z; c.sc->abD = z; c.sc->abL = z; c.sc->bbD = bbD; c.sc->bbL = bbL;
      c.sc->fslotA = ci; c.sc->fslotB = cj;
    }
    for (int s = tid; s < cap; s += c.nthr) c.szL[s] = (s == ci) ? 0 : (s == cj ? szf : c.sizes[s]);   // sizes of the merged state
    csync(c);
  }
  const double ll_fin = loglik_eval(c, c.szL);                              // :462-464
  if (tid == 0) { c.sc->fslotA = -1; c.sc->fslotB = -1; }
  const double ll_cur = loglik_cur(c);
  if (tid == 0) {
    const double log_lik_ratio = ll_fin - ll_cur;
    const double lar = rc_min0(log_prior_ratio + log_lik_ratio - log_proposal_ratio);   // :467-468
    const double lu = rc_log(rc_draw1(c.key, it, RC_SITE_SM_ACCEPT, mh, 0, 0));
    c.sc->itmp[1] = lu < lar ? 1 : 0;                                                   // :469-472
  }
  csync(c);
  if (commit && c.sc->itmp[1]) {
    // the proposed state becomes the local state of the remaining proposals of this iteration
    if (!c.sc->forked) {                                   // first accepted proposal: keep the chain's own block sums
      for (int t = tid; t < cap * cap; t += c.nthr) { c.WDbak[t] = c.WD[t]; c.WLbak[t] = c.WL[t]; }
      csync(c);
      if (tid == 0) c.sc->forked = 1;
    }
    const rc_i128* rows = c.prows;   // [rowA_D | rowA_L | rowB_D | rowB_L] x cap
    const int A = split ? ca : ci, B = split ? cb : cj;
    for (int t = tid; t < cap; t += c.nthr) {
      if (t != A && t != B) {
        c.WD[tri(A, t, cap)] = rows[0 * cap + t]; c.WL[tri(A, t, cap)] = rows[1 * cap + t];
        c.WD[tri(B, t, cap)] = rows[2 * cap + t]; c.WL[tri(B, t, cap)] = rows[3 * cap + t];
      }
    }
    if (tid == 0) {
      c.WD[tri(A, A, cap)] = c.sc->aaD; c.WL[tri(A, A, cap)] = c.sc->aaL;
      c.WD[tri(A, B, cap)] = c.sc->abD; c.WL[tri(A, B, cap)] = c.sc->abL;
      c.WD[tri(B, B, cap)] = c.sc->bbD; c.WL[tri(B, B, cap)] = c.sc->bbL;
      c.sc->K = split ? K + 1 : K - 1;
    }
    if (!split)
      for (int q = tid; q < nS + 2; q += c.nthr) c.labL[c.Slist[q]] = (uint8_t)cj;     // :436-445 (split: labels are final in place)
    for (int s = tid; s < cap; s += c.nthr) c.sizes[s] = c.szL[s];
    csync(c);                                   // the row sums follow the members that changed slot
    for (int q = 0; q < nS + 2; ++q) {
      const int y = c.Slist[q], from = c.origM[q], to = c.labL[y];
      if (from != to) inc_update_S(c, y, from, to);
    }
    const unsigned m = c.inc->clk + 1;                                      // cached per-slot terms: all stale
    csync(c);
    for (int s2 = tid; s2 < cap; s2 += c.nthr) c.tchg[s2] = m;
    if (tid == 0) c.inc->clk = m;
  } else {
    // restore the labels of the members (the proposal lived in place)
    for (int q = tid; q < nS + 2; q += c.nthr) c.labL[c.Slist[q]] = c.origM[q];
  }
  csync(c);
  unswap();
  if (tid == 0) st_add(c, ST_MH_LOGLIK, RC_CLOCK() - tm2);
}

// sortlabels (utils.jl:69-74): first-appearance relabelling to 1..K.
__device__ void record_labels(const Ctx& c, uint8_t* out) {
  const int tid = c.ctid;
  for (int s = tid; s < c.cap; s += c.nthr) c.itmp[s] = 0x7fffffff;
  csync(c);
  for (int j = tid; j < c.n; j += c.nthr) atomicMin(&c.itmp[c.lab[j]], j);
  csync(c);
  for (int s = tid; s < c.cap; s += c.nthr) {
    const int f = c.itmp[s];
    int id = 1;
    for (int t = 0; t < c.cap; ++t) id += c.itmp[t] < f;
    c.clist[s] = (uint8_t)id;
  }
  csync(c);
  for (int j = tid; j < c.n; j += c.nthr) out[j] = c.clist[c.lab[j]];
  csync(c);
}

// ------------------------------------------------------------------------------------------------
// The full Gibbs scan (mcmc.jl:158-256) WITHOUT streaming the matrix.
//   S[k][x] = sum_{j in k} DL[x][j] is kept per chain in global memory ([cap][n], exact integers).  Row x's candidate
//   sums are then cap 16-byte loads instead of a 16 n-byte row; a move of point i from a to b streams row i once and
//   updates S[a][.] and S[b][.] (inc_update_S).  The threads of the chain evaluate consecutive rows at once (one row per
//   thread) on the assumption that none of the earlier ones moves its point; the rows up to and including the first one
//   that moves are exactly what the sequential scan computes and are committed, the rest is evaluated again after the
//   move has been applied.  Every committed row sees the inputs of the sequential scan, so the results are the same bits as the
//   oracle's.
// ------------------------------------------------------------------------------------------------

// One row of the scan is evaluated by a GROUP of G adjacent lanes (G = 4: 8 rows per warp, slots < 64; G = 8: 4 rows per
// warp, slots < 128).  Lane g of the group owns the slots k = g + G j, j = 0..15, and keeps their terms in registers, so
// every term is loaded once, all of a lane's loads are in flight together, and a batch of nthr / G consecutive rows costs
// one memory round trip plus a few hundred instructions -- short enough for a chain that moves, wide enough (the whole
// CTA works on consecutive rows: one 128-byte segment per slot and 8 rows) for one that does not.
//
// Per-slot terms are CACHED across sweeps: L1 and L2' of (slot k, point i) depend only on S[k][i] and the size of k, i.e.
// on cluster k alone.  The chain counts its state changes (clk: moves of the scan, committed proposals); every slot
// remembers the count at which it last gained or lost a point (tchg[k]) and every point the count at which its row was
// last evaluated (tw[i]) -- an evaluation leaves the entry of EVERY live slot of that point valid (kept or recomputed and
// stored).  Entry (k, i) is therefore what a fresh evaluation would give (same formula, same inputs, same bits) exactly
// when tchg[k] <= tw[i]; anything else is recomputed.  The point's own slot (evaluated with the point detached) is never
// cached.  A chain at equilibrium spends two logarithms per row instead of two per (row, cluster), and validity costs
// one 4-byte count per point (shared memory when it fits) instead of a tag per entry.
#define RC_NZMAX 37.0   // Gumbel noise -log(-log u) <= 36.74 for every 53-bit u < 1: candidates further than this below the leader cannot win
#define RC_NP 16        // slots per lane of a row group
// What a row evaluation reads, passed BY VALUE: inc_eval_row is deliberately not inlined (its register allocation stays
// its own) and a reference to the kernel's Ctx would force that whole structure into local memory.
struct RowCtx {
  int n, cap, qD, qL;
  const longlong2* DL;
  const longlong2* S;
  const uint8_t* lab;
  const int* sizes;
  const uint8_t* rank;       // [cap] number of live slots below each slot (chain state)
  const double* tabs;
  const IncShared* inc;
  const Scal* sc;
  const rc_kparams* kp;
  unsigned long long key;
  double2* Cc;               // [cap][n] cached per-slot terms (L1, L2') of every point attached elsewhere
  RowSum* Rs;                // [n] row summaries (written when inc->mksum)
  unsigned* tw;              // [n] change count at which the point's cached entries were last all valid (0: never)
  const unsigned* tchg;      // [cap] change count at which each slot last changed (shared memory)
};
// Out of line on purpose: a row evaluation is unrolled over the lane's slots, and these two bodies (a Philox block and two
// logarithms each) are reached by a few slots per row only -- sixteen inlined copies of each made the evaluator larger than
// the instruction cache (ncu: 15 % of the kernel's stall samples were instruction fetches at exactly these branches).
__device__ __noinline__ double inc_noise_ool(unsigned long long key, unsigned it, int i, int kk) {  // utils.jl:4-5
  const rc_draw dr = rc_draw2(key, it, RC_SITE_SCAN, 0, (uint32_t)i, (uint32_t)(kk >> 1));
  return -rc_log(-rc_log((kk & 1) ? dr.u1 : dr.u0));
}
__device__ __forceinline__ double inc_noise(const RowCtx& c, unsigned it, int i, int kk) { return inc_noise_ool(c.key, it, i, kk); }
// per-slot terms (L1, L2') of one (slot, point) from its row sum and size (:206-242)
__device__ __noinline__ double2 inc_terms_ool(const rc_kparams* kpp, long long sx, long long sy, int szs, double lgA, double lgZ, int qD, int qL) {
  const rc_kparams& kp = *kpp;
  const rc_params& P = kp.P;
  const double szd = (double)szs;
  const double sD = rc_dequant(sx, qD), sL = rc_dequant(sy, qL);
  const double a_i = P.alpha + P.delta1 * szd, b_i = P.beta + sD;
  const double z_i = P.zeta + P.delta2 * szd, g_i = P.gamma + sD;
  double2 o;
  o.x = lgA + kp.abratio - a_i * rc_log(b_i) + (P.delta1 - 1) * sL - szd * kp.lgd1;
  o.y = lgZ - z_i * rc_log(g_i) + kp.zgratio + (P.delta2 - 1) * sL - szd * kp.lgd2;
  return o;
}
// Returns the chosen slot (the same value in the G lanes of the row's group), or -2 when a new cluster is a candidate
// and no slot is free.  All G lanes of a group call it with the same i; groups are independent of each other.
template <int G>
__device__ __noinline__ int inc_eval_row(const RowCtx c, unsigned it, int i) {
  const rc_kparams& kp = *c.kp;
  const rc_params& P = kp.P;
  const int n = c.n, cap = c.cap;
  const IncShared* sh = c.inc;
  const int lane = threadIdx.x & 31, g = lane & (G - 1), gbase = lane & ~(G - 1);
  const unsigned gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << gbase;
  const int nlive = sh->nlive;
  const int li = c.lab[i];
  const longlong2 self = __ldg(c.DL + (size_t)i * n + i);
  const bool single = c.sizes[li] == 1;
  const int Ki = nlive - (single ? 1 : 0);                                  // :195-196, i detached
  int e = sh->e0;
  if (single && (e < 0 || li < e)) e = li;                                  // findfirst(clustsizes .== 0), :199
  const bool hasnew = (P.maxK == 0 || Ki < P.maxK) && Ki < n;               // :198
  if (hasnew && e < 0) return -2;
  const double* __restrict__ tabs = c.tabs;
  // the point's own slot is always evaluated from its row sum: that load starts now
  longlong2 own_s = make_longlong2(0, 0);
  if (!single && (li & (G - 1)) == g) own_s = c.S[(size_t)li * n + i];
  // ---- the lane's slots: liveness (i detached), cached terms or row sums, all loads up front ----
  unsigned live = 0u, fresh = 0u;                                           // bit j: slot g + G j is a live candidate / must be recomputed
  const unsigned twi = c.tw[i], clk = sh->clk;
#pragma unroll
  for (int j = 0; j < RC_NP; ++j) {
    const int k = g + G * j;
    const bool lv = k < cap && c.sizes[k] - (k == li ? 1 : 0) > 0;
    live |= (lv ? 1u : 0u) << j;
  }
  double va[RC_NP], vb[RC_NP];                                              // (L1, L2') -- or the raw row sums until they are evaluated
#pragma unroll
  for (int j = 0; j < RC_NP; ++j) {
    const int k = g + G * j;
    // one 16-byte load per live slot, without a branch (all of the lane's loads are in flight together): the cached terms
    // when slot k has not changed since they were made, else its row sum
    const bool lv = (live >> j) & 1u, own = k == li;
    const bool hit = lv && !own && c.tchg[k] <= twi;
    const size_t idx = (size_t)k * n + i;
    const longlong2* src = hit ? reinterpret_cast<const longlong2*>(c.Cc + idx) : c.S + idx;
    longlong2 t = make_longlong2(0, 0);
    if (lv && !own) t = *src;
    if (own) t = own_s;
    va[j] = __longlong_as_double(t.x); vb[j] = __longlong_as_double(t.y);
    if (lv && !hit) fresh |= 1u << j;
  }
  // ---- per-slot terms (:206-242) of the slots that have no valid cached entry (always the point's own slot) ----
#pragma unroll
  for (int j = 0; j < RC_NP; ++j) {
    if (!((fresh >> j) & 1u)) continue;
    const int k = g + G * j;
    const bool own = k == li;
    long long sx = __double_as_longlong(va[j]), sy = __double_as_longlong(vb[j]);
    if (own) { sx -= self.x; sy -= self.y; }                                // :193-194 detach i
    const int szs = c.sizes[k] - (own ? 1 : 0);
    const double lgA = own ? tabs[3 * cap + k] : tabs[k];
    const double lgZ = own ? tabs[4 * cap + k] : tabs[cap + k];
    const double2 tv = inc_terms_ool(c.kp, sx, sy, szs, lgA, lgZ, c.qD, c.qL);
    va[j] = tv.x; vb[j] = tv.y;
    if (!own) c.Cc[(size_t)k * n + i] = make_double2(va[j], vb[j]);
  }
  if (g == 0 && twi != clk) c.tw[i] = clk;                                  // every live slot's entry of this point is valid as of now
  // ---- vecsum(L2', C_i) in the canonical order (:243): slot s in class s % 32, ascending within a class, then the
  //      xor-butterfly tree over the 32 classes (16, 8, 4, 2, 1).  A lane owns the classes g + G q entirely, so the tree
  //      levels with offset >= G are local and the last log2(G) levels are shuffles inside the group ----
  double L2i;
  {
    constexpr int NQ = 32 / G;                                              // classes per lane; class q has the slots j = q, q + NQ, ...
    double a[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      a[q] = 0.0;
#pragma unroll
      for (int j = q; j < RC_NP; j += NQ)
        if ((live >> j) & 1u) a[q] += vb[j];
    }
#pragma unroll
    for (int h = NQ / 2; h >= 1; h >>= 1)                                   // class offsets 16, 8, ... down to G
#pragma unroll
      for (int q = 0; q < h; ++q) a[q] = a[q] + a[q + h];
    double t = a[0];
#pragma unroll
    for (int off = G / 2; off >= 1; off >>= 1) t = t + __shfl_xor_sync(gmask, t, off);
    L2i = t;
  }
  // ---- log-probabilities (:244-247), their minimum, the leader ----
  const double r = c.sc->r, log1mp = c.sc->log1mp;
  unsigned have = live;
  const bool ownsnew = hasnew && (e & (G - 1)) == g;
  const int jnew = e / G;
  bool anynan = false;
  double mn = RC_INF, toplp = -RC_INF, topc = 0.0;
  int topj = -1;
#pragma unroll
  for (int j = 0; j < RC_NP; ++j) {
    const int k = g + G * j;
    if ((live >> j) & 1u) {
      const double L2 = L2i - vb[j];
      vb[j] = va[j] + (P.repulsion ? L2 : copysign(0.0, L2));               // c_k: everything but the (r, p)-dependent prior term
      va[j] = (k == li ? tabs[5 * cap + k] : tabs[2 * cap + k]) + vb[j];
    } else if (ownsnew && j == jnew) {                                      // :228-230 new cluster
      const double L2 = L2i - 0.0;
      va[j] = (kp.LOGN[Ki + 1] + r * log1mp) + (0.0 + (P.repulsion ? L2 : copysign(0.0, L2)));
      have |= 1u << j;
    } else continue;
    if (rc_isnan(va[j])) anynan = true;
    else {
      if (va[j] < mn) mn = va[j];
      if (va[j] > toplp) { toplp = va[j]; topj = j; topc = vb[j]; }
    }
  }
  // group-wide minimum / NaN flag / leader (highest log-probability; ties: lowest lane, then lowest j)
  int toplane = topj >= 0 ? g : -1;
#pragma unroll
  for (int off = G / 2; off >= 1; off >>= 1) {
    const double om = __shfl_xor_sync(gmask, mn, off);
    const int on = __shfl_xor_sync(gmask, (int)anynan, off);
    const double ot = __shfl_xor_sync(gmask, toplp, off);
    const int oj = __shfl_xor_sync(gmask, topj, off), ol = __shfl_xor_sync(gmask, toplane, off);
    const double oc = __shfl_xor_sync(gmask, topc, off);
    if (om < mn) mn = om;
    anynan = anynan || on != 0;
    if (ol >= 0 && (toplane < 0 || ot > toplp || (ot == toplp && (ol < toplane || (ol == toplane && oj < topj))))) { toplp = ot; topj = oj; toplane = ol; topc = oc; }
  }
  if (anynan) mn = RC_NAN;                                                  // Julia minimum propagates NaN
  // candidate index of the lane's slot j (position among the candidates in ascending slot order, new cluster last)
  auto cand_index = [&](int j) -> int {
    const int k = g + G * j;
    if (!((live >> j) & 1u)) return Ki;
    return (int)c.rank[k] - ((single && k > li) ? 1 : 0);
  };
  // ---- Gumbel-max (utils.jl:2-6): argmax of noise + shifted log-probability, first index wins ties ----
  double bg = 0.0; int bkk = 0x7fffffff, bslot = -1; bool bnan = false;    // the lane's best candidate
  const bool fast = !anynan && mn > -RC_INF && mn < RC_INF && toplp < RC_INF && toplane >= 0;     // uniform over the group
  if (fast && sh->mksum && !single) {
    // row summary (RowSum): the leader when it is a live slot, its term, the largest term among the other live slots
    double c2 = -RC_INF;
#pragma unroll
    for (int j = 0; j < RC_NP; ++j)
      if (((live >> j) & 1u) && !(g == toplane && j == topj) && vb[j] > c2) c2 = vb[j];
#pragma unroll
    for (int off = G / 2; off >= 1; off >>= 1) { const double o = __shfl_xor_sync(gmask, c2, off); if (o > c2) c2 = o; }
    const int leadlive = __shfl_sync(gmask, (g == toplane) ? (int)((live >> topj) & 1u) : 0, gbase + toplane);
    if (g == 0) {
      RowSum rs; rs.cT = topc; rs.c2 = c2; rs.L2i = L2i; rs.T = toplane + G * topj; rs.stamp = leadlive ? clk : 0u;
      c.Rs[i] = rs;
    }
  }
  if (fast) {
    // every shifted log-probability is finite: a candidate whose value plus the largest possible noise stays below the
    // leader's exact value cannot be the arg-max, so its noise is never drawn (same result, far fewer logarithms)
    double gtop = 0.0;
    if (g == toplane) {
      bkk = cand_index(topj);
      bg = inc_noise(c, it, i, bkk) + (toplp - mn);
      bslot = g + G * topj;
      gtop = bg;
    }
    gtop = __shfl_sync(gmask, gtop, gbase + toplane);
#pragma unroll
    for (int j = 0; j < RC_NP; ++j) {
      if (!((have >> j) & 1u) || (g == toplane && j == topj)) continue;
      const double lpm = va[j] - mn;
      if (lpm + RC_NZMAX >= gtop) {
        const int kk = cand_index(j);
        const double gg = inc_noise(c, it, i, kk) + lpm;
        if (bslot < 0 || gg > bg || (gg == bg && kk < bkk)) { bg = gg; bkk = kk; bslot = g + G * j; }
      }
    }
  } else {
    // general path (NaN / infinities among the log-probabilities): every candidate draws its noise; NaN is maximal for
    // argmax and the first NaN (lowest candidate index) wins
#pragma unroll
    for (int j = 0; j < RC_NP; ++j) {
      if (!((have >> j) & 1u)) continue;
      const int kk = cand_index(j);
      const double gg = inc_noise(c, it, i, kk) + (va[j] - mn);
      const bool gn = rc_isnan(gg);
      bool better;
      if (bslot < 0) better = true;
      else if (gn) better = !bnan || kk < bkk;
      else if (bnan) better = false;
      else better = gg > bg || (gg == bg && kk < bkk);
      if (better) { bg = gg; bkk = kk; bslot = g + G * j; bnan = gn; }
    }
  }
#pragma unroll
  for (int off = G / 2; off >= 1; off >>= 1) {
    const double og = __shfl_xor_sync(gmask, bg, off);
    const int ok = __shfl_xor_sync(gmask, bkk, off);
    const int os = __shfl_xor_sync(gmask, bslot, off);
    const int on = __shfl_xor_sync(gmask, (int)bnan, off);
    bool better;
    if (os < 0) better = false;
    else if (bslot < 0) better = true;
    else if (on) better = !bnan || ok < bkk;
    else if (bnan) better = false;
    else better = og > bg || (og == bg && ok < bkk);
    if (better) { bg = og; bkk = ok; bslot = os; bnan = on != 0; }
  }
  return bslot;
}

// (Re)build the chain's slot tables in shared memory from the sizes: the live list, the first empty slot and the
// size-dependent terms at the current size / at size - 1.  Warp 0.
__device__ void inc_build_tables(const Ctx& c, int only_a = -1, int only_b = -1) {
  const rc_kparams& kp = *c.kp;
  IncShared* sh = c.inc;
  const int cap = c.cap, lane = c.lane;
  int base = 0, e0 = -1;
  for (int w = 0; w * 32 < cap; ++w) {
    const int s = w * 32 + lane;
    const int sz = s < cap ? c.sizes[s] : 0;
    const bool live = s < cap && sz > 0;
    const unsigned m = __ballot_sync(0xffffffffu, live);
    const unsigned em = __ballot_sync(0xffffffffu, s < cap && sz == 0);
    if (live) c.live[base + __popc(m & ((1u << lane) - 1u))] = (uint8_t)s;
    if (s < cap) c.rank[s] = (uint8_t)(base + __popc(m & ((1u << lane) - 1u)));      // live slots below s
    base += __popc(m);
    if (e0 < 0 && em) e0 = w * 32 + __ffs(em) - 1;
    if (s < cap && (only_a < 0 || s == only_a || s == only_b)) {
      c.tabs[s] = kp.LGA[sz]; c.tabs[cap + s] = kp.LGZ[sz]; c.tabs[2 * cap + s] = lpr_at(c, sz > 0 ? sz : 1);
      c.tabs[3 * cap + s] = kp.LGA[sz > 0 ? sz - 1 : 0]; c.tabs[4 * cap + s] = kp.LGZ[sz > 0 ? sz - 1 : 0];
      c.tabs[5 * cap + s] = lpr_at(c, sz > 1 ? sz - 1 : 1);
    }
  }
  if (only_a >= 0 && lane == 0) { const unsigned m = ++sh->clk; c.tchg[only_a] = m; c.tchg[only_b] = m; }   // clusters a and b changed: their cached terms are stale
  if (lane == 0) {
    sh->nlive = base; sh->e0 = e0;
    const int hi = max(base > 0 ? (int)c.live[base - 1] : 0, e0 >= 0 ? e0 : cap - 1);   // highest slot a row of the scan can meet
    sh->narrow = hi < 64 ? 4 : (hi < 128 ? 8 : 16);
  }
  __syncwarp();
  {
    // the row summaries' bound: the largest prior term over the live slots (at the slot's size and at size - 1), all finite
    double mx = -RC_INF; bool ok = true;
    for (int s = lane; s < cap; s += 32)
      if (c.sizes[s] > 0) {
        const double t2 = c.tabs[2 * cap + s], t5 = c.tabs[5 * cap + s];
        if (!(t2 > -RC_INF && t2 < RC_INF && t5 > -RC_INF && t5 < RC_INF)) ok = false;       // (false for NaN too)
        else mx = fmax(mx, fmax(t2, t5));
      }
    for (int off = 16; off; off >>= 1) { mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off)); ok = __shfl_xor_sync(0xffffffffu, (int)ok, off) && ok; }
    if (lane == 0) { sh->maxtab = mx; sh->tabs_ok = ok ? 1 : 0; }
  }
  __syncwarp();
}

// bar.red.or over the team: true when v holds in any thread (a barrier like csync)
__device__ __forceinline__ bool team_any(int barid, int nthr, bool v) {
  int r;
  asm volatile("{\n .reg .pred p, q;\n setp.ne.s32 p, %1, 0;\n bar.red.or.pred q, %2, %3, p;\n selp.s32 %0, 1, 0, q;\n}"
               : "=r"(r) : "r"((int)v), "r"(barid), "r"(nthr) : "memory");
  return r != 0;
}
// doubles <-> 64-bit integers of the same order (finite values), for min / max by integer atomics
__device__ __forceinline__ long long ord_key(double x) { const long long b = __double_as_longlong(x); return b >= 0 ? b : b ^ 0x7fffffffffffffffLL; }
__device__ __forceinline__ double ord_val(long long k) { return __longlong_as_double(k >= 0 ? k : k ^ 0x7fffffffffffffffLL); }
#define RC_CM_BIG 0x1p1000       // magnitudes below this: no sum of four such values overflows

// Per-slot margins of the row summaries.  Of the row-summary test (RowSum) only tab_T, maxtab and the new-cluster base
// A = LOGN[Ki + 1] + r log(1 - p) depend on (r, p); everything per row is fixed while the chain's state is.  So when every
// row's summary is current, its leader is its own slot T and that slot keeps at least two points, slot T stores over its rows
//   Cm[T].x = min fl(cT - c2),   Cm[T].y = min fl(cT - L2i) (repulsion) / min cT (none),   Cm[T].z = max(|cT|, |c2|, |L2i|)
// and a scan tests O(K) slots instead of n summaries (inc_scan_by_margins).  Min and max are exact, so the order in which
// rows are reduced does not matter.  Built after a committed scan that moved no point; a failed build is not retried until
// the state changes (Cms = {change count, ok}).  red: [3][cap] shared-memory scratch.  Whole team.
__device__ __noinline__ void inc_margins_build(const RowCtx rc, IncShared* sh, double4* Cm, unsigned* Cms, long long* red,
                                               int tid, int NT, int barid) {
  const int n = rc.n, cap = rc.cap;
  const unsigned clk = sh->clk;
  const bool rep = rc.kp->P.repulsion;
  for (int s = tid; s < cap; s += NT) { red[s] = LLONG_MAX; red[cap + s] = LLONG_MAX; red[2 * cap + s] = 0; }
  asm volatile("bar.sync %0, %1;" ::"r"(barid), "r"(NT) : "memory");
  bool ok = true;
  int cs = -1;                                                              // the thread's current slot and its running values
  double ma = 0.0, mb = 0.0, mg = 0.0;
  auto flush = [&]() {
    if (cs < 0) return;
    atomicMin(red + cs, ord_key(ma)); atomicMin(red + cap + cs, ord_key(mb));
    atomicMax(red + 2 * cap + cs, __double_as_longlong(mg));              // (mg >= 0: its bits order like the value)
  };
  for (int i = tid; i < n; i += NT) {
    const RowSum rs = rc.Rs[i];
    const int T = rs.T;
    // (comparisons are false for NaN: a NaN term fails like an infinite one)
    if (rs.stamp != clk || T != (int)rc.lab[i] || rc.sizes[T] < 2 ||
        !(fabs(rs.cT) < RC_CM_BIG && fabs(rs.c2) < RC_CM_BIG && fabs(rs.L2i) < RC_CM_BIG)) { ok = false; break; }
    const double a = rs.cT - rs.c2, b = rep ? rs.cT - rs.L2i : rs.cT;
    const double m = fmax(fabs(rs.cT), fmax(fabs(rs.c2), fabs(rs.L2i)));
    if (T != cs) { flush(); cs = T; ma = a; mb = b; mg = m; }
    else { ma = fmin(ma, a); mb = fmin(mb, b); mg = fmax(mg, m); }
  }
  if (ok) flush();
  ok = !team_any(barid, NT, !ok);
  if (ok)
    for (int s = tid; s < cap; s += NT) Cm[s] = make_double4(ord_val(red[s]), ord_val(red[cap + s]), __longlong_as_double(red[2 * cap + s]), 0.0);
  if (tid == 0) { Cms[0] = clk; Cms[1] = ok ? 1u : 0u; sh->cm_clk = clk; sh->cm_ok = ok ? 1 : 0; }
  asm volatile("bar.sync %0, %1;" ::"r"(barid), "r"(NT) : "memory");
}

// A whole scan decided by the per-slot margins: true when every row would be decided by its summary and stays where it is.
// Every warp tests every live slot T (t5 = tab_T at size - 1, the point detached) against
//   (1)  fl(fl(t5 - maxtab) + Cm[T].x) > 41 + eps1,   eps1 = 2^-46 (E1 + 64),  E1 = Cm[T].z + |t5| + |maxtab|
//   (2)  fl(fl(t5 - A)      + Cm[T].y) > 41 + eps2,   eps2 = 2^-46 (E2 + 64),  E2 = Cm[T].z + |t5| + |A|   (new cluster possible)
// and then every row's leader uniform is drawn and checked to be > 0, as the row-summary path does.
// Proof that (1) implies the row test tab_T + cT - (maxtab + c2) > 41, i.e. fl(fl(t5 + cT) - fl(maxtab + c2)) > 41, for every
// row of T (for (2) replace maxtab by A and c2 by L2i, or by +-0 without repulsion, where lpnew = A exactly; A is computed
// by the same operations as in the row test).  u = 2^-53, M = Cm[T].z, all magnitudes below 2^1000 (checked, so nothing
// overflows and every term is finite):  with d = fl(cT - c2) >= Cm[T].x (the minimum is exact)
//   fl(t5 + cT) - fl(maxtab + c2) >= t5 - maxtab + cT - c2 - u(|t5| + |cT| + |maxtab| + |c2|)
//   cT - c2 >= d - u(|cT| + |c2|) >= Cm[T].x - 2uM
//   t5 - maxtab + Cm[T].x >= w - u(|t5| + |maxtab|) - u(1 + u)(|t5| + |maxtab| + 2M(1 + u))   (w: the left side of (1))
// so the row's exact difference is >= w - u(3|t5| + 3|maxtab| + 6M)(1 + 2u) > w - 2^-50 E1 > 41 + 2^-46 E1 + 2^-40 - 2^-50 E1
// (computing eps and its sum with 41 loses less than 2^-96 E1 + 2^-47), hence > 41 + 2^-41, and its rounding stays above
// 41 (ulp(41) = 2^-47).  Rows of T pass the row test, so the new path decides a subset of what the row summaries decide,
// with the same outcome (no move), and no output changes.  Whole team; one barrier.
__device__ __noinline__ bool inc_scan_by_margins(const RowCtx rc, const double4* Cm, unsigned it, int tid, int NT, int barid) {
  const rc_params& P = rc.kp->P;
  const IncShared* sh = rc.inc;
  const int n = rc.n, cap = rc.cap;
  const int Ki = sh->nlive;
  const bool hasnew = (P.maxK == 0 || Ki < P.maxK) && Ki < n;               // :198 (every point's own cluster survives)
  const double maxtab = sh->maxtab;
  if (hasnew && sh->e0 < 0) return false;                                   // (the row evaluation reports the missing slot)
  const double A = rc.kp->LOGN[Ki + 1] + rc.sc->r * rc.sc->log1mp;          // (as in the row test)
  bool fail = false;
  for (int s = tid & 31; s < cap; s += 32)
    if (rc.sizes[s] > 0) {
      const double4 m = Cm[s];
      const double t5 = rc.tabs[5 * cap + s];
      const double e1 = m.z + fabs(t5) + fabs(maxtab);
      bool pass = e1 < RC_CM_BIG && (t5 - maxtab) + m.x > RC_SUM_MARGIN + 0x1p-46 * (e1 + 64.0);
      if (hasnew) {
        const double e2 = m.z + fabs(t5) + fabs(A);
        pass = pass && e2 < RC_CM_BIG && (t5 - A) + m.y > RC_SUM_MARGIN + 0x1p-46 * (e2 + 64.0);
      }
      if (!pass) fail = true;
    }
  fail = __any_sync(0xffffffffu, fail);
  if (!fail)
    for (int i = tid; i < n; i += NT) {                                     // the leader's own uniform must be > 0 (else its noise is -Inf)
      const int kk = (int)rc.rank[rc.lab[i]];
      const rc_draw dr = rc_draw2(rc.key, it, RC_SITE_SCAN, 0, (uint32_t)i, (uint32_t)(kk >> 1));
      if (!(((kk & 1) ? dr.u1 : dr.u0) > 0.0)) fail = true;
    }
  return !team_any(barid, NT, fail);
}

// The full scan (mcmc.jl:192-253) from row istart in batches of up to nthr / G consecutive rows (G lanes per row), by the
// team described by c (the whole CTA, or the warps that have nothing to do during the restricted scans).
// dry: nothing is committed -- the scan stops at the first row that would move its point (or overflow) and leaves that
// row in dry_stop; every row before it stands exactly as the sequential scan would leave it (it does not move).
__device__ void inc_full_scan(const Ctx& c, unsigned it, int istart, bool dry) {
  IncShared* sh = c.inc;
  const int n = c.n, cap = c.cap, NT = c.nthr, tid = c.ctid, lane = c.lane;
  if (tid == 0) {
    sh->sfirst[0] = RC_INC_NONE; sh->sfirst[1] = RC_INC_NONE; sh->sfirst[2] = RC_INC_NONE;
    sh->fa[0] = RC_INC_NONE; sh->fa[1] = RC_INC_NONE; sh->fa[2] = RC_INC_NONE; sh->fm[0] = RC_INC_NONE; sh->fm[1] = RC_INC_NONE; sh->fm[2] = RC_INC_NONE;
    if (!dry) sh->nmoves = 0; else sh->dry_stop = n;
  }
  if (c.cwarp == 0) inc_build_tables(c);
  csync(c);
  RowCtx rc;
  rc.n = n; rc.cap = cap; rc.qD = c.qD; rc.qL = c.qL; rc.DL = c.DL; rc.S = c.S; rc.lab = c.lab; rc.sizes = c.sizes; rc.rank = c.rank;
  rc.tabs = c.tabs; rc.inc = c.inc; rc.sc = c.sc; rc.kp = c.kp; rc.key = c.key; rc.Cc = c.Cc; rc.tw = c.tw; rc.tchg = c.tchg; rc.Rs = c.Rs;
  int batch = 0, i0 = istart;
  // Rows per batch follow the observed run length between moves (rows behind a move are evaluated again).
  int nrows = sh->hint > 0 ? sh->hint : NT, streak = 0;
  int skipA = 0;                                                            // batches to go before the summaries are tried again
  long long nfast = 0;
  // a committed scan whose per-slot margins are current: decided as a whole when they prove that no row moves
  if (!dry && istart == 0 && sh->mksum && sh->tabs_ok && sh->cm_ok && sh->cm_clk == sh->clk &&
      inc_scan_by_margins(rc, c.Cm, it, tid, NT, c.barid)) {
    i0 = n; nfast = n;
#ifdef RC_NO_STATS
    if (tid == 0) st_add(c, ST_BULK_REDUCE, 1);                             // (default library: scans decided by the margins)
#endif
  }
  while (i0 < n) {
    const int slot3 = batch % 3;
    if (tid == 0) { const int nx = (batch + 1) % 3; sh->sfirst[nx] = RC_INC_NONE; sh->fa[nx] = RC_INC_NONE; sh->fm[nx] = RC_INC_NONE; }
    ++batch;
    int F = RC_INC_NONE;
    bool fromA = false;
    if (sh->mksum && sh->tabs_ok && skipA == 0) {
      // ---- rows decided by their summaries (RowSum), one thread per row ----
      const int nbA = min(NT, n - i0);
      if (tid < nbA) {
        const int i = i0 + tid;
        if (i + NT < n) asm volatile("prefetch.global.L1 [%0];" ::"l"(c.Rs + i + NT));        // the next batch's summary
        const RowSum rs = c.Rs[i];
        int r = -3;                                                         // undecided
        if (rs.stamp == sh->clk) {
          const rc_kparams& kp = *c.kp;
          const rc_params& P = kp.P;
          const int li = c.lab[i], T = rs.T;
          const int Ki = sh->nlive;
          const bool hasnew = (P.maxK == 0 || Ki < P.maxK) && Ki < n;       // :198 (the point's own cluster survives: not single)
          if (c.sizes[li] > 1 && !(hasnew && sh->e0 < 0)) {
            const double lpT = (T == li ? c.tabs[5 * cap + T] : c.tabs[2 * cap + T]) + rs.cT;
            const double bound = sh->maxtab + rs.c2;
            const double lpnew = (kp.LOGN[Ki + 1] + c.sc->r * c.sc->log1mp) + (0.0 + (P.repulsion ? rs.L2i : copysign(0.0, rs.L2i)));
            if (lpT - bound > RC_SUM_MARGIN && (!hasnew || (lpT - lpnew > RC_SUM_MARGIN && lpnew > -RC_INF)) && lpT < RC_INF && lpT > -RC_INF) {
              const int kk = (int)c.rank[T];                                 // the leader's own uniform must be > 0 (else its noise is -Inf)
              const rc_draw dr = rc_draw2(c.key, it, RC_SITE_SCAN, 0, (uint32_t)i, (uint32_t)(kk >> 1));
              if (((kk & 1) ? dr.u1 : dr.u0) > 0.0) r = T;
            }
          }
        }
        c.res[tid] = r;
        if (r == -3) atomicMin(&sh->fa[slot3], tid);
        else if (r != (int)c.lab[i]) atomicMin(&sh->fm[slot3], tid);
      }
      csync(c);
      const int U = min(sh->fa[slot3], nbA), M = sh->fm[slot3];
      if (M < U) { F = M; fromA = true; nfast += M; }                        // a decided row moves its point: committed below like any move
      else {
        i0 += U; nfast += U;                                                // the rows before U stand
        skipA = U == 0 ? 4 : 0;
        if (U == nbA) continue;
      }
    } else if (skipA > 0) --skipA;
    if (!fromA) {
      const int G = sh->narrow;                                             // lanes per row: 4 / 8 / 16 when every candidate slot is below 64 / 128 / 256
      const int nb = min(nrows, NT / G);                                    // rows of this batch
      const long long te0 = RC_CLOCK();
      {
        const int row = tid / G, i = i0 + row;
        if (row < nb && i < n) {
          const int cnew = G == 4 ? inc_eval_row<4>(rc, it, i) : (G == 8 ? inc_eval_row<8>(rc, it, i) : inc_eval_row<16>(rc, it, i));
          if ((tid & (G - 1)) == 0) {
            c.res[row] = cnew;
            if (cnew != (int)c.lab[i]) atomicMin(&sh->sfirst[slot3], row);
          }
        }
      }
      if (tid == 0) st_add(c, ST_REBUILDS, RC_CLOCK() - te0);               // (incremental mode: cycles of thread 0 in the row evaluations)
      csync(c);
      F = sh->sfirst[slot3];
      if (F == RC_INC_NONE) {                                               // nobody moved: the whole batch stands
        i0 += nb;
        streak += nb;
        if (streak >= nrows) { nrows = min(NT, nrows * 2); streak = 0; }
        continue;
      }
    }
    const int mi = i0 + F, b = c.res[F];
    if (dry) { if (tid == 0) sh->dry_stop = mi; break; }                    // the committing scan resumes here
    if (b < 0) { if (tid == 0) c.sc->status = RC_ERR_SLOTS; break; }        // slot capacity exhausted at row mi
    const int a = c.lab[mi];
    const long long tu0 = RC_CLOCK();
    if (c.cwarp == 0) {
      // ---- the point moved (:250-252): block sums from row mi's sums over the live slots, then labels, sizes, tables ----
      const longlong2 self = __ldg(c.DL + (size_t)mi * n + mi);
      long long bd[RC_NSI], bl[RC_NSI];
      bool live[RC_NSI];
#pragma unroll
      for (int w = 0; w < RC_NSI; ++w) {
        const int s = w * 32 + lane;
        bd[w] = 0; bl[w] = 0;
        live[w] = s < cap && c.sizes[s] - (s == a ? 1 : 0) > 0;
        if (live[w]) { const longlong2 t = c.S[(size_t)s * n + mi]; bd[w] = t.x; bl[w] = t.y; if (s == a) { bd[w] -= self.x; bl[w] -= self.y; } }
      }
      __syncwarp();
#pragma unroll
      for (int w = 0; w < RC_NSI; ++w) {
        const int s = w * 32 + lane;
        if (s >= cap) continue;
        if (s == a) {
          const int ix = tri(a, a, cap);
          rc_i128 x = c.WD[ix]; rc_sub128(x, rc_make128(2 * bd[w] + self.x)); c.WD[ix] = x;
          rc_i128 y = c.WL[ix]; rc_sub128(y, rc_make128(2 * bl[w] + self.y)); c.WL[ix] = y;
          const size_t o = (size_t)a * n + mi;                              // S[a][mi] loses the point's own entry (inc_update_S skips x = mi)
          longlong2 t = c.S[o]; t.x -= self.x; t.y -= self.y; c.S[o] = t;
        } else if (live[w]) {
          const int ix = tri(a, s, cap);
          rc_i128 x = c.WD[ix]; rc_sub128(x, rc_make128(bd[w])); c.WD[ix] = x;
          rc_i128 y = c.WL[ix]; rc_sub128(y, rc_make128(bl[w])); c.WL[ix] = y;
        }
      }
      __syncwarp();
#pragma unroll
      for (int w = 0; w < RC_NSI; ++w) {
        const int s = w * 32 + lane;
        if (s >= cap) continue;
        if (s == b) {
          const int ix = tri(b, b, cap);
          rc_i128 x = c.WD[ix]; rc_add128(x, rc_make128(2 * bd[w] + self.x)); c.WD[ix] = x;
          rc_i128 y = c.WL[ix]; rc_add128(y, rc_make128(2 * bl[w] + self.y)); c.WL[ix] = y;
          const size_t o = (size_t)b * n + mi;
          longlong2 t = c.S[o]; t.x += self.x; t.y += self.y; c.S[o] = t;
        } else if (live[w]) {
          const int ix = tri(b, s, cap);
          rc_i128 x = c.WD[ix]; rc_add128(x, rc_make128(bd[w])); c.WD[ix] = x;
          rc_i128 y = c.WL[ix]; rc_add128(y, rc_make128(bl[w])); c.WL[ix] = y;
        }
      }
      __syncwarp();
      if (lane == 0) { c.lab[mi] = (uint8_t)b; c.sizes[a] -= 1; c.sizes[b] += 1; sh->nmoves += 1; }
      __syncwarp();
      inc_build_tables(c, a, b);
    }
    inc_update_S(c, mi, a, b, mi, NT > 32 ? 32 : 0);
    csync(c);
    if (tid == 0) st_add(c, ST_BULK_PATCH, RC_CLOCK() - tu0);               // (incremental mode: cycles in the move updates)
    i0 = mi + 1;
    nrows = min(NT, max(8, (2 * (streak + F + 1) + 7) & ~7));
    streak = 0;
  }
  csync(c);
#ifdef RC_NO_STATS
  if (tid == 0) st_add(c, ST_BULK_ROWS, nfast);                             // (default library: rows decided by their summaries)
#endif
  if (tid == 0) {
    if (dry) sh->nfast_dry = (int)nfast;
    else { sh->scanfast = 2 * ((istart > 0 ? sh->nfast_dry : 0) + nfast) >= n ? 1 : 0; sh->nfast_dry = 0; }
  }
  if (dry) return;
  if (c.cwarp == 0) {                                                       // :254
    int K = 0;
    for (int s = lane; s < cap; s += 32) K += c.sizes[s] > 0;
    for (int off = 16; off; off >>= 1) K += __shfl_xor_sync(0xffffffffu, K, off);
    if (lane == 0) { c.sc->K = K; st_add(c, ST_MOVES, sh->nmoves); sh->hint = nrows; sh->mksum = (sh->nmoves <= 2 && c.kp->shortcuts) ? 1 : 0; }
  }
  csync(c);
  // nothing moved and the margins are not current: build them (in the split-merge member scratch, dead here) while every
  // row's summary is fresh
  if (sh->nmoves == 0 && sh->mksum && sh->cm_clk != sh->clk && 4 * c.mcap >= 3 * cap)
    inc_margins_build(rc, sh, c.Cm, c.Cms, reinterpret_cast<long long*>(c.mAB), tid, NT, c.barid);
}

struct IncLayout { size_t prows, sc, inc, sizes, szL, itmp, clist, lab, labL, live, rank, tabs, res, ep, tw, mAB, mDG, mL2s, total; };
__host__ __device__ inline IncLayout inc_layout(int n, int cap, int mcap, int tw_smem) {
  IncLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t p = o; o += (bytes + 15) & ~(size_t)15; return p; };
  L.prows = take(sizeof(rc_i128) * 4 * cap);        // rows of the proposed state during a split-merge step
  L.sc = take(sizeof(Scal));
  L.inc = take(sizeof(IncShared));
  L.sizes = take(sizeof(int) * cap);
  L.szL = take(sizeof(int) * cap);
  L.itmp = take(sizeof(int) * (cap > 64 ? cap : 64));
  L.clist = take(cap);
  L.lab = take(n);
  L.labL = take(n);
  L.live = take(cap);
  L.rank = take(cap);
  L.tabs = take(sizeof(double) * 6 * cap);
  L.res = take(sizeof(int) * 512);
  L.ep = take(sizeof(unsigned) * cap);
  L.tw = take(tw_smem ? sizeof(unsigned) * n : 0);
  L.mAB = take(sizeof(longlong4) * mcap);
  L.mDG = take(sizeof(longlong2) * mcap);
  L.mL2s = take(sizeof(double2) * mcap);
  L.total = (o + 127) & ~(size_t)127;
  return L;
}

// One CTA = one chain = the team; blockDim.x = kp.inc_nthr (a multiple of 32, at most 512).  S and W are built by
// k_init_S / k_initw_from_S before the first launch.
__global__ void __launch_bounds__(512, 1) k_chain_inc(const __grid_constant__ rc_kparams kp) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int chain = blockIdx.x;
  const int n = kp.n, cap = kp.cap;
  Ctx c;
  c.n = n; c.cap = cap; c.qD = kp.qD; c.qL = kp.qL; c.DL = kp.DL; c.kp = &kp;
  c.ctid = threadIdx.x; c.cwarp = c.ctid >> 5; c.lane = c.ctid & 31; c.barid = 1;
  c.nthr = blockDim.x; c.nwarp = blockDim.x >> 5;
  {
    const IncLayout L = inc_layout(n, cap, kp.inc_mcap, kp.tw_smem);
    c.mcap = kp.inc_mcap;
    c.mAB = reinterpret_cast<longlong4*>(smem + L.mAB);
    c.mDG = reinterpret_cast<longlong2*>(smem + L.mDG);
    c.mL2s = reinterpret_cast<double2*>(smem + L.mL2s);
    c.live = smem + L.live;
    c.rank = smem + L.rank;
    c.tabs = reinterpret_cast<double*>(smem + L.tabs);
    c.res = reinterpret_cast<int*>(smem + L.res);
    c.tchg = reinterpret_cast<unsigned*>(smem + L.ep);
    c.tw = kp.tw_smem ? reinterpret_cast<unsigned*>(smem + L.tw) : kp.Vv + (size_t)chain * n;
    c.Rs = kp.Rs + (size_t)chain * n;
    c.LLF = kp.LLF + (size_t)chain * cap * cap; c.LLFs = kp.LLFs + (size_t)chain * cap * cap;
    c.Cm = kp.Cm + (size_t)chain * cap; c.Cms = kp.Cms + (size_t)chain * 2;
    c.prows = reinterpret_cast<rc_i128*>(smem + L.prows);
    c.sc = reinterpret_cast<Scal*>(smem + L.sc);
    c.inc = reinterpret_cast<IncShared*>(smem + L.inc);
    c.sizes = reinterpret_cast<int*>(smem + L.sizes);
    c.szL = reinterpret_cast<int*>(smem + L.szL);
    c.itmp = reinterpret_cast<int*>(smem + L.itmp);
    c.clist = smem + L.clist;
    c.lab = smem + L.lab;
    c.labL = (kp.numMH == 1 && kp.ovl_min_thr > 0 && (int)blockDim.x >= kp.ovl_min_thr) ? smem + L.labL : c.lab;   // one proposal per iteration: the proposal works on a copy (scan beside the restricted scans)
  }
  const int ch = chain;
  c.WD = kp.WD + (size_t)ch * cap * cap;
  c.WL = kp.WL + (size_t)ch * cap * cap;
  c.S = kp.S + (size_t)ch * cap * n;
  c.Cc = kp.Cc + (size_t)ch * cap * n;
  c.WDbak = kp.WDbak ? kp.WDbak + (size_t)ch * cap * cap : nullptr;
  c.WLbak = kp.WLbak ? kp.WLbak + (size_t)ch * cap * cap : nullptr;
  c.labbak = kp.labbak ? kp.labbak + (size_t)ch * n : nullptr;
  c.szbak = kp.szbak ? kp.szbak + (size_t)ch * (cap + 1) : nullptr;
  c.Slist = kp.Slist + (size_t)ch * (n + 2);
  c.origM = kp.origM + (size_t)ch * (n + 2);
  c.AB = kp.AB + (size_t)ch * (n + 2);
  c.L2s = kp.L2s + (size_t)ch * n;
  c.NZ = kp.NZ + (size_t)ch * (kp.numGibbs + 1) * n;
  c.DG = kp.DG + (size_t)ch * (n + 2);
  c.stats = kp.stats + (size_t)ch * 16;
  c.terms = kp.terms + (size_t)ch * kp.terms_stride;
  c.key = rc_chain_key(kp.seed, (unsigned long long)(kp.chain_offset + ch));
  const int tid = c.ctid, nt = c.nthr;

  for (int j = tid; j < n; j += nt) c.lab[j] = kp.labels[(size_t)chain * n + j];
  for (int s = tid; s < cap; s += nt) { c.sizes[s] = kp.sizes[(size_t)chain * cap + s]; c.tchg[s] = kp.epochs[(size_t)chain * (cap + 1) + s]; }
  if (kp.tw_smem) for (int j = tid; j < n; j += nt) c.tw[j] = kp.Vv[(size_t)chain * n + j];
  if (tid == 0) { c.inc->clk = kp.epochs[(size_t)chain * (cap + 1) + cap]; c.inc->mksum = kp.shortcuts ? 1 : 0; c.inc->tabs_ok = 0; c.inc->maxtab = 0.0; c.inc->nfast_dry = 0; c.inc->scanfast = 0; c.sc->llclk = 0u; c.sc->llcur = 0.0; c.inc->cm_clk = c.Cms[0]; c.inc->cm_ok = (int)c.Cms[1]; }
  if (tid == 0) {
    Scal& s = *c.sc;
    s.r = kp.r[chain]; s.p = kp.p[chain];
    s.logp = rc_log(s.p); s.log1mp = rc_log(1 - s.p);
    s.status = kp.status[chain]; s.fslotA = -1; s.fslotB = -1; s.ltp = 0.0; s.forked = 0;
    c.inc->hint = 0;
    int K = 0;
    for (int q = 0; q < cap; ++q) K += kp.sizes[(size_t)chain * cap + q] > 0;
    s.K = K;
  }
  csync(c);
  if (kp.loglik_only) {                                                      // rc_loglik: the loaded state's log-likelihood only
    const double ll = loglik_cur(c);
    if (tid == 0) kp.out_ll[chain] = ll;
    return;
  }

  for (long long iter = kp.it0 + 1; iter <= kp.it1; ++iter) {
    const unsigned it = (unsigned)iter;
    const long long ti0 = RC_CLOCK();
    csync(c);
    if (c.sc->status != 0) break;                                            // the chain stopped (slot capacity)
    bool do_scan = true;
    if (tid == 0) c.inc->dry_stop = 0;
    if (c.cwarp == 0) {
      const bool ra = update_r(c, it);                                       // mcmc.jl:538
      if (tid == 0) {
        kp.r_acc[(size_t)chain * kp.numiters + (iter - 1)] = ra ? 1 : 0;
        update_p(c, it);                                                     // :539
      }
    }
    csync(c);
    // (the size-dependent prior terms are evaluated where they are needed: lpr_at)
    if (tid == 0) st_add(c, ST_RP, RC_CLOCK() - ti0);
    // sample_labels! (:540)
    const bool multi = kp.numMH > 1;
    if (multi) {                                             // the chain's own state, in case a proposal is accepted and committed
      for (int j = tid; j < n; j += nt) c.labbak[j] = c.lab[j];
      for (int s = tid; s < cap; s += nt) c.szbak[s] = c.sizes[s];
      if (tid == 0) { c.szbak[cap] = c.sc->K; c.sc->forked = 0; }
      csync(c);
    }
    for (unsigned mh = 0; mh < (unsigned)kp.numMH; ++mh) {
      splitmerge_step(c, it, mh, mh + 1 < (unsigned)kp.numMH);
      if (c.sc->status) { do_scan = false; break; }
      const int acc = c.sc->itmp[1], spl = c.sc->itmp[2];
      if (tid == 0) {
        kp.sm_acc[((size_t)chain * kp.numiters + (iter - 1)) * kp.numMH + mh] = (uint8_t)acc;
        kp.sm_split[((size_t)chain * kp.numiters + (iter - 1)) * kp.numMH + mh] = (uint8_t)spl;
      }
      csync(c);
      // Quirk Q1 (SURVEY.md A.6): an accepted proposal rebinds sample_labels!'s LOCAL state; the remaining
      // proposals and the final scan (:477) run on that local object and the caller's labels are untouched this
      // iteration.  The scan's draws are independent of everything kept (structured stream), so it is skipped.
      if (acc) do_scan = false;
    }
    if (multi && c.sc->status == 0) {                        // back to the chain's own state
      if (c.sc->forked) {
        for (int t = tid; t < cap * cap; t += nt) { c.WD[t] = c.WDbak[t]; c.WL[t] = c.WLbak[t]; }
        for (int j = 0; j < n; ++j) {                        // the row sums follow every point back to its own slot
          const int from = c.lab[j], to = c.labbak[j];
          if (from != to) inc_update_S(c, j, from, to);
        }
        const unsigned m = c.inc->clk + 1;                       // cached per-slot terms: all stale
        csync(c);
        for (int s2 = tid; s2 < cap; s2 += nt) c.tchg[s2] = m;
        if (tid == 0) c.inc->clk = m;
        csync(c);
        for (int j = tid; j < n; j += nt) c.lab[j] = c.labbak[j];
        for (int s = tid; s < cap; s += nt) c.sizes[s] = c.szbak[s];
        if (tid == 0) c.sc->K = c.szbak[cap];
      }
      csync(c);
    }
    const long long ts0 = RC_CLOCK();
    if (do_scan) inc_full_scan(c, it, c.inc->dry_stop, false);         // (rows before dry_stop were scanned beside the restricted scans and stand)
    const long long ts1 = RC_CLOCK();
    if (tid == 0) st_add(c, ST_SCAN_TOTAL, ts1 - ts0);
    csync(c);
    if (c.sc->status == 0 && iter > kp.burnin && (iter - kp.burnin) % kp.thin == 0) {    // :546-554
      const long long j = (iter - kp.burnin) / kp.thin - 1;
      if (j < kp.numsamples) {
        record_labels(c, kp.out_labels + ((size_t)chain * kp.numsamples + j) * n);
        const double ll = loglik_cur(c);
        if (c.cwarp == 0) {
          const double lpv = logprior_eval(c);
          if (tid == 0) {
            const size_t o = (size_t)chain * kp.numsamples + j;
            kp.out_K[o] = c.sc->K; kp.out_r[o] = c.sc->r; kp.out_p[o] = c.sc->p;
            kp.out_ll[o] = ll; kp.out_lp[o] = ll + lpv;
          }
        }
        csync(c);
      }
    }
    if (tid == 0) { st_add(c, ST_RECORD, RC_CLOCK() - ts1); st_add(c, ST_ITER_TOTAL, RC_CLOCK() - ti0); }
  }
  csync(c);
  for (int j = tid; j < n; j += nt) kp.labels[(size_t)chain * n + j] = c.lab[j];
  for (int s = tid; s < cap; s += nt) { kp.sizes[(size_t)chain * cap + s] = c.sizes[s]; kp.epochs[(size_t)chain * (cap + 1) + s] = c.tchg[s]; }
  if (kp.tw_smem) for (int j = tid; j < n; j += nt) kp.Vv[(size_t)chain * n + j] = c.tw[j];
  if (tid == 0) kp.epochs[(size_t)chain * (cap + 1) + cap] = c.inc->clk;
  if (tid == 0) { kp.r[chain] = c.sc->r; kp.p[chain] = c.sc->p; kp.status[chain] = c.sc->status; }
}

// ---- incremental mode: S and W from scratch (first launch) ----------------------------------------------
// S[ch][t][x] = sum over columns j with label t of DL[x][j].  One CTA per row x at a time; every thread walks a
// contiguous strip of the row keeping a running sum while the label stays the same (one pair of shared-memory atomics
// per label run).  Zero entries are not written (S is zero-filled before).
__global__ void __launch_bounds__(256) k_init_S(const longlong2* __restrict__ DL, int n, const uint8_t* __restrict__ labels, int cap,
                                                longlong2* __restrict__ S, int nch) {
  extern __shared__ unsigned long long sbins[];          // [cap] D sums, [cap] L sums
  for (int t = threadIdx.x; t < 2 * cap; t += blockDim.x) sbins[t] = 0ull;
  __syncthreads();
  const int w = (n + blockDim.x - 1) / blockDim.x;
  const int j0 = threadIdx.x * w, j1 = min(n, j0 + w);
  for (int x = blockIdx.x; x < n; x += gridDim.x) {
    const longlong2* row = DL + (size_t)x * n;
    for (int ch = blockIdx.y; ch < nch; ch += gridDim.y) {
      const uint8_t* lab = labels + (size_t)ch * n;
      int cur = -1; long long d = 0, l = 0;
      for (int j = j0; j < j1; ++j) {
        const int lb = lab[j];
        if (lb != cur) {
          if (cur >= 0) { atomicAdd(&sbins[cur], (unsigned long long)d); atomicAdd(&sbins[cap + cur], (unsigned long long)l); }
          cur = lb; d = 0; l = 0;
        }
        const longlong2 v = row[j];
        d += v.x; l += v.y;
      }
      if (cur >= 0) { atomicAdd(&sbins[cur], (unsigned long long)d); atomicAdd(&sbins[cap + cur], (unsigned long long)l); }
      __syncthreads();
      longlong2* Sc = S + (size_t)ch * cap * n;
      for (int t = threadIdx.x; t < cap; t += blockDim.x) {
        const long long bd = (long long)sbins[t], bl = (long long)sbins[cap + t];
        sbins[t] = 0ull; sbins[cap + t] = 0ull;
        if (bd != 0 || bl != 0) Sc[(size_t)t * n + x] = make_longlong2(bd, bl);
      }
      __syncthreads();
    }
  }
}
__global__ void k_replicate_S(longlong2* __restrict__ S, size_t per_chain, int64_t nchains) {
  const size_t total = per_chain * (size_t)(nchains - 1);
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x)
    S[per_chain + t] = S[t % per_chain];
}
// W[ch][k][t] (k <= t) = sum over x with label k of S[ch][t][x]: the block sums loglik needs (mcmc.jl:1-56).
// One CTA per (slot t, chain); 128-bit totals by carry-propagating 64-bit atomics; W is zero-filled before.
__device__ __forceinline__ void atomic_add128g(rc_i128* a, const rc_i128& v) {
  const unsigned long long old = atomicAdd(&a->lo, v.lo);
  const long long hi = v.hi + ((old + v.lo) < old ? 1LL : 0LL);
  if (hi) atomicAdd(reinterpret_cast<unsigned long long*>(&a->hi), (unsigned long long)hi);
}
__global__ void __launch_bounds__(256) k_initw_from_S(const longlong2* __restrict__ S, int n, const uint8_t* __restrict__ labels,
                                                      const int* __restrict__ sizes, int cap, rc_i128* __restrict__ WD,
                                                      rc_i128* __restrict__ WL) {
  const int t = blockIdx.x, ch = blockIdx.y;
  if (sizes[(size_t)ch * cap + t] == 0) return;
  const uint8_t* lab = labels + (size_t)ch * n;
  const longlong2* St = S + ((size_t)ch * cap + t) * n;
  rc_i128* wd = WD + (size_t)ch * cap * cap;
  rc_i128* wl = WL + (size_t)ch * cap * cap;
  const int w = (n + blockDim.x - 1) / blockDim.x;
  const int x0 = threadIdx.x * w, x1 = min(n, x0 + w);
  int cur = -1;
  rc_i128 d, l; d.lo = 0; d.hi = 0; l.lo = 0; l.hi = 0;
  for (int x = x0; x < x1; ++x) {
    const int k = lab[x];
    if (k != cur) {
      if (cur >= 0 && cur <= t) { atomic_add128g(&wd[cur * cap + t], d); atomic_add128g(&wl[cur * cap + t], l); }
      cur = k; d.lo = 0; d.hi = 0; l.lo = 0; l.hi = 0;
    }
    const longlong2 v = St[x];
    rc_add128(d, v.x); rc_add128(l, v.y);
  }
  if (cur >= 0 && cur <= t) { atomic_add128g(&wd[cur * cap + t], d); atomic_add128g(&wl[cur * cap + t], l); }
}

// sample_rp (mcmc.jl:592-636): the (r, p)-only chain fitprior runs on the cluster sizes of its notional clustering
// (prior.jl:80).  One warp; update_r / update_p are the sampler's own (mcmc.jl:80-155); the initial r is drawn with
// SCALE sigma (mcmc.jl:617: rand(Gamma(eta, sigma)), where runsampler uses 1/sigma -- reproduced as written).
__global__ void __launch_bounds__(32) k_sample_rp(const __grid_constant__ rc_kparams kp, int* sizes, int K, double* terms, double* out_r,
                                                  double* out_p, uint8_t* out_acc) {
  __shared__ Scal sc;
  Ctx c;
  c.n = kp.n; c.cap = K; c.kp = &kp; c.sizes = sizes; c.sc = &sc; c.terms = terms;
  c.ctid = threadIdx.x; c.cwarp = 0; c.lane = threadIdx.x; c.nthr = 32; c.nwarp = 1; c.barid = 1;
  c.key = rc_chain_key(kp.seed, (unsigned long long)kp.chain_offset);
  if (threadIdx.x == 0) {
    const rc_params& P = kp.P;
    sc.r = rc_gamma_mt(P.eta, c.key, 0, RC_SITE_INIT, 2) * P.sigma;
    sc.p = rc_beta(P.u, P.v, c.key, 0);
    sc.K = K; sc.status = 0;
  }
  __syncwarp();
  long long j = 0;
  for (long long iter = 1; iter <= kp.numiters; ++iter) {
    const bool ra = update_r(c, (unsigned)iter);
    if (threadIdx.x == 0) {
      update_p(c, (unsigned)iter);
      if (out_acc) out_acc[iter - 1] = ra ? 1 : 0;
      if (iter > kp.burnin && (iter - kp.burnin) % kp.thin == 0 && j < kp.numsamples) { out_r[j] = sc.r; out_p[j] = sc.p; ++j; }
    }
    j = __shfl_sync(0xffffffffu, j, 0);
    __syncwarp();
  }
}

__global__ void k_tables(rc_params P, int n, double* LGA, double* LGZ, double* LOGN) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s <= n + 1; s += gridDim.x * blockDim.x) {
    const double sd = (double)s;
    LGA[s] = rc_lgamma(P.alpha + P.delta1 * sd);
    LGZ[s] = rc_lgamma(P.zeta + P.delta2 * sd);
    LOGN[s] = rc_log(sd);
  }
}

}  // namespace

size_t rc_sampler_inc_smem_bytes(int n, int cap, int mcap, int tw_smem) { return inc_layout(n, cap, mcap, tw_smem).total; }

// Incremental mode: (re)build S (and W) of every chain from the labels, then one launch of k_chain_inc.
int rc_launch_inc_init(const rc_kparams& kp, bool shared_labels, cudaStream_t st) {
  const size_t per = (size_t)kp.cap * kp.n;
  const size_t nS = shared_labels ? 1 : (size_t)kp.nchains;
  if (cudaMemsetAsync(kp.S, 0, sizeof(longlong2) * per * nS, st) != cudaSuccess) return 1;
  if (cudaMemsetAsync(kp.WD, 0, sizeof(rc_i128) * (size_t)kp.cap * kp.cap * kp.nchains, st) != cudaSuccess) return 1;
  if (cudaMemsetAsync(kp.WL, 0, sizeof(rc_i128) * (size_t)kp.cap * kp.cap * kp.nchains, st) != cudaSuccess) return 1;
  const int gy = (int)std::min<size_t>(nS, 64);
  const int gx = std::max(1, std::min(kp.n, (148 * 8 + gy - 1) / gy));
  k_init_S<<<dim3(gx, gy), 256, sizeof(unsigned long long) * 2 * kp.cap, st>>>(kp.DL, kp.n, kp.labels, kp.cap, kp.S, (int)nS);
  if (shared_labels && kp.nchains > 1) k_replicate_S<<<148 * 8, 256, 0, st>>>(kp.S, per, kp.nchains);
  k_initw_from_S<<<dim3(kp.cap, kp.nchains), 256, 0, st>>>(kp.S, kp.n, kp.labels, kp.sizes, kp.cap, kp.WD, kp.WL);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
// Self-check of the incrementally maintained sums (compute-sanitizer is not available on the target pool, so the
// invariant is checked directly): rebuild S and W of every chain from its labels into scratch and count the entries
// that differ from the maintained ones.  Exact integers: any lost or doubled update shows up as a mismatch.
__global__ void k_count_diff(const unsigned long long* __restrict__ a, const unsigned long long* __restrict__ b, size_t words,
                             unsigned long long* __restrict__ ndiff) {
  unsigned long long local = 0;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < words; t += (size_t)gridDim.x * blockDim.x) local += a[t] != b[t];
  if (local) atomicAdd(ndiff, local);
}
int rc_inc_check(const rc_kparams& kp, long long* mismatches_S, long long* mismatches_W, cudaStream_t st) {
  const size_t per = (size_t)kp.cap * kp.n, perW = (size_t)kp.cap * kp.cap;
  longlong2* S2 = nullptr; rc_i128 *WD2 = nullptr, *WL2 = nullptr; unsigned long long* nd = nullptr;
  if (cudaMalloc(&S2, sizeof(longlong2) * per * kp.nchains) != cudaSuccess || cudaMalloc(&WD2, sizeof(rc_i128) * perW * kp.nchains) != cudaSuccess ||
      cudaMalloc(&WL2, sizeof(rc_i128) * perW * kp.nchains) != cudaSuccess || cudaMalloc(&nd, 2 * sizeof(unsigned long long)) != cudaSuccess) {
    cudaFree(S2); cudaFree(WD2); cudaFree(WL2); cudaFree(nd); return 1;
  }
  rc_kparams k2 = kp;
  k2.S = S2; k2.WD = WD2; k2.WL = WL2;
  int rc = rc_launch_inc_init(k2, false, st);
  cudaMemsetAsync(nd, 0, 2 * sizeof(unsigned long long), st);
  // W: only the entries (k <= t) of live slots are maintained / rebuilt; dead slots hold zeros in both
  k_count_diff<<<1024, 256, 0, st>>>((const unsigned long long*)kp.S, (const unsigned long long*)S2, per * kp.nchains * 2, nd);
  k_count_diff<<<256, 256, 0, st>>>((const unsigned long long*)kp.WD, (const unsigned long long*)WD2, perW * kp.nchains * 2, nd + 1);
  k_count_diff<<<256, 256, 0, st>>>((const unsigned long long*)kp.WL, (const unsigned long long*)WL2, perW * kp.nchains * 2, nd + 1);
  unsigned long long h[2] = {0, 0};
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaMemcpy(h, nd, sizeof(h), cudaMemcpyDeviceToHost) != cudaSuccess) rc = 1;
  cudaFree(S2); cudaFree(WD2); cudaFree(WL2); cudaFree(nd);
  *mismatches_S = (long long)h[0]; *mismatches_W = (long long)h[1];
  return rc;
}

void rc_launch_chain_inc(const rc_kparams& kp, size_t smem, int nthr, cudaStream_t st) {
  cudaFuncSetAttribute(k_chain_inc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k_chain_inc<<<kp.nchains, nthr, smem, st>>>(kp);
}

void rc_launch_sample_rp(const rc_kparams& kp, int* sizes, int K, double* terms, double* out_r, double* out_p, uint8_t* out_acc, cudaStream_t st) {
  k_sample_rp<<<1, 32, 0, st>>>(kp, sizes, K, terms, out_r, out_p, out_acc);
}

void rc_launch_tables(const rc_params& P, int n, double* LGA, double* LGZ, double* LOGN, cudaStream_t st) {
  k_tables<<<(n + 2 + 255) / 256, 256, 0, st>>>(P, n, LGA, LGZ, LOGN);
}