/* rcb200.h -- C ABI of librcb200.so: the B200-native sampler hot path of RedClust.
 *
 * The reference (RedClust.jl v1.2.2) is pure Julia and has NO FFI/plugin boundary
 * (SURVEY.md section 8b); the drop-in boundary is its exported Julia API
 * (/root/reference/src/RedClust.jl:32-66).  This header is what a `ccall`-based Julia host
 * (redclust.jl_b200/julia/RedClustB200.jl) or the Python ctypes mirror
 * (redclust.jl_b200/host.py) binds.  Each entry point cites the reference code it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative rc_status otherwise; rc_last_error()
 *     returns a thread-local message (the host wrapper turns it into ErrorException /
 *     ArgumentError exactly where the reference throws, src/types.jl:40-54,149-153).
 *   - matrices are dense fp64; D is symmetric so row-/column-major are the same bytes.
 *   - labels crossing the ABI are 1-based int64 (Julia `Vector{Int}`), Bool vectors are 1 byte.
 *   - the caller owns every host buffer; the library keeps no host pointer after returning.
 *   - handles are opaque, bound to one CUDA device, and not thread-safe per handle.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     RC_ERR_CUDA.
 */
#ifndef RCB200_H
#define RCB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCB200_VERSION 100 /* 0.1.0 */

typedef enum rc_status {
  RC_OK = 0,
  RC_ERR_ARG = -1,       /* invalid argument (null pointer, bad size, bad option)          */
  RC_ERR_CUDA = -2,      /* CUDA runtime failure / no device                               */
  RC_ERR_NOTSYM = -3,    /* "D must be symmetric."              (src/types.jl:149-151)     */
  RC_ERR_DOMAIN = -4,    /* non-finite entry or non-positive off-diagonal dissimilarity    */
  RC_ERR_SLOTS = -5,     /* a chain needed more live cluster slots than the slot capacity  */
  RC_ERR_STATE = -6      /* handle used out of order                                        */
} rc_status;

/* MCMCOptionsList, src/types.jl:26-58 (numsamples is derived: floor((numiters-burnin)/thin)). */
typedef struct rc_options {
  int64_t numiters, burnin, thin, numGibbs, numMH;
} rc_options;

/* PriorHyperparamsList, src/types.jl:93-108. */
typedef struct rc_params {
  double delta1, delta2, alpha, beta, zeta, gamma, eta, sigma, proposalsd_r, u, v;
  int64_t K_initial;
  int64_t maxK;
  int32_t repulsion;
  int32_t _pad;
} rc_params;

typedef struct rc_data rc_data;       /* MCMCData: device-resident D / log D   (src/types.jl:145-162) */
typedef struct rc_sampler rc_sampler; /* chains' MCMCState + MCMCResult traces (src/types.jl:131-137,193-248) */

int32_t rc_version(void);
const char* rc_last_error(void);
int32_t rc_device_count(void);

/* ---- MCMCData -------------------------------------------------------------------------- */
/* MCMCData(D): src/types.jl:148-156.  Validates squareness/symmetry, builds
 * logD = log.(D - Diagonal(D) + I) and the fixed-point images the kernels stream.            */
int32_t rc_data_from_dist(const double* D, int64_t n, int32_t device, rc_data** out);
/* MCMCData(points): src/types.jl:159-162 = pairwise(Euclidean(), X, dims=2) with X dim x n
 * column-major (point i = X[i*dim .. i*dim+dim-1]); also src/utils.jl:144-145, src/prior.jl:51,180. */
int32_t rc_data_from_points(const double* X, int64_t dim, int64_t n, int32_t device, rc_data** out);
/* Multi-GPU distance build (row blocks + all-gather): rows [row0, row0 + nrows) of pairwise(Euclidean(), X) into a
 * caller DEVICE buffer of nrows x n fp64, bit-equal to the same rows of rc_data_from_points' matrix; and MCMCData(D)
 * from a complete matrix that already lives on the device (src/types.jl:148-162 across GPUs). */
int32_t rc_distm_rows_dev(const double* X, int64_t dim, int64_t n, int64_t row0, int64_t nrows, int32_t device, void* D_rows_dev);
int32_t rc_data_from_dist_dev(const void* D_dev, int64_t n, int32_t device, rc_data** out);
/* The oracle co-clustering matrix of generatemixture (src/utils.jl:130-143) for given points and Dirichlet draws:
 * out[i][j] = (1 / numiters) sum_t (P_t' P_t)[i][j], P_t[k][i] = W[t][k] N(x_i; radius e_k, sigma^2 I) normalised over k.
 * X: n x dim row-major, W: numiters x K, out: n x n, all host fp64.  The stacked posteriors of a chunk of draws form one
 * Gram product on the FP64 tensor cores (the kernel of the distance build).                                          */
int32_t rc_oracle_coclustering(const double* X, int64_t dim, int64_t n, int64_t K, double radius, double sigma, const double* W,
                               int64_t numiters, int32_t device, double* out);
int64_t rc_data_n(const rc_data* d);
/* data.D and data.logD back to the host as n x n fp64. */
int32_t rc_data_copy_dist(const rc_data* d, double* D_out);
int32_t rc_data_copy_logdist(const rc_data* d, double* logD_out);
/* Fixed-point scales of the images the sampler streams: Dq = round(D * 2^qD), Lq = round(logD * 2^qL)
 * (largest q <= 50 with n * max|.| * 2^q < 2^61, so that every cluster sum is an exact 64-bit integer). */
int32_t rc_data_scales(const rc_data* d, int32_t* qD, int32_t* qL);
/* One row of data.D (the k-medoids++ seeding of the host draws its weights from medoid rows). */
int32_t rc_data_copy_row(const rc_data* d, int64_t i, double* row_out);

/* ---- the O(n^2) parts of fitprior (src/prior.jl:22-128) on the device-resident matrix ---------------
 * rc_kmedoids: Clustering.kmedoids(dissM, k; maxiter) as called at src/prior.jl:55-71 (elbow scan and notional
 * clustering) and src/mcmc.jl:519-527 (default init of runsampler): alternate nearest-medoid assignment (first
 * minimum) and medoid update (member with the smallest sum of dissimilarities to its cluster, lowest index on
 * ties) from the given initial medoids (0-based) until nothing changes or maxiter updates were made.  The sums
 * run over the fixed-point image Dq, so ties and near-ties resolve identically on every machine.
 * assignments: n, 1-based cluster ids; medoids: k, 0-based; totalcost = sum_i D[medoid(i)][i].
 * rc_pair_stats: per row i the exact sums over j > i of (Dq, Lq) within i's cluster and over all j > i, and the
 * number of within pairs -- rows_out is n x 5 int64 {within Dq, within Lq, all Dq, all Lq, within count}.  Their
 * totals are the sufficient statistics of the Gamma fits to A and B (src/prior.jl:73-110). */
int32_t rc_kmedoids(const rc_data* d, int64_t k, const int64_t* init_medoids, int64_t maxiter, int64_t* assignments,
                    int64_t* medoids, double* totalcost, int32_t* converged, int64_t* iterations);
/* rc_kmedoids_seed: Clustering.jl's default seeding of kmedoids (:kmpp on the costs) on the resident matrix, driven by k
 * uniforms: u01[0] picks the first medoid uniformly, u01[t] the t-th in proportion to the dissimilarity to the nearest
 * medoid so far.  medoids_out: k, 0-based -- the init_medoids of rc_kmedoids.                                        */
int32_t rc_kmedoids_seed(const rc_data* d, int64_t k, const double* u01, int64_t* medoids_out);
int32_t rc_pair_stats(const rc_data* d, const int64_t* labels, int64_t* rows_out);
/* rc_kmeans: Clustering.kmeans(x, k; maxiter) as called at src/prior.jl:63-69 (algo = "k-means": elbow scan and notional
 * clustering on the points).  X: n x dim row-major host points.  Seeding: the k points init_idx (0-based) when given, else
 * k-means++ driven by the k uniforms u01 (u01[0] picks the first centre uniformly, u01[t] the t-th in proportion to the
 * squared distance to the nearest centre so far).  Lloyd iterations (nearest centre, first minimum on ties; centre = mean
 * of its members, an empty cluster keeps its centre) until no label changes or the objective moves by less than tol
 * (Clustering.jl's criterion; its default tol is 1e-6) or maxiter updates were made.  All sums run in a fixed order: the
 * result is a function of the arguments alone.  assignments: n, 1-based; centers (may be NULL): k x dim row-major;
 * totalcost = sum of squared distances to the assigned centres.                                                       */
int32_t rc_kmeans(const double* X, int64_t n, int64_t dim, int64_t k, const int64_t* init_idx, const double* u01, int64_t maxiter,
                  double tol, int32_t device, int64_t* assignments, double* centers, double* totalcost, int32_t* converged,
                  int64_t* iterations);
/* sample_rp(clustsizes, options, params): src/mcmc.jl:592-636, called by fitprior at src/prior.jl:80 -- the (r, p)-only
 * chain on fixed cluster sizes (sample_r / sample_p of src/mcmc.jl:94-155; initial r ~ Gamma(eta, scale sigma) as
 * written at :617).  r_out / p_out: numsamples values; r_acc_out (numiters bytes) may be NULL.                      */
int32_t rc_sample_rp(const int64_t* clustsizes, int64_t nsizes, const rc_options* opt, const rc_params* par, uint64_t seed,
                     int32_t device, double* r_out, double* p_out, uint8_t* r_acc_out);
void rc_data_destroy(rc_data* d);

/* ---- runsampler ------------------------------------------------------------------------ */
/* r ~ Gamma(eta, 1/sigma), p ~ Beta(u, v): src/mcmc.jl:524-525, drawn on the structured stream. */
int32_t rc_init_rp(const rc_params* params, uint64_t seed, int64_t chain_id, double* r, double* p);

/* Allocate `nchains` independent chains (global chain ids chain_offset .. chain_offset+nchains-1)
 * on the data's device.  init_labels: nchains x n, 1-based, any slot ids in 1..n (src/types.jl:131-137);
 * init_r / init_p: nchains values.  slot_cap: max simultaneously live clusters per chain
 * (0 = default = 128, at most 255) -- the reference allows up to n (SURVEY.md H4); initial labels must lie in
 * 1..slot_cap (relabel with sortlabels first).             */
int32_t rc_sampler_create(const rc_data* d, const rc_options* opt, const rc_params* par,
                          int64_t nchains, int64_t chain_offset, const int64_t* init_labels,
                          const double* init_r, const double* init_p, uint64_t seed,
                          int32_t slot_cap, rc_sampler** out);
/* Advance every chain by `iters` iterations of the loop at src/mcmc.jl:537-555
 * (iters < 0: run to numiters).  One persistent kernel launch per call, or one per launch group when the chains'
 * row sums do not all fit the device (each group rebuilds them from its labels first; same results).          */
int32_t rc_sampler_run(rc_sampler* s, int64_t iters);
/* Seconds of device time (CUDA events) spent in rc_sampler_run so far, and iterations done:
 * MCMCResult.runtime / mean_iter_time, src/mcmc.jl:536,586-587.                                */
int32_t rc_sampler_progress(const rc_sampler* s, int64_t* iters_done, double* device_seconds);
int64_t rc_sampler_numsamples(const rc_sampler* s);
int64_t rc_sampler_n(const rc_sampler* s);
int64_t rc_sampler_nchains(const rc_sampler* s);
/* Recorded samples of one chain (src/mcmc.jl:546-554): labels numsamples x n (sortlabels'd,
 * 1-based), K, r, p, loglik, logposterior.  Any pointer may be NULL.                          */
int32_t rc_sampler_copy_samples(const rc_sampler* s, int64_t chain, int64_t* labels, int64_t* K,
                                double* r, double* p, double* loglik, double* logposterior);
/* The same for EVERY chain in one call (labels nchains x numsamples x n, traces nchains x numsamples, acceptances
 * nchains x numiters [x numMH]): one device-to-host copy per array, labels widened by all host threads.            */
int32_t rc_sampler_copy_all(const rc_sampler* s, int64_t* labels, int64_t* K, double* r, double* p, double* loglik,
                            double* logposterior, uint8_t* r_acc, uint8_t* sm_acc, uint8_t* sm_split);
/* r_acceptances (numiters), splitmerge_acceptances / splitmerge_splits (numiters*numMH):
 * src/mcmc.jl:538-543.                                                                         */
int32_t rc_sampler_copy_acceptances(const rc_sampler* s, int64_t chain, uint8_t* r_acc,
                                    uint8_t* sm_acc, uint8_t* sm_split);
/* Current MCMCState of one chain: labels (n, 1-based slot ids), r, p -- the `init` argument of
 * a resumed run (src/mcmc.jl:504,519-529).                                                     */
int32_t rc_sampler_copy_state(const rc_sampler* s, int64_t chain, int64_t* labels, double* r, double* p);
/* Profiling aid (no reference equivalent): 16 SM-cycle counters per chain accumulated by the chain kernel.
 * out: nchains x 16 int64.  Only librcb200_stats.so carries the clock reads; the default library returns the
 * move / rebuild counts, zeros for the cycle slots, and two counts of the incremental kernel's exact shortcuts: slot 4 the
 * rows decided by their stored summaries, slot 0 the merge proposals rejected by their acceptance bound. */
int32_t rc_sampler_copy_stats(const rc_sampler* s, int64_t* out);
/* Per-chain status after a run: 0 ok, RC_ERR_SLOTS if the chain needed more than slot_cap simultaneously live
 * clusters and stopped there (the reference allows up to n, src/types.jl:135, src/mcmc.jl:199; see INTEGRATION.md).
 * rc_sampler_run fails with RC_ERR_SLOTS only when EVERY chain stopped; otherwise the healthy chains' results are
 * valid and rc_sampler_overflowed tells how many chains to skip.                                 */
int32_t rc_sampler_chain_status(const rc_sampler* s, int64_t chain);
int64_t rc_sampler_overflowed(const rc_sampler* s);
/* Diagnostic (no reference equivalent): the sampler keeps, per chain, the sums of every row of D / log D by cluster and
 * the cluster-by-cluster block sums incrementally (exact integers).  This rebuilds both from the current labels and
 * counts the 64-bit words that differ -- 0 / 0 unless an update was lost; -1 / -1 before the first run.  With launch
 * groups only the chains of the group launched last still have their row sums: those are checked.                */
int32_t rc_sampler_check_sums(const rc_sampler* s, int64_t* mismatches_S, int64_t* mismatches_W);
/* Posterior co-clustering counts of the device-resident samples of chains [chain0, chain0+nch):
 * sum(adjacencymatrix.(clusts)) (src/mcmc.jl:560, src/utils.jl:59-63) as exact int32 counts in a
 * DEVICE buffer of n*n int32 (e.g. a torch tensor's data_ptr, so the caller can all-reduce it
 * over NCCL before dividing).                                                                  */
int32_t rc_sampler_psm_counts_dev(const rc_sampler* s, int64_t chain0, int64_t nch, void* counts_dev);
/* Same, divided by the number of samples, into a host n x n fp64 matrix.                       */
int32_t rc_sampler_psm(const rc_sampler* s, int64_t chain0, int64_t nch, double* psm_out);
void rc_sampler_destroy(rc_sampler* s);

/* ---- posterior predictive allocation of new observations (no reference equivalent) -------------------------------------
 * For new point x (row x of Dnew, m x n: dissimilarities to the training points in data order, finite and > 0) and sample s,
 * P_s(x, k) is the full Gibbs scan's conditional for x as point n + 1 of the augmented data in state (labels_s, r_s, p_s)
 * (src/mcmc.jl:193-247) normalised as sample_logweights draws from it (src/utils.jl:2-6): candidates are the slots 1..K_s
 * of sortlabels(labels_s) and, when maxK == 0 or K_s < maxK, the new slot K_s + 1.  Outputs (host):
 *   cocl_out[x][j] = (1/S) sum_s P_s(x, c_s(j))   (m x n),   newcl_out[x] = (1/S) sum_s P_s(x, K_s + 1)   (m)
 * summed in ascending sample order; S = 0 gives NaN.  lp_out (NULL or S x m x 256) receives the un-normalised
 * log-probabilities of the candidates, slot k at index k - 1, NaN beyond the last candidate.  More than 255 clusters in a
 * sample: RC_ERR_SLOTS; r <= 0 or p outside (0, 1): RC_ERR_ARG; a bad entry of Dnew: RC_ERR_DOMAIN.                     */
int32_t rc_predict(const rc_data* d, const rc_params* par, const double* Dnew, int64_t m, const int64_t* labels, const double* r,
                   const double* p, int64_t S, double* cocl_out, double* newcl_out, double* lp_out);
/* The same over the device-resident recorded samples of chains [chain0, chain0 + nch) (chain-major, sample-minor) with the
 * sampler's hyperparameters (src/mcmc.jl:193-247, src/utils.jl:2-6).  Needs a run to numiters (RC_ERR_STATE before: the
 * samples are not all recorded) and chains that did not stop at the slot capacity (RC_ERR_SLOTS).                        */
int32_t rc_sampler_predict(const rc_sampler* s, const double* Dnew, int64_t m, int64_t chain0, int64_t nch, double* cocl_out,
                           double* newcl_out);
/* Dissimilarities of new points Y (m x dim) to training points X (n x dim), both row-major host fp64, into out (m x n):
 * bit-equal to rows n.., columns ..n of rc_data_from_points on the stacked points (the rows of rc_distm_rows_dev). */
int32_t rc_crossdist(const double* X, int64_t n, const double* Y, int64_t m, int64_t dim, int32_t device, double* out);

/* ---- stand-alone pieces ------------------------------------------------------------------ */
/* loglik(data, state, params) and logprior(state, params) for one host label vector:
 * src/mcmc.jl:1-78.                                                                            */
int32_t rc_loglik(const rc_data* d, const rc_params* par, const int64_t* labels, double* out);
/* PSM of host label vectors (S x n, any positive labels): src/mcmc.jl:560.                    */
int32_t rc_psm(const int64_t* labels, int64_t S, int64_t n, int32_t device, double* psm_out);
/* The same counts (not divided) for S host label vectors into a caller DEVICE buffer of n x n int32: one rank's share
 * of a PSM whose samples are sharded over GPUs; all-reduce(SUM) the buffers, divide by the global sample count. */
int32_t rc_psm_counts_dev(const int64_t* labels, int64_t S, int64_t n, int32_t device, void* counts_dev);
/* MPEL search of getpointestimate (src/pointestimate.jl:34-59): loss_sums[i] = sum_j loss(c_i,c_j),
 * *best = first argmin (0-based).  loss: 0 binder (Mirkin), 1 omARI, 2 VI, 3 ID (un-normalised). */
int32_t rc_mpel(const int64_t* labels, int64_t S, int64_t n, int32_t loss, int32_t device,
                double* loss_sums, int64_t* best);
/* Multi-GPU MPEL (candidates sharded over GPUs): rows row_first, row_first + row_stride, ... (nrows of them) of the
 * strict upper triangle of the pairwise loss matrix into a caller DEVICE buffer (nrows x S fp64); after an
 * all-gather of the blocks into the S x S upper triangle, rc_mpel_finish_dev sums the columns in ascending row
 * order and returns the first argmin -- bit-equal to rc_mpel on one GPU (src/pointestimate.jl:34-59). */
int32_t rc_mpel_rows_dev(const int64_t* labels, int64_t S, int64_t n, int32_t loss, int32_t device, int64_t row_first,
                         int64_t row_stride, int64_t nrows, void* M_rows_dev);
int32_t rc_mpel_finish_dev(const void* M_upper_dev, int64_t S, int32_t device, double* loss_sums, int64_t* best);
/* MPEL with the Binder loss over pooled samples, from the co-clustering counts N alone (src/pointestimate.jl:34-59,68-76,
 * counts of src/mcmc.jl:560): with P_s = sum_k C(n_k, 2) and W_s = sum_{a<b} N_ab [c_s(a) == c_s(b)], the disagreeing pairs
 * of sample s summed over every sample t are T_s = S P_s + sum_t P_t - 2 W_s, an exact integer.  loss_sums[s] = T_s / C(n, 2)
 * (rc_mpel's binder column sums up to its fp64 rounding), *best = first argmin of T (0-based), totals[s] = T_s.  O(S n^2)
 * work and no S x S matrix.  Needs 1 <= S < 2^31 and n <= 65 535.  loss_sums, best and totals may each be NULL.       */
int32_t rc_binder_mpel(const int64_t* labels, int64_t S, int64_t n, int32_t device, double* loss_sums, int64_t* best, int64_t* totals);
/* The same over the device-resident samples of chains [chain0, chain0 + nch) (chain-major, sample-minor: *best indexes
 * them in that order); nothing is copied to the host.  RC_ERR_STATE before a run to numiters, RC_ERR_SLOTS when a chain
 * of the range stopped at the slot capacity, RC_ERR_ARG for a bad range.                                                */
int32_t rc_sampler_binder_mpel(const rc_sampler* s, int64_t chain0, int64_t nch, double* loss_sums, int64_t* best, int64_t* totals);

/* ---- multi-GPU exchange steps (SURVEY.md 8e) -------------------------------------------------------
 * One process per GPU.  The sampler needs no collective (independent chains: chain_offset above).  The three steps
 * that exchange data run over an NCCL communicator owned by an rc_comm handle: rank 0 calls rc_comm_unique_id, the
 * launcher (torch.distributed, MPI, Julia Distributed, ...) hands the 128 bytes to every rank, every rank calls
 * rc_comm_init.  NCCL is resolved at run time (libnccl.so.2), so the library loads without it.
 *   rc_comm_data_from_points  MCMCData(points), src/types.jl:159-162: row blocks of pairwise(Euclidean()) + all-gather
 *   rc_comm_sampler_psm       src/mcmc.jl:560 over the chains of every rank: int32 counts + ONE all-reduce + divide
 *   rc_comm_psm               the same for host label vectors sharded over the ranks (S_local of them on this rank)
 *   rc_comm_mpel              src/pointestimate.jl:49-57 with the candidate rows dealt cyclically + all-gather
 *   rc_comm_sampler_binder_mpel  src/pointestimate.jl:34-59,68-76 over the chains of every rank (src/mcmc.jl:560): the
 *                             all-reduced counts, per-rank int64 W and P, ONE all-gather; every rank gets T over all
 *                             samples in rank order (= global chain order; *best indexes that concatenation)
 * psm_out (host, n x n fp64) and counts_dev_out (device, n x n int32) may each be NULL.  Results are bit-equal to the
 * single-GPU entry points.                                                                              */
typedef struct rc_comm rc_comm;
int32_t rc_comm_unique_id(uint8_t* id128);
int32_t rc_comm_init(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, rc_comm** out);
int32_t rc_comm_info(const rc_comm* c, int32_t* rank, int32_t* world);
void rc_comm_destroy(rc_comm* c);
int32_t rc_comm_allreduce_i32(rc_comm* c, void* buf_dev, int64_t count);
int32_t rc_comm_data_from_points(rc_comm* c, const double* X, int64_t dim, int64_t n, rc_data** out);
int32_t rc_comm_sampler_psm(rc_comm* c, const rc_sampler* s, double* psm_out, void* counts_dev_out);
int32_t rc_comm_psm(rc_comm* c, const int64_t* labels, int64_t S_local, int64_t n, double* psm_out, void* counts_dev_out);
int32_t rc_comm_mpel(rc_comm* c, const int64_t* labels, int64_t S, int64_t n, int32_t loss, double* loss_sums, int64_t* best);
int32_t rc_comm_sampler_binder_mpel(rc_comm* c, const rc_sampler* s, double* loss_sums, int64_t* best, int64_t* totals);

#ifdef __cplusplus
}
#endif
#endif /* RCB200_H */
