"""Host-side mirror of RedClust.jl's public API for the sampler hot path (the reference is pure Julia and
Julia is not installed in this image, so -- as the task allows -- the host side above the C ABI is written
in Python; julia/RedClustB200.jl is the `ccall` twin of this file).

Names, argument meaning and error behaviour follow the reference:
  MCMCOptionsList        /root/reference/src/types.jl:26-58
  PriorHyperparamsList   /root/reference/src/types.jl:93-108
  MCMCData               /root/reference/src/types.jl:145-162
  MCMCResult             /root/reference/src/types.jl:193-248
  runsampler             /root/reference/src/mcmc.jl:501-590
  getpointestimate       /root/reference/src/pointestimate.jl:17-60
  binderloss / infodist  /root/reference/src/pointestimate.jl:68-98
  adjacencymatrix / sortlabels / makematrix / generatemixture   /root/reference/src/utils.jl:59-156

All heavy work happens in librcb200.so on the GPU.  Nothing here falls back to the CPU: without the
library or a device the calls raise.  The extra keyword arguments (`nchains`, `seed`, `device`,
`slot_cap`) are additions the reference has no equivalent for (it runs one chain per call on the
task-local RNG)."""
import ctypes as C
import math
import time
import os

import numpy as np

from . import _lib
from ._lib import RCError, rc_options, rc_params, rc_rhat_summary, check, ptr, lib


class ArgumentError(ValueError):
    """Julia's ArgumentError."""


# ------------------------------------------------------------------------------------------------
class MCMCOptionsList:
    def __init__(self, numiters=5000, burnin=None, thin=1, numGibbs=5, numMH=1):
        if burnin is None:
            burnin = int(math.floor(0.2 * numiters))
        for name, v in (("numiters", numiters), ("burnin", burnin), ("thin", thin), ("numGibbs", numGibbs), ("numMH", numMH)):
            if not isinstance(v, (int, np.integer)):
                raise TypeError(f"{name} must be an integer")
        if numiters < 1:
            raise RCError(_lib.RC_ERR_ARG, "numiters must be ≥ 1.")
        if burnin > numiters:
            raise RCError(_lib.RC_ERR_ARG, "burnin must be < numiters")
        if thin < 1:
            raise RCError(_lib.RC_ERR_ARG, "thin must be positive.")
        if numGibbs < 0:
            raise RCError(_lib.RC_ERR_ARG, "numGibbs must be non-negative.")
        if numMH < 0:
            raise RCError(_lib.RC_ERR_ARG, "numMH must be non-negative.")
        self.numiters, self.burnin, self.thin, self.numGibbs, self.numMH = int(numiters), int(burnin), int(thin), int(numGibbs), int(numMH)
        self.numsamples = int(math.floor((numiters - burnin) / thin))

    def _c(self):
        return rc_options(self.numiters, self.burnin, self.thin, self.numGibbs, self.numMH)

    def __repr__(self):
        return (f"MCMC Options: {self.numiters} iterations, {self.burnin} burnin, {self.numsamples} samples, "
                f"{self.numGibbs} restricted Gibbs steps per split-merge, {self.numMH} split-merge steps per iteration")


class PriorHyperparamsList:
    _fields = ("delta1", "alpha", "beta", "delta2", "zeta", "gamma", "eta", "sigma", "proposalsd_r", "u", "v",
               "K_initial", "repulsion", "maxK")
    _greek = {"δ1": "delta1", "δ2": "delta2", "α": "alpha", "β": "beta", "ζ": "zeta", "γ": "gamma", "η": "eta", "σ": "sigma"}

    def __init__(self, **kw):
        kw = {self._greek.get(k, k): v for k, v in kw.items()}
        d = dict(delta1=1.0, alpha=1.0, beta=1.0, delta2=1.0, zeta=1.0, gamma=1.0, eta=1.0, sigma=1.0,
                 proposalsd_r=None, u=1.0, v=1.0, K_initial=1, repulsion=True, maxK=0)
        for k in kw:
            if k not in d:
                raise TypeError(f"unknown hyperparameter {k}")
        d.update(kw)
        if d["proposalsd_r"] is None:
            d["proposalsd_r"] = math.sqrt(d["eta"]) / d["sigma"]      # types.jl:102
        for k, v in d.items():
            setattr(self, k, v)

    def _c(self):
        return rc_params(float(self.delta1), float(self.delta2), float(self.alpha), float(self.beta), float(self.zeta),
                         float(self.gamma), float(self.eta), float(self.sigma), float(self.proposalsd_r), float(self.u),
                         float(self.v), int(self.K_initial), int(self.maxK), int(bool(self.repulsion)), 0)

    def __repr__(self):
        return "PriorHyperparamsList(" + ", ".join(f"{k}={getattr(self, k)!r}" for k in self._fields) + ")"


class Comm:
    """The NCCL communicator of the three exchange steps (rc_comm_* of include/rcb200.h): one per process, one process
    per GPU.  torch.distributed (or anything else) is only the launcher that hands rank 0's 128-byte id to the others."""

    _cache = {}

    def __init__(self, unique_id, rank, world, device):
        self._h = C.c_void_p()
        self.rank, self.world, self.device, self.group = rank, world, device, None
        idb = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
        check(lib().rc_comm_init(ptr(idb), rank, world, device, C.byref(self._h)))

    @staticmethod
    def unique_id():
        idb = np.zeros(128, np.uint8)
        check(lib().rc_comm_unique_id(ptr(idb)))
        return idb.tobytes()

    @classmethod
    def from_torch(cls, group=None, device=None):
        """Communicator over the ranks of a torch.distributed process group (cached per group and device); a world of
        one without an initialised process group."""
        import torch
        import torch.distributed as dist
        dev = torch.cuda.current_device() if device is None else device
        key = (id(group), dev)
        if key in cls._cache:
            return cls._cache[key]
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(group), dist.get_world_size(group)
            box = [cls.unique_id() if rank == 0 else None]
            src = dist.get_global_rank(group, 0) if group is not None else 0
            dist.broadcast_object_list(box, src=src, group=group)
            c = cls(box[0], rank, world, dev)
            c.group = group
        else:
            c = cls(cls.unique_id(), 0, 1, dev)
        cls._cache[key] = c
        return c

    def all_ranks(self, obj):
        """obj of every rank in rank order, exchanged over the torch.distributed group of from_torch ([obj] in a world of
        one)."""
        if self.world == 1:
            return [obj]
        import torch.distributed as dist
        out = [None] * self.world
        dist.all_gather_object(out, obj, group=self.group)
        return out

    def close(self):
        L = getattr(_lib, "_lib", None)
        if getattr(self, "_h", None) and L is not None:
            L.rc_comm_destroy(self._h)
            self._h = None


class MCMCData:
    """Device-resident dissimilarity matrix (D, log D and their fixed-point images)."""

    def __init__(self, data, device=0):
        self._h = C.c_void_p()
        self.device = device
        if isinstance(data, np.ndarray) and data.ndim == 2 and data.dtype == np.float64 and not getattr(data, "_rc_points", False):
            D = data
            if D.shape[0] != D.shape[1]:
                raise RCError(_lib.RC_ERR_ARG, "D must be a square matrix.")
            D = np.ascontiguousarray(D)
            check(lib().rc_data_from_dist(ptr(D), D.shape[0], device, C.byref(self._h)))
        else:
            X = makematrix(data)                      # dim x n, as the reference
            Xt = np.ascontiguousarray(X.T)            # point-major for the kernel
            check(lib().rc_data_from_points(ptr(Xt), Xt.shape[1], Xt.shape[0], device, C.byref(self._h)))
        self.n = int(lib().rc_data_n(self._h))

    @classmethod
    def from_points(cls, points, device=0):
        """MCMCData(points): points is a sequence of n observation vectors (or an n x dim array)."""
        obj = cls.__new__(cls)
        obj._h = C.c_void_p()
        obj.device = device
        P = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
        check(lib().rc_data_from_points(ptr(P), P.shape[1], P.shape[0], device, C.byref(obj._h)))
        obj.n = int(lib().rc_data_n(obj._h))
        return obj

    @classmethod
    def from_points_sharded(cls, points, group=None, device=None, comm=None):
        """MCMCData(points) with the distance build split over the ranks (SURVEY 8e): rank r computes a block of rows,
        one ncclAllGather gives every GPU the whole matrix, which stays on the device (rc_comm_data_from_points).
        Bit-equal to from_points on one GPU."""
        comm = comm or Comm.from_torch(group, device)
        P = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
        obj = cls.__new__(cls)
        obj._h = C.c_void_p()
        obj.device = comm.device
        check(lib().rc_comm_data_from_points(comm._h, ptr(P), P.shape[1], P.shape[0], C.byref(obj._h)))
        obj.n = int(lib().rc_data_n(obj._h))
        return obj

    @property
    def D(self):
        out = np.empty((self.n, self.n))
        check(lib().rc_data_copy_dist(self._h, ptr(out)))
        return out

    @property
    def logD(self):
        out = np.empty((self.n, self.n))
        check(lib().rc_data_copy_logdist(self._h, ptr(out)))
        return out

    def scales(self):
        a, b = C.c_int32(), C.c_int32()
        check(lib().rc_data_scales(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def __del__(self):
        h = getattr(self, "_h", None)
        L = getattr(_lib, "_lib", None)               # the module is already torn down at interpreter exit
        if h and L is not None:
            L.rc_data_destroy(h)
            self._h = None

    def __repr__(self):
        return f"MCMC data : {self.n}×{self.n} dissimilarity matrix."


class MCMCState:
    """clusts (1-based labels), r, p -- the `init` argument of runsampler (types.jl:131-137)."""

    def __init__(self, clusts, r, p):
        self.clusts = np.asarray(clusts, dtype=np.int64)
        self.r, self.p = float(r), float(p)


class MCMCResult:
    """Fields of the reference's MCMCResult (types.jl:193-224)."""

    def __repr__(self):
        return (f"MCMC Summary: {self.options.numiters} iterations, {len(self.K)} samples, "
                f"acceptance rate r {self.r_acceptance_rate:.3f}, split-merge {self.splitmerge_acceptance_rate:.3f}, "
                f"runtime {self.runtime:.3f} s")


def _autocor(x):
    """StatsBase.autocor(x): demeaned, lags 0:min(S-1, round(10 log10 S))."""
    x = np.asarray(x, dtype=np.float64)
    S = x.size
    if S == 0:
        return np.zeros(0)
    lags = np.arange(0, min(S - 1, int(round(10 * math.log10(S)))) + 1)
    z = x - x.mean()
    zz = float(z @ z)
    return np.array([float(z[:S - l] @ z[l:]) / zz if zz != 0 else float("nan") for l in lags])


def iac_ess_acf(x):
    acf = _autocor(x)
    iac = acf.sum() * 2
    return iac, len(x) / iac if iac != 0 else float("nan"), acf


class Sampler:
    """Thin owner of an rc_sampler handle: `nchains` chains of one data set on one device."""

    def __init__(self, data, options, params, init_labels, init_r, init_p, seed=0, chain_offset=0, slot_cap=0):
        self.data, self.options, self.params = data, options, params
        lab = np.ascontiguousarray(np.asarray(init_labels, dtype=np.int64).reshape(-1, data.n))
        self.nchains = lab.shape[0]
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(init_r, dtype=np.float64), (self.nchains,)))
        p = np.ascontiguousarray(np.broadcast_to(np.asarray(init_p, dtype=np.float64), (self.nchains,)))
        self._h = C.c_void_p()
        o, q = options._c(), params._c()
        check(lib().rc_sampler_create(data._h, C.byref(o), C.byref(q), self.nchains, chain_offset, ptr(lab), ptr(r), ptr(p),
                                      seed, slot_cap, C.byref(self._h)))

    def run(self, iters=-1):
        check(lib().rc_sampler_run(self._h, iters))

    def chain_status(self, chain=0):
        """0, or RC_ERR_SLOTS (-5) when the chain needed more than slot_cap simultaneously live clusters and stopped."""
        return int(lib().rc_sampler_chain_status(self._h, chain))

    def check_sums(self):
        """(mismatching words of the row sums, of the block sums) after rebuilding both from the labels: (0, 0) when the
        incremental updates kept them exact, (-1, -1) before the first run.  With launch groups (chains whose row sums do
        not all fit the device) the chains of the group launched last are checked."""
        a, b = C.c_int64(), C.c_int64()
        check(lib().rc_sampler_check_sums(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def overflowed(self):
        """Number of chains stopped by the slot capacity (run() raises only when every chain stopped)."""
        return int(lib().rc_sampler_overflowed(self._h))

    def progress(self):
        a, b = C.c_int64(), C.c_double()
        check(lib().rc_sampler_progress(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def samples(self, chain=0):
        S, n = int(lib().rc_sampler_numsamples(self._h)), self.data.n
        out = dict(labels=np.zeros((S, n), np.int64), K=np.zeros(S, np.int64), r=np.zeros(S), p=np.zeros(S),
                   loglik=np.zeros(S), logposterior=np.zeros(S))
        check(lib().rc_sampler_copy_samples(self._h, chain, ptr(out["labels"]), ptr(out["K"]), ptr(out["r"]), ptr(out["p"]),
                                            ptr(out["loglik"]), ptr(out["logposterior"])))
        ni, nm = self.options.numiters, self.options.numiters * self.options.numMH
        out["r_acc"] = np.zeros(ni, np.uint8)
        out["sm_acc"] = np.zeros(nm, np.uint8)
        out["sm_split"] = np.zeros(nm, np.uint8)
        check(lib().rc_sampler_copy_acceptances(self._h, chain, ptr(out["r_acc"]), ptr(out["sm_acc"]), ptr(out["sm_split"])))
        return out

    def samples_all(self):
        """The recorded outputs of every chain in one call: dict of arrays with a leading chain axis."""
        S, n, Cn = int(lib().rc_sampler_numsamples(self._h)), self.data.n, self.nchains
        ni, nm = self.options.numiters, self.options.numiters * self.options.numMH
        out = dict(labels=np.empty((Cn, S, n), np.int64), K=np.empty((Cn, S), np.int64), r=np.empty((Cn, S)), p=np.empty((Cn, S)),
                   loglik=np.empty((Cn, S)), logposterior=np.empty((Cn, S)), r_acc=np.zeros((Cn, ni), np.uint8),
                   sm_acc=np.zeros((Cn, nm), np.uint8), sm_split=np.zeros((Cn, nm), np.uint8))
        check(lib().rc_sampler_copy_all(self._h, ptr(out["labels"]), ptr(out["K"]), ptr(out["r"]), ptr(out["p"]), ptr(out["loglik"]),
                                        ptr(out["logposterior"]), ptr(out["r_acc"]), ptr(out["sm_acc"]), ptr(out["sm_split"])))
        return out

    def state(self, chain=0):
        lab = np.zeros(self.data.n, np.int64)
        r, p = C.c_double(), C.c_double()
        check(lib().rc_sampler_copy_state(self._h, chain, ptr(lab), C.byref(r), C.byref(p)))
        return MCMCState(lab, r.value, p.value)

    # Cycle counters in librcb200_stats.so.  In the default library the timing slots stay 0 and three slots count events:
    # dec_wait the merge proposals rejected by their bound, bulk_rows the rows decided by their summaries, bulk_reduce the
    # scans decided as a whole by the per-slot margins.
    STAT_NAMES = ("dec_wait", "dec_work", "bulk_wait_consumed", "bulk_wait_full", "bulk_rows", "bulk_patch", "moves", "rebuilds",
                  "mh_setup", "mh_rscan", "mh_loglik", "scan_total", "record", "iter_total", "rp", "bulk_reduce")

    def stats(self):
        """Cycle counters of the chain kernel (profiling aid): dict name -> array over chains."""
        out = np.zeros((self.nchains, 16), np.int64)
        check(lib().rc_sampler_copy_stats(self._h, ptr(out)))
        return {k: out[:, i] for i, k in enumerate(self.STAT_NAMES)}

    def psm(self, chain0=0, nch=None):
        nch = self.nchains - chain0 if nch is None else nch
        out = np.zeros((self.data.n, self.data.n))
        check(lib().rc_sampler_psm(self._h, chain0, nch, ptr(out)))
        return out

    def psm_counts_dev(self, counts_ptr, chain0=0, nch=None):
        nch = self.nchains - chain0 if nch is None else nch
        check(lib().rc_sampler_psm_counts_dev(self._h, chain0, nch, C.c_void_p(counts_ptr)))

    def _comm(self, group, device, comm):
        """The communicator of an *_allreduce call: comm, else the one of the process group on this sampler's device."""
        return comm or Comm.from_torch(group, self.data.device if device is None else device)

    def psm_allreduce(self, group=None, device=None, comm=None):
        """PSM over the samples of every rank (mcmc.jl:560 across chain shards): per-rank exact int32 co-clustering
        counts stay on the device, ONE ncclAllReduce(sum) of the n x n matrix combines them, then a single divide by
        the global number of samples (rc_comm_sampler_psm)."""
        comm = self._comm(group, device, comm)
        out = np.empty((self.data.n, self.data.n))
        check(lib().rc_comm_sampler_psm(comm._h, self._h, ptr(out), None))
        return out

    def predict(self, newdist, chain0=0, nch=None):
        """predictivecoclustering over the recorded samples of chains chain0 .. chain0 + nch - 1 (chain-major, as
        samples_all()) without copying them to the host: dict(coclustering = m x n, newcluster = m)."""
        nch = self.nchains - chain0 if nch is None else nch
        Dn = _newdist(self.data.n, newdist)
        m = Dn.shape[0]
        out = dict(coclustering=np.empty((m, self.data.n)), newcluster=np.empty(m))
        check(lib().rc_sampler_predict(self._h, ptr(Dn), m, chain0, nch, ptr(out["coclustering"]), ptr(out["newcluster"])))
        return out

    def binder_pointestimate(self, chain0=0, nch=None):
        """getpointestimate(method="MPEL", loss="binder") over the pooled recorded samples of chains chain0 .. chain0 + nch
        - 1, from their co-clustering counts on the device (rc_sampler_binder_mpel): dict(clust = the winning partition,
        chain, index = its sample within that chain, sums = expected Binder loss sums of every sample (chain-major),
        totals = the same as exact integer counts of disagreeing pairs)."""
        nch = self.nchains - chain0 if nch is None else nch
        S = int(lib().rc_sampler_numsamples(self._h))
        total = max(nch, 0) * S
        sums, totals, best = np.empty(total), np.empty(total, np.int64), C.c_int64()
        check(lib().rc_sampler_binder_mpel(self._h, chain0, nch, ptr(sums), C.byref(best), ptr(totals)))
        chain, index = chain0 + best.value // S, best.value % S
        return dict(clust=self.samples(chain)["labels"][index], chain=chain, index=index, sums=sums, totals=totals)

    def binder_pointestimate_allreduce(self, group=None, device=None, comm=None):
        """binder_pointestimate over the chains of every rank (rc_comm_sampler_binder_mpel): the all-reduced counts, one
        ncclAllGather of the per-rank totals; equal to one GPU over the same chains.  dict(best = index into the samples
        of all ranks in rank order, sums, totals, and clust / chain / index of the winner on the rank that holds it, None
        on the others)."""
        comm = self._comm(group, device, comm)
        S = int(lib().rc_sampler_numsamples(self._h))
        mine = self.nchains * S
        sizes = comm.all_ranks(mine)
        total = sum(sizes)
        sums, totals, best = np.empty(total), np.empty(total, np.int64), C.c_int64()
        check(lib().rc_comm_sampler_binder_mpel(comm._h, self._h, ptr(sums), C.byref(best), ptr(totals)))
        out = dict(best=best.value, sums=sums, totals=totals, clust=None, chain=None, index=None)
        local = best.value - sum(sizes[:comm.rank])
        if 0 <= local < mine:
            out.update(chain=local // S, index=local % S)
            out["clust"] = self.samples(out["chain"])["labels"][out["index"]]
        return out

    def _traces(self, chain0, nch):
        """K, r, p, loglik and logposterior of chains chain0 .. chain0 + nch - 1 as nch x numsamples arrays."""
        S = int(lib().rc_sampler_numsamples(self._h))
        out = {k: np.empty((nch, S)) for k in _TRACES}
        K = np.empty(S, np.int64)
        for i, c in enumerate(range(chain0, chain0 + nch)):
            check(lib().rc_sampler_copy_samples(self._h, c, None, ptr(K), *(ptr(out[k][i]) for k in _TRACES[1:])))
            out["K"][i] = K
        return out

    def convergencediagnostics(self, chain0=0, nch=None, matrix=False):
        """Convergence across chains chain0 .. chain0 + nch - 1 (rc_sampler_cocl_rhat): the split-R-hat of every point pair's
        co-clustering indicator, computed from the device-resident samples, and each chain's distance from the pooled PSM,
        with the split-R-hat of the traces K, r, p, loglik and logposterior.  Returns dict(rhat_max, rhat_pair = (a, b)
        0-based, pairs_above = pairs with R-hat > 1.01, chain_meandev / chain_maxdev = mean and largest |p_c - pbar| over
        the pairs per chain, rhat = the n x n matrix when matrix=True else None, traces = {name: split-R-hat})."""
        nch = self.nchains - chain0 if nch is None else nch
        n, k = self.data.n, max(nch, 0)
        sm, md, xd = rc_rhat_summary(), np.empty(k), np.empty(k)
        R = np.empty((n, n)) if matrix else None
        check(lib().rc_sampler_cocl_rhat(self._h, chain0, nch, C.byref(sm), ptr(R), ptr(md), ptr(xd)))
        tr = self._traces(chain0, nch)
        return _rhat_dict(sm, R, md, xd, {name: _split_rhat(x) for name, x in tr.items()})

    def convergencediagnostics_allreduce(self, group=None, device=None, comm=None, matrix=False):
        """convergencediagnostics over the chains of every rank (rc_comm_sampler_cocl_rhat): the all-reduced co-clustering
        counts, one ncclAllReduce of the squared group counts and one ncclAllGather of the chain deviations; equal to one
        GPU over the same chains.  chain_meandev / chain_maxdev and the traces cover every rank's chains in rank order."""
        comm = self._comm(group, device, comm)
        n, total = self.data.n, sum(comm.all_ranks(self.nchains))
        sm, md, xd = rc_rhat_summary(), np.empty(total), np.empty(total)
        R = np.empty((n, n)) if matrix else None
        check(lib().rc_comm_sampler_cocl_rhat(comm._h, self._h, C.byref(sm), ptr(R), ptr(md), ptr(xd)))
        parts = comm.all_ranks(self._traces(0, self.nchains))
        tr = {k: np.concatenate([p[k] for p in parts]) for k in _TRACES}
        return _rhat_dict(sm, R, md, xd, {name: _split_rhat(x) for name, x in tr.items()})

    def _partition_dists(self, refs, chain0, nch, loss):
        """partitiondistances over the device-resident samples of chains chain0 .. chain0 + nch - 1 (rc_sampler_partition_dists)."""
        code = _loss_code(loss)
        P = _partitions(refs, self.data.n, "the partitions")
        out = _dists_out(P.shape[0], max(nch, 0) * int(lib().rc_sampler_numsamples(self._h)), loss)
        check(lib().rc_sampler_partition_dists(self._h, ptr(P), P.shape[0], chain0, nch, code, ptr(out["dist"]), ptr(out["pairs"]),
                                               ptr(out["K"])))
        return out

    def expectedloss(self, partitions, chain0=0, nch=None, loss="VI"):
        """expectedloss over the recorded samples of chains chain0 .. chain0 + nch - 1 (chain-major), from the device-resident
        samples: dict(expectedloss, totals)."""
        nch = self.nchains - chain0 if nch is None else nch
        return _expected(self._partition_dists(partitions, chain0, nch, loss), loss)

    def credibleball(self, estimate, chain0=0, nch=None, loss="VI", alpha=0.05):
        """credibleball over the recorded samples of chains chain0 .. chain0 + nch - 1 (chain-major: indices count the
        samples of chain0 first), from the device-resident samples."""
        _check_alpha(alpha)
        nch = self.nchains - chain0 if nch is None else nch
        S = int(lib().rc_sampler_numsamples(self._h))
        out = self._partition_dists(_estimate(estimate, self.data.n), chain0, nch, loss)
        return _ball_result(out, alpha, self._labels_of(lambda i: (chain0 + i // S, i % S)))

    def credibleball_allreduce(self, estimate, loss="VI", alpha=0.05, group=None, device=None, comm=None):
        """credibleball over the chains of every rank (rc_comm_sampler_partition_dists): each rank computes its own samples,
        one ncclAllGather assembles the distances, equal to one GPU over the same chains.  Indices count every rank's
        samples in rank order; a bound's clust is filled on the rank that holds its first sample, None on the others."""
        _check_alpha(alpha)
        code = _loss_code(loss)
        P = np.ascontiguousarray(_estimate(estimate, self.data.n))
        comm = self._comm(group, device, comm)
        S = int(lib().rc_sampler_numsamples(self._h))
        mine = self.nchains * S
        sizes = comm.all_ranks(mine)
        out = _dists_out(1, sum(sizes), loss)
        check(lib().rc_comm_sampler_partition_dists(comm._h, self._h, ptr(P), 1, code, ptr(out["dist"]), ptr(out["pairs"]), ptr(out["K"])))
        first = sum(sizes[:comm.rank])
        return _ball_result(out, alpha, self._labels_of(lambda i: ((i - first) // S, (i - first) % S) if 0 <= i - first < mine else None))

    def alignedallocation(self, estimate, chain0=0, nch=None, maps=False):
        """alignedallocation over the recorded samples of chains chain0 .. chain0 + nch - 1 (chain-major), from the
        device-resident samples (rc_sampler_aligned_alloc)."""
        est = np.ascontiguousarray(_estimate(estimate, self.data.n))
        nch = self.nchains - chain0 if nch is None else nch
        out, clusters = _aligned_out(est, max(nch, 0) * int(lib().rc_sampler_numsamples(self._h)), maps)
        check(lib().rc_sampler_aligned_alloc(self._h, ptr(est), chain0, nch, ptr(out["counts"]), ptr(out["matched"]),
                                             ptr(out["K"]), ptr(out["maps"])))
        return _aligned_result(out, clusters, est)

    def alignedallocation_allreduce(self, estimate, maps=False, group=None, device=None, comm=None):
        """alignedallocation over the chains of every rank (rc_comm_sampler_aligned_alloc): each rank aligns its own samples,
        one ncclAllReduce sums the counts and one ncclAllGather assembles the per-sample outputs in rank order, equal to one
        GPU over the same chains."""
        est = np.ascontiguousarray(_estimate(estimate, self.data.n))
        comm = self._comm(group, device, comm)
        out, clusters = _aligned_out(est, sum(comm.all_ranks(self.nchains * int(lib().rc_sampler_numsamples(self._h)))), maps)
        check(lib().rc_comm_sampler_aligned_alloc(comm._h, self._h, ptr(est), ptr(out["counts"]), ptr(out["matched"]),
                                                  ptr(out["K"]), ptr(out["maps"])))
        return _aligned_result(out, clusters, est)

    def _labels_of(self, where):
        """clust_of for _ball_result: where(i) = (chain, sample) of pooled sample i on this sampler, or None.  Each chain's
        labels are copied to the host once (labels only, not the traces)."""
        S, n, chains = int(lib().rc_sampler_numsamples(self._h)), self.data.n, {}

        def clust_of(i):
            w = where(i)
            if w is None:
                return None
            c, t = w
            if c not in chains:
                chains[c] = np.empty((S, n), np.int64)
                check(lib().rc_sampler_copy_samples(self._h, c, ptr(chains[c]), None, None, None, None, None))
            return chains[c][t].copy()
        return clust_of

    def close(self):
        L = getattr(_lib, "_lib", None)
        if getattr(self, "_h", None) and L is not None:
            L.rc_sampler_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def init_rp(params, seed, chain):
    r, p = C.c_double(), C.c_double()
    q = params._c()
    check(lib().rc_init_rp(C.byref(q), seed, chain, C.byref(r), C.byref(p)))
    return r.value, p.value


def _result_from(samples, options, params, psm, runtime):
    res = MCMCResult()
    res.clusts = [samples["labels"][j] for j in range(samples["labels"].shape[0])]
    res.posterior_coclustering = psm
    for name in ("K", "r", "p"):
        x = samples[name]
        setattr(res, name, x)
        iac, ess, acf = iac_ess_acf(x)                                         # mcmc.jl:564-573
        setattr(res, name + "_iac", iac); setattr(res, name + "_ess", ess); setattr(res, name + "_acf", acf)
        setattr(res, name + "_mean", float(np.mean(x)) if len(x) else float("nan"))
        setattr(res, name + "_variance", float(np.var(x, ddof=1)) if len(x) > 1 else float("nan"))
    res.splitmerge_acceptances = samples["sm_acc"].astype(bool)
    res.splitmerge_splits = samples["sm_split"].astype(bool)
    res.r_acceptances = samples["r_acc"].astype(bool)
    res.splitmerge_acceptance_rate = float(res.splitmerge_acceptances.mean()) if options.numMH > 0 else 0.0   # :576-580
    res.r_acceptance_rate = float(res.r_acceptances.mean())
    res.loglik, res.logposterior = samples["loglik"], samples["logposterior"]
    res.options, res.params = options, params
    res.runtime = runtime
    res.mean_iter_time = runtime / options.numiters
    return res


def runsampler(data, options=None, params=None, init=None, verbose=True, nchains=1, seed=0, slot_cap=0):
    """runsampler(data, options, params, init; verbose) -> MCMCResult   (mcmc.jl:501-590).
    With nchains > 1 returns a list of MCMCResult (independent chains, one persistent kernel)."""
    if options is None:
        options = MCMCOptionsList()
    if params is None:
        from .prior import fitprior
        params = fitprior(data, "k-medoids", True, verbose=verbose)          # runs on the device-resident matrix
    n = data.n
    if init is None:                                                           # mcmc.jl:519-527
        from .prior import kmedoids
        k0 = min(params.maxK, params.K_initial) if params.maxK > 0 else params.K_initial
        lab0 = kmedoids(data, int(k0), maxiter=1000)["assignments"]         # rc_kmedoids on the resident matrix
        labs = np.tile(lab0, (nchains, 1))
        rp = [init_rp(params, seed, c) for c in range(nchains)]
        r0 = np.array([x[0] for x in rp]); p0 = np.array([x[1] for x in rp])
    else:
        inits = init if isinstance(init, (list, tuple)) else [init] * nchains
        labs = np.stack([sortlabels(s.clusts) if np.max(s.clusts) > (slot_cap or 128) else np.asarray(s.clusts) for s in inits])
        r0 = np.array([s.r for s in inits]); p0 = np.array([s.p for s in inits])
    if verbose:
        print("Run MCMC")
        print(f"Setup: {options.numiters} iterations, {options.numsamples} samples, {n} observations.")
    smp = Sampler(data, options, params, labs, r0, p0, seed=seed, slot_cap=slot_cap)
    smp.run(-1)
    _, runtime = smp.progress()
    if verbose:
        print("Computing summary statistics and diagnostics.")
    results = []
    for c in range(nchains):
        if smp.overflowed() and smp.chain_status(c) != 0:
            # the chain needed more than slot_cap live clusters (the reference allows up to n, src/mcmc.jl:199): its
            # trace is incomplete, the other chains are unaffected
            import warnings
            warnings.warn(f"chain {c} needed more than slot_cap = {slot_cap or 128} simultaneously live clusters and was stopped; "
                          "its result is None (raise slot_cap, or set maxK in the hyperparameters)")
            results.append(None)
            continue
        s = smp.samples(c)
        psm = smp.psm(c, 1) if options.numsamples > 0 else np.full((n, n), np.nan)   # mcmc.jl:560
        results.append(_result_from(s, options, params, psm, runtime))
    smp.close()
    return results[0] if nchains == 1 else results


# ------------------------------------------------------------------------------------------------
def prettytime(t):
    """utils.jl:158-187: human-readable duration (Dates.canonicalize splits whole seconds into weeks / days / hours /
    minutes / seconds; only days and below are named by the reference)."""
    if t < 1e-6:
        return "%.2f ns" % (t * 1e9)
    if t < 1e-3:
        return "%.2f μs" % (t * 1e6)
    if t < 1:
        return "%.2f ms" % (t * 1e3)
    if t < 60:
        return "%.2f s" % t
    sec = int(math.floor(t))
    parts = []
    for name, span in (("day", 86400), ("hr", 3600), ("min", 60)):
        v, sec = divmod(sec, span)
        if v:
            parts.append(f"{v} {name}" + ("s" if v != 1 else ""))
    if sec:
        parts.append(f"{sec} s")
    return " ".join(parts)


def prettynumber(x):
    """utils.jl:189."""
    return "%.3e" % x if x < 1 else "%.3f" % x


def makematrix(x):
    """utils.jl:154-156: vector of vectors -> matrix whose COLUMNS are the vectors."""
    return np.asarray([np.asarray(v, dtype=np.float64) for v in x], dtype=np.float64).T.copy()


def adjacencymatrix(clusts):
    c = np.asarray(clusts)
    return c[:, None] == c[None, :]


def sortlabels(x):
    x = np.asarray(x)
    _, first, inv = np.unique(x, return_index=True, return_inverse=True)
    order = np.argsort(np.argsort(first))
    return (order[inv] + 1).astype(np.int64)


def uppertriangle(M):
    M = np.asarray(M)
    i, j = np.triu_indices(M.shape[0], 1)
    return M[i, j]


def psm(labels, device=0):
    """sum(adjacencymatrix.(clusts)) ./ numsamples on the GPU (mcmc.jl:560) for host label vectors."""
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    out = np.zeros((L.shape[1], L.shape[1]))
    check(lib().rc_psm(ptr(L), L.shape[0], L.shape[1], device, ptr(out)))
    return out


# ---- posterior predictive allocation of new observations (no reference equivalent; the conditional of the full Gibbs
# scan, mcmc.jl:193-247, for a point that is not in the data, normalised as sample_logweights draws from it, utils.jl:2-6)
def _newdist(n, newdist):
    Dn = np.asarray(newdist, dtype=np.float64)
    if Dn.ndim == 1:
        Dn = Dn[None, :]
    if Dn.ndim != 2 or Dn.shape[0] < 1 or Dn.shape[1] != n:
        raise ArgumentError(f"newdist must be an m × {n} matrix: one row per new point, one column per training point.")
    return np.ascontiguousarray(Dn)


def crossdistances(points, newpoints, device=0):
    """Euclidean distances of m new points to the n training points (m x n), bit-equal to the rows of the new points in
    MCMCData.from_points(vstack(points, newpoints)).D -- the `newdist` argument of the predictive calls."""
    X = np.ascontiguousarray(np.asarray(points, dtype=np.float64))
    Y = np.ascontiguousarray(np.asarray(newpoints, dtype=np.float64))
    if Y.ndim == 1:
        Y = Y[None, :]
    if X.ndim != 2 or Y.ndim != 2 or X.shape[1] != Y.shape[1] or X.shape[0] < 1 or Y.shape[0] < 1:
        raise ArgumentError("points and newpoints must be n × dim and m × dim with the same dim.")
    out = np.empty((Y.shape[0], X.shape[0]))
    check(lib().rc_crossdist(ptr(X), X.shape[0], ptr(Y), Y.shape[0], X.shape[1], device, ptr(out)))
    return out


def predictive_from_labels(data, newdist, labels, r, p, params, logprobs=False):
    """The predictive of S label vectors (S x n, any positive labels; each is relabelled by sortlabels) with their r and
    p: dict(coclustering = m x n, newcluster = m), and with logprobs=True the S x m x 256 un-normalised log-probabilities
    of the candidate slots (slot k at index k - 1, NaN beyond the last candidate)."""
    Dn = _newdist(data.n, newdist)
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64).reshape(-1, data.n))
    S, m = L.shape[0], Dn.shape[0]
    rr = np.ascontiguousarray(np.asarray(r, dtype=np.float64).reshape(-1))
    pp = np.ascontiguousarray(np.asarray(p, dtype=np.float64).reshape(-1))
    if rr.size != S or pp.size != S:
        raise ArgumentError("r and p must hold one value per sample.")
    out = dict(coclustering=np.empty((m, data.n)), newcluster=np.empty(m))
    lp = np.empty((S, m, 256)) if logprobs else None
    q = params._c()
    check(lib().rc_predict(data._h, C.byref(q), ptr(Dn), m, ptr(L), ptr(rr), ptr(pp), S, ptr(out["coclustering"]),
                           ptr(out["newcluster"]), ptr(lp)))
    if logprobs:
        out["logprobs"] = lp
    return out


def predictivecoclustering(samples, data, newdist):
    """Posterior predictive allocation of new observations: for each new point x (row of newdist, m x n dissimilarities to
    the training points of `data`) coclustering[x, j] is the posterior probability that x joins the cluster of training
    point j, newcluster[x] that it opens a cluster of its own -- the scan step's conditional (mcmc.jl:193-247) averaged
    over the samples.  `samples` is an MCMCResult or a list of them (pooled in list order, sampled with the same
    hyperparameters).  Returns dict(coclustering = m x n, newcluster = m)."""
    res = list(samples) if isinstance(samples, (list, tuple)) else [samples]
    if not res:
        raise ArgumentError("samples must hold at least one MCMCResult.")
    params = res[0].params
    for x in res[1:]:
        if bytes(x.params._c()) != bytes(params._c()):
            raise ArgumentError("the results to pool were sampled with different hyperparameters.")
    labs = [np.asarray(c, dtype=np.int64) for x in res for c in x.clusts]
    if any(c.shape != (data.n,) for c in labs):
        raise ArgumentError(f"the samples must label the {data.n} points of data.")
    L = np.stack(labs) if labs else np.zeros((0, data.n), np.int64)
    r = np.concatenate([np.asarray(x.r, dtype=np.float64) for x in res])
    p = np.concatenate([np.asarray(x.p, dtype=np.float64) for x in res])
    return predictive_from_labels(data, newdist, L, r, p, params)


def allocationprobabilities(data, newdist, clusts, r, p, params):
    """Allocation probabilities of new points for one partition `clusts` (such as a point estimate) with its r and p:
    m x (K + 1), column k for the k-th distinct label in ascending order, the last column for a new cluster (0 when maxK
    leaves no room for one).  These are the kernel's probabilities of the one-sample predictive."""
    c = np.asarray(clusts, dtype=np.int64)
    if c.shape != (data.n,):
        raise ArgumentError(f"clusts must label the {data.n} points of data.")
    out = predictive_from_labels(data, newdist, c[None, :], [r], [p], params)
    _, first = np.unique(c, return_index=True)
    return np.column_stack([out["coclustering"][:, first], out["newcluster"]])


_LOSS = {"binder": 0, "omARI": 1, "VI": 2, "ID": 3}


def mpel_loss_sums(labels, loss, device=0):
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    sums = np.zeros(L.shape[0])
    best = C.c_int64()
    check(lib().rc_mpel(ptr(L), L.shape[0], L.shape[1], _LOSS[loss], device, ptr(sums), C.byref(best)))
    return sums, best.value


def psm_counts_dev(labels, counts_ptr, device=0):
    """Exact co-clustering counts (mcmc.jl:560, not divided) of host label vectors (S x n) into a caller DEVICE buffer of
    n x n int32 (e.g. a torch tensor's data_ptr()): one rank's share of a PSM whose samples are sharded over GPUs."""
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    check(lib().rc_psm_counts_dev(ptr(L), L.shape[0], L.shape[1], device, C.c_void_p(counts_ptr)))


def psm_sharded(labels, group=None, device=None, total=None, comm=None):
    """PSM of label vectors that are sharded over the ranks (SURVEY 8e, BASELINE configs[4]): `labels` is THIS rank's
    S_r x n share; exact int32 counts per rank on the device, one ncclAllReduce(sum) of the n x n matrix, one divide by
    the global number of samples (rc_comm_psm).  Every rank returns the full PSM."""
    comm = comm or Comm.from_torch(group, device)
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    S, n = L.shape
    out = np.empty((n, n))
    check(lib().rc_comm_psm(comm._h, ptr(L), S, n, ptr(out), None))
    return out


def cyclic_rows(rank, world, S):
    """Rows of an S-row matrix owned by `rank` when they are dealt out cyclically (row i -> rank i % world), and the
    padded per-rank row count every rank allocates for the all_gather."""
    per = (S + world - 1) // world
    return list(range(rank, S, world)), per


def assemble_cyclic_rows(allrows, S):
    """Inverse of the cyclic deal: allrows[r, k] is row r + k * world (all_gather output, world x per x S) -> S x S."""
    world, per, cols = allrows.shape
    return allrows.permute(1, 0, 2).reshape(per * world, cols)[:S].contiguous()


def mpel_loss_sums_sharded(labels, loss, group=None, device=None, comm=None):
    """mpel_loss_sums with the candidate samples split over the ranks (SURVEY 8e): rank r evaluates rows r, r + world,
    ... of the upper triangle of the pairwise loss matrix (cyclic, so the ranks do equal work), one ncclAllGather
    assembles it on every GPU, the column sums run in ascending row order -- bit-equal to the single-GPU result
    (rc_comm_mpel)."""
    comm = comm or Comm.from_torch(group, device)
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    sums = np.zeros(L.shape[0]); best = C.c_int64()
    check(lib().rc_comm_mpel(comm._h, ptr(L), L.shape[0], L.shape[1], _LOSS[loss], ptr(sums), C.byref(best)))
    return sums, int(best.value)


def binder_loss_sums(labels, device=0):
    """Expected Binder loss of every sample against all of them (S x n host labels), from their co-clustering counts on
    the device (rc_binder_mpel): (sums, best, totals) with sums[s] = totals[s] / C(n, 2), totals the exact integer counts
    of disagreeing pairs summed over the samples, best their first argmin.  O(S n^2) work and no S x S matrix, so it
    takes pooled chains; sums agree with mpel_loss_sums(labels, "binder") up to that call's fp64 rounding."""
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    if L.ndim != 2:
        raise ArgumentError("labels must be an S × n matrix.")
    sums, totals, best = np.empty(L.shape[0]), np.empty(L.shape[0], np.int64), C.c_int64()
    check(lib().rc_binder_mpel(ptr(L), L.shape[0], L.shape[1], device, ptr(sums), C.byref(best), ptr(totals)))
    return sums, int(best.value), totals


# ---- convergence across chains (no reference equivalent: the reference's diagnostics are per chain, mcmc.jl:564-573) ----
_TRACES = ("K", "r", "p", "loglik", "logposterior")


def _split_rhat(x):
    """Split-R-hat (BDA3 11.4) of a C x S trace: the first and last floor(S / 2) samples of every chain are the 2C groups
    (the middle sample of an odd S is dropped); sqrt(var+ / W) with W the mean within-group sample variance (ddof = 1) and
    B / L the sample variance of the group means.  W = 0 means every group is constant, decided by comparing the values:
    1 when they all hold the same value, +Inf otherwise."""
    x = np.asarray(x, dtype=np.float64)
    S = x.shape[1]
    if S < 4:
        raise ArgumentError("split-R-hat needs at least 4 samples per chain.")
    L = S // 2
    g = np.concatenate([x[:, :L], x[:, S - L:]])
    if np.all(g == g[:, :1]):
        return 1.0 if np.all(g == g[0, 0]) else math.inf
    W = float(np.mean(np.var(g, axis=1, ddof=1)))
    B = L * float(np.var(np.mean(g, axis=1), ddof=1))
    return math.sqrt(((L - 1) / L * W + B / L) / W)


def _rhat_dict(sm, R, meandev, maxdev, traces):
    return dict(rhat_max=float(sm.max), rhat_pair=(int(sm.a), int(sm.b)), pairs_above=int(sm.above), chain_meandev=meandev,
                chain_maxdev=maxdev, rhat=R, traces=traces)


def cocl_rhat(labels, device=0, matrix=False):
    """The co-clustering part of convergencediagnostics for host label vectors, labels = C chains x S samples x n points
    (any positive labels; rc_cocl_rhat): dict(rhat_max, rhat_pair, pairs_above, chain_meandev, chain_maxdev, rhat)."""
    L = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    if L.ndim != 3:
        raise ArgumentError("labels must be a chains × samples × n array.")
    Cn, S, n = L.shape
    sm, md, xd = rc_rhat_summary(), np.empty(Cn), np.empty(Cn)
    R = np.empty((n, n)) if matrix else None
    check(lib().rc_cocl_rhat(ptr(L), Cn, S, n, device, C.byref(sm), ptr(R), ptr(md), ptr(xd)))
    out = _rhat_dict(sm, R, md, xd, None)
    del out["traces"]
    return out


def convergencediagnostics(results, device=0, matrix=False):
    """Convergence across the chains of a list of MCMCResult (runsampler with nchains > 1): the split-R-hat of every point
    pair's co-clustering indicator (labels switch between chains, these indicators do not) and each chain's distance from
    the pooled PSM, on the device, with the split-R-hat of the traces K, r, p, loglik and logposterior on the host.  Returns
    the dict of Sampler.convergencediagnostics.  Chains that sample another mode of the partition show as pairs with
    R-hat above 1.01 and as a chain whose chain_meandev stands out."""
    res = list(results) if isinstance(results, (list, tuple)) else [results]
    if not res:
        raise ArgumentError("results must hold at least one MCMCResult.")
    if any(r is None for r in res):
        raise ArgumentError("a chain stopped at the slot capacity (its result is None); drop it before the diagnostics.")
    if len({len(r.clusts) for r in res}) > 1:
        raise ArgumentError("the results hold different numbers of samples.")
    if len({np.asarray(c).shape for r in res for c in r.clusts}) > 1:
        raise ArgumentError("the results label different numbers of points.")
    out = cocl_rhat(np.stack([np.stack(r.clusts) for r in res]), device, matrix)
    out["traces"] = {k: _split_rhat(np.stack([np.asarray(getattr(r, k)) for r in res])) for k in _TRACES}
    return out


# ---- distances from given partitions to the samples: posterior expected loss and credible balls (no reference call; Wade &
# Ghahramani 2018, Bayesian Analysis 13(2), section 4, as mcclust.ext::credibleball) ----
def _loss_code(loss):
    if not (isinstance(loss, str) and loss in _LOSS):
        raise ArgumentError('loss must be one of "binder", "omARI", "VI" and "ID" (a function-valued loss is not supported here).')
    return _LOSS[loss]


def _check_alpha(alpha):
    if not 0 < alpha < 1:
        raise ArgumentError("alpha must lie in (0, 1).")


def _estimate(estimate, n):
    est = np.asarray(estimate, dtype=np.int64)
    if est.shape != (n,):
        raise ArgumentError(f"estimate must label the {n} points of the samples.")
    return est


def _partitions(parts, n, what):
    """nref x n int64 label array of one partition (length n) or several (nref x n)."""
    P = np.asarray(parts, dtype=np.int64)
    if P.ndim == 1:
        P = P[None, :]
    if P.ndim != 2 or P.shape[0] < 1 or P.shape[1] != n:
        raise ArgumentError(f"{what} must label the {n} points of the samples.")
    return np.ascontiguousarray(P)


def _sample_labels(samples):
    """S x n int64 labels of an MCMCResult, a list of them (pooled in list order) or an S x n label array."""
    if isinstance(samples, (list, tuple)):
        if not samples:
            raise ArgumentError("samples must hold at least one MCMCResult.")
        if any(r is None for r in samples):
            raise ArgumentError("a chain stopped at the slot capacity (its result is None); drop it before pooling.")
        clusts = [c for r in samples for c in r.clusts]
    elif isinstance(samples, MCMCResult):
        clusts = list(samples.clusts)
    else:
        L = np.asarray(samples, dtype=np.int64)
        if L.ndim != 2 or L.shape[0] == 0:
            raise ArgumentError("samples must be an MCMCResult, a list of them or a non-empty S × n label array.")
        return np.ascontiguousarray(L)
    if not clusts:
        raise ArgumentError("samples hold no sample.")
    if len({np.asarray(c).shape for c in clusts}) > 1:
        raise ArgumentError("the results to pool label different numbers of points.")
    return np.ascontiguousarray(np.stack(clusts).astype(np.int64, copy=False))


def _dists_out(nref, S, loss):
    """Output arrays of the partition-distance calls; the exact Binder counts only with loss="binder" (else None: the kernel
    then skips their integer sums)."""
    return dict(dist=np.empty((nref, S)), pairs=np.empty((nref, S), np.int64) if loss == "binder" else None, K=np.empty(S, np.int32))


def _expected(out, loss):
    """(sum_t d_t) / S per partition, the sum in ascending sample order from +0.0 (np.cumsum adds sequentially): bit-equal
    to rc_mpel's loss_sums[0] / S for a partition stacked before the samples."""
    d = out["dist"]
    sums = np.cumsum(np.hstack([np.zeros((d.shape[0], 1)), d]), axis=1)[:, -1]
    return dict(expectedloss=sums / d.shape[1], totals=out["pairs"].sum(axis=1) if loss == "binder" else None)


def _credibleball(d, K, alpha):
    """The credible ball of Wade & Ghahramani (2018, section 4) from the distances d of the S samples to the estimate and
    their numbers of clusters K.  radius: the smallest sample distance e with #{t: d_t <= e} / S >= 1 - alpha (fp64 division
    and comparison); the ball is every sample with d_t <= radius, ties included.  horizontal: the ball's samples at the
    largest distance; upper: among the ball's samples with the fewest clusters, those at the largest distance; lower: the
    same among those with the most clusters.  Each bound is dict(dist, K = the first one's, indices = every sample attaining
    it, ascending)."""
    d = np.asarray(d, dtype=np.float64)
    K = np.asarray(K, dtype=np.int64)
    ds = np.sort(d)
    frac = np.searchsorted(ds, ds, side="right") / np.float64(d.size)
    radius = float(ds[int(np.argmax(frac >= 1.0 - alpha))])
    inball = d <= radius

    def bound(mask):
        far = d[mask].max()
        idx = np.flatnonzero(mask & (d == far))
        return dict(dist=float(far), K=int(K[idx[0]]), indices=idx)
    return dict(radius=radius, inball=int(inball.sum()), horizontal=bound(inball), upper=bound(inball & (K == K[inball].min())),
                lower=bound(inball & (K == K[inball].max())))


def _ball_result(out, alpha, clust_of):
    """credibleball's dict from the distances of one estimate (partitiondistances' dict); clust_of(i) gives the labels of
    pooled sample i (or None where they are not held)."""
    ball = _credibleball(out["dist"][0], out["K"], alpha)
    for name in ("horizontal", "upper", "lower"):
        ball[name]["clust"] = clust_of(int(ball[name]["indices"][0]))
    ball["expectedloss"] = float(_expected(out, None)["expectedloss"][0])
    ball["dist"] = out["dist"][0]
    return ball


def partitiondistances(refs, samples, loss="VI", device=0):
    """Distances from reference partitions (one of length n, or nref x n; any positive labels, at most 255 clusters each)
    to every sample, with the losses of getpointestimate: one contingency table per (reference, sample) on the device
    (rc_partition_dists).  `samples` is an MCMCResult, a list of them (pooled in list order) or an S x n label array.
    Returns dict(dist = nref x S, pairs = with loss="binder" the nref x S exact counts of disagreeing pairs, else None,
    K = clusters per sample)."""
    code = _loss_code(loss)
    L = _sample_labels(samples)
    S, n = L.shape
    P = _partitions(refs, n, "refs")
    out = _dists_out(P.shape[0], S, loss)
    check(lib().rc_partition_dists(ptr(P), P.shape[0], ptr(L), S, n, code, device, ptr(out["dist"]), ptr(out["pairs"]), ptr(out["K"])))
    return out


def expectedloss(partitions, samples, loss="VI", device=0):
    """Posterior expected loss of given partitions (the MAP sample, a point estimate, a k-medoids clustering, the true labels
    of a simulation, ...) over the samples: dict(expectedloss = (sum_t d_t) / S per partition, summed in ascending pooled
    order; totals = with loss="binder" the exact int64 total of disagreeing pairs per partition, else None).  O(S n) per
    partition, so it scores pooled chains under any of the four losses."""
    _loss_code(loss)
    L = _sample_labels(samples)
    return _expected(partitiondistances(_partitions(partitions, L.shape[1], "partitions"), L, loss, device), loss)


def credibleball(estimate, samples, loss="VI", alpha=0.05, device=0):
    """Credible ball around a point estimate (Wade & Ghahramani 2018, section 4; mcclust.ext::credibleball): the smallest
    ball in the given loss around `estimate` that holds 1 - alpha of the samples, and its bounds.  Returns dict(radius,
    inball = samples in the ball, expectedloss of the estimate, dist = the S distances, horizontal / upper / lower =
    dict(dist, K, indices = pooled sample indices attaining the bound, clust = labels of the first))."""
    _loss_code(loss)
    _check_alpha(alpha)
    L = _sample_labels(samples)
    out = partitiondistances(_estimate(estimate, L.shape[1]), L, loss, device)
    return _ball_result(out, alpha, lambda i: L[i].copy())


# ---- allocation probabilities to the clusters of a point estimate (no reference call; the pivot method of the ECR algorithm,
# Papastamoulis & Iliopoulos 2010, JCGS 19(2), as label.switching::ecr) ----
def _aligned_out(est, S, maps):
    """Output arrays of the aligned-allocation calls, and the estimate's labels in first-appearance order (the columns).
    With more than 255 clusters the library refuses before it writes, so the counts never need more than 256 columns."""
    first = np.sort(np.unique(est, return_index=True)[1])
    kh = min(first.size, 255)
    return dict(counts=np.empty((est.size, kh + 1), np.int32), matched=np.empty(S, np.int64), K=np.empty(S, np.int32),
                maps=np.empty((S, 255), np.uint8) if maps else None), est[first]


def _aligned_result(out, clusters, est):
    S = out["matched"].size
    prob = out["counts"] / np.float64(S)
    col = np.argsort(clusters)[np.unique(est, return_inverse=True)[1]]    # the column of each point's estimate cluster
    res = dict(prob=prob, clusters=clusters, self=prob[np.arange(est.size), col], counts=out["counts"], matched=out["matched"],
               K=out["K"])
    if out["maps"] is not None:
        res["maps"] = out["maps"]
    return res


def alignedallocation(estimate, samples, maps=False, device=0):
    """Allocation probabilities of every point to the clusters of a point estimate: each sample's clusters are matched to
    the estimate's by the assignment that maximises the number of agreeing points (the ECR pivot method, Papastamoulis &
    Iliopoulos 2010; ties resolved by one canonical Hungarian method), then prob[i, k] = the share of samples in which point
    i's matched cluster is estimate cluster k.  `samples` is an MCMCResult, a list of them (pooled in list order) or an S x n
    label array; the estimate takes any positive labels (at most 255 clusters).  Returns dict(prob = n x (K + 1) fp64, the
    last column the samples in which the point's cluster was unmatched; clusters = the estimate's labels in column order;
    self = prob[i, column of estimate(i)]; counts = the n x (K + 1) int32 counts, rows summing to S; matched = agreeing points
    per sample, n - matched the transfer distance; K = clusters per sample; maps = with maps=True the S x 255 uint8
    sigma_t(l) at [t, l - 1], 0 for unmatched and beyond K_t)."""
    L = _sample_labels(samples)
    S, n = L.shape
    est = np.ascontiguousarray(_estimate(estimate, n))
    out, clusters = _aligned_out(est, S, maps)
    check(lib().rc_aligned_alloc(ptr(est), ptr(L), S, n, device, ptr(out["counts"]), ptr(out["matched"]), ptr(out["K"]),
                                 ptr(out["maps"])))
    return _aligned_result(out, clusters, est)


_PAIRWISE_BYTES = 64 << 30          # the S x S fp64 loss matrix of the pairwise MPEL path must stay below this


def _pooled_pointestimate(results, method, loss, device):
    """getpointestimate over a list of MCMCResult (runsampler with nchains > 1), pooled in list order."""
    if not results:
        raise ArgumentError("samples must hold at least one MCMCResult.")
    if any(r is None for r in results):
        raise ArgumentError("a chain stopped at the slot capacity (its result is None); drop it before pooling.")
    clusts = [c for r in results for c in r.clusts]
    if len({np.asarray(c).shape for c in clusts}) > 1:
        raise ArgumentError("the results to pool label different numbers of points.")
    if method == "MAP":
        i = int(np.argmax(np.concatenate([np.asarray(r.logposterior) for r in results])))
    elif method == "MLE":
        i = int(np.argmax(np.concatenate([np.asarray(r.loglik) for r in results])))
    elif isinstance(loss, str) and loss == "binder":
        _, i, _ = binder_loss_sums(np.stack(clusts), device)
    else:
        S = len(clusts)
        if 8 * S * S > _PAIRWISE_BYTES:
            raise ArgumentError(f"{S} pooled samples need a {8 * S * S / 2**30:.0f} GiB pairwise loss matrix for loss={loss!r}; "
                                'loss="binder" takes pooled samples without one.')
        pooled = MCMCResult()
        pooled.clusts = clusts
        return getpointestimate(pooled, method, loss, device)
    return clusts[i], i


def getpointestimate(samples, method="MAP", loss="VI", device=0):
    """getpointestimate(samples; method, loss) -> (clust, i)   (pointestimate.jl:17-60); i is 0-based here.  `samples` is
    an MCMCResult or a list of them (runsampler with nchains > 1), pooled in list order with i indexing the
    concatenation; MPEL with loss="binder" over a list runs from the pooled co-clustering counts (binder_loss_sums)."""
    if method == "MPEL" and isinstance(loss, str) and loss not in _LOSS:
        raise ArgumentError("Invalid loss function specifier.")
    if method not in ("MAP", "MLE", "MPEL"):
        raise ArgumentError("Invalid method specifier.")
    if isinstance(samples, (list, tuple)):
        return _pooled_pointestimate(list(samples), method, loss, device)
    if method == "MAP":
        i = int(np.argmax(samples.logposterior))
    elif method == "MLE":
        i = int(np.argmax(samples.loglik))
    elif isinstance(loss, str):
        _, i = mpel_loss_sums(np.stack(samples.clusts), loss, device)
    else:                                                   # user-supplied loss: host loop, as the reference
        cl = samples.clusts
        S = len(cl)
        M = np.zeros((S, S))
        for a in range(S):
            for b in range(a + 1, S):
                M[a, b] = loss(cl[a], cl[b])
        i = int(np.argmin((M + M.T).sum(0)))
    return samples.clusts[i], i


def _pair_loss(a, b, loss):
    sums, _ = mpel_loss_sums(np.stack([np.asarray(a, np.int64), np.asarray(b, np.int64)]), loss)
    return float(sums[0])


def binderloss(a, b, normalised=True):
    if len(a) != len(b):
        raise ArgumentError("Length of the input vectors must be equal.")
    n = len(a)
    return _pair_loss(a, b, "binder") * (1 if normalised else n * (n - 1) // 2)


def infodist(a, b, normalised=True):
    if len(a) != len(b):
        raise ArgumentError("Length of the input vectors must be equal.")
    d = _pair_loss(a, b, "ID")
    if not normalised:
        return d
    n = len(a)
    def H(x):
        c = np.unique(x, return_counts=True)[1] / n
        return float(-(c * np.log(c)).sum())
    m = max(H(a), H(b))
    return 1 - (m - d) / m if m > 0 else float("nan")


def evaluateclustering(clusts, truth, device=0):
    """evaluateclustering(clusts, truth) (summaries.jl:13-24): nbloss, ari, vi, nvi, id, nid, nmi -- the four pair losses
    come from the contingency-table kernel (rc_mpel on the two label vectors), the entropies for the normalised
    mutual information (Clustering.mutualinfo: I / sqrt(H(a) H(b))) from the label counts."""
    a = np.asarray(clusts, dtype=np.int64); b = np.asarray(truth, dtype=np.int64)
    if a.size != b.size:
        raise ArgumentError("Length of inputs must be equal.")
    n = a.size
    two = np.stack([a, b])
    val = {loss: float(mpel_loss_sums(two, loss, device)[0][0]) for loss in ("binder", "omARI", "VI", "ID")}

    def entropy(x):
        c = np.bincount(np.unique(x, return_inverse=True)[1]).astype(np.float64)
        return float(math.log(n) - (c * np.log(c)).sum() / n)

    Ha, Hb = entropy(a), entropy(b)
    I = (Ha + Hb - val["VI"]) / 2
    nmi = I / math.sqrt(Ha * Hb) if Ha > 0 and Hb > 0 else (1.0 if Ha == Hb else 0.0)
    logn = math.log(n)
    return dict(nbloss=val["binder"], ari=1 - val["omARI"], vi=val["VI"], nvi=val["VI"] / logn, id=val["ID"], nid=val["ID"] / logn, nmi=nmi)


def summarise(clusts, truth, io=None, device=0):
    """summarise([io], clusts, truth) (summaries.jl:31-44)."""
    import sys as _sys
    out = _sys.stdout if io is None else io
    t = evaluateclustering(clusts, truth, device)
    print("Clustering summary", file=out)
    print(f"Number of clusters : {len(np.unique(np.asarray(clusts)))}", file=out)
    print(f"Normalised Binder loss : {t['nbloss']}", file=out)
    print(f"Adjusted Rand Index : {t['ari']}", file=out)
    print(f"Normalised Variation of Information (NVI) distance : {t['nvi']}", file=out)
    print(f"Normalised Information Distance (NID) : {t['nid']}", file=out)
    print(f"Normalised Mutual Information : {t['nmi']}", file=out)


def _oracle_coclustering(pts, K, alpha, radius, sigma, g, device, numiters=5000):
    """utils.jl:130-143: average over 5000 Dirichlet draws w of P' P, P[j, i] = w_j N(x_i; c_j, sigma^2 I) normalised
    over j.  The draws come from the host generator; the posteriors and the Gram products (chunks of draws stacked into
    one n x (B K) operand, FP64 tensor cores) run in librcb200 (rc_oracle_coclustering)."""
    X = np.ascontiguousarray(np.asarray(pts, dtype=np.float64))
    N, dim = X.shape
    W = np.ascontiguousarray(g.dirichlet(np.full(K, float(alpha)), size=numiters))             # numiters x K
    out = np.empty((N, N))
    check(lib().rc_oracle_coclustering(ptr(X), dim, N, K, float(radius), float(sigma), ptr(W), numiters, device, ptr(out)))
    return out


def generatemixture(N, K, alpha=None, dim=None, radius=1.0, sigma=0.1, rng=None, device=0, oracle=None):
    """generatemixture(N, K; α, dim, radius, σ, rng) (utils.jl:101-147): Dirichlet weights, sorted labels,
    simplex-vertex centres, isotropic normal points, Euclidean distance matrix (built on the GPU), and the oracle
    co-clustering matrix (utils.jl:130-143, always computed as in the reference -- about a second at N = 10 000;
    oracle=False skips it, it is not consumed by the sampler)."""
    alpha = K if alpha is None else alpha
    dim = K if dim is None else dim
    if N < 1:
        raise ArgumentError("N must be greater than 1.")
    if K < 1 or K > N:
        raise ArgumentError("K must satisfy 1 ≤ K ≤ N.")
    if alpha <= 0:
        raise ArgumentError("α must be positive.")
    if dim < K:
        raise ArgumentError("dim must be ≥ K.")
    if radius <= 0:
        raise ArgumentError("radius must be positive.")
    if sigma <= 0:
        raise ArgumentError("σ must be positive.")
    g = rng if isinstance(rng, np.random.Generator) else np.random.default_rng(rng)
    probs = g.dirichlet(np.full(K, float(alpha)))
    clusts = np.sort(g.choice(K, size=N, p=probs)) + 1
    pts = g.normal(0.0, sigma, size=(N, dim))
    pts[np.arange(N), clusts - 1] += radius
    data = MCMCData.from_points(pts, device=device)
    want = True if oracle is None else bool(oracle)
    occ = _oracle_coclustering(pts, K, alpha, radius, sigma, g, device) if want else None
    return dict(points=[pts[i] for i in range(N)], distancematrix=data.D, clusts=clusts.astype(np.int64), probs=probs,
                oracle_coclustering=occ, data=data)


class _NpzDatasets:
    """The package's own copy of the example data sets behind the interface of an open HDF5 file
    (handle["example1"]["points"], keys(), close())."""

    def __init__(self, path):
        self._z = np.load(path)

    def keys(self):
        return sorted({k.split("/")[0] for k in self._z.files})

    def __getitem__(self, group):
        if group not in self.keys():
            raise KeyError(group)
        z = self._z

        class _G:
            def keys(self_):
                return sorted(k.split("/")[1] for k in z.files if k.startswith(group + "/"))

            def __getitem__(self_, name):
                return z[f"{group}/{name}"]
        return _G()

    def close(self):
        self._z.close()


def example_datasets(path=None):
    """example_datasets() (example_data.jl:33-35): a read-only handle to the example data sets of the main paper; close
    it when done.  `path` (or the environment variable REDCLUST_EXAMPLE_DATA) names an HDF5 file of the reference's
    layout -- RedClust.jl's own data/example_datasets.h5 -- which is read by the package's minimal HDF5 reader
    (h5min.py); without it the package's own copy of the same arrays is opened.  Datasets come back in HDF5 dimension
    order (a Julia dim x N matrix as N x dim)."""
    path = path or os.environ.get("REDCLUST_EXAMPLE_DATA")
    if path:
        from .h5min import H5File
        return H5File(path)
    return _NpzDatasets(os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "example_datasets.npz"))


def example_dataset(n, path=None):
    """example_dataset(n) (example_data.jl:56-71): the n-th simulated example of the main paper (generated by the
    reference with seed 44, K = 10, N = 100, sigma = 0.25 / 0.2 / 0.18, dim = 10 / 50 / 10) as a dict with the fields of
    the reference's named tuple: points (list of N vectors), distmatrix, clusts, probs, oracle_coclustering."""
    if n not in (1, 2, 3):
        raise ArgumentError("n must be 1, 2, or 3.")
    f = example_datasets(path)
    try:
        eg = f["example" + str(n)]
        x = np.asarray(eg["points"])                                   # N x dim here = Julia's dim x N, column i = point i
        return dict(points=[x[i].copy() for i in range(x.shape[0])], distmatrix=np.asarray(eg["distance_matrix"]),
                    clusts=np.asarray(eg["cluster_labels"]).astype(np.int64), probs=np.asarray(eg["cluster_weights"]),
                    oracle_coclustering=np.asarray(eg["oracle_coclustering_probabilities"]))
    finally:
        f.close()


def pair_stats(data, labels):
    """Sufficient statistics of the within-cluster (A) and between-cluster (B) upper-triangle dissimilarities of a
    device-resident MCMCData for the Gamma fits of fitprior (prior.jl:73-110): counts, sums and sums of logs.
    The device returns exact integer row sums of the fixed-point images; they are added here as Python integers."""
    lab = np.ascontiguousarray(np.asarray(labels, dtype=np.int64))
    rows = np.zeros((data.n, 5), np.int64)
    check(lib().rc_pair_stats(data._h, ptr(lab), ptr(rows)))
    qD, qL = data.scales()
    wd, wl, ad, al, nw = (sum(map(int, rows[:, c])) for c in range(5))
    n = data.n
    nA, nB = nw, n * (n - 1) // 2 - nw
    return dict(nA=nA, sA=wd / 2.0 ** qD, lA=wl / 2.0 ** qL, nB=nB, sB=(ad - wd) / 2.0 ** qD, lB=(al - wl) / 2.0 ** qL)


def params_from_labels(D, labels, eta=None, sigma=None, u=None, v=None, **kw):
    """Hyperparameters from a notional clustering, exactly as fitprior does after its clustering step
    (prior.jl:73-110): Gamma MLE shapes of within / between distances, alpha = |A| delta1, beta = sum(A),
    zeta = |B| delta2, gamma = sum(B).  eta, sigma, u, v default to moment matches of (r, p) ~ NegBin fit."""
    from .prior import gamma_shape_from_stats
    labels = np.asarray(labels)
    K = len(np.unique(labels))
    if isinstance(D, MCMCData):                      # device path: one pass over the resident matrix
        st = pair_stats(D, labels)
        nA, sA, lA, nB, sB, lB = st["nA"], st["sA"], st["lA"], st["nB"], st["sB"], st["lB"]
        return _params_from_stats(nA, sA, lA, nB, sB, lB, K, eta, sigma, u, v, kw)
    D = np.asarray(D)
    n = D.shape[0]
    # sufficient statistics of the within-cluster (A) and between-cluster (B) upper-triangle distances
    tot_s, tot_l = 0.0, 0.0
    for i0 in range(0, n, 1024):
        blk = D[i0:i0 + 1024]
        tot_s += float(blk.sum())
        with np.errstate(divide="ignore"):
            lg = np.log(blk)
        lg[np.arange(blk.shape[0]), np.arange(i0, i0 + blk.shape[0])] = 0.0
        tot_l += float(lg.sum())
    tot_s = (tot_s - float(np.trace(D))) / 2; tot_l /= 2
    nA, sA, lA = 0, 0.0, 0.0
    for k in np.unique(labels):
        mem = np.where(labels == k)[0]
        if mem.size < 2:
            continue
        sub = D[np.ix_(mem, mem)]
        iu = np.triu_indices(mem.size, 1)
        vals = sub[iu]
        nA += vals.size; sA += float(vals.sum()); lA += float(np.log(vals).sum())
    nB, sB, lB = n * (n - 1) // 2 - nA, tot_s - sA, tot_l - lA
    return _params_from_stats(nA, sA, lA, nB, sB, lB, K, eta, sigma, u, v, kw)


def _params_from_stats(nA, sA, lA, nB, sB, lB, K, eta, sigma, u, v, kw):
    from .prior import gamma_shape_from_stats
    if nA:
        d1 = gamma_shape_from_stats(sA / nA, lA / nA); al, be = nA * d1, sA
    else:
        d1, al, be = 1.0, 1.0, 1.0
    if nB:
        d2 = gamma_shape_from_stats(sB / nB, lB / nB); ze, ga = nB * d2, sB
    else:
        d2, ze, ga = 1.0, 1.0, 1.0
    p = dict(delta1=d1, alpha=al, beta=be, delta2=d2, zeta=ze, gamma=ga, eta=4.0 if eta is None else eta,
             sigma=2.0 if sigma is None else sigma, u=2.0 if u is None else u, v=20.0 if v is None else v, K_initial=K)
    p.update(kw)
    return PriorHyperparamsList(**p)
