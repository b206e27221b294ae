"""ctypes binding of the CPU oracle (oracle/rc_oracle.cpp) plus numpy restatements of the
PSM and point-estimate code.  TEST INFRASTRUCTURE ONLY: imported by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs; the product
path (redclust.jl_b200/) never imports it.

Reference lines restated here in numpy:
  adjacencymatrix / PSM      /root/reference/src/utils.jl:59-63, src/mcmc.jl:560
  getpointestimate (MPEL)    /root/reference/src/pointestimate.jl:17-60
  binderloss / infodist      /root/reference/src/pointestimate.jl:68-98
  randindex / varinfo / mutualinfo are Clustering.jl (0.13.5-0.15, not vendored): restated from
  their published definitions (SURVEY.md Appendix B).
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_LOCK = __import__("threading").Lock()          # the tests call the oracle from a thread pool: build / load once


class Options(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("numiters", "burnin", "thin", "numGibbs", "numMH")]


class Params(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("delta1", "delta2", "alpha", "beta", "zeta", "gamma", "eta", "sigma",
                                         "proposalsd_r", "u", "v")] + [
        ("K_initial", C.c_int64), ("maxK", C.c_int64), ("repulsion", C.c_int32), ("_pad", C.c_int32)]


def build(force=False):
    so = os.path.join(_HERE, "librc_oracle.so")
    src = os.path.join(_HERE, "rc_oracle.cpp")
    deps = [src, os.path.join(_HERE, "..", "include", "rcb200.h"),
            os.path.join(_HERE, "..", "redclust.jl_b200", "csrc", "rc_math.h"),
            os.path.join(_HERE, "..", "redclust.jl_b200", "csrc", "rc_rng.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["make", "-C", _HERE, "-B", "librc_oracle.so"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        L = C.CDLL(build())
        dp = C.POINTER(C.c_double)
        L.rco_run.restype = C.c_int
        L.rco_loglik.restype = C.c_double
        L.rco_logprior.restype = C.c_double
        L.rco_time_chains.restype = C.c_double
        for f in ("rco_log", "rco_exp", "rco_log1p", "rco_lgamma", "rco_erfc", "rco_normcdf", "rco_norminv"):
            getattr(L, f).restype = C.c_double
            getattr(L, f).argtypes = [C.c_double]
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def make_options(numiters=5000, burnin=None, thin=1, numGibbs=5, numMH=1):
    if burnin is None:
        burnin = int(np.floor(0.2 * numiters))
    return Options(numiters, burnin, thin, numGibbs, numMH)


def make_params(**kw):
    d = dict(delta1=1.0, delta2=1.0, alpha=1.0, beta=1.0, zeta=1.0, gamma=1.0, eta=1.0, sigma=1.0,
             proposalsd_r=None, u=1.0, v=1.0, K_initial=1, maxK=0, repulsion=1)
    d.update(kw)
    if d["proposalsd_r"] is None:
        d["proposalsd_r"] = np.sqrt(d["eta"]) / d["sigma"]
    return Params(d["delta1"], d["delta2"], d["alpha"], d["beta"], d["zeta"], d["gamma"], d["eta"], d["sigma"],
                  d["proposalsd_r"], d["u"], d["v"], int(d["K_initial"]), int(d["maxK"]), int(bool(d["repulsion"])), 0)


def numsamples(o):
    return int(np.floor((o.numiters - o.burnin) / o.thin))


def run_chain(D, options, params, init_labels, init_r, init_p, seed=0, chain=0, sum_mode=0):
    """runsampler loop for one chain (mcmc.jl:537-555).  Returns a dict of traces."""
    D = np.ascontiguousarray(D, dtype=np.float64)
    n = D.shape[0]
    S = numsamples(options)
    out = dict(labels=np.zeros((S, n), np.int64), K=np.zeros(S, np.int64), r=np.zeros(S), p=np.zeros(S),
               loglik=np.zeros(S), logposterior=np.zeros(S), r_acc=np.zeros(options.numiters, np.uint8),
               sm_acc=np.zeros(options.numiters * options.numMH, np.uint8),
               sm_split=np.zeros(options.numiters * options.numMH, np.uint8),
               final_labels=np.zeros(n, np.int64), final_rp=np.zeros(2))
    init = np.ascontiguousarray(init_labels, dtype=np.int64)
    lib().rco_run(_p(D, C.c_double), C.c_int64(n), C.byref(options), C.byref(params), _p(init, C.c_int64),
                  C.c_double(init_r), C.c_double(init_p), C.c_uint64(seed), C.c_uint64(chain), C.c_int(sum_mode),
                  _p(out["labels"], C.c_int64), _p(out["K"], C.c_int64), _p(out["r"], C.c_double),
                  _p(out["p"], C.c_double), _p(out["loglik"], C.c_double), _p(out["logposterior"], C.c_double),
                  _p(out["r_acc"], C.c_uint8), _p(out["sm_acc"], C.c_uint8), _p(out["sm_split"], C.c_uint8),
                  _p(out["final_labels"], C.c_int64), _p(out["final_rp"], C.c_double))
    return out


def time_chains(D, options, params, init_labels, init_r, init_p, seed=0, chain0=0, nthreads=1, sum_mode=0):
    """Timed multi-chain run (bench.py cpu_baseline / --impl reference).  Returns (seconds in the loops, final K)."""
    D = np.ascontiguousarray(D, dtype=np.float64)
    n = D.shape[0]
    r = np.ascontiguousarray(init_r, dtype=np.float64); p = np.ascontiguousarray(init_p, dtype=np.float64)
    init = np.ascontiguousarray(init_labels, dtype=np.int64)
    K = np.zeros(r.size, np.int64)
    secs = lib().rco_time_chains(_p(D, C.c_double), C.c_int64(n), C.byref(options), C.byref(params), _p(init, C.c_int64),
                                 _p(r, C.c_double), _p(p, C.c_double), C.c_uint64(seed), C.c_int64(chain0),
                                 C.c_int64(r.size), C.c_int(nthreads), C.c_int(sum_mode), _p(K, C.c_int64))
    return secs, K


def loglik(D, params, labels, sum_mode=0):
    D = np.ascontiguousarray(D, dtype=np.float64)
    lab = np.ascontiguousarray(labels, dtype=np.int64)
    return lib().rco_loglik(_p(D, C.c_double), C.c_int64(D.shape[0]), C.byref(params), _p(lab, C.c_int64), C.c_int(sum_mode))


def logprior(params, labels, r, p):
    lab = np.ascontiguousarray(labels, dtype=np.int64)
    return lib().rco_logprior(C.c_int64(lab.size), C.byref(params), _p(lab, C.c_int64), C.c_double(r), C.c_double(p))


def logdist(D):
    D = np.ascontiguousarray(D, dtype=np.float64)
    out = np.zeros_like(D)
    lib().rco_logdist(_p(D, C.c_double), C.c_int64(D.shape[0]), _p(out, C.c_double))
    return out


def init_rp(params, seed, chain):
    r, p = C.c_double(), C.c_double()
    lib().rco_init_rp(C.byref(params), C.c_uint64(seed), C.c_uint64(chain), C.byref(r), C.byref(p))
    return r.value, p.value


def distm(points):
    """points: (n, dim) array (row i = observation i) -> n x n Euclidean distance matrix."""
    X = np.ascontiguousarray(points, dtype=np.float64)
    n, dim = X.shape
    D = np.zeros((n, n))
    lib().rco_distm(_p(X, C.c_double), C.c_int64(dim), C.c_int64(n), _p(D, C.c_double))
    return D


DIST_TAU = 2.0 ** -6        # rc_dist_unresolved's threshold (rc_math.h)


def distm_longdouble(X, Y=None):
    """sqrt(sum_t (x_it - y_jt)^2) in np.longdouble (x86 extended: 63-bit mantissa), one row at a time: the difference
    form, free of the Gram form's cancellation.  Y defaults to X."""
    assert np.finfo(np.longdouble).nmant >= 63, "np.longdouble is no wider than fp64 here"
    X = np.asarray(X, dtype=np.longdouble)
    Y = X if Y is None else np.asarray(Y, dtype=np.longdouble)
    R = np.empty((Y.shape[0], X.shape[0]), dtype=np.longdouble)
    for i in range(Y.shape[0]):
        R[i] = np.sqrt(((X - Y[i]) ** 2).sum(axis=1))
    return R


def distm_bound(dim):
    """Relative error every off-diagonal distance entry must meet: (dim + 4) u / tau, u = 2^-53 (DESIGN section 4)."""
    return (dim + 4) * 2.0 ** -53 / DIST_TAU


def distm_within_bound(D, R, dim):
    """Largest |D - R| / R over the entries with R > 0, over distm_bound(dim); entries with R == 0 must be exactly 0."""
    R = np.asarray(R, dtype=np.longdouble)
    pos = R > 0
    assert np.all(D[~pos] == 0), "identical points with a non-zero distance"
    assert np.all(D[pos] > 0), "distinct points with a zero distance"
    return float((np.abs(np.asarray(D, dtype=np.longdouble)[pos] - R[pos]) / R[pos]).max(initial=0) / distm_bound(dim))


def distance_family(name, n, dim, rng):
    """n x dim points on which the Gram form of the Euclidean distance loses accuracy to a different degree:
    centred        normal(0, 1);
    offset1e2/1e4  normal(0, 1) + 1e2 / 1e4 in every coordinate;
    utm            5e6 + normal(0, 100): projected geographic coordinates in metres (dim 2 in the tests);
    planted        centred points, pairs at separations 1e-3 ... 1e-9 of their norm;
    mixed          one coordinate near 1e6 (three distinct values, so many pairs share it), the others near 1e-3;
    collinear      a + t b for one random a, b."""
    if name == "centred":
        return rng.normal(size=(n, dim))
    if name in ("offset1e2", "offset1e4"):
        return rng.normal(size=(n, dim)) + float(name[6:])
    if name == "utm":
        return 5e6 + 100.0 * rng.normal(size=(n, dim))
    if name == "planted":
        X = rng.normal(size=(n, dim))
        for k, i in enumerate(range(0, n - 1, max(2, n // 8))):
            u = rng.normal(size=dim)
            X[i + 1] = X[i] + 10.0 ** -(3 + k % 7) * np.linalg.norm(X[i]) * u / np.linalg.norm(u)
        return X
    if name == "mixed":
        X = 1e-3 * rng.normal(size=(n, dim))
        X[:, 0] = 1e6 + rng.integers(0, 3, size=n)
        return X
    if name == "collinear":
        return rng.normal(size=dim)[None, :] + rng.uniform(-1, 1, size=n)[:, None] * rng.normal(size=dim)[None, :]
    raise ValueError(name)


DISTANCE_FAMILIES = ("centred", "offset1e2", "offset1e4", "utm", "planted", "mixed", "collinear")


def philox(ctr, key):
    c = np.asarray(ctr, np.uint32); k = np.asarray(key, np.uint32); o = np.zeros(4, np.uint32)
    lib().rco_philox(_p(c, C.c_uint32), _p(k, C.c_uint32), _p(o, C.c_uint32))
    return o


def draw2(seed, chain, it, site, mh, a, b):
    o = np.zeros(2)
    lib().rco_draw2(C.c_uint64(seed), C.c_uint64(chain), C.c_uint32(it), C.c_uint32(site), C.c_uint32(mh),
                    C.c_uint32(a), C.c_uint32(b), _p(o, C.c_double))
    return o


# ---------------------------------------------------------------------------------------------
# numpy restatements (integer / small fp work)
# ---------------------------------------------------------------------------------------------
def sortlabels(x):
    """utils.jl:69-74: first-appearance relabelling to 1..K."""
    m = {}
    out = np.empty(len(x), np.int64)
    for i, v in enumerate(x):
        out[i] = m.setdefault(int(v), len(m) + 1)
    return out


def adjacencymatrix(c):
    c = np.asarray(c)
    return c[:, None] == c[None, :]


def psm_counts(labels):
    """sum(adjacencymatrix.(clusts)) as exact integer counts (mcmc.jl:560)."""
    labels = np.asarray(labels)
    S, n = labels.shape
    cnt = np.zeros((n, n), np.int64)
    for s in range(S):
        cnt += adjacencymatrix(labels[s])
    return cnt


def psm(labels):
    labels = np.asarray(labels)
    return psm_counts(labels) / labels.shape[0]


def _contingency(a, b):
    a = np.asarray(a); b = np.asarray(b)
    ua, ia = np.unique(a, return_inverse=True)
    ub, ib = np.unique(b, return_inverse=True)
    c = np.zeros((ua.size, ub.size), np.int64)
    np.add.at(c, (ia, ib), 1)
    return c


def randindex(a, b):
    """Clustering.randindex -> (ARI, RI, Mirkin, Hubert)."""
    c = _contingency(a, b).astype(np.float64)
    n = c.sum()
    nis = (c.sum(1) ** 2).sum(); njs = (c.sum(0) ** 2).sum()
    t1 = n * (n - 1) / 2; t2 = (c ** 2).sum(); t3 = 0.5 * (nis + njs)
    nc = (n * (n ** 2 + 1) - (n + 1) * nis - (n + 1) * njs + 2 * (nis * njs) / n) / (2 * (n - 1))
    A = t1 + t2 - t3; Dg = -t2 + t3
    ari = 0.0 if t1 == nc else (A - nc) / (t1 - nc)
    return ari, A / t1, Dg / t1, (A - Dg) / t1


def _entropy(p):
    p = p[p > 0]
    return float(-(p * np.log(p)).sum())


def mutualinfo(a, b):
    c = _contingency(a, b).astype(np.float64)
    n = c.sum()
    pij = c / n; pi = pij.sum(1, keepdims=True); pj = pij.sum(0, keepdims=True)
    m = pij > 0
    return float((pij[m] * np.log(pij[m] / (pi @ pj)[m])).sum())


def varinfo(a, b):
    c = _contingency(a, b).astype(np.float64)
    n = c.sum()
    return _entropy(c.sum(1) / n) + _entropy(c.sum(0) / n) - 2 * mutualinfo(a, b)


def binderloss(a, b, normalised=True):
    if len(a) != len(b):
        raise ValueError("Length of the input vectors must be equal.")
    n = len(a)
    return randindex(a, b)[2] * (1 if normalised else n * (n - 1) // 2)


def infodist(a, b, normalised=True):
    if len(a) != len(b):
        raise ValueError("Length of the input vectors must be equal.")
    n = len(a)
    hu = _entropy(np.unique(a, return_counts=True)[1] / n)
    hv = _entropy(np.unique(b, return_counts=True)[1] / n)
    mi = mutualinfo(a, b)
    return 1 - mi / max(hu, hv) if normalised else max(hu, hv) - mi


LOSSES = {
    "binder": lambda x, y: randindex(x, y)[2],
    "omARI": lambda x, y: 1 - randindex(x, y)[0],
    "VI": varinfo,
    "ID": lambda x, y: infodist(x, y, normalised=False),
}


def mpel_loss_sums(labels, loss):
    """pointestimate.jl:49-57: column sums of the symmetrised S x S loss matrix."""
    fn = LOSSES[loss] if isinstance(loss, str) else loss
    S = len(labels)
    M = np.zeros((S, S))
    for i in range(S):
        for j in range(i + 1, S):
            M[i, j] = fn(labels[i], labels[j])
    M = M + M.T
    return M.sum(0)


def getpointestimate(result, method="MAP", loss="VI"):
    if method == "MPEL" and isinstance(loss, str) and loss not in LOSSES:
        raise ValueError("Invalid loss function specifier.")
    if method not in ("MAP", "MLE", "MPEL"):
        raise ValueError("Invalid method specifier.")
    if method == "MAP":
        i = int(np.argmax(result["logposterior"]))
    elif method == "MLE":
        i = int(np.argmax(result["loglik"]))
    else:
        i = int(np.argmin(mpel_loss_sums(result["labels"], loss)))
    return result["labels"][i], i


# ---- fitprior pieces (SURVEY 8f rank 1) ------------------------------------------------------------------
def kmedoids_fixed_point(D, q, init, maxiter=1000):
    """Clustering.kmedoids(dissM, k; maxiter) as used at /root/reference/src/prior.jl:55-71 and src/mcmc.jl:519-527
    (third-party code, restated: alternate nearest-medoid assignment -- first minimum -- and medoid update -- member
    with the smallest sum of dissimilarities to its cluster, lowest index on ties -- until nothing changes), with the
    medoid sums over the fixed-point image Dq = round(D 2^q) so that they are exact integers.
    Returns (assignments 1-based, medoids 0-based, converged, total cost as an integer in units of 2^-q)."""
    D = np.asarray(D, dtype=np.float64)
    Dq = np.rint(D * 2.0 ** q).astype(np.int64)
    med = np.array(init, dtype=np.int64)
    k = med.size
    assign = np.argmin(D[med], axis=0)
    conv = False
    for _ in range(maxiter):
        newmed = med.copy()
        for c in range(k):
            mem = np.where(assign == c)[0]
            if mem.size:
                newmed[c] = mem[np.argmin(Dq[np.ix_(mem, mem)].sum(0))]
        newassign = np.argmin(D[newmed], axis=0)
        same = np.array_equal(newmed, med) and np.array_equal(newassign, assign)
        med, assign = newmed, newassign
        if same:
            conv = True
            break
    return assign + 1, med, conv, int(Dq[med[assign], np.arange(D.shape[0])].sum())


def pair_stats(D, labels):
    """A = uppertriangle(dissM)[adjacency], B = the rest (/root/reference/src/prior.jl:73-75): counts, sums, log-sums."""
    D = np.asarray(D, dtype=np.float64); labels = np.asarray(labels)
    iu = np.triu_indices(D.shape[0], 1)
    adj = (labels[:, None] == labels[None, :])[iu]
    ut = D[iu]
    A, B = ut[adj], ut[~adj]
    return dict(nA=int(A.size), sA=float(A.sum()), lA=float(np.log(A).sum()), nB=int(B.size), sB=float(B.sum()), lB=float(np.log(B).sum()))


# ---- probes used by tests/test_oracle_pins.py ------------------------------------------------------------------
def scan_only(D, params, labels, r, p, iters, seed=0, chain=0, sum_mode=0):
    """`iters` full Gibbs scans (mcmc.jl:158-256) at fixed (r, p); returns the sortlabels'd state after each scan."""
    D = np.ascontiguousarray(D, dtype=np.float64)
    n = D.shape[0]
    lab = np.ascontiguousarray(labels, dtype=np.int64)
    out = np.zeros((iters, n), np.int64)
    lib().rco_scan_only(_p(D, C.c_double), C.c_int64(n), C.byref(params), _p(lab, C.c_int64), C.c_double(r), C.c_double(p),
                        C.c_uint64(seed), C.c_uint64(chain), C.c_int64(iters), C.c_int(sum_mode), _p(out, C.c_int64))
    return out


def gibbs_logprobs(D, params, labels, r, p, i, sum_mode=1):
    """Candidate slots (1-based, the reference's order) and the un-normalised log-probabilities of the scan step of
    point i (0-based) in the given state (mcmc.jl:193-247)."""
    D = np.ascontiguousarray(D, dtype=np.float64)
    n = D.shape[0]
    lab = np.ascontiguousarray(labels, dtype=np.int64)
    cand = np.zeros(n + 1, np.int64); lp = np.zeros(n + 1)
    L = lib()
    L.rco_gibbs_logprobs.restype = C.c_int64
    m = L.rco_gibbs_logprobs(_p(D, C.c_double), C.c_int64(n), C.byref(params), _p(lab, C.c_int64), C.c_double(r), C.c_double(p),
                             C.c_int64(i), C.c_int(sum_mode), _p(cand, C.c_int64), _p(lp, C.c_double))
    return cand[:m].copy(), lp[:m].copy()


def draws(kind, a, b, count, seed=0):
    """Raw draws of the shared samplers: kind 'gamma' (shape a), 'beta' (a, b), 'truncnorm' (mean a, sd b, lower 0),
    'randint' (1..a)."""
    k = {"gamma": 0, "beta": 1, "truncnorm": 2, "randint": 3}[kind]
    out = np.zeros(count)
    lib().rco_draws(C.c_int(k), C.c_double(a), C.c_double(b), C.c_uint64(seed), C.c_int64(count), _p(out, C.c_double))
    return out


def sample_rp(clustsizes, options, params, seed=0):
    """mcmc.jl:592-636 on the CPU: dict(r, p, r_acc)."""
    cs = np.ascontiguousarray(clustsizes, dtype=np.int64)
    S = numsamples(options)
    out = dict(r=np.zeros(S), p=np.zeros(S), r_acc=np.zeros(options.numiters, np.uint8))
    lib().rco_sample_rp(_p(cs, C.c_int64), C.c_int64(cs.size), C.byref(options), C.byref(params), C.c_uint64(seed),
                        _p(out["r"], C.c_double), _p(out["p"], C.c_double), _p(out["r_acc"], C.c_uint8))
    return out


def kmeans_lloyd(X, init, maxiter=1000, tol=1e-6):
    """Lloyd iterations of Clustering.kmeans from the given seeds (numpy; checker of rc_kmeans): X n x dim points, init 0-based
    seed points.  Nearest centre (first minimum), centre = mean of members (an empty cluster keeps its centre), stop when no
    label changes or the objective moves by less than tol.  Returns 1-based assignments, centres (k x dim), cost, converged, iterations."""
    P = np.asarray(X, dtype=np.float64)
    cent = P[np.asarray(init)].copy()
    k = cent.shape[0]

    def assign_pass():
        d = ((P[:, None, :] - cent[None, :, :]) ** 2).sum(2)
        a = np.argmin(d, axis=1)
        return a, float(d[np.arange(P.shape[0]), a].sum())
    a, obj = assign_pass()
    conv, it = False, 0
    while not conv and it < maxiter:
        it += 1
        for c in range(k):
            m = a == c
            if m.any():
                cent[c] = P[m].mean(0)
        na, nobj = assign_pass()
        if k == 1 or np.array_equal(na, a) or abs(nobj - obj) < tol:
            conv = True
        a, obj = na, nobj
    return a + 1, cent, obj, conv, it
