"""The fixed-point images across the scale of the data.

Every path that sums dissimilarities (the chain kernel, rc_loglik, the predictive scan step, k-medoids, the pair statistics
of fitprior) reads {Dq, Lq} = {round(D 2^qD), round(log D 2^qL)}, q = rc_choose_q(max|.|, n): the largest q with
n max|.| 2^q < 2^61.  Kernels and oracle share rc_choose_q, so their bit parity says nothing about it; here D is scaled by c
from 2^-60 to 2^60 (and by three factors that are not powers of two), beta and gamma with it, and the results are checked
  * against an mpmath (50 digits) statement of the scan conditional (src/mcmc.jl:193-247) and of loglik (mcmc.jl:1-56),
    into which the fp64 distances and hyperparameters go exactly;
  * against three exact properties of the model:
    (1) c = 2^k scales D exactly and qD shifts by -k, so the D image is bit-identical: every D-side integer sum is the
        same integer and its value is exactly 2^k times the unscaled one (k-medoids, the pair statistics, beta, gamma);
    (2) with repulsion on, every candidate of the scan shifts by the same -(n - 1) log c, so its probabilities do not
        depend on the scale (with repulsion off the shift is -n_k log c; that case is checked against mpmath only);
    (3) loglik(cD, beta c, gamma c) = loglik(D) - C(n, 2) log c with repulsion on.
"""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest
from mpmath import mp, mpf

POW2 = [-60, -40, -20, 0, 20, 40, 60]
OTHER = [1e-12, 3.3e-7, 7e11]
SCALES = [2.0 ** k for k in POW2] + OTHER
SCALE_IDS = [f"2^{k}" for k in POW2] + [repr(c) for c in OTHER]
BASE = dict(delta1=2.5, delta2=3.0, alpha=40.0, beta=30.0, zeta=50.0, gamma=120.0, eta=4.0, sigma=2.0, u=2.0, v=8.0,
            K_initial=2, maxK=0)


def scaled(d, c):
    """Hyperparameters for the data c D: the Gamma rates beta and gamma carry the unit of D."""
    return dict(d, beta=d["beta"] * c, gamma=d["gamma"] * c)


def mixture(n, K, dim, sigma, seed):
    g = np.random.default_rng(seed)
    lab = np.sort(g.choice(K, size=n, p=g.dirichlet(np.full(K, float(K))))) + 1
    lab = (np.unique(lab, return_inverse=True)[1] + 1).astype(np.int64)
    X = g.normal(0, sigma, size=(n, dim))
    X[np.arange(n), lab - 1] += 1.0
    return X, lab


def dist(X):
    sq = (X * X).sum(1)
    D = np.sqrt(np.maximum(sq[:, None] + sq[None, :] - 2 * X @ X.T, 0))
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0.0)
    return D


def oracle_scales(orc, D):
    import ctypes as C
    D = np.ascontiguousarray(D)
    qd, ql = C.c_int(), C.c_int()
    orc.lib().rco_fixedpoint_scales(D.ctypes.data_as(C.POINTER(C.c_double)), C.c_int64(D.shape[0]), C.byref(qd), C.byref(ql))
    return qd.value, ql.value


# ---- the mpmath statements ------------------------------------------------------------------------------------------
def mp_conditional(D, d, labels, r, p, i):
    """Candidates (ascending slots, then the first empty slot) and log-probabilities of the scan step of point i,
    src/mcmc.jl:193-247, in 50-digit arithmetic."""
    mp.dps = 50
    n = D.shape[0]
    lab = np.array(labels).copy()
    lab[i] = -1
    slots = sorted(set(lab[lab > 0].tolist()))
    Ki = len(slots)
    cand = list(slots)
    if (d["maxK"] == 0 or Ki < d["maxK"]) and Ki < n:
        cand.append(min(s for s in range(1, n + 1) if s not in slots))
    al, be, ze, ga, d1, d2 = (mpf(float(d[k])) for k in ("alpha", "beta", "zeta", "gamma", "delta1", "delta2"))
    r, p = mpf(float(r)), mpf(float(p))
    abr = al * mp.log(be) - mp.loggamma(al)
    zgr = ze * mp.log(ga) - mp.loggamma(ze)
    L1, L2p, pri = {}, {}, {}
    for k in slots:
        mem = np.flatnonzero(lab == k)
        nk = len(mem)
        vals = [mpf(float(D[i, j])) for j in mem]
        s, l = mp.fsum(vals), mp.fsum(mp.log(v) for v in vals)
        a_i, b_i, z_i, g_i = al + d1 * nk, be + s, ze + d2 * nk, ga + s
        L1[k] = mp.loggamma(a_i) + abr - a_i * mp.log(b_i) + (d1 - 1) * l - nk * mp.loggamma(d1)
        L2p[k] = mp.loggamma(z_i) - z_i * mp.log(g_i) + zgr + (d2 - 1) * l - nk * mp.loggamma(d2)
        pri[k] = mp.log(nk + 1) + mp.log(p) + mp.log(nk - 1 + r) - mp.log(nk)
    L2i = mp.fsum(L2p.values())
    rep = bool(d["repulsion"])
    lp = [pri[k] + L1[k] + ((L2i - L2p[k]) if rep else 0) if k in L1 else mp.log(Ki + 1) + r * mp.log(1 - p) + (L2i if rep else 0)
          for k in cand]
    return np.array(cand), lp


def mp_normalised(lp):
    """lp - logsumexp(lp) in 50 digits, as float64."""
    mp.dps = 50
    v = [mpf(x) for x in lp]
    lse = mp.log(mp.fsum(mp.exp(x) for x in v))
    return np.array([float(x - lse) for x in v])


def mp_loglik(D, d, labels):
    """loglik, src/mcmc.jl:1-56 (the model's log-likelihood of the clustering), in 50-digit arithmetic."""
    mp.dps = 50
    n = D.shape[0]
    ks = sorted(set(np.asarray(labels).tolist()))
    idx = {k: t for t, k in enumerate(ks)}
    c = np.array([idx[k] for k in labels])
    K = len(ks)
    S = [[mpf(0)] * K for _ in range(K)]
    L = [[mpf(0)] * K for _ in range(K)]
    for i in range(n):
        for j in range(i + 1, n):
            v = mpf(float(D[i, j]))
            a, b = min(c[i], c[j]), max(c[i], c[j])
            S[a][b] += v
            L[a][b] += mp.log(v)
    size = np.bincount(c, minlength=K)
    al, be, ze, ga, d1, d2 = (mpf(float(d[k])) for k in ("alpha", "beta", "zeta", "gamma", "delta1", "delta2"))
    tot = mpf(0)
    for a in range(K):
        pairs = int(size[a]) * (int(size[a]) - 1) // 2
        A, B = al + d1 * pairs, be + S[a][a]
        tot += (d1 - 1) * L[a][a] - pairs * mp.loggamma(d1) + al * mp.log(be) - mp.loggamma(al) + mp.loggamma(A) - A * mp.log(B)
        if d["repulsion"]:
            for b in range(a + 1, K):
                pairs = int(size[a]) * int(size[b])
                Z, G = ze + d2 * pairs, ga + S[a][b]
                tot += (d2 - 1) * L[a][b] - pairs * mp.loggamma(d2) + ze * mp.log(ga) - mp.loggamma(ze) + mp.loggamma(Z) - Z * mp.log(G)
    return tot


# ---- problems (built once per session) -------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def conditional_problems():
    """(D, labels, r, p, points): three mixtures of n = 50, 160 and 400 points, two label states each (the generating
    labels and a random state with arbitrary slot ids), three points per state."""
    g = np.random.default_rng(17)
    out = []
    for n, K, seed in ((50, 3, 1), (160, 5, 2), (400, 8, 3)):
        X, lab = mixture(n, K, 10, 0.2, seed)
        D = dist(X)
        ids = g.choice(np.arange(1, n + 1), size=K + 2, replace=False)
        for labels in (lab, ids[g.integers(0, K + 2, size=n)]):
            out.append((D, labels, float(g.gamma(2.0)) + 0.05, float(g.uniform(0.05, 0.95)), g.choice(n, 3, replace=False)))
    return out


def golden_states(golden):
    """Example set 1 with its generating labels and a random labelling in 1..6."""
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"].astype(np.int64)
    return D, (lab, np.random.default_rng(1).integers(1, 7, size=lab.size).astype(np.int64))


_MP_LOGLIK = {}


def mp_loglik_cached(D, d, labels, c):
    key = (D.tobytes(), np.asarray(labels).tobytes(), c, bool(d["repulsion"]))
    if key not in _MP_LOGLIK:
        _MP_LOGLIK[key] = mp_loglik(D * c, scaled(d, c), labels)
    return _MP_LOGLIK[key]


# ---- CPU: the oracle ---------------------------------------------------------------------------------------------------
def expected_q(m, n):
    """rc_choose_q's rule: the largest q with n m 2^q < 2^61 (the product n m taken in fp64, as the C code does)."""
    v = m * n
    if v == 0:
        return 50
    q = 61 - math.frexp(v)[1]
    return min(max(q, -1022), 1022)


@pytest.mark.parametrize("which", ["example1", "mixture2000"])
def test_fixedpoint_scales_follow_the_data(orc, golden, which):
    D = golden[1]["distance_matrix"] if which == "example1" else dist(mixture(2000, 10, 10, 0.25, 5)[0])
    n = D.shape[0]
    q0 = oracle_scales(orc, D)
    for k, c in zip(POW2 + [None] * len(OTHER), SCALES):
        Dc = D * c
        qD, qL = oracle_scales(orc, Dc)
        mD, mL = np.abs(Dc).max(), np.abs(orc.logdist(Dc)).max()
        assert (qD, qL) == (expected_q(mD, n), expected_q(mL, n)), c
        for q, m in ((qD, mD), (qL, mL)):                   # every sum of n entries fits, at no more than 2 bits short
            assert Fraction(m) * n * Fraction(2) ** q < 2 ** 61 <= Fraction(m) * n * Fraction(2) ** (q + 2), (c, q)
        if k is not None:
            assert qD == q0[0] - k, (k, qD, q0)


def test_fixedpoint_scale_limits(orc):
    assert oracle_scales(orc, np.zeros((1, 1))) == (50, 50)                     # all-zero data: any q is exact
    D = np.array([[0.0, 2.0 ** -1000], [2.0 ** -1000, 0.0]])
    assert oracle_scales(orc, D)[0] == 1022                                     # n max|D| < 2^-961: the upper clamp
    D = np.array([[0.0, 1e300], [1e300, 0.0]])
    assert oracle_scales(orc, D)[0] == 61 - math.frexp(2e300)[1]


@pytest.mark.parametrize("repulsion", [1, 0])
@pytest.mark.parametrize("c", SCALES, ids=SCALE_IDS)
def test_oracle_conditional_against_mpmath(orc, c, repulsion):
    """Oracle scan step (sum_mode 0, the kernels' fixed-point sums) at scale c: normalised log-probabilities within 1e-9
    of the 50-digit statement; with repulsion on, within 1e-10 of the unscaled conditional (property 2)."""
    d = dict(BASE, repulsion=repulsion)
    dc = scaled(d, c)
    P, P1 = orc.make_params(**dc), orc.make_params(**d)
    worst = worst_scale = 0.0
    for D, labels, r, p, points in conditional_problems():
        Dc = D * c
        for i in points:
            cand, lp = orc.gibbs_logprobs(Dc, P, labels, r, p, int(i), sum_mode=0)
            cand_mp, lp_mp = mp_conditional(Dc, dc, labels, r, p, int(i))
            assert np.array_equal(cand, cand_mp)
            err = np.abs(mp_normalised(lp) - mp_normalised(lp_mp)).max()
            worst = max(worst, err)
            if repulsion:
                _, lp1 = orc.gibbs_logprobs(D, P1, labels, r, p, int(i), sum_mode=0)
                worst_scale = max(worst_scale, np.abs(mp_normalised(lp) - mp_normalised(lp1)).max())
    assert worst <= 1e-9, worst
    assert worst_scale <= 1e-10, worst_scale


@pytest.mark.parametrize("c", SCALES, ids=SCALE_IDS)
def test_oracle_loglik_against_mpmath(orc, golden, c):
    """Oracle loglik (sum_mode 0) within 1e-12 relative of the 50-digit statement at scale c, and property 3."""
    D, states = golden_states(golden)
    for rep in (1, 0):
        d = dict(BASE, repulsion=rep)
        for labels in states:
            got = orc.loglik(D * c, orc.make_params(**scaled(d, c)), labels, sum_mode=0)
            ref = mp_loglik_cached(D, d, labels, c)
            assert abs(got - float(ref)) <= 1e-12 * abs(float(ref)), (rep, got, float(ref))
            if rep:
                n = D.shape[0]
                base = orc.loglik(D, orc.make_params(**d), labels, sum_mode=0)
                shift = n * (n - 1) // 2 * math.log(c)
                assert abs(got - (base - shift)) <= 1e-12 * (abs(base) + abs(shift)), (got, base, shift)


def test_oracle_loglik_shift_larger_mixture(orc):
    """Property 3 on n = 400 at every scale (the oracle alone)."""
    X, lab = mixture(400, 8, 10, 0.2, 7)
    D = dist(X)
    d = dict(BASE, repulsion=1)
    base = orc.loglik(D, orc.make_params(**d), lab, sum_mode=0)
    for c in SCALES:
        got = orc.loglik(D * c, orc.make_params(**scaled(d, c)), lab, sum_mode=0)
        shift = 400 * 399 // 2 * math.log(c)
        assert abs(got - (base - shift)) <= 1e-12 * (abs(base) + abs(shift)), (c, got, base - shift)


def test_kmedoids_fixed_point_power_of_two_scales(orc, golden):
    """Property 1 for the k-medoids restatement the device kernel is checked against: the same assignments, medoids
    and integer cost at every 2^k, the cost exactly 2^k times."""
    D = golden[1]["distance_matrix"]
    init = np.random.default_rng(4).choice(100, size=10, replace=False)
    q0 = oracle_scales(orc, D)[0]
    a0, m0, c0, cost0 = orc.kmedoids_fixed_point(D, q0, init)
    for k in POW2:
        Dk = D * 2.0 ** k
        q = oracle_scales(orc, Dk)[0]
        a, m, conv, cost = orc.kmedoids_fixed_point(Dk, q, init)
        assert np.array_equal(a, a0) and np.array_equal(m, m0) and conv == c0, k
        assert cost == cost0 and cost / 2.0 ** q == 2.0 ** k * (cost0 / 2.0 ** q0), (k, cost, cost0)


def test_oracle_chain_power_of_two_scales(orc):
    """Properties 2 and 3 through a whole chain of the oracle (repulsion on, same seed): at 2^-40 and 2^40 every
    decision is the unscaled chain's and the loglik trace is shifted by C(n, 2) k ln 2."""
    X, lab = mixture(200, 5, 10, 0.2, 9)
    D = dist(X)
    d = dict(BASE, repulsion=1)
    opts = orc.Options(20, 0, 1, 3, 2)
    ref = orc.run_chain(D, opts, orc.make_params(**d), lab, 1.3, 0.4, seed=3)
    for k in (-40, 40):
        got = orc.run_chain(D * 2.0 ** k, opts, orc.make_params(**scaled(d, 2.0 ** k)), lab, 1.3, 0.4, seed=3)
        assert_same_decisions(got, ref)
        assert_loglik_shift(got["loglik"], ref["loglik"], 200, k)


def assert_same_decisions(got, ref):
    for f in ("r_acc", "sm_acc", "sm_split", "K", "labels", "r", "p"):
        bad = np.flatnonzero(np.asarray(got[f] != ref[f]).reshape(len(got[f]), -1).any(1))
        assert bad.size == 0, (f, "first difference at record", bad[:1])


def assert_loglik_shift(got, ref, n, k):
    shift = n * (n - 1) // 2 * k * math.log(2)
    rel = np.abs(got - (ref - shift)) / np.abs(ref - shift)
    assert rel.max() <= 1e-12, (k, rel.max())


# ---- device ------------------------------------------------------------------------------------------------------------
def dev_loglik(pkg, data, params, labels):
    import ctypes as C
    from redclust_jl_b200._lib import lib, check, ptr
    out = C.c_double()
    q = params._c()
    check(lib().rc_loglik(data._h, C.byref(q), ptr(np.ascontiguousarray(labels, dtype=np.int64)), C.byref(out)))
    return out.value


@pytest.mark.gpu
def test_device_scales_equal_oracle(pkg, orc, golden):
    D = golden[1]["distance_matrix"]
    for c in SCALES:
        assert pkg.MCMCData(D * c).scales() == oracle_scales(orc, D * c), c
    assert pkg.MCMCData(np.zeros((1, 1))).scales() == (50, 50)
    huge = np.array([[0.0, 1e308], [1e308, 0.0]])                 # n max|D| overflows fp64
    with pytest.raises(pkg.RCError, match="too large"):
        pkg.MCMCData(huge)
    assert pkg.MCMCData(huge / 1e8).scales()[0] == oracle_scales(orc, huge / 1e8)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("c", SCALES, ids=SCALE_IDS)
def test_device_loglik_at_scale(pkg, orc, golden, c):
    """rc_loglik bit-equal to the oracle and within 1e-12 relative of the 50-digit statement."""
    D, states = golden_states(golden)
    data = pkg.MCMCData(D * c)
    for rep in (1, 0):
        d = dict(BASE, repulsion=rep)
        dc = scaled(d, c)
        for labels in states:
            got = dev_loglik(pkg, data, pkg.PriorHyperparamsList(**dc), labels)
            assert got == orc.loglik(D * c, orc.make_params(**dc), labels, sum_mode=0)
            ref = float(mp_loglik_cached(D, d, labels, c))
            assert abs(got - ref) <= 1e-12 * abs(ref), (rep, got, ref)


def sortlabels(x):
    _, first, inv = np.unique(x, return_index=True, return_inverse=True)
    return (np.argsort(np.argsort(first))[inv] + 1).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("repulsion", [1, 0])
def test_device_predictive_at_scale(pkg, orc, golden, repulsion):
    """predictive_from_labels with D and Dnew scaled together: log-probabilities bit-equal to the oracle's scan step on
    the augmented data and within 1e-9 (normalised) of the 50-digit statement; with repulsion on the probabilities
    agree with the unscaled run's to 1e-10 (property 2)."""
    X = golden[1]["points"]
    held = np.array([3, 41, 77, 98])
    keep = np.setdiff1d(np.arange(X.shape[0]), held)
    Dfull = dist(X)
    D, Dn = np.ascontiguousarray(Dfull[np.ix_(keep, keep)]), np.ascontiguousarray(Dfull[np.ix_(held, keep)])
    n = D.shape[0]
    g = np.random.default_rng(8)
    labs = np.stack([golden[1]["cluster_labels"][keep], g.integers(1, 7, size=n)]).astype(np.int64)
    r, p = np.array([1.3, 0.6]), np.array([0.4, 0.8])
    d = dict(BASE, repulsion=repulsion)
    base = pkg.predictive_from_labels(pkg.MCMCData(D), Dn, labs, r, p, pkg.PriorHyperparamsList(**d))
    for c in SCALES:
        dc = scaled(d, c)
        out = pkg.predictive_from_labels(pkg.MCMCData(D * c), Dn * c, labs, r, p, pkg.PriorHyperparamsList(**dc), logprobs=True)
        P = orc.make_params(**dc)
        for s in range(labs.shape[0]):
            for x in range(Dn.shape[0]):
                Da = np.zeros((n + 1, n + 1))
                Da[:n, :n] = D * c; Da[n, :n] = Dn[x] * c; Da[:n, n] = Dn[x] * c
                la = np.append(sortlabels(labs[s]), 1)
                cand, lp = orc.gibbs_logprobs(Da, P, la, r[s], p[s], n, sum_mode=0)
                got = out["logprobs"][s, x][: cand.size]
                assert np.array_equal(got.view(np.int64), lp.view(np.int64)), (c, s, x)
                _, lp_mp = mp_conditional(Da, dc, la, r[s], p[s], n)
                assert np.abs(mp_normalised(got) - mp_normalised(lp_mp)).max() <= 1e-9, (c, s, x)
        if repulsion:
            for f in ("coclustering", "newcluster"):
                assert np.abs(out[f] - base[f]).max() <= 1e-10, (c, f, np.abs(out[f] - base[f]).max())


def run_device(pkg, D, lab, d, opts, seed, nchains):
    params = pkg.PriorHyperparamsList(**d)
    data = pkg.MCMCData(np.ascontiguousarray(D))
    rp = [pkg.init_rp(params, seed, ch) for ch in range(nchains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (nchains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=seed)
    smp.run(-1)
    assert smp.check_sums() == (0, 0)
    return [smp.samples(ch) for ch in range(nchains)], rp


@pytest.mark.gpu
def test_device_sampler_at_scale(pkg, orc):
    """Four chains of n = 500 (numGibbs 3, numMH 2, repulsion on) at 2^-40 and 2^40: every output bit-identical to the
    oracle (k_build_dl, the cached terms and the 128-bit block totals at the new q), and every decision the unscaled
    run's with the loglik trace shifted by C(n, 2) k ln 2 (properties 2 and 3)."""
    X, lab = mixture(500, 8, 10, 0.3, 11)
    D = dist(X)
    fit = pkg.params_from_labels(D, lab)
    d = {f: getattr(fit, f) for f in fit._fields}
    lab = np.random.default_rng(2).integers(1, 4, size=500).astype(np.int64)   # a start from which the chain moves
    opts = pkg.MCMCOptionsList(numiters=24, burnin=4, thin=1, numGibbs=3, numMH=2)
    base, _ = run_device(pkg, D, lab, d, opts, 21, 4)
    for k in (-40, 40):
        dc = scaled(d, 2.0 ** k)
        got, rp = run_device(pkg, D * 2.0 ** k, lab, dc, opts, 21, 4)
        for ch in range(4):
            ref = orc.run_chain(D * 2.0 ** k, orc.Options(24, 4, 1, 3, 2), orc.make_params(**dc), lab, rp[ch][0], rp[ch][1],
                                seed=21, chain=ch)
            for f in ("r_acc", "sm_acc", "sm_split", "K", "labels", "r", "p", "loglik", "logposterior"):
                assert np.array_equal(got[ch][f], ref[f]), (k, ch, f)
            assert_same_decisions(got[ch], base[ch])
            assert_loglik_shift(got[ch]["loglik"], base[ch]["loglik"], 500, k)


@pytest.mark.gpu
def test_device_kmedoids_and_pair_stats_power_of_two_scales(pkg, orc, golden):
    """kmedoids_device, pair_stats and params_from_labels(data) at every 2^k: property 1 (same assignments, medoids and
    convergence, cost exactly 2^k times, equal to the restatement), sA and sB (beta, gamma) exactly 2^k times, the
    Gamma shapes delta1, delta2 and alpha, zeta within 1e-12 relative."""
    from redclust_jl_b200.prior import kmedoids_device
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    init = np.random.default_rng(4).choice(100, size=10, replace=False)
    data0 = pkg.MCMCData(D)
    km0, st0, pr0 = kmedoids_device(data0, 10, init_medoids=init), pkg.pair_stats(data0, lab), pkg.params_from_labels(data0, lab)
    for k in POW2:
        c = 2.0 ** k
        data = pkg.MCMCData(D * c)
        qD = data.scales()[0]
        km = kmedoids_device(data, 10, init_medoids=init)
        a, med, conv, cost_q = orc.kmedoids_fixed_point(D * c, qD, init)
        assert np.array_equal(km["assignments"], a) and np.array_equal(km["medoids"], med) and km["converged"] == conv
        assert km["totalcost"] == cost_q / 2.0 ** qD
        assert np.array_equal(km["assignments"], km0["assignments"]) and np.array_equal(km["medoids"], km0["medoids"])
        assert km["totalcost"] == c * km0["totalcost"], (k, km["totalcost"], km0["totalcost"])
        st = pkg.pair_stats(data, lab)
        assert st["nA"] == st0["nA"] and st["sA"] == c * st0["sA"] and st["sB"] == c * st0["sB"], k
        pr = pkg.params_from_labels(data, lab)
        assert pr.beta == c * pr0.beta and pr.gamma == c * pr0.gamma, k
        for f in ("delta1", "delta2", "alpha", "zeta"):
            assert abs(getattr(pr, f) - getattr(pr0, f)) <= 1e-12 * abs(getattr(pr0, f)), (k, f)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [None, "dmma32", "exact"])
def test_device_from_points_power_of_two_scales(pkg, golden, monkeypatch, mode):
    """MCMCData.from_points(2^k X) is bit-equal to 2^k from_points(X) on every distance path: the Gram form scales by
    2^2k exactly and the recompute test compares relative sizes."""
    if mode is None:
        monkeypatch.delenv("RCB200_DISTM", raising=False)
    else:
        monkeypatch.setenv("RCB200_DISTM", mode)
    for X in (golden[1]["points"], np.random.default_rng(6).normal(size=(300, 37)) + 10.0):
        a = pkg.MCMCData.from_points(X)
        D0, q0 = a.D, a.scales()[0]
        for k in (-100, -20, 20, 100):
            b = pkg.MCMCData.from_points(X * 2.0 ** k)
            assert np.array_equal(b.D, D0 * 2.0 ** k), (mode, k)
            assert b.scales()[0] == q0 - k


@pytest.mark.gpu
def test_device_fitprior_kmeans_upscaled(pkg, golden):
    """fitprior(points 2^k, "k-means"): the k-means++ weights, the Lloyd centres and distances and the knee of the
    elbow scale exactly, so the same clustering and hyperparameters come out, beta and gamma exactly 2^k times.  Only
    k > 0: Clustering.jl's kmeans (restated as is) stops when the objective moves by less than an absolute 1e-6, which at
    2^-20 ends every run after its first pass."""
    pts = golden[1]["points"]
    p0 = pkg.fitprior(list(pts), "k-means", False, Kmin=1, Kmax=15, verbose=False, rng=1)
    for k in (20, 40):
        c = 2.0 ** k
        pk = pkg.fitprior(list(pts * c), "k-means", False, Kmin=1, Kmax=15, verbose=False, rng=1)
        assert pk.K_initial == p0.K_initial, k
        assert pk.beta == c * p0.beta and pk.gamma == c * p0.gamma, k
        for f in ("eta", "sigma", "u", "v", "proposalsd_r"):
            assert getattr(pk, f) == getattr(p0, f), (k, f)
        for f in ("delta1", "delta2", "alpha", "zeta"):
            assert abs(getattr(pk, f) - getattr(p0, f)) <= 1e-12 * abs(getattr(p0, f)), (k, f)
