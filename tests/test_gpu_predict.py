"""Posterior predictive allocation of new observations (rc_predict, rc_sampler_predict, rc_crossdist): the scan step's
conditional (mcmc.jl:193-247) for a point that is not in the data, bit-identical to the oracle's scan step on the augmented
data, its softmax (utils.jl:2-6), and the ascending-order averages over samples."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def dist(X):
    D = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1))
    return (D + D.T) / 2


def split(X, held):
    """Training matrix, held-out rows (m x n) of the full matrix, training indices."""
    keep = np.setdiff1d(np.arange(X.shape[0]), held)
    D = dist(X)
    return np.ascontiguousarray(D[np.ix_(keep, keep)]), np.ascontiguousarray(D[np.ix_(held, keep)]), keep


def random_params(g, K):
    d = dict(delta1=float(g.uniform(1, 4)), delta2=float(g.uniform(1, 4)), alpha=float(g.uniform(1, 8)), beta=float(g.uniform(1, 8)),
             zeta=float(g.uniform(1, 8)), gamma=float(g.uniform(1, 8)), eta=4.0, sigma=2.0, u=2.0, v=8.0, K_initial=2,
             maxK=int(g.choice([0, K, K + 1])), repulsion=int(g.integers(0, 2)))
    return d


def sortlabels(x):
    _, first, inv = np.unique(x, return_index=True, return_inverse=True)
    return (np.argsort(np.argsort(first))[inv] + 1).astype(np.int64)


def oracle_lp(orc, D, drow, P, lab, r, p):
    """The oracle's scan step of point n of the augmented data, which carries an existing label."""
    n = D.shape[0]
    Da = np.zeros((n + 1, n + 1))
    Da[:n, :n] = D; Da[n, :n] = drow; Da[:n, n] = drow
    la = np.append(sortlabels(lab), 1)
    return orc.gibbs_logprobs(Da, P, la, r, p, n, sum_mode=0)


def problems(golden):
    g = np.random.default_rng(11)
    for t in range(60):
        if t % 4 == 3:                                       # held-out points of the reference's example data
            X = golden[1 + (t // 4) % 3]["points"]
            held = g.choice(X.shape[0], size=int(g.integers(2, 5)), replace=False)
        else:                                                # points as in test_oracle_pins.small_problem
            n = int(g.integers(5, 301)); m = int(g.integers(1, 4))
            X = g.normal(size=(n + m, 3)); X[: (n + m) // 2] += 2.0
            held = np.arange(n, n + m)
        D, Dn, _ = split(X, held)
        n = D.shape[0]
        K = int(g.integers(1, min(12, n) + 1))
        S = int(g.integers(1, 4))
        labs = []
        for _ in range(S):
            base = np.concatenate([np.arange(1, K + 1), g.integers(1, K + 1, size=n - K)])
            g.shuffle(base)
            ids = g.choice(np.arange(1, 1000), size=K, replace=False)   # arbitrary positive labels
            labs.append(ids[base - 1])
        d = random_params(g, K)
        r = g.gamma(2.0, size=S) + 0.05
        p = g.uniform(0.05, 0.95, size=S)
        yield D, Dn, np.stack(labs), r, p, d


def test_logprobs_bit_identical_to_oracle_scan_step(pkg, orc, golden):
    checked = 0
    for D, Dn, labs, r, p, d in problems(golden):
        data = pkg.MCMCData(D)
        out = pkg.predictive_from_labels(data, Dn, labs, r, p, pkg.PriorHyperparamsList(**d), logprobs=True)
        P = orc.make_params(**d)
        for s in range(labs.shape[0]):
            for x in range(Dn.shape[0]):
                cand, lp = oracle_lp(orc, D, Dn[x], P, labs[s], r[s], p[s])
                got = out["logprobs"][s, x]
                assert np.count_nonzero(~np.isnan(got)) == cand.size
                assert np.array_equal(cand, np.arange(1, cand.size + 1))
                assert np.array_equal(got[: cand.size].view(np.int64), lp.view(np.int64)), (got[: cand.size], lp)
                checked += 1
    assert checked > 150


def softmax(lp):
    e = np.exp(lp - lp.max())
    return e / e.sum()


def test_probabilities_are_the_softmax_of_the_logprobs(pkg, golden):
    for D, Dn, labs, r, p, d in problems(golden):
        data = pkg.MCMCData(D)
        params = pkg.PriorHyperparamsList(**d)
        lp = pkg.predictive_from_labels(data, Dn, labs, r, p, params, logprobs=True)["logprobs"]
        for s in range(labs.shape[0]):
            A = pkg.allocationprobabilities(data, Dn, labs[s], r[s], p[s], params)
            K = len(np.unique(labs[s]))
            assert A.shape == (Dn.shape[0], K + 1)
            assert np.all(np.abs(A.sum(1) - 1) < 1e-14)
            for x in range(Dn.shape[0]):
                row = lp[s, x][~np.isnan(lp[s, x])]
                P = softmax(row)
                slot_of_col = sortlabels(labs[s])[np.unique(labs[s], return_index=True)[1]] - 1
                assert np.all(np.abs(A[x, :K] - P[slot_of_col]) < 1e-14)
                assert abs(A[x, K] - (P[K] if P.size == K + 1 else 0.0)) < 1e-14


def golden_split(golden, k, nheld):
    X, lab = golden[k]["points"], golden[k]["cluster_labels"]
    step = X.shape[0] // nheld
    held = np.arange(nheld) * step + step // 2
    D, Dn, keep = split(X, held)
    return X, lab, held, D, Dn, keep


def run_chain(pkg, D, lab, iters, burnin, seed, nchains=1):
    params = pkg.params_from_labels(D, lab)
    data = pkg.MCMCData(D)
    opts = pkg.MCMCOptionsList(numiters=iters, burnin=burnin)
    res = pkg.runsampler(data, opts, params, init=pkg.MCMCState(lab, 1.5, 0.9), verbose=False, seed=seed, nchains=nchains)
    return data, params, res


def test_averages_against_numpy_statement(pkg, golden):
    X, lab, held, D, Dn, keep = golden_split(golden, 1, 20)
    data, params, res = run_chain(pkg, D, lab[keep], 250, 50, seed=3)
    labs, S = np.stack(res.clusts), len(res.clusts)
    assert S == 200
    got = pkg.predictivecoclustering(res, data, Dn)
    lp = pkg.predictive_from_labels(data, Dn, labs, res.r, res.p, params, logprobs=True)["logprobs"]
    m, n = Dn.shape
    acc, accn = np.zeros((m, n)), np.zeros(m)
    for s in range(S):
        for x in range(m):
            P = softmax(lp[s, x][~np.isnan(lp[s, x])])
            acc[x] += P[labs[s] - 1]
            accn[x] += P[labs[s].max()] if P.size > labs[s].max() else 0.0
    assert np.all(np.abs(got["coclustering"] - acc / S) < 1e-13)
    assert np.all(np.abs(got["newcluster"] - accn / S) < 1e-13)
    same = np.all(labs[:, :, None] == labs[:, None, :], axis=0)
    i, j = np.nonzero(np.triu(same, 1))
    assert i.size > 0
    assert np.array_equal(got["coclustering"][:, i], got["coclustering"][:, j])


def test_batch_invariance_and_permutation(pkg, golden):
    X, lab, held, D, Dn, keep = golden_split(golden, 2, 10)
    data, params, res = run_chain(pkg, D, lab[keep], 60, 10, seed=5)
    all_ = pkg.predictivecoclustering(res, data, Dn)
    for x in range(Dn.shape[0]):
        one = pkg.predictivecoclustering(res, data, Dn[x:x + 1])
        assert np.array_equal(one["coclustering"][0], all_["coclustering"][x])
        assert np.array_equal(one["newcluster"][0], all_["newcluster"][x])
    perm = np.random.default_rng(1).permutation(Dn.shape[0])
    pp = pkg.predictivecoclustering(res, data, Dn[perm])
    assert np.array_equal(pp["coclustering"], all_["coclustering"][perm])
    assert np.array_equal(pp["newcluster"], all_["newcluster"][perm])


@pytest.mark.parametrize("grouped", [False, True])
def test_device_samples_equal_host_path(pkg, golden, monkeypatch, grouped):
    if grouped:
        monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", "1")
    X, lab, held, D, Dn, keep = golden_split(golden, 3, 10)
    params = pkg.params_from_labels(D, lab[keep])
    data = pkg.MCMCData(D)
    nch, seed = 4, 2
    rp = [pkg.init_rp(params, seed, c) for c in range(nch)]
    smp = pkg.Sampler(data, pkg.MCMCOptionsList(numiters=40, burnin=10), params, np.tile(lab[keep], (nch, 1)),
                      [x[0] for x in rp], [x[1] for x in rp], seed=seed)
    smp.run(-1)
    sa = smp.samples_all()
    n = data.n
    for c0, k in ((0, 3), (1, 2)):
        dev = smp.predict(Dn, c0, k)
        host = pkg.predictive_from_labels(data, Dn, sa["labels"][c0:c0 + k].reshape(-1, n), sa["r"][c0:c0 + k].ravel(),
                                          sa["p"][c0:c0 + k].ravel(), params)
        assert np.array_equal(dev["coclustering"], host["coclustering"])
        assert np.array_equal(dev["newcluster"], host["newcluster"])
    smp.close()


def test_sample_chunks_do_not_change_results(pkg, golden, monkeypatch):
    """The samples are processed in chunks whose running fp64 sums carry over (RCB200_PREDICT_CHUNK caps the chunk size):
    chunks of 7 samples, host and device samples, and the log-probabilities of every chunk equal the one-chunk call."""
    X, lab, held, D, Dn, keep = golden_split(golden, 1, 10)
    params = pkg.params_from_labels(D, lab[keep])
    data = pkg.MCMCData(D)
    nch, seed = 3, 4
    rp = [pkg.init_rp(params, seed, c) for c in range(nch)]
    smp = pkg.Sampler(data, pkg.MCMCOptionsList(numiters=60, burnin=10), params, np.tile(lab[keep], (nch, 1)),
                      [x[0] for x in rp], [x[1] for x in rp], seed=seed)
    smp.run(-1)
    sa = smp.samples_all()
    L, r, p = sa["labels"].reshape(-1, data.n), sa["r"].ravel(), sa["p"].ravel()
    one = pkg.predictive_from_labels(data, Dn, L, r, p, params, logprobs=True)
    dev_one = smp.predict(Dn, 1, 2)
    monkeypatch.setenv("RCB200_PREDICT_CHUNK", "7")
    many = pkg.predictive_from_labels(data, Dn, L, r, p, params, logprobs=True)
    dev_many = smp.predict(Dn, 1, 2)
    for k in ("coclustering", "newcluster"):
        assert np.array_equal(one[k], many[k])
        assert np.array_equal(dev_one[k], dev_many[k])
    assert np.array_equal(one["logprobs"].view(np.int64), many["logprobs"].view(np.int64))
    smp.close()


def test_sampler_predict_needs_complete_samples(pkg, golden):
    """Samples are recorded only by a run to numiters: before that, the device path refuses instead of reading unwritten labels."""
    X, lab, held, D, Dn, keep = golden_split(golden, 2, 5)
    params = pkg.params_from_labels(D, lab[keep])
    smp = pkg.Sampler(pkg.MCMCData(D), pkg.MCMCOptionsList(numiters=30, burnin=5), params, lab[keep], 1.5, 0.9, seed=1)
    smp.run(10)
    with pytest.raises(pkg.RCError) as e:
        smp.predict(Dn)
    assert e.value.status == -6
    smp.run(-1)
    assert np.all(np.isfinite(smp.predict(Dn)["coclustering"]))
    smp.close()


def test_crossdistances_bit_equal_to_stacked_build(pkg, golden):
    for k in (1, 2, 3):
        X = golden[k]["points"]
        held = np.arange(3, X.shape[0], 9)
        keep = np.setdiff1d(np.arange(X.shape[0]), held)
        got = pkg.crossdistances(X[keep], X[held])
        full = pkg.MCMCData.from_points(np.vstack([X[keep], X[held]])).D
        assert np.array_equal(got, full[keep.size:, :keep.size])


def test_errors(pkg, golden):
    X, lab, held, D, Dn, keep = golden_split(golden, 1, 4)
    data = pkg.MCMCData(D)
    params = pkg.params_from_labels(D, lab[keep])
    L = lab[keep][None, :]
    with pytest.raises(pkg.ArgumentError):
        pkg.predictive_from_labels(data, Dn[:, :-1], L, [1.0], [0.5], params)
    for bad in (0.0, -1.0, np.nan, np.inf, -np.inf):
        B = Dn.copy(); B[1, 7] = bad
        with pytest.raises(pkg.RCError) as e:
            pkg.predictive_from_labels(data, B, L, [1.0], [0.5], params)
        assert e.value.status == -4 and "strictly positive" in str(e.value)
    data_big = pkg.MCMCData(dist(np.random.default_rng(0).normal(size=(300, 3))))   # one cluster per point: 300 labels
    with pytest.raises(pkg.RCError) as e:
        pkg.predictive_from_labels(data_big, np.ones((1, 300)), np.arange(1, 301)[None, :], [1.0], [0.5], params)
    assert e.value.status == -5
    for r, p in ((0.0, 0.5), (-1.0, 0.5), (np.nan, 0.5), (1.0, 0.0), (1.0, 1.0), (1.0, np.nan)):
        with pytest.raises(pkg.RCError) as e:
            pkg.predictive_from_labels(data, Dn, L, [r], [p], params)
        assert e.value.status == -1
    out = pkg.predictive_from_labels(data, Dn, np.zeros((0, data.n), np.int64), [], [], params)
    assert np.all(np.isnan(out["coclustering"])) and np.all(np.isnan(out["newcluster"]))


@pytest.mark.parametrize("k", [1, 2, 3])
def test_predictive_against_reference_held_oracle_coclustering(pkg, golden, k):
    """Held-out points of the reference's example data: their predictive co-clustering with the training points against the
    rows the reference ships (`oracle_coclustering_probabilities`, src/utils.jl:130-143) -- the generating mixture's true
    co-clustering probabilities.  2500 iterations on the other 90 points, hyperparameters from the true labels.  Measured:
    mean absolute difference 0.040 / 0.016 / 1.2e-5, correlation 0.82 / 0.94 / 1.00; the bounds leave Monte Carlo room."""
    X, lab, held, D, Dn, keep = golden_split(golden, k, 10)
    data, params, res = run_chain(pkg, D, lab[keep], 2500, 500, seed=k)
    got = pkg.predictivecoclustering(res, data, Dn)["coclustering"]
    cc = golden[k]["oracle_coclustering_probabilities"][np.ix_(held, keep)]
    mad = np.abs(got - cc).mean()
    cor = np.corrcoef(got.ravel(), cc.ravel())[0, 1]
    print(f"example{k}: mean |diff| {mad:.4g}, correlation {cor:.4g}")
    assert mad < 0.06
    assert cor > 0.7
