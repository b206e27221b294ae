"""GPU parity tests of the persistent chain kernel against the CPU oracle (same structured random stream):
label trajectories, K, r, p, acceptances bit-exact; loglik / logposterior bit-exact (the block sums are
exact integers, so the fp64 evaluation sees identical inputs) -- the north-star tolerance is 1e-10 relative."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def oparams(orc, params):
    return orc.make_params(**{k: getattr(params, k) for k in params._fields})


def run_both(pkg, orc, D, labels, params, numiters, burnin, thin, numGibbs, numMH, seed, nchains=1, slot_cap=0):
    opts = pkg.MCMCOptionsList(numiters=numiters, burnin=burnin, thin=thin, numGibbs=numGibbs, numMH=numMH)
    data = pkg.MCMCData(np.ascontiguousarray(D))
    labs = np.tile(np.asarray(labels, np.int64), (nchains, 1))
    rp = [pkg.init_rp(params, seed, c) for c in range(nchains)]
    smp = pkg.Sampler(data, opts, params, labs, [x[0] for x in rp], [x[1] for x in rp], seed=seed, slot_cap=slot_cap)
    smp.run(-1)
    assert smp.check_sums() == (0, 0)                        # incrementally maintained sums == a rebuild from the labels
    out = []
    for c in range(nchains):
        got = smp.samples(c)
        ref = orc.run_chain(D, orc.Options(numiters, burnin, thin, numGibbs, numMH), oparams(orc, params), labels,
                            rp[c][0], rp[c][1], seed=seed, chain=c)
        st = smp.state(c)
        out.append((got, ref, st))
    return out, smp


def assert_same(got, ref, st=None):
    assert np.array_equal(got["r_acc"], ref["r_acc"])
    assert np.array_equal(got["sm_split"], ref["sm_split"])
    assert np.array_equal(got["sm_acc"], ref["sm_acc"])
    assert np.array_equal(got["K"], ref["K"])
    assert np.array_equal(got["labels"], ref["labels"])
    for k in ("r", "p", "loglik", "logposterior"):
        assert np.array_equal(got[k], ref[k]), (k, got[k][:4], ref[k][:4])
    if st is not None:
        assert np.array_equal(st.clusts, ref["final_labels"])
        assert st.r == ref["final_rp"][0] and st.p == ref["final_rp"][1]


def mixture(n, K, dim, sigma, seed):
    g = np.random.default_rng(seed)
    w = g.dirichlet(np.full(K, float(K)))
    lab = np.sort(g.choice(K, size=n, p=w)) + 1
    lab = (np.unique(lab, return_inverse=True)[1] + 1).astype(np.int64)
    X = g.normal(0, sigma, size=(n, dim))
    X[np.arange(n), lab - 1] += 1.0
    return X, lab


def test_loglik_matches_oracle(pkg, orc, golden):
    for k in (1, 2, 3):
        D, lab = golden[k]["distance_matrix"], golden[k]["cluster_labels"]
        params = pkg.params_from_labels(D, lab)
        data = pkg.MCMCData(D)
        import ctypes as C
        out = C.c_double()
        q = params._c()
        from redclust_jl_b200._lib import lib, check, ptr
        for labels in (lab, np.random.default_rng(k).integers(1, 7, size=lab.size)):
            labels = np.ascontiguousarray(labels, dtype=np.int64)
            check(lib().rc_loglik(data._h, C.byref(q), ptr(labels), C.byref(out)))
            assert out.value == orc.loglik(D, oparams(orc, params), labels)


def test_fixture_gibbs_only(pkg, orc, golden):
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    (res,), _ = run_both(pkg, orc, D, lab, params, 60, 10, 1, 5, 0, seed=11)
    assert_same(*res)


def test_fixture_default_options(pkg, orc, golden):
    for k in (1, 2, 3):
        D, lab = golden[k]["distance_matrix"], golden[k]["cluster_labels"]
        params = pkg.params_from_labels(D, lab)
        (res,), _ = run_both(pkg, orc, D, lab, params, 150, 30, 3, 5, 1, seed=100 + k)
        assert_same(*res)
        assert res[1]["sm_split"].sum() > 0 and (1 - res[1]["sm_split"]).sum() > 0      # both move types exercised


def test_single_cluster_start_and_no_repulsion(pkg, orc, golden):
    D = golden[3]["distance_matrix"]
    lab = np.ones(100, np.int64)
    params = pkg.params_from_labels(D, golden[3]["cluster_labels"], repulsion=False)
    (res,), _ = run_both(pkg, orc, D, lab, params, 80, 0, 1, 3, 1, seed=5)
    assert_same(*res)


def test_maxK_and_numGibbs0(pkg, orc, golden):
    D, lab = golden[2]["distance_matrix"], golden[2]["cluster_labels"]
    params = pkg.params_from_labels(D, lab, maxK=10)
    (res,), _ = run_both(pkg, orc, D, lab, params, 80, 0, 1, 0, 1, seed=9)
    assert_same(*res)
    assert res[0]["K"].max() <= 10


def test_multichain_n1000(pkg, orc):
    X, lab = mixture(1000, 20, 50, 0.18, 3)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    res, smp = run_both(pkg, orc, D, lab, params, 12, 2, 2, 5, 1, seed=77, nchains=4)
    for got, ref, st in res:
        assert_same(got, ref, st)
    allc = smp.samples_all()                               # one-call read-back of every chain == the per-chain reads
    for c, (got, _, _) in enumerate(res):
        for k in got:
            assert np.array_equal(allc[k][c], got[k]), k
    # PSM counts of the device-resident samples are exact integers
    S = res[0][1]["labels"].shape[0]
    psm = smp.psm(0, 4)
    cnt = sum(orc.psm_counts(r[1]["labels"]) for r in res)
    assert np.array_equal(psm, cnt / (4 * S))


def test_multitile_n2500_resume(pkg, orc):
    X, lab = mixture(2500, 12, 20, 0.2, 8)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=6, burnin=0, thin=1)
    r0, p0 = pkg.init_rp(params, 1, 0)
    smp = pkg.Sampler(data, opts, params, lab, r0, p0, seed=1)
    smp.run(2); smp.run(1); smp.run(-1)                   # resumable: three launches == one run
    got = smp.samples(0)
    ref = orc.run_chain(D, orc.Options(6, 0, 1, 5, 1), oparams(orc, params), lab, r0, p0, seed=1, chain=0)
    assert_same(got, ref, smp.state(0))


def test_slot_overflow_is_reported(pkg, golden):
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1)
    smp = pkg.Sampler(pkg.MCMCData(D), opts, params, lab, 1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError) as e:
        smp.run(-1)
    assert e.value.status == -5


def test_slot_overflow_stops_only_the_chain_that_overflowed(pkg, orc, golden):
    """With several chains the run succeeds as long as one chain is healthy; rc_sampler_chain_status names the stopped
    ones and the healthy chains still match the oracle bit for bit."""
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=40, burnin=0, thin=1)
    nch = 24
    rp = [pkg.init_rp(params, 2, c) for c in range(nch)]
    for cap in (12, 13, 14, 15, 16, 17, 18, 11):
        smp = pkg.Sampler(pkg.MCMCData(D), opts, params, np.tile(lab, (nch, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=2, slot_cap=cap)
        try:
            smp.run(-1)
        except pkg.RCError as e:
            assert e.status == -5 and smp.overflowed() == nch
            continue
        st = [smp.chain_status(c) for c in range(nch)]
        assert sum(1 for x in st if x) == smp.overflowed() < nch
        if 0 < smp.overflowed():
            for c in range(nch):
                if st[c] == 0:
                    ref = orc.run_chain(D, orc.Options(40, 0, 1, 5, 1), oparams(orc, params), lab, rp[c][0], rp[c][1], seed=2, chain=c)
                    assert_same(smp.samples(c), ref, smp.state(c))
            return
    pytest.skip("no slot capacity in 11..18 stopped some but not all of the chains")


@pytest.mark.parametrize("m", [1, 2])
def test_launch_groups_are_bit_identical(pkg, orc, golden, monkeypatch, m):
    """Chains run in launch groups of m (the mode of chains whose row sums do not all fit the device): every launch rebuilds
    the row sums from the labels with every cache stale, and the results do not change a bit; 3 chains leave a ragged last
    group for m = 2.  check_sums covers the last group."""
    monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", str(m))
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    res, _ = run_both(pkg, orc, D, lab, params, 60, 0, 2, 5, 1, seed=31 + m, nchains=3)
    for got, ref, st in res:
        assert_same(got, ref, st)


def test_launch_groups_resume_n2500(pkg, orc, monkeypatch):
    """One chain per launch group at n = 2500, resumed: every call rebuilds each group's state, and three calls equal one run."""
    monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", "1")
    X, lab = mixture(2500, 12, 20, 0.2, 8)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=4, burnin=0, thin=1)
    rp = [pkg.init_rp(params, 2, c) for c in range(2)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (2, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=2)
    smp.run(2); smp.run(1); smp.run(-1)
    assert smp.check_sums() == (0, 0)
    for c in range(2):
        ref = orc.run_chain(D, orc.Options(4, 0, 1, 5, 1), oparams(orc, params), lab, rp[c][0], rp[c][1], seed=2, chain=c)
        assert_same(smp.samples(c), ref, smp.state(c))


def test_several_proposals_per_iteration(pkg, orc, golden):
    """numMH > 1: an accepted proposal becomes the local state of the remaining proposals of the iteration (and, by
    quirk Q1, never reaches the chain's own state)."""
    D = golden[3]["distance_matrix"]
    params = pkg.params_from_labels(D, golden[3]["cluster_labels"], repulsion=False)
    (res,), _ = run_both(pkg, orc, D, np.ones(100, np.int64), params, 60, 0, 1, 3, 4, seed=5)   # splits accepted often
    assert_same(*res)
    assert res[1]["sm_acc"].sum() > 10
    for k in (1, 2):
        D, lab = golden[k]["distance_matrix"], golden[k]["cluster_labels"]
        params = pkg.params_from_labels(D, lab)
        (res,), _ = run_both(pkg, orc, D, lab, params, 80, 10, 2, 5, 3, seed=60 + k)
        assert_same(*res)


def test_tiny_problems_and_many_slots(pkg, orc):
    """n = 2 ... 65 with weak priors: chains wander between 1 and n clusters, i.e. through the empty-slot allocation, the
    switch from 4 to 8 lanes per row of the scan once a slot beyond 63 is live, singleton split / merge proposals and
    numMH in {0, 1, 3}."""
    rng = np.random.default_rng(0)
    params = pkg.PriorHyperparamsList(delta1=2.0, alpha=5.0, beta=3.0, delta2=2.5, zeta=6.0, gamma=4.0, eta=4.0, sigma=2.0,
                                      u=2.0, v=10.0, K_initial=2)
    P = oparams(orc, params)
    seen = set()
    for n in (2, 3, 5, 33, 65):
        X = rng.normal(size=(n, 3)); X[: n // 2] += 3
        data = pkg.MCMCData.from_points(X)
        D = data.D
        lab = np.array([1] * (n // 2) + [2] * (n - n // 2), dtype=np.int64)
        for numMH in (0, 1, 3):
            opts = pkg.MCMCOptionsList(numiters=30, burnin=3, thin=2, numGibbs=2, numMH=numMH)
            r0, p0 = pkg.init_rp(params, 9, 0)
            smp = pkg.Sampler(data, opts, params, lab, r0, p0, seed=9)
            smp.run(-1)
            got = smp.samples(0)
            ref = orc.run_chain(D, orc.Options(30, 3, 2, 2, numMH), P, lab, r0, p0, seed=9, chain=0)
            assert_same(got, ref, smp.state(0))
            seen.update(int(k) for k in got["K"])
    assert 1 in seen and max(seen) >= 60            # from a single cluster to (nearly) one cluster per point


def test_points_in_random_order(pkg, orc):
    """Cluster members scattered over the points (no cluster is a contiguous run of rows) and a start that is 4 % off:
    three chains."""
    X, lab = mixture(3000, 25, 30, 0.15, 21)
    perm = np.random.default_rng(4).permutation(lab.size)
    X, lab = X[perm], orc.sortlabels(lab[perm])
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(data, lab)
    g = np.random.default_rng(6)
    init = lab.copy(); idx = g.choice(lab.size, 120, replace=False); init[idx] = g.integers(1, lab.max() + 1, size=idx.size)
    res, smp = run_both(pkg, orc, D, init, params, 5, 0, 1, 5, 1, seed=13, nchains=3)
    for got, ref, st in res:
        assert_same(got, ref, st)


@pytest.mark.parametrize("env", [
    dict(RCB200_INC_THREADS="256"),                                                       # the bench configuration: 64 threads on the restricted scans
    dict(RCB200_INC_THREADS="256", RCB200_RS_TEAM="32"),
    dict(RCB200_INC_THREADS="256", RCB200_OVERLAP_MIN_THREADS="0"),                       # scan after the restricted scans
    dict(RCB200_INC_THREADS="256", RCB200_TW_SMEM="0"),                                   # validity counts of the cached terms in global memory
    dict(RCB200_INC_THREADS="512", RCB200_RS_TEAM="256"),
    dict(RCB200_INC_THREADS="128"),
    dict(RCB200_INC_THREADS="64", RCB200_OVERLAP_MIN_THREADS="64", RCB200_RS_TEAM="32"),
])
def test_team_shapes_are_bit_identical(pkg, orc, monkeypatch, env):
    """The chain kernel's team shapes (threads per chain, threads on the restricted scans, scan beside or after them,
    where the cached terms' validity counts live) change the schedule, never a bit: a chain that moves points, splits and
    merges (loose mixture, wrong initial labels), three chains, against the oracle; the maintained sums equal a rebuild."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    X, lab = mixture(700, 9, 12, 0.45, 21)
    g = np.random.default_rng(3)
    init = lab.copy()
    flip = g.random(lab.size) < 0.3
    init[flip] = g.integers(1, 10, size=int(flip.sum()))
    init = (np.unique(init, return_inverse=True)[1] + 1).astype(np.int64)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab, maxK=40)          # (the loose mixture would open hundreds of clusters)
    res, smp = run_both(pkg, orc, D, init, params, 25, 0, 1, 5, 1, seed=5, nchains=3)
    assert smp.check_sums() == (0, 0)
    moved = 0
    for got, ref, st in res:
        assert_same(got, ref, st)
        moved += int((np.diff(ref["labels"].astype(np.int64), axis=0) != 0).sum())
    splits = sum(int(r[1]["sm_split"].sum()) for r in res)
    assert moved > 200 and 0 < splits < 75                       # the run moved points and proposed both splits and merges


@pytest.mark.parametrize("shortcuts", ["1", "0"])
def test_shortcuts_fire_and_change_nothing(pkg, orc, monkeypatch, shortcuts):
    """Row summaries (a row whose stored leader margin proves the Gumbel-max outcome is not evaluated) and the bound that
    rejects hopeless merge proposals without their restricted scans: on a well separated mixture most rows and most merge
    proposals take the shortcut, and every output still equals the oracle's -- as it does with RCB200_SHORTCUTS=0."""
    monkeypatch.setenv("RCB200_SHORTCUTS", shortcuts)
    X, lab = mixture(600, 6, 10, 0.12, 4)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    iters, nch = 40, 2
    res, smp = run_both(pkg, orc, D, lab, params, iters, 0, 1, 5, 1, seed=9, nchains=nch)
    assert smp.check_sums() == (0, 0)
    for got, ref, st in res:
        assert_same(got, ref, st)
    st = smp.stats()
    fast_rows, quick_rejects = int(st["bulk_rows"].sum()), int(st["dec_wait"].sum())     # (counts in the default library)
    merges = sum(int((r[1]["sm_split"] == 0).sum()) for r in res)
    if shortcuts == "1":
        assert fast_rows > 0.5 * iters * nch * 600, fast_rows
        assert quick_rejects > 0.5 * merges, (quick_rejects, merges)
    else:
        assert fast_rows == 0 and quick_rejects == 0
    # a chain that moves (loose mixture, wrong start): summaries are invalidated by every move, proposals are sometimes accepted
    X2, lab2 = mixture(500, 8, 10, 0.4, 11)
    g = np.random.default_rng(1)
    init = g.integers(1, 5, size=500)
    init = (np.unique(init, return_inverse=True)[1] + 1).astype(np.int64)
    data2 = pkg.MCMCData.from_points(X2)
    params2 = pkg.params_from_labels(data2.D, lab2, maxK=30)
    res2, smp2 = run_both(pkg, orc, data2.D, init, params2, 30, 0, 1, 5, 1, seed=2, nchains=2)
    assert smp2.check_sums() == (0, 0)
    for got, ref, st in res2:
        assert_same(got, ref, st)
