"""GPU parity at the BASELINE.json configurations (sizes the CPU oracle still finishes in seconds on the box's cores):
  configs[1]  n = 1000, K = 20, dim = 50, 64 chains -- shortened replay (300 of the 10 000 iterations), EVERY chain
              compared bit for bit with the oracle on the same structured random stream;
  configs[3]  n = 2000, many chains -- 128 chains (one GPU's share of the 1024) x 20 iterations, every chain compared;
  configs[4]  n = 50 000 is a PSM / point-estimate case: exact co-clustering counts at n = 20 000 on sampled rows and the
              MPEL search at S = 512 candidate samples against a vectorised numpy statement of pointestimate.jl:34-59.
Launch groups (the mode of chains whose row sums do not all fit the device) are exercised where it is cheap."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from test_gpu_sampler import assert_same, mixture, oparams  # noqa: E402


def oracle_chains(orc, D, opts, P, lab, rp, seed, chains):
    """The oracle for many chains at once: one chain per host thread (ctypes releases the GIL)."""
    def one(c):
        return orc.run_chain(D, orc.Options(*opts), P, lab, rp[c][0], rp[c][1], seed=seed, chain=c)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        return list(ex.map(one, chains))


def replay(pkg, orc, n, K, dim, sigma, nchains, iters, burnin, thin, seed, chains_per_group=None):
    X, lab = mixture(n, K, dim, sigma, seed)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=iters, burnin=burnin, thin=thin, numGibbs=5, numMH=1)
    rp = [pkg.init_rp(params, seed, c) for c in range(nchains)]
    old = os.environ.get("RCB200_CHAINS_PER_GROUP")
    if chains_per_group:
        os.environ["RCB200_CHAINS_PER_GROUP"] = str(chains_per_group)
    try:
        smp = pkg.Sampler(data, opts, params, np.tile(lab, (nchains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=seed)
    finally:
        if chains_per_group:
            os.environ.pop("RCB200_CHAINS_PER_GROUP") if old is None else os.environ.__setitem__("RCB200_CHAINS_PER_GROUP", old)
    smp.run(-1)
    assert smp.check_sums() == (0, 0)
    refs = oracle_chains(orc, D, (iters, burnin, thin, 5, 1), oparams(orc, params), lab, rp, seed, range(nchains))
    moved = 0
    for c in range(nchains):
        got = smp.samples(c)
        assert_same(got, refs[c], smp.state(c))
        moved += int((np.diff(refs[c]["labels"], axis=0) != 0).sum())
    smp.close()
    return moved, refs


def test_config1_replay_every_chain(pkg, orc):
    """BASELINE configs[1] (generatemixture n = 1000, K = 20, dim = 50, 64 chains), sigma = 0.2 so that the chains move
    (K wanders well above 20), 300 iterations, all 64 chains bit-identical to the oracle."""
    moved, refs = replay(pkg, orc, 1000, 20, 50, 0.2, 64, 300, 60, 4, seed=44)
    assert moved > 1000                                   # the chains are not frozen
    assert max(int(r["K"].max()) for r in refs) > 20
    assert sum(int(r["sm_split"].sum()) for r in refs) > 0 and sum(int((1 - r["sm_split"]).sum()) for r in refs) > 0


def test_config1_replay_launch_groups(pkg, orc):
    """The same replay in launch groups of 3 chains (8 chains x 60 iterations: groups of 3, 3 and 2)."""
    replay(pkg, orc, 1000, 20, 50, 0.2, 8, 60, 10, 5, seed=45, chains_per_group=3)


def test_config3_many_chains_n2000(pkg, orc):
    """BASELINE configs[3] (n = 2000, 1024 chains over 8 GPUs): one GPU's share, 128 chains x 20 iterations, every
    chain compared."""
    moved, _ = replay(pkg, orc, 2000, 20, 50, 0.17, 128, 20, 0, 2, seed=46)
    assert moved > 0


def test_config4_psm_exact_counts_n20000(pkg):
    """Exact co-clustering counts (mcmc.jl:560) at n = 20 000, S = 200 samples of up to 90 clusters, checked on 48
    sampled rows against direct label comparison; plus symmetry and the diagonal."""
    import torch
    g = np.random.default_rng(5)
    n, S = 20000, 200
    base = g.integers(1, 61, size=n)
    L = np.tile(base, (S, 1))
    flip = g.random((S, n)) < 0.15
    L[flip] = g.integers(1, 91, size=int(flip.sum()))
    L = np.ascontiguousarray(L, dtype=np.int64)
    cnt = torch.zeros((n, n), dtype=torch.int32, device="cuda")
    pkg.psm_counts_dev(L, cnt.data_ptr())
    torch.cuda.synchronize()
    rows = g.choice(n, size=48, replace=False)
    got = cnt[torch.from_numpy(rows).cuda()].cpu().numpy()
    for t, i in enumerate(rows):
        assert np.array_equal(got[t], (L == L[:, [i]]).sum(0))
    assert bool((torch.diagonal(cnt) == S).all())
    blk = cnt[:4096, :4096]
    assert bool((blk == blk.T).all())


def _contingency_all(Lc, K, i):
    """Contingency tables of sample i against every sample: (K, S, K) int64."""
    S, n = Lc.shape
    Zi = np.zeros((K, n)); Zi[Lc[i], np.arange(n)] = 1.0
    Zall = np.zeros((n, S * K))
    Zall[np.repeat(np.arange(n), S), (np.arange(S)[None, :] * K + Lc.T).ravel()] = 1.0
    return np.rint(Zi @ Zall).astype(np.int64).reshape(K, S, K)


def numpy_mpel_sums(L, loss):
    """pointestimate.jl:49-57 with Clustering.jl's randindex / varinfo / mutualinfo definitions, vectorised over j."""
    S, n = L.shape
    Lc = np.stack([np.unique(r, return_inverse=True)[1] for r in L])
    K = int(Lc.max()) + 1
    M = np.zeros((S, S))
    xlogx = lambda c: np.where(c > 0, c * np.log(np.where(c > 0, c, 1)), 0.0)   # noqa: E731
    for i in range(S):
        c = _contingency_all(Lc, K, i).astype(np.float64)            # (K, S, K)
        a = c.sum(2)                                                 # (K, S)   row sums (sample i's clusters)
        b = c.sum(0)                                                 # (S, K)   column sums (sample j's clusters)
        t2 = (c ** 2).sum((0, 2)); nis = (a ** 2).sum(0); njs = (b ** 2).sum(1)
        t1 = n * (n - 1) / 2; t3 = 0.5 * (nis + njs)
        if loss == "binder":
            M[i] = (t3 - t2) / t1
        elif loss == "omARI":
            nc = (n * (n ** 2 + 1) - (n + 1) * nis - (n + 1) * njs + 2 * (nis * njs) / n) / (2 * (n - 1))
            A = t1 + t2 - t3
            M[i] = 1 - np.where(t1 == nc, 0.0, (A - nc) / (t1 - nc))
        else:
            ha = np.log(n) - xlogx(a).sum(0) / n; hb = np.log(n) - xlogx(b).sum(1) / n
            hab = np.log(n) - xlogx(c).sum((0, 2)) / n
            mi = ha + hb - hab
            M[i] = (ha + hb - 2 * mi) if loss == "VI" else (np.maximum(ha, hb) - mi)
        M[i, i] = 0.0
    M = np.triu(M, 1); M = M + M.T
    return M.sum(0)


@pytest.mark.parametrize("loss", ["binder", "omARI", "VI", "ID"])
def test_config4_mpel_S512(pkg, orc, loss):
    g = np.random.default_rng(8)
    S, n = 512, 600
    base = np.sort(g.integers(1, 9, size=n))
    L = np.tile(base, (S, 1))
    flip = g.random((S, n)) < 0.1
    L[flip] = g.integers(1, 11, size=int(flip.sum()))
    ref = numpy_mpel_sums(L, loss)
    small = orc.mpel_loss_sums(L[:16], loss)                           # the vectorised statement against the plain oracle
    assert np.allclose(numpy_mpel_sums(L[:16], loss), small, rtol=1e-10, atol=1e-12)
    got, best = pkg.mpel_loss_sums(L, loss)
    assert np.allclose(got, ref, rtol=1e-10, atol=1e-10)
    assert abs(ref[best] - ref.min()) <= 1e-10 * max(1.0, abs(ref.min()))


def test_more_than_128_live_clusters(pkg, orc):
    """The sampler takes up to 255 simultaneously live clusters (byte labels; the reference allows n): sigma = 0.25 at n = 2000 opens well over 128 clusters within four sweeps -- every sweep
    bit-identical to the oracle, 16 lanes per row once a slot beyond 127 is live."""
    X, lab = mixture(2000, 20, 50, 0.25, 44)
    data = pkg.MCMCData.from_points(X)
    D = data.D
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=4, burnin=0, thin=1, numGibbs=5, numMH=1)
    rp = [pkg.init_rp(params, 3, c) for c in range(2)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (2, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=3, slot_cap=255)
    smp.run(-1)
    assert smp.check_sums() == (0, 0)
    refs = oracle_chains(orc, D, (4, 0, 1, 5, 1), oparams(orc, params), lab, rp, 3, range(2))
    for c in range(2):
        assert_same(smp.samples(c), refs[c], smp.state(c))
    assert max(int(r["K"].max()) for r in refs) > 128
