"""Convergence across chains (rc_cocl_rhat, rc_sampler_cocl_rhat, rc_comm_sampler_cocl_rhat): the split-R-hat of every
point pair's co-clustering indicator and each chain's distance from the pooled PSM, bit for bit against a numpy statement
from one-hot counts, closed forms, the agreement of the host-label, sampler and world-of-one paths, and the refusals."""
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def group_counts(L):
    """N_g (m x n x n int64) of C x S x n labels: groups 2c and 2c + 1 are chain c's first and last floor(S / 2) samples."""
    C, S, n = L.shape
    h = S // 2
    out = []
    for c in range(C):
        for part in (L[c, :h], L[c, S - h:]):
            codes = np.unique(part, return_inverse=True)[1].reshape(part.shape)
            K = int(codes.max()) + 1
            Y = np.zeros((n, h * K))
            Y[np.tile(np.arange(n), h), (np.arange(h)[:, None] * K + codes).ravel()] = 1.0
            out.append(np.rint(Y @ Y.T).astype(np.int64))
    return np.stack(out)


def reference(L):
    """R matrix, summary and deviations from integer N and Q, with the operation order of the definition."""
    C, S, n = L.shape
    h, m = S // 2, 2 * C
    Ng = group_counts(L)
    N, Q = Ng.sum(0), (Ng * Ng).sum(0)
    Wn, Bn = h * N - Q, m * Q - N * N
    f = np.float64
    with np.errstate(divide="ignore", invalid="ignore"):
        R = np.sqrt(f(h - 1) / f(h) + (f(h - 1) * Bn.astype(f)) / (f(m - 1) * f(h) * Wn.astype(f)))
    R = np.where(Wn > 0, R, np.where(Bn == 0, 1.0, np.inf))
    np.fill_diagonal(R, 1.0)
    iu = np.triu_indices(n, 1)
    vals = R[iu]
    k = int(np.argmax(vals == vals.max()))
    d = np.abs(m * (Ng[0::2] + Ng[1::2]) - 2 * N)[:, iu[0], iu[1]]
    pairs = n * (n - 1) // 2
    meandev = np.array([f(int(x)) / (f(2 * m * h) * f(pairs)) for x in d.sum(1)])
    maxdev = np.array([f(int(x)) / f(2 * m * h) for x in d.max(1)])
    return dict(rhat=R, rhat_max=float(vals.max()), rhat_pair=(int(iu[0][k]), int(iu[1][k])), pairs_above=int((vals > 1.01).sum()),
                chain_meandev=meandev, chain_maxdev=maxdev)


def bits(x):
    return np.asarray(x, np.float64).view(np.int64)


def assert_same(got, ref, matrix=True):
    assert got["rhat_pair"] == ref["rhat_pair"] and got["pairs_above"] == ref["pairs_above"]
    assert bits(got["rhat_max"]) == bits(ref["rhat_max"])
    assert np.array_equal(bits(got["chain_meandev"]), bits(ref["chain_meandev"]))
    assert np.array_equal(bits(got["chain_maxdev"]), bits(ref["chain_maxdev"]))
    if matrix:
        assert np.array_equal(bits(got["rhat"]), bits(ref["rhat"]))


def chain_labels(g, C, S, n, K, flip=0.2, spread=0.1):
    """Each chain perturbs a common base partition a little, and every sample redraws a fraction of its chain's labels."""
    base = g.integers(1, K + 1, size=n)
    out = np.empty((C, S, n), np.int64)
    for c in range(C):
        cb = base.copy()
        moved = g.random(n) < spread
        cb[moved] = g.integers(1, K + 1, size=int(moved.sum()))
        L = np.tile(cb, (S, 1))
        f = g.random(L.shape) < flip
        L[f] = g.integers(1, K + 1, size=int(f.sum()))
        out[c] = L * 7 + 3                                     # arbitrary positive labels
    return out


@pytest.mark.parametrize("C, S, n, K", [(4, 20, 97, 6), (3, 21, 131, 9), (1, 9, 70, 4), (2, 12, 300, 200), (2, 4, 2, 2), (5, 7, 64, 3)])
def test_bits_against_numpy(pkg, C, S, n, K):
    g = np.random.default_rng(100 * C + S + n)
    L = chain_labels(g, C, S, n, K)
    ref = reference(L)
    got = pkg.cocl_rhat(L, matrix=True)
    assert_same(got, ref)
    assert got["rhat"] is not None and np.array_equal(got["rhat"], got["rhat"].T)
    lean = pkg.cocl_rhat(L)                                    # the summary does not need the matrix
    assert lean["rhat"] is None
    assert_same(lean, ref, matrix=False)


@pytest.mark.parametrize("S", [16, 17])
def test_identical_groups(pkg, S):
    """Every group holds the same label vectors: R = sqrt((L - 1) / L) exactly on the pairs that vary, 1 on the others."""
    g = np.random.default_rng(S)
    n, h, C = 83, S // 2, 3
    G = g.integers(1, 6, size=(h, n))
    L = np.stack([np.concatenate([G, g.integers(1, 6, size=(S - 2 * h, n)), G]) for _ in range(C)])
    got = pkg.cocl_rhat(L, matrix=True)
    same = (G[:, :, None] == G[:, None, :]).sum(0)
    varies = (same > 0) & (same < h)
    np.fill_diagonal(varies, False)
    assert varies.any() and (~varies).sum() > n
    want = np.where(varies, np.sqrt(np.float64(h - 1) / np.float64(h)), 1.0)
    assert np.array_equal(bits(got["rhat"]), bits(want))
    assert np.all(got["chain_meandev"] == 0) and np.all(got["chain_maxdev"] == 0)
    assert got["pairs_above"] == 0 and got["rhat_max"] == 1.0


def test_constant_chains_that_differ(pkg):
    g = np.random.default_rng(4)
    n, S = 150, 10
    P = [g.integers(1, 4, size=n) for _ in range(2)]
    parts = [P[0], P[0], P[1], P[0]]
    L = np.stack([np.tile(p, (S, 1)) for p in parts])
    got = pkg.cocl_rhat(L, matrix=True)
    co = [p[:, None] == p[None, :] for p in P]
    differ = co[0] != co[1]
    want = np.where(differ, np.inf, 1.0)
    assert np.array_equal(got["rhat"], want)
    iu = np.triu_indices(n, 1)
    k = int(np.argmax(differ[iu]))
    assert got["rhat_max"] == np.inf and got["rhat_pair"] == (int(iu[0][k]), int(iu[1][k]))
    assert got["pairs_above"] == int(differ[iu].sum())
    assert int(np.argmax(got["chain_meandev"])) == 2


def run_sampler(pkg, golden, nch=4, numiters=40, burnin=10, example=3, **kw):
    D, lab = golden[example]["distance_matrix"], golden[example]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    rp = [pkg.init_rp(params, 2, c) for c in range(nch)]
    return pkg.Sampler(pkg.MCMCData(D), pkg.MCMCOptionsList(numiters=numiters, burnin=burnin), params, np.tile(lab, (nch, 1)),
                       [x[0] for x in rp], [x[1] for x in rp], seed=2, **kw)


def fake_results(pkg, sa, chains):
    out = []
    for c in chains:
        r = pkg.MCMCResult()
        r.clusts = [x for x in sa["labels"][c]]
        for k in ("K", "r", "p", "loglik", "logposterior"):
            setattr(r, k, sa[k][c])
        out.append(r)
    return out


@pytest.mark.parametrize("burnin", [10, 9])
def test_sampler_path_equals_host_labels(pkg, golden, burnin):
    host = importlib.import_module(pkg.__name__ + ".host")
    smp = run_sampler(pkg, golden, burnin=burnin)
    smp.run(-1)
    sa = smp.samples_all()
    for c0, k in ((0, 4), (1, 2), (3, 1)):
        dev = smp.convergencediagnostics(c0, k, matrix=True)
        ref = pkg.cocl_rhat(sa["labels"][c0:c0 + k], matrix=True)
        assert_same(dev, ref)
        assert_same(dev, reference(sa["labels"][c0:c0 + k]))
        lst = pkg.convergencediagnostics(fake_results(pkg, sa, range(c0, c0 + k)), matrix=True)
        assert_same(lst, ref)
        for name in ("K", "r", "p", "loglik", "logposterior"):
            want = host._split_rhat(sa[name][c0:c0 + k].astype(np.float64))
            assert dev["traces"][name] == want and lst["traces"][name] == want, name
    one = smp.convergencediagnostics()
    red = smp.convergencediagnostics_allreduce(comm=pkg.Comm.from_torch(device=0))
    assert_same(red, one, matrix=False)
    assert red["traces"] == one["traces"]
    smp.close()


def test_a_chain_in_another_partition(pkg, golden):
    smp = run_sampler(pkg, golden, nch=4, numiters=60, burnin=10)
    smp.run(-1)
    L = smp.samples_all()["labels"].copy()
    smp.close()
    g = np.random.default_rng(3)
    other = g.permutation(L[2, 0])                              # the same cluster sizes over other points
    L[2] = other
    got = pkg.cocl_rhat(L)
    assert int(np.argmax(got["chain_meandev"])) == 2
    assert got["rhat_max"] > 1.01 and got["pairs_above"] > 0
    assert_same(got, reference(L), matrix=False)


def test_refusals(pkg, golden):
    from redclust_jl_b200._lib import lib

    def refused(status, fn, *args, **kw):
        with pytest.raises(pkg.RCError) as e:
            fn(*args, **kw)
        assert e.value.status == status, str(e.value)
        return str(e.value)

    smp = run_sampler(pkg, golden, nch=2, numiters=30, burnin=5)
    smp.run(10)
    refused(-6, smp.convergencediagnostics)
    refused(-6, smp.convergencediagnostics_allreduce, comm=pkg.Comm.from_torch(device=0))
    smp.run(-1)
    for c0, k in ((-1, 1), (0, 0), (1, 2), (2, 1)):
        refused(-1, smp.convergencediagnostics, c0, k)
    assert np.isfinite(smp.convergencediagnostics()["rhat_max"])
    smp.close()
    short = run_sampler(pkg, golden, nch=2, numiters=13, burnin=10)     # 3 samples per chain
    short.run(-1)
    refused(-1, short.convergencediagnostics)
    short.close()
    D1, lab1 = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    stopped = pkg.Sampler(pkg.MCMCData(D1), pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1), pkg.params_from_labels(D1, lab1),
                          lab1, 1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError):
        stopped.run(-1)
    refused(-5, stopped.convergencediagnostics)
    stopped.close()
    L = np.ones((2, 6, 5), np.int64)
    refused(-1, pkg.cocl_rhat, L[:, :3])
    refused(-1, pkg.cocl_rhat, L[:, :, :1])
    assert "out of range" in refused(-1, pkg.cocl_rhat, L, device=int(lib().rc_device_count()))


def test_buffers_that_do_not_fit_are_refused(pkg):
    """With the device nearly full the call refuses and names the sizes; the device stays usable."""
    import torch
    n = 8000
    free, _ = torch.cuda.mem_get_info()
    hog = torch.empty(free - (1 << 30), dtype=torch.uint8, device="cuda")
    try:
        L = np.tile(np.arange(n) % 5 + 1, (2, 4, 1))
        msg = str(pytest.raises(pkg.RCError, pkg.cocl_rhat, L).value)
        assert "GB of device memory" in msg and "Q 0.51 GB" in msg, msg
    finally:
        del hog
        torch.cuda.empty_cache()
    assert pkg.cocl_rhat(np.tile(np.arange(50) % 5 + 1, (2, 4, 1)))["rhat_max"] == 1.0
