"""Allocation probabilities to the clusters of a point estimate (rc_aligned_alloc, rc_sampler_aligned_alloc,
rc_comm_sampler_aligned_alloc): every sample's map equals the canonical assignment's restatement bit for bit, matched
equals scipy's optimum, the counts equal a bincount through the maps; closed forms; the agreement of the host-label,
list, sampler (also in launch groups) and world-of-one paths; and the refusals."""
import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from test_gpu_credibleball import label_set, labels_255, run_sampler, fake_results
from test_host_alignment import canonical

pytestmark = pytest.mark.gpu


def first_appearance(x):
    """Labels 1..K in first-appearance order, and the original labels in that order."""
    u, first, inv = np.unique(x, return_index=True, return_inverse=True)
    order = np.argsort(first)
    rank = np.empty(u.size, np.int64)
    rank[order] = np.arange(1, u.size + 1)
    return rank[inv], u[order]


def table(e, c):
    T = np.zeros((e.max(), c.max()), np.int64)
    np.add.at(T, (e - 1, c - 1), 1)
    return T


def expected(est, L):
    """maps, matched, K and counts from the restatement, numpy tables and a bincount through the maps."""
    e, _ = first_appearance(est)
    kh, n = e.max(), e.size
    S = L.shape[0]
    maps, matched, K = np.zeros((S, 255), np.uint8), np.zeros(S, np.int64), np.zeros(S, np.int32)
    counts = np.zeros((n, kh + 1), np.int64)
    for t in range(S):
        c, _ = first_appearance(L[t])
        T = table(e, c)
        sigma, m = canonical(T)
        r, cc = linear_sum_assignment(T, maximize=True)
        assert m == T[r, cc].sum()
        maps[t, :c.max()] = sigma[1:]
        matched[t], K[t] = m, c.max()
        col = sigma[c]
        col = np.where(col == 0, kh, col - 1)
        counts[np.arange(n), col] += 1
    return maps, matched, K, counts


def estimate_for(k, refs):
    """Estimates with fewer, as many and more clusters than the samples (up to 255), with arbitrary positive labels."""
    g = np.random.default_rng(77 + k)
    n = refs.shape[1]
    if k % 3 == 0:
        return refs[0]
    if k % 3 == 1:
        return (refs[0] % 7) * 13 + 2
    return labels_255(g, n) * 3 + 1 if n >= 255 else g.permutation(n) + 5


@pytest.mark.parametrize("k", range(32))
def test_against_the_restatement(pkg, k):
    refs, L = label_set(k)
    est = estimate_for(k, refs)
    if max(len(np.unique(est)), max(len(np.unique(x)) for x in L)) > 100:
        L = L[:10]                                             # the restatement's O(N^3) host time
    out = pkg.alignedallocation(est, L, maps=True)
    maps, matched, K, counts = expected(est, L)
    S = L.shape[0]
    assert np.array_equal(out["maps"], maps)
    assert np.array_equal(out["matched"], matched)
    assert np.array_equal(out["K"], K) and np.array_equal(K, [len(np.unique(x)) for x in L])
    assert np.array_equal(out["counts"], counts) and np.all(out["counts"].sum(1) == S)
    assert np.array_equal(out["prob"], counts / np.float64(S))
    _, clusters = first_appearance(est)
    assert np.array_equal(out["clusters"], clusters)
    e, _ = first_appearance(est)
    assert np.array_equal(out["self"], out["prob"][np.arange(est.size), e - 1])
    assert "maps" not in pkg.alignedallocation(est, L)


def test_wide_tables(pkg):
    """n > 65 535: the 32-bit table cells."""
    g = np.random.default_rng(9)
    n = 70001
    est = g.integers(1, 9, size=n) * 5
    L = np.where(g.random((3, n)) < 0.7, est[None, :] // 5 % 4 + 1, g.integers(1, 5, size=(3, n)))
    out = pkg.alignedallocation(est, L, maps=True)
    maps, matched, K, counts = expected(est, L)
    assert np.array_equal(out["maps"], maps) and np.array_equal(out["matched"], matched)
    assert np.array_equal(out["K"], K) and np.array_equal(out["counts"], counts)


def test_closed_forms(pkg):
    g = np.random.default_rng(4)
    n, kh, S = 600, 9, 30
    est = g.integers(1, kh + 1, size=n)
    e, clusters = first_appearance(est)
    # label permutations of the estimate: one-hot prob, every point sure of its own cluster, matched = n
    L = np.stack([g.permutation(np.arange(100, 100 + kh))[est - 1] for _ in range(S)])
    out = pkg.alignedallocation(est, L)
    assert np.all(out["matched"] == n) and np.all(out["self"] == 1.0)
    assert np.array_equal(out["prob"], np.eye(kh + 1)[e - 1])
    # a one-cluster sample matches the largest estimate cluster, the first in column order on ties
    sizes = np.bincount(e)[1:]
    one = pkg.alignedallocation(est, np.ones((2, n), np.int64), maps=True)
    assert np.all(one["maps"][:, 0] == 1 + np.argmax(sizes)) and np.all(one["maps"][:, 1:] == 0)
    assert np.all(one["matched"] == sizes.max())
    tie = np.repeat([4, 9, 2, 7], [10, 30, 30, 5])                # clusters 9 and 2 tie: 9 comes first
    assert pkg.alignedallocation(tie, np.ones((1, 75)), maps=True)["maps"][0, 0] == 2
    # perturbed permuted copies recover each sample's permutation; a point's matched cluster is its own in most samples
    perms = [g.permutation(kh) + 1 for _ in range(S)]
    L = np.stack([p[e - 1] for p in perms])
    flip = g.random(L.shape) < 0.05
    L[flip] = g.integers(1, kh + 1, size=int(flip.sum()))
    out = pkg.alignedallocation(est, L, maps=True)
    for t in range(S):
        c, labs = first_appearance(L[t])
        for l in range(1, labs.size + 1):
            assert out["maps"][t, l - 1] == 1 + int(np.flatnonzero(perms[t] == labs[l - 1])[0]), (t, l)
    assert np.array_equal(np.argmax(out["prob"], axis=1), e - 1) and out["self"].mean() > 0.9


@pytest.mark.parametrize("grouped", [False, True])
def test_paths_agree(pkg, golden, monkeypatch, grouped):
    if grouped:
        monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", "1")
    smp = run_sampler(pkg, golden, numiters=60)
    smp.run(-1)
    sa = smp.samples_all()
    n = sa["labels"].shape[2]
    est = golden[3]["cluster_labels"] * 11 + 4

    def same(x, y):
        assert set(x) == set(y)
        for key in x:
            assert np.array_equal(x[key], y[key]), key
    for c0, k in ((0, 4), (1, 2), (3, 1)):
        host = sa["labels"][c0:c0 + k].reshape(-1, n)
        dev = smp.alignedallocation(est, c0, k, maps=True)
        same(dev, pkg.alignedallocation(est, host, maps=True))
        same(dev, pkg.alignedallocation(est, fake_results(pkg, sa, range(c0, c0 + k)), maps=True))
        assert np.array_equal(dev["K"], sa["K"][c0:c0 + k].ravel())
    red = smp.alignedallocation_allreduce(est, maps=True, comm=pkg.Comm.from_torch(device=0))
    same(red, smp.alignedallocation(est, maps=True))
    smp.close()


def test_refusals(pkg, golden):
    from redclust_jl_b200._lib import lib, ptr

    def refused(status, fn, *args, **kw):
        with pytest.raises(pkg.RCError) as e:
            fn(*args, **kw)
        assert e.value.status == status, str(e.value)
        return str(e.value)

    est = golden[3]["cluster_labels"]
    smp = run_sampler(pkg, golden, nch=2, numiters=30, burnin=5)
    smp.run(10)
    refused(-6, smp.alignedallocation, est)
    refused(-6, smp.alignedallocation_allreduce, est, comm=pkg.Comm.from_torch(device=0))
    smp.run(-1)
    for c0, k in ((-1, 1), (0, 0), (1, 2), (2, 1)):
        refused(-1, smp.alignedallocation, est, c0, k)
    many = np.arange(est.size) % 256 + 1
    if est.size >= 256:
        assert "more than 255 clusters" in refused(-5, smp.alignedallocation, many)
    E = np.ascontiguousarray(est, dtype=np.int64)
    counts = np.empty((est.size, len(np.unique(est)) + 1), np.int32)
    assert lib().rc_sampler_aligned_alloc(smp._h, ptr(E), 0, 2, None, None, None, None) == -1
    assert lib().rc_sampler_aligned_alloc(smp._h, ptr(E), 0, 2, ptr(counts), None, None, None) == 0
    assert np.array_equal(counts, smp.alignedallocation(est)["counts"])
    # the sharded entry point refuses in its status exchange; the communicator then still serves a complete call
    comm = pkg.Comm.from_torch(device=0)
    assert lib().rc_comm_sampler_aligned_alloc(comm._h, smp._h, None, ptr(counts), None, None, None) == -1
    assert lib().rc_comm_sampler_aligned_alloc(comm._h, smp._h, ptr(E), ptr(counts), None, None, None) == 0
    assert np.array_equal(counts, smp.alignedallocation(est)["counts"])
    smp.close()
    D1, lab1 = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    stopped = pkg.Sampler(pkg.MCMCData(D1), pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1), pkg.params_from_labels(D1, lab1),
                          lab1, 1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError):
        stopped.run(-1)
    refused(-5, stopped.alignedallocation, lab1)
    stopped.close()
    g = np.random.default_rng(1)
    L = g.integers(1, 4, size=(5, 300))
    assert "more than 255 clusters" in refused(-5, pkg.alignedallocation, np.arange(300) % 256 + 1, L)
    assert "out of range" in refused(-1, pkg.alignedallocation, L[0], L, device=int(lib().rc_device_count()))
    Lc = np.ascontiguousarray(L, dtype=np.int64)
    c = np.empty((300, 4), np.int32)
    assert lib().rc_aligned_alloc(ptr(Lc), ptr(Lc), 5, 300, 0, None, None, None, None) == -1
    assert lib().rc_aligned_alloc(ptr(Lc), ptr(Lc), 0, 300, 0, ptr(c), None, None, None) == -1
    assert lib().rc_aligned_alloc(ptr(Lc), ptr(Lc), 1 << 31, 300, 0, ptr(c), None, None, None) == -1
    assert lib().rc_aligned_alloc(None, ptr(Lc), 5, 300, 0, ptr(c), None, None, None) == -1
    # a table that does not fit: the message of pair_geometry, as the credible ball gives it
    n = 70001
    big = labels_255(g, n)
    msg = refused(-5, pkg.alignedallocation, big, np.tile(big, (2, 1)))
    assert "does not fit shared memory" in msg and "255 x 255" in msg


def pooled_labels(g, n, kh, S):
    """An estimate and S samples in which most points keep their cluster for long runs of samples, some switch cluster at
    random times (runs of 1 to several hundred samples) and some change in every sample; every sample carries its own
    label values, and one sample in ten has an extra small cluster (K_t = kh + 1)."""
    est = g.integers(1, kh + 1, size=n)
    base = np.tile(est, (S, 1))
    often = g.random(n) < 0.1
    base[:, often] = g.integers(1, kh + 1, size=(S, int(often.sum())))
    runs = ~often & (g.random(n) < 0.25)
    seg = np.cumsum(g.random((S, int(runs.sum()))) < 0.0125, axis=0)
    base[:, runs] = g.integers(1, kh + 1, size=(seg.max() + 1, int(runs.sum())))[seg, np.arange(int(runs.sum()))]
    extra = g.random(S) < 0.1
    base[np.ix_(extra, np.arange(40))] = kh + 1
    L = np.stack([g.permutation(np.arange(100, 101 + kh))[b - 1] for b in base])
    return est * 3 + 7, L


def test_pooled_slices(pkg, capfd, monkeypatch):
    """Sample slices of k_align_count well above its 64-sample sigma chunk and 16-label load group: the counts equal a
    bincount through the returned maps, and the maps equal the restatement."""
    g = np.random.default_rng(21)
    n, kh, S = 10000, 12, 4000
    est, L = pooled_labels(g, n, kh, S)
    monkeypatch.setenv("RCB200_VERBOSE", "1")
    out = pkg.alignedallocation(est, L, maps=True)
    line = [x for x in capfd.readouterr().err.splitlines() if "aligned allocation:" in x][-1]
    gy = int(line.split("k_align_count")[1].split("x")[1].split(")")[0])
    assert S / gy > 2 * 64, line                                # more than two sigma chunks per slice
    e, _ = first_appearance(est)
    cols = np.empty((S, n), np.int64)
    for t in range(S):
        c, _ = first_appearance(L[t])
        m = out["maps"][t][c - 1].astype(np.int64)
        cols[t] = np.where(m == 0, kh, m - 1)
    counts = np.bincount((np.arange(n)[None, :] * (kh + 1) + cols).ravel(), minlength=n * (kh + 1)).reshape(n, kh + 1)
    assert np.array_equal(out["counts"], counts) and np.all(out["counts"].sum(1) == S)
    assert 0 < counts[:, kh].sum() and np.any(counts[:, :kh].max(1) < S)   # unmatched and changing points occur
    maps, matched, K, _ = expected(est, L)
    assert np.array_equal(out["maps"], maps) and np.array_equal(out["matched"], matched) and np.array_equal(out["K"], K)


@pytest.mark.parametrize("k", [0, 3, 7, 11, 14, 19, 26, 31])
def test_64bit_argmin(pkg, monkeypatch, k):
    """RCB200_ALIGN_KEY64=1 runs every argmin through the 64-bit (value, column) reduction: the same maps as the 32-bit key
    and as the restatement."""
    refs, L = label_set(k)
    est = estimate_for(k, refs)
    if max(len(np.unique(est)), max(len(np.unique(x)) for x in L)) > 100:
        L = L[:10]
    fast = pkg.alignedallocation(est, L, maps=True)
    monkeypatch.setenv("RCB200_ALIGN_KEY64", "1")
    wide = pkg.alignedallocation(est, L, maps=True)
    for key in fast:
        assert np.array_equal(fast[key], wide[key]), key
    assert np.array_equal(wide["maps"], expected(est, L)[0])


def test_buffers_that_do_not_fit_are_refused(pkg):
    """With the device nearly full the host-label call refuses before it allocates, and its sizes include the device copy
    of the sample labels; the device stays usable."""
    import torch
    n, S = 1000, 60000
    L = np.tile(np.arange(n) % 5 + 1, (S, 1))
    free, _ = torch.cuda.mem_get_info()
    hog = torch.empty(free - (64 << 20), dtype=torch.uint8, device="cuda")
    try:
        e = pytest.raises(pkg.RCError, pkg.alignedallocation, L[0], L).value
        assert e.status == -2 and "GB of device memory" in str(e) and "sample labels 0.06 GB" in str(e), str(e)
    finally:
        del hog
        torch.cuda.empty_cache()
    assert np.all(pkg.alignedallocation(L[0], L[:3])["self"] == 1.0)
