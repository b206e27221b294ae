"""Posterior expected Binder loss over pooled samples from the co-clustering counts (rc_binder_mpel,
rc_sampler_binder_mpel, rc_comm_sampler_binder_mpel): exact integer totals against contingency tables, agreement with the
pairwise MPEL search (pointestimate.jl:34-59,68-76), the device-resident path, its refusals, and getpointestimate over a
list of results."""
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def pairs(x):
    x = np.asarray(x, np.int64)
    return x * (x - 1) // 2


def totals_from_tables(L):
    """T_s = sum_t #pairs on which samples s and t disagree, from the S x S contingency tables (int64)."""
    S, n = L.shape
    C = np.stack([np.unique(l, return_inverse=True)[1] for l in L])            # 0 .. K_s - 1
    K = int(C.max()) + 1
    P = np.array([pairs(np.bincount(c, minlength=K)).sum() for c in C])
    T = np.zeros(S, np.int64)
    for s in range(S):
        code = C[s][None, :] * K + C + (np.arange(S) * K * K)[:, None]         # (t, i, j) cell of every point
        both = pairs(np.bincount(code.ravel(), minlength=S * K * K).reshape(S, K * K)).sum(1)
        T[s] = (P[s] + P - 2 * both).sum()
    return T


def label_sets():
    """>= 40 sets: n over 2 .. 700 (not multiples of 4 / 16 / 64 included), S over 1 .. 300, from one cluster to all
    singletons and up to 255 clusters, with arbitrary positive labels and duplicated samples."""
    g = np.random.default_rng(21)
    fixed = [(2, 1, "one"), (2, 3, "single"), (3, 2, "rand"), (5, 5, "rand"), (7, 1, "rand"), (63, 4, "rand"), (64, 64, "rand"),
             (65, 65, "rand"), (129, 3, "single"), (255, 5, "single"), (300, 7, "k255"), (700, 300, "rand"), (700, 13, "k255"),
             (97, 300, "one"), (16, 17, "dup"), (201, 40, "dup"), (511, 2, "rand"), (4, 130, "rand")]
    for n, S, kind in fixed:
        yield n, S, kind
    for _ in range(30):
        yield int(g.integers(2, 701)), int(g.choice([1, 2, 3, 5, 8, 31, 66, 127, 200, 257])), str(g.choice(["rand", "rand", "dup", "one"]))


def make_labels(g, n, S, kind):
    if kind == "one":
        L = np.full((S, n), 7, np.int64)
        L[1::2, : n // 2] = 3                                  # a second cluster in every other sample
        return L
    if kind == "single":
        return np.stack([g.permutation(n) + 1 for _ in range(S)]).astype(np.int64)
    if kind == "k255":
        L = []
        for _ in range(S):
            base = np.concatenate([np.arange(255), g.integers(0, 255, size=n - 255)])
            L.append(g.permutation(base))
        return (np.stack(L) * 3 + 11).astype(np.int64)          # 255 arbitrary positive labels
    K = int(g.integers(1, min(n, 40) + 1))
    L = g.integers(1, K + 1, size=(S, n)) * 1000 + 5
    if kind == "dup" and S > 2:
        h = S // 2
        L[h:2 * h] = L[:h].copy()                              # sample h + i repeats sample i; an odd S keeps one unique last sample
    return L.astype(np.int64)


def test_exact_totals_and_agreement_with_pairwise_mpel(pkg):
    g = np.random.default_rng(5)
    done = 0
    for n, S, kind in label_sets():
        L = make_labels(g, n, S, kind)
        sums, best, totals = pkg.binder_loss_sums(L)
        T = totals_from_tables(L)
        assert np.array_equal(totals, T), (n, S, kind)
        assert np.array_equal(sums.view(np.int64), (T / (n * (n - 1) // 2)).view(np.int64)), (n, S, kind)
        assert best == int(np.argmin(T))
        ref, rbest = pkg.mpel_loss_sums(L, "binder")
        assert np.allclose(sums, ref, rtol=1e-12, atol=1e-15), (n, S, kind)
        order = np.sort(sums)                                  # gap to the runner-up sample: exact ties are rc_mpel's rounding
        if order.size == 1 or order[1] - order[0] > 1e-12 * order[0]:
            assert rbest == best, (n, S, kind)
        if kind == "dup" and S > 2:                            # sample h + i repeats sample i: ties go to the first index
            h = S // 2
            assert np.array_equal(T[h:2 * h], T[:h])
            assert not (h <= best < 2 * h) and not (h <= rbest < 2 * h)
        done += 1
    assert done >= 40


def test_larger_exact_case_from_counts(pkg):
    """n = 1000, S = 2000: the totals against W_s summed from the device's co-clustering counts by masked sums."""
    import torch
    g = np.random.default_rng(8)
    n, S = 1000, 2000
    base = np.sort(g.integers(1, 13, size=n))
    L = np.tile(base, (S, 1))
    flip = g.random(L.shape) < 0.15
    L[flip] = g.integers(1, 13, size=int(flip.sum()))
    cnt = torch.zeros((n, n), dtype=torch.int32, device="cuda")
    pkg.psm_counts_dev(L, cnt.data_ptr())
    N = cnt.cpu().numpy().astype(np.float64)
    Z = np.zeros((n, S * 12))                                  # one-hot image of every sample's labels
    Z[np.repeat(np.arange(n)[None, :], S, 0).ravel(), (np.arange(S)[:, None] * 12 + L - 1).ravel()] = 1.0
    blk = ((N @ Z) * Z).sum(0).reshape(S, 12).sum(1)           # sum over same-cluster (a, b) of N_ab, diagonal included
    W = ((np.rint(blk).astype(np.int64) - n * S) // 2)         # N_aa = S; a < b only
    P = np.array([pairs(np.bincount(l)).sum() for l in L])
    T = S * P + P.sum() - 2 * W
    _, best, totals = pkg.binder_loss_sums(L)
    assert np.array_equal(totals, T)
    assert best == int(np.argmin(T))


def run_sampler(pkg, golden, nch=4, numiters=40, burnin=10):
    D, lab = golden[3]["distance_matrix"], golden[3]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    rp = [pkg.init_rp(params, 2, c) for c in range(nch)]
    return pkg.Sampler(pkg.MCMCData(D), pkg.MCMCOptionsList(numiters=numiters, burnin=burnin), params, np.tile(lab, (nch, 1)),
                       [x[0] for x in rp], [x[1] for x in rp], seed=2)


@pytest.mark.parametrize("grouped", [False, True])
def test_device_samples_equal_host_path(pkg, golden, monkeypatch, grouped):
    if grouped:
        monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", "1")
    smp = run_sampler(pkg, golden)
    smp.run(-1)
    sa = smp.samples_all()
    n, S = smp.data.n, sa["labels"].shape[1]
    for c0, k in ((0, 4), (1, 2), (3, 1)):
        dev = smp.binder_pointestimate(c0, k)
        sums, best, totals = pkg.binder_loss_sums(sa["labels"][c0:c0 + k].reshape(-1, n))
        assert np.array_equal(dev["sums"], sums) and np.array_equal(dev["totals"], totals)
        assert (dev["chain"] - c0) * S + dev["index"] == best
        assert np.array_equal(dev["clust"], sa["labels"][dev["chain"], dev["index"]])
    smp.close()


def test_sampler_path_refusals(pkg, golden):
    smp = run_sampler(pkg, golden, nch=2, numiters=30, burnin=5)
    smp.run(10)
    with pytest.raises(pkg.RCError) as e:
        smp.binder_pointestimate()
    assert e.value.status == -6
    smp.run(-1)
    for c0, k in ((-1, 1), (0, 0), (1, 2), (2, 1)):
        with pytest.raises(pkg.RCError) as e:
            smp.binder_pointestimate(c0, k)
        assert e.value.status == -1
    assert np.all(np.isfinite(smp.binder_pointestimate()["sums"]))
    smp.close()
    # the chain stops at a capacity of 10 live clusters on the 10-cluster example (as in test_gpu_sampler)
    D, lab = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    stopped = pkg.Sampler(pkg.MCMCData(D), pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1), pkg.params_from_labels(D, lab), lab,
                          1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError):
        stopped.run(-1)
    with pytest.raises(pkg.RCError) as e:
        stopped.binder_pointestimate()
    assert e.value.status == -5
    stopped.close()


def pooled_results(pkg, golden):
    D, lab = golden[2]["distance_matrix"], golden[2]["cluster_labels"]
    params = pkg.params_from_labels(D, lab)
    data = pkg.MCMCData(D)
    res = pkg.runsampler(data, pkg.MCMCOptionsList(numiters=120, burnin=20), params, verbose=False, nchains=3, seed=4)
    one = pkg.MCMCResult()
    one.clusts = [c for r in res for c in r.clusts]
    one.logposterior = np.concatenate([r.logposterior for r in res])
    one.loglik = np.concatenate([r.loglik for r in res])
    return res, one


def test_getpointestimate_over_a_list(pkg, golden):
    res, one = pooled_results(pkg, golden)
    for method, loss in [("MAP", "VI"), ("MLE", "VI")] + [("MPEL", l) for l in ("binder", "omARI", "VI", "ID")]:
        c1, i1 = pkg.getpointestimate(res, method, loss)
        c2, i2 = pkg.getpointestimate(one, method, loss)
        assert i1 == i2, (method, loss)
        assert np.array_equal(c1, c2)
    for bad in ([], [res[0], None], [res[0], type("R", (), {"clusts": [np.ones(7, np.int64)], "loglik": [0.0], "logposterior": [0.0]})()]):
        with pytest.raises(pkg.ArgumentError):
            pkg.getpointestimate(bad, "MPEL", "binder")
    host = importlib.import_module(pkg.__name__ + ".host")
    saved = host._PAIRWISE_BYTES
    host._PAIRWISE_BYTES = 8
    try:
        with pytest.raises(pkg.ArgumentError, match='loss="binder"'):
            pkg.getpointestimate(res, "MPEL", "VI")
        assert pkg.getpointestimate(res, "MPEL", "binder")[1] == pkg.getpointestimate(one, "MPEL", "binder")[1]
    finally:
        host._PAIRWISE_BYTES = saved


def test_world_of_one_equals_single_gpu(pkg, golden):
    smp = run_sampler(pkg, golden, nch=3)
    smp.run(-1)
    one = smp.binder_pointestimate()
    comm = pkg.Comm.from_torch(device=0)
    red = smp.binder_pointestimate_allreduce(comm=comm)
    S = smp.samples(0)["K"].size
    assert np.array_equal(red["sums"], one["sums"]) and np.array_equal(red["totals"], one["totals"])
    assert red["best"] == one["chain"] * S + one["index"]
    assert np.array_equal(red["clust"], one["clust"])
    smp.close()
