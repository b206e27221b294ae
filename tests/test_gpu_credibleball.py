"""Distances from given partitions to the samples (rc_partition_dists, rc_sampler_partition_dists,
rc_comm_sampler_partition_dists), the posterior expected loss and the credible ball built on them: bit-equality with
rc_mpel's loss matrix and sums on the stacked label set, exact Binder counts against numpy contingency tables and
rc_binder_mpel's totals, closed forms, the agreement of the host-label, list, sampler and world-of-one paths, and the
refusals."""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LOSSES = ("binder", "omARI", "VI", "ID")


def bits(x):
    return np.asarray(x, np.float64).view(np.int64)


def labels_255(g, n):
    return g.permutation(np.arange(n) % 255 + 1)


def label_set(k):
    """Label set k of 32: n = 2, n a multiple of 16 (16-byte label rows) and not, up to 255 clusters in the references and the samples, S = 1,
    several references, the first reference with labels far outside 1..K and the samples with arbitrary positive labels."""
    g = np.random.default_rng(1000 + k)
    n = [2, 2, 5, 15, 17, 31, 33, 63, 100, 129, 300, 256, 513, 1024, 2049, 4097][k % 16]
    S = [1, 2, 7, 40, 1, 13, 64, 100][k % 8]
    nref = 1 + k % 3
    K = min(n, [2, 5, 20, 255][k % 4])

    def one():
        return labels_255(g, n) if K == 255 and n >= 255 else g.integers(1, K + 1, size=n)
    refs = np.stack([one() for _ in range(nref)])
    refs[0] = refs[0] * 1_000_003 + 10**12
    samples = np.stack([one() for _ in range(S)])
    if k % 2:
        samples = samples * 7 + 3
    return refs, samples


def mpel_row0(pkg, L, loss):
    """Row 0 of rc_mpel's loss matrix on L (rc_mpel_rows_dev with row_first = 0)."""
    import torch
    from redclust_jl_b200._lib import lib, check, ptr
    L = np.ascontiguousarray(L, dtype=np.int64)
    buf = torch.zeros((1, L.shape[0]), dtype=torch.float64, device="cuda")
    check(lib().rc_mpel_rows_dev(ptr(L), L.shape[0], L.shape[1], LOSSES.index(loss), 0, 0, 1, 1, C.c_void_p(buf.data_ptr())))
    return buf.cpu().numpy()[0]


def binder_pairs(a, b):
    """Disagreeing pairs of two label vectors from their int64 contingency table."""
    ca, cb = np.unique(a, return_inverse=True)[1], np.unique(b, return_inverse=True)[1]
    T = np.zeros((ca.max() + 1, cb.max() + 1), np.int64)
    np.add.at(T, (ca, cb), 1)
    return int(((T.sum(1) ** 2).sum() + (T.sum(0) ** 2).sum()) // 2 - (T ** 2).sum())


@pytest.mark.parametrize("k", range(32))
def test_bits_against_mpel(pkg, k):
    refs, L = label_set(k)
    S = L.shape[0]
    for loss in LOSSES:
        out = pkg.partitiondistances(refs, L, loss)
        el = pkg.expectedloss(refs, L, loss)
        for r in range(refs.shape[0]):
            stacked = np.concatenate([refs[r:r + 1], L])
            assert np.array_equal(bits(out["dist"][r]), bits(mpel_row0(pkg, stacked, loss)[1:])), (loss, r)
            sums, _ = pkg.mpel_loss_sums(stacked, loss)
            assert bits(el["expectedloss"][r]) == bits(sums[0] / S), (loss, r)
        assert (el["totals"] is not None) == (loss == "binder") and (out["pairs"] is not None) == (loss == "binder")
        if loss == "binder":
            binder = out
    want = np.array([[binder_pairs(a, b) for b in L] for a in refs])
    assert np.array_equal(binder["pairs"], want)
    assert np.array_equal(out["K"], [len(np.unique(x)) for x in L])
    assert np.array_equal(pkg.expectedloss(refs, L, "binder")["totals"], want.sum(1))


def test_binder_totals_equal_pooled_counts(pkg):
    g = np.random.default_rng(5)
    n, S = 700, 300
    base = g.integers(1, 30, size=n)
    L = np.tile(base, (S, 1))
    f = g.random(L.shape) < 0.2
    L[f] = g.integers(1, 40, size=int(f.sum()))
    _, _, totals = pkg.binder_loss_sums(L)
    idx = [0, 17, 299]
    got = pkg.expectedloss(L[idx], L, "binder")["totals"]
    assert np.array_equal(got, totals[idx])


def test_closed_form_all_equal(pkg):
    g = np.random.default_rng(2)
    est = g.integers(1, 6, size=90)
    L = np.tile(est * 3 + 1, (25, 1))                           # the same partition under other labels
    for loss in LOSSES:
        b = pkg.credibleball(est, L, loss)
        assert b["radius"] == 0.0 and b["inball"] == 25 and b["expectedloss"] == 0.0
        for name in ("horizontal", "upper", "lower"):
            assert b[name]["dist"] == 0.0 and b[name]["K"] == len(np.unique(est))
            assert np.array_equal(b[name]["indices"], np.arange(25))
            assert np.array_equal(pkg.sortlabels(b[name]["clust"]), pkg.sortlabels(est))


@pytest.mark.parametrize("f", [0.02, 0.1, 0.3])
def test_closed_form_one_merge(pkg, f):
    n, S, alpha = 120, 200, 0.05
    est = np.repeat(np.arange(1, 5), [30, 25, 40, 25])           # clusters 2 (25 points) and 4 (25 points) merge
    merged = np.where(est == 4, 2, est)
    a, b = 25, 25
    g = np.random.default_rng(int(f * 100))
    which = np.zeros(S, bool)
    which[g.choice(S, size=int(round(f * S)), replace=False)] = True
    L = np.where(which[:, None], merged[None, :], est[None, :])
    ball = pkg.credibleball(est, L, "binder", alpha)
    dm = (a * b) / (n * (n - 1) / 2)
    assert np.array_equal(np.flatnonzero(ball["dist"] > 0), np.flatnonzero(which))
    assert np.all(ball["dist"][which] == dm)
    if f < alpha:
        assert ball["radius"] == 0.0 and ball["upper"]["K"] == 4
    else:
        assert ball["radius"] == dm
        assert ball["upper"]["K"] == 3 and np.array_equal(ball["upper"]["indices"], np.flatnonzero(which))
        assert np.array_equal(ball["upper"]["clust"], merged)
        assert ball["lower"]["dist"] == 0.0 and ball["lower"]["K"] == 4
    el = pkg.expectedloss(est, L, "binder")
    assert el["totals"][0] == a * b * int(which.sum())


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
        out.append(r)
    return out


def same_ball(x, y):
    assert bits(x["radius"]) == bits(y["radius"]) and x["inball"] == y["inball"]
    assert bits(x["expectedloss"]) == bits(y["expectedloss"])
    assert np.array_equal(bits(x["dist"]), bits(y["dist"]))
    for name in ("horizontal", "upper", "lower"):
        assert x[name]["dist"] == y[name]["dist"] and x[name]["K"] == y[name]["K"], name
        assert np.array_equal(x[name]["indices"], y[name]["indices"]), name
        assert np.array_equal(x[name]["clust"], y[name]["clust"]), name


def test_paths_agree(pkg, golden):
    smp = run_sampler(pkg, golden, numiters=60)
    smp.run(-1)
    sa = smp.samples_all()
    S = sa["labels"].shape[1]
    est = golden[3]["cluster_labels"]
    for loss in LOSSES:
        for c0, k in ((0, 4), (1, 2), (3, 1)):
            host = sa["labels"][c0:c0 + k].reshape(-1, sa["labels"].shape[2])
            dev = smp.credibleball(est, c0, k, loss, 0.1)
            lst = pkg.credibleball(est, fake_results(pkg, sa, range(c0, c0 + k)), loss, 0.1)
            same_ball(dev, lst)
            d = pkg.partitiondistances(est, host, loss)
            assert np.array_equal(bits(d["dist"][0]), bits(dev["dist"]))
            assert np.array_equal(d["K"], sa["K"][c0:c0 + k].ravel())
            e1 = smp.expectedloss(np.stack([est, host[3]]), c0, k, loss)
            e2 = pkg.expectedloss(np.stack([est, host[3]]), host, loss)
            assert np.array_equal(bits(e1["expectedloss"]), bits(e2["expectedloss"]))
            if loss == "binder":
                assert np.array_equal(e1["totals"], e2["totals"])
            i = int(dev["upper"]["indices"][0])
            assert np.array_equal(dev["upper"]["clust"], sa["labels"][c0 + i // S][i % S])
        red = smp.credibleball_allreduce(est, loss, 0.1, comm=pkg.Comm.from_torch(device=0))
        same_ball(red, smp.credibleball(est, loss=loss, alpha=0.1))
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
    refused(-6, smp.credibleball, est)
    refused(-6, smp.expectedloss, est)
    refused(-6, smp.credibleball_allreduce, est, comm=pkg.Comm.from_torch(device=0))
    smp.run(-1)
    for c0, k in ((-1, 1), (0, 0), (1, 2), (2, 1)):
        refused(-1, smp.credibleball, est, c0, k)
    S = 2 * 25
    P = np.ascontiguousarray(est[None, :], dtype=np.int64)
    dist = np.empty(S)
    for bad in (-1, 4):
        assert lib().rc_sampler_partition_dists(smp._h, ptr(P), 1, 0, 2, bad, ptr(dist), None, None) == -1
    assert lib().rc_sampler_partition_dists(smp._h, ptr(P), 0, 0, 2, 2, ptr(dist), None, None) == -1
    assert lib().rc_sampler_partition_dists(smp._h, ptr(P), 1, 0, 2, 2, None, None, None) == -1
    assert lib().rc_sampler_partition_dists(smp._h, ptr(P), 1, 0, 2, 2, ptr(dist), None, None) == 0
    # the sharded entry point refuses in its status exchange; the communicator then still serves a complete call
    comm = pkg.Comm.from_torch(device=0)
    assert lib().rc_comm_sampler_partition_dists(comm._h, smp._h, ptr(P), 1, 7, ptr(dist), None, None) == -1
    assert lib().rc_comm_sampler_partition_dists(comm._h, smp._h, ptr(P), 0, 2, ptr(dist), None, None) == -1
    pairs, K = np.empty(S, np.int64), np.empty(S, np.int32)
    assert lib().rc_comm_sampler_partition_dists(comm._h, smp._h, ptr(P), 1, 0, ptr(dist), ptr(pairs), ptr(K)) == 0
    one = smp._partition_dists(est, 0, 2, "binder")
    assert np.array_equal(dist, one["dist"][0]) and np.array_equal(pairs, one["pairs"][0]) and np.array_equal(K, one["K"])
    assert np.array_equal(dist, smp.credibleball(est)["dist"])
    smp.close()
    D1, lab1 = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    stopped = pkg.Sampler(pkg.MCMCData(D1), pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1), pkg.params_from_labels(D1, lab1),
                          lab1, 1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError):
        stopped.run(-1)
    refused(-5, stopped.credibleball, lab1)
    stopped.close()
    g = np.random.default_rng(1)
    L = g.integers(1, 4, size=(5, 300))
    many = np.arange(300) % 256 + 1                              # 256 clusters
    assert "more than 255 clusters" in refused(-5, pkg.partitiondistances, many, L)
    refused(-5, pkg.credibleball, many, L)
    assert "out of range" in refused(-1, pkg.partitiondistances, L[0], L, device=int(lib().rc_device_count()))
    Lc = np.ascontiguousarray(L, dtype=np.int64)
    out = np.empty((1, 5))
    for bad in (-1, 4):
        assert lib().rc_partition_dists(ptr(Lc), 1, ptr(Lc), 5, 300, bad, 0, ptr(out), None, None) == -1
    assert lib().rc_partition_dists(ptr(Lc), 1, ptr(Lc), 5, 300, 2, 0, None, None, None) == -1
    assert lib().rc_partition_dists(ptr(Lc), 0, ptr(Lc), 5, 300, 2, 0, ptr(out), None, None) == -1
    assert lib().rc_partition_dists(ptr(Lc), 1, ptr(Lc), 0, 300, 2, 0, ptr(out), None, None) == -1


def test_wide_tables_and_table_limit(pkg):
    """n > 65 535 takes the 32-bit table cells of rc_mpel and gives its bits; a table that does not fit is refused."""
    g = np.random.default_rng(9)
    n = 70001
    L = g.integers(1, 4, size=(3, n))
    ref = g.integers(1, 6, size=n)
    out = pkg.partitiondistances(ref, L, "VI")
    row = mpel_row0(pkg, np.concatenate([ref[None], L]), "VI")
    assert np.array_equal(bits(out["dist"][0]), bits(row[1:]))
    assert out["pairs"] is None
    assert np.array_equal(pkg.partitiondistances(ref, L, "binder")["pairs"][0], [binder_pairs(ref, x) for x in L])
    big = labels_255(g, n)
    msg = str(pytest.raises(pkg.RCError, pkg.partitiondistances, big, np.tile(big, (2, 1))).value)
    assert "does not fit shared memory" in msg and "255 x 255" in msg
    assert not math.isnan(pkg.expectedloss(ref, L)["expectedloss"][0])
