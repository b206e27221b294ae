"""The two ways post-processing reaches samples.  The sampler's recorded samples: every entry point that reads them (PSM,
device counts, Binder MPEL, predictive, and the PSM over every rank) refuses before a run to numiters (RC_ERR_STATE),
over a bad chain range (RC_ERR_ARG) and over a chain stopped at the slot capacity (RC_ERR_SLOTS), since nothing wrote
those samples.  Host label vectors: a device index out of range is RC_ERR_ARG from every entry point that takes one."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

METHODS = ["psm", "psm_counts_dev", "binder_pointestimate", "predict", "psm_allreduce"]


@pytest.fixture(scope="module")
def held_out(golden):
    """Example 3 without every 30th point: training distances, the held-out points' rows and the training labels."""
    X, lab = golden[3]["points"], golden[3]["cluster_labels"]
    held = np.arange(0, X.shape[0], 30)
    keep = np.setdiff1d(np.arange(X.shape[0]), held)
    D = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1))
    D = (D + D.T) / 2
    return np.ascontiguousarray(D[np.ix_(keep, keep)]), np.ascontiguousarray(D[np.ix_(held, keep)]), lab[keep]


@pytest.fixture(scope="module")
def comm(pkg):
    return pkg.Comm.from_torch(device=0)


def read(smp, method, comm, newdist, *chains):
    """What `method` computes from the sampler's samples of chains[0] .. chains[0] + chains[1] - 1 (all by default)."""
    import torch
    n = smp.data.n
    if method == "psm":
        return smp.psm(*chains)
    if method == "psm_counts_dev":
        cnt = torch.zeros((n, n), dtype=torch.int32, device="cuda")
        smp.psm_counts_dev(cnt.data_ptr(), *chains)
        return cnt.cpu().numpy()
    if method == "binder_pointestimate":
        return smp.binder_pointestimate(*chains)["sums"]
    if method == "predict":
        return smp.predict(newdist, *chains)["coclustering"]
    assert not chains
    return smp.psm_allreduce(comm=comm)


def refused(pkg, status, fn, *args):
    with pytest.raises(pkg.RCError) as e:
        fn(*args)
    assert e.value.status == status, str(e.value)


@pytest.mark.parametrize("method", METHODS)
def test_sampler_samples_need_a_complete_run(pkg, golden, held_out, comm, method):
    D, Dn, lab = held_out
    params = pkg.params_from_labels(D, lab)
    rp = [pkg.init_rp(params, 2, c) for c in range(2)]
    smp = pkg.Sampler(pkg.MCMCData(D), pkg.MCMCOptionsList(numiters=30, burnin=5), params, np.tile(lab, (2, 1)),
                      [x[0] for x in rp], [x[1] for x in rp], seed=2)
    smp.run(10)
    refused(pkg, -6, read, smp, method, comm, Dn)
    smp.run(-1)
    if method != "psm_allreduce":                          # the other methods take a chain range
        for c0, k in ((-1, 1), (0, 0), (1, 2), (2, 1)):
            refused(pkg, -1, read, smp, method, comm, Dn, c0, k)
    assert np.all(np.isfinite(read(smp, method, comm, Dn)))
    smp.close()
    # the chain stops at a capacity of 10 live clusters on the 10-cluster example (as in test_gpu_sampler)
    D1, lab1 = golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    stopped = pkg.Sampler(pkg.MCMCData(D1), pkg.MCMCOptionsList(numiters=50, burnin=0, thin=1), pkg.params_from_labels(D1, lab1),
                          lab1, 1.0, 0.5, seed=2, slot_cap=10)
    with pytest.raises(pkg.RCError):
        stopped.run(-1)
    refused(pkg, -5, read, stopped, method, comm, np.ones((1, D1.shape[0])))
    stopped.close()


def test_device_out_of_range(pkg, golden):
    import torch
    from redclust_jl_b200._lib import lib
    bad = int(lib().rc_device_count())                     # one past the last device
    L = np.tile(golden[1]["cluster_labels"], (3, 1))
    X = golden[1]["points"]
    n = L.shape[1]
    cnt = torch.zeros((n, n), dtype=torch.int32, device="cuda")
    calls = [(pkg.psm, L), (pkg.psm_counts_dev, L, cnt.data_ptr()), (pkg.mpel_loss_sums, L, "binder"), (pkg.binder_loss_sums, L),
             (pkg.crossdistances, X[2:], X[:2]), (pkg.kmeans, X.T, 2)]
    for fn, *args in calls:
        with pytest.raises(pkg.RCError) as e:
            fn(*args, device=bad)
        assert e.value.status == -1 and "out of range" in str(e.value), (fn.__name__, str(e.value))
