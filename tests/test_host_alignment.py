"""The host side of the aligned allocation: a restatement of the canonical assignment (the shortest-augmenting-path
Hungarian method with int64 potentials whose tie rule defines which optimum alignedallocation returns) against scipy's
optimum on tables full of ties, rectangular both ways, from 1 x 1 to 255 x 255; and the argument errors of
alignedallocation / Sampler.alignedallocation, which are raised before any device call."""
import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment


def canonical(T):
    """sigma (index 0 unused, sigma[l] in 0..Kh, 0 = unmatched) and matched of the Kh x Kt overlap table T (rows = estimate
    clusters): e-maxx Hungarian on the square N = max(Kh, Kt) cost -T (0 in the padding), rows added in ascending order;
    in each Dijkstra step over the unused columns `cur < minv` (strict) updates minv / way and the first column of the
    smallest minv is taken.  The loop over the columns is vectorised; each column's update is independent of the others."""
    Kh, Kt = T.shape
    N = max(Kh, Kt)
    a = np.zeros((N + 1, N + 1), np.int64)
    a[1:Kh + 1, 1:Kt + 1] = -np.asarray(T, np.int64)
    INF = np.iinfo(np.int64).max // 4
    u, v = np.zeros(N + 1, np.int64), np.zeros(N + 1, np.int64)
    p, way = np.zeros(N + 1, np.int64), np.zeros(N + 1, np.int64)
    for i in range(1, N + 1):
        p[0], j0 = i, 0
        minv, used = np.full(N + 1, INF, np.int64), np.zeros(N + 1, bool)
        while True:
            used[j0] = True
            i0, free = p[j0], ~used
            cur = a[i0] - u[i0] - v
            upd = free & (cur < minv)
            minv[upd], way[upd] = cur[upd], j0
            cand = np.where(free, minv, INF + 1)
            j1 = int(np.argmin(cand))                      # the first column of the smallest minv
            delta = cand[j1]
            u[p[used]] += delta
            v[used] -= delta
            minv[free] -= delta
            j0 = j1
            if p[j0] == 0:
                break
        while j0:
            j1 = way[j0]
            p[j0] = p[j1]
            j0 = j1
    sigma = np.zeros(Kt + 1, np.int64)
    for l in range(1, Kt + 1):
        k = p[l]
        if k <= Kh and T[k - 1, l - 1] > 0:
            sigma[l] = k
    matched = int(sum(T[sigma[l] - 1, l - 1] for l in range(1, Kt + 1) if sigma[l]))
    return sigma, matched


def tables():
    g = np.random.default_rng(3)
    out = [np.array([[0]]), np.array([[5]]), np.array([[0, 0, 0]]), np.array([[2], [2], [1]])]
    for _ in range(300):
        kh, kt = (int(x) for x in g.integers(1, 12, size=2))
        out.append(g.integers(0, 4, size=(kh, kt)))
    for kh, kt in ((255, 255), (255, 3), (2, 255), (40, 200), (180, 17)):
        out.append(g.integers(0, 3, size=(kh, kt)) * g.integers(0, 2, size=(kh, kt)))
    out.append(np.ones((255, 255), np.int64))                  # every assignment is optimal
    return out


def test_restatement_reaches_the_optimum():
    for T in tables():
        sigma, matched = canonical(T)
        r, c = linear_sum_assignment(T, maximize=True)
        assert matched == T[r, c].sum(), T.shape
        used = sigma[sigma > 0]
        assert len(set(used.tolist())) == used.size            # one sample cluster per estimate cluster
        assert all(T[sigma[l] - 1, l - 1] > 0 for l in range(1, T.shape[1] + 1) if sigma[l])


def test_restatement_ties_go_to_the_first():
    sigma, matched = canonical(np.array([[3], [5], [5], [1]]))
    assert sigma.tolist() == [0, 2] and matched == 5
    sigma, _ = canonical(np.ones((3, 3), np.int64))
    assert sigma.tolist() == [0, 1, 2, 3]


def fake(pkg, S, n, seed=0):
    g = np.random.default_rng(seed)
    r = pkg.MCMCResult()
    r.clusts = [g.integers(1, 4, size=n) for _ in range(S)]
    return r


def test_argument_errors(pkg):
    a = fake(pkg, 6, 20)
    L = np.stack(a.clusts)
    est = L[0]
    bad = [
        (lambda: pkg.alignedallocation(est[:-1], a), "estimate must label the 20 points"),
        (lambda: pkg.alignedallocation(np.stack([est, est]), a), "estimate must label"),
        (lambda: pkg.alignedallocation(est, []), "at least one MCMCResult"),
        (lambda: pkg.alignedallocation(est, [a, None]), r"slot capacity \(its result is None\); drop it before pooling"),
        (lambda: pkg.alignedallocation(est, np.zeros((0, 20), np.int64)), "non-empty"),
        (lambda: pkg.alignedallocation(est, [fake(pkg, 0, 20)]), "no sample"),
        (lambda: pkg.alignedallocation(est, [a, fake(pkg, 3, 21)]), "different numbers of points"),
        (lambda: pkg.alignedallocation(est, L[:, :19]), "estimate must label the 19 points"),
    ]
    for fn, what in bad:
        with pytest.raises(pkg.ArgumentError, match=what):
            fn()


def test_sampler_argument_errors(pkg):
    """The Sampler methods check the estimate against the sampler's n before any call into the library."""
    smp = pkg.Sampler.__new__(pkg.Sampler)

    class _Data:
        n = 20
    smp.data = _Data()
    for fn in (lambda: smp.alignedallocation(np.ones(19, np.int64)), lambda: smp.alignedallocation_allreduce(np.ones((2, 20)))):
        with pytest.raises(pkg.ArgumentError, match="estimate must label the 20 points"):
            fn()
