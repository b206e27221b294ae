"""The host side of the credible ball: _credibleball against an independent loop-based statement of Wade & Ghahramani
(2018, section 4) on constructed distances with ties at the radius, several samples at the extreme numbers of clusters
and alpha near 0 and 1, and the argument errors of credibleball / expectedloss / partitiondistances, which are raised
before any device call."""
import importlib

import numpy as np
import pytest


@pytest.fixture(scope="module")
def host(pkg):
    return importlib.import_module(pkg.__name__ + ".host")


def ball_loop(d, K, alpha):
    """The definition, one sample at a time: the radius is the smallest sample distance e whose ball holds at least
    1 - alpha of the samples; each bound lists every sample of the ball that attains it."""
    S = len(d)
    radius = None
    for e in sorted(set(d)):
        if sum(1 for x in d if x <= e) / S >= 1 - alpha:
            radius = e
            break
    ball = [t for t in range(S) if d[t] <= radius]

    def farthest(ts):
        far = max(d[t] for t in ts)
        return far, [t for t in ts if d[t] == far]
    kmin, kmax = min(K[t] for t in ball), max(K[t] for t in ball)
    return dict(radius=radius, inball=len(ball), horizontal=farthest(ball), upper=farthest([t for t in ball if K[t] == kmin]),
                lower=farthest([t for t in ball if K[t] == kmax]))


def assert_ball(got, want, K):
    assert got["radius"] == want["radius"] and got["inball"] == want["inball"]
    for name in ("horizontal", "upper", "lower"):
        far, idx = want[name]
        assert got[name]["dist"] == far, name
        assert got[name]["indices"].tolist() == idx, name
        assert got[name]["K"] == K[idx[0]], name


def cases():
    g = np.random.default_rng(11)
    out = []
    # ties at the radius: four samples at 0.25 straddle the 1 - alpha point
    d = np.array([0.0, 0.1, 0.25, 0.25, 0.25, 0.25, 0.4, 0.5, 0.1, 0.0])
    K = np.array([3, 3, 2, 5, 2, 5, 1, 6, 4, 3])
    out += [(d, K, a) for a in (0.05, 0.2, 0.3, 0.5, 0.6, 0.65, 0.8)]
    # several samples at the fewest / most clusters, at different distances
    d = np.array([0.3, 0.1, 0.3, 0.2, 0.05, 0.3, 0.2, 0.1])
    K = np.array([2, 2, 7, 7, 4, 2, 7, 3])
    out += [(d, K, a) for a in (0.01, 0.1, 0.3, 0.5)]
    # alpha near 0 (the whole sample) and near 1 (the nearest samples only)
    for a in (1e-12, 1e-3, 1 - 1e-3, 1 - 1e-12):
        d = g.choice([0.0, 0.125, 0.5, 0.75, 1.0], size=200)
        out.append((d, g.integers(1, 9, size=200), a))
    # random distances from a small set of values (many ties), random K
    for _ in range(20):
        S = int(g.integers(1, 300))
        out.append((g.choice(g.random(6), size=S), g.integers(1, 12, size=S), float(g.random())))
    return out


@pytest.mark.parametrize("k", range(len(cases())))
def test_ball_against_the_definition(host, k):
    d, K, alpha = cases()[k]
    assert_ball(host._credibleball(d, K, alpha), ball_loop(list(d), list(K), alpha), K)


def test_ball_edge_values(host):
    d, K = np.array([0.5, 0.0, 0.5, 0.0]), np.array([3, 1, 3, 1])
    b = host._credibleball(d, K, 0.5)                           # exactly half the samples at distance 0
    assert b["radius"] == 0.0 and b["inball"] == 2 and b["upper"]["indices"].tolist() == [1, 3]
    b = host._credibleball(d, K, 0.49)
    assert b["radius"] == 0.5 and b["inball"] == 4 and b["lower"]["indices"].tolist() == [0, 2] and b["lower"]["K"] == 3
    one = host._credibleball(np.array([0.7]), np.array([4]), 0.05)
    assert one["radius"] == 0.7 and all(one[x]["indices"].tolist() == [0] for x in ("horizontal", "upper", "lower"))


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
        (lambda: pkg.credibleball(est[:-1], a), "estimate must label the 20 points"),
        (lambda: pkg.credibleball(np.stack([est, est]), a), "estimate must label"),
        (lambda: pkg.credibleball(est, a, alpha=0.0), r"alpha must lie in \(0, 1\)"),
        (lambda: pkg.credibleball(est, a, alpha=1.0), "alpha"),
        (lambda: pkg.credibleball(est, a, alpha=-0.5), "alpha"),
        (lambda: pkg.credibleball(est, a, loss="vi"), "loss must be one of"),
        (lambda: pkg.credibleball(est, a, loss=lambda x, y: 0.0), "function-valued"),
        (lambda: pkg.expectedloss(est, a, loss="Binder"), "loss must be one of"),
        (lambda: pkg.partitiondistances(est, a, loss=2), "loss must be one of"),
        (lambda: pkg.credibleball(est, []), "at least one MCMCResult"),
        (lambda: pkg.credibleball(est, [a, None]), r"slot capacity \(its result is None\); drop it before pooling"),
        (lambda: pkg.credibleball(est, np.zeros((0, 20), np.int64)), "non-empty"),
        (lambda: pkg.expectedloss(est, [fake(pkg, 0, 20)]), "no sample"),
        (lambda: pkg.expectedloss(est, [a, fake(pkg, 3, 21)]), "different numbers of points"),
        (lambda: pkg.expectedloss(est[:5], L), "partitions must label the 20 points"),
        (lambda: pkg.partitiondistances(np.zeros((0, 20), np.int64), L), "refs must label"),
    ]
    for fn, what in bad:
        with pytest.raises(pkg.ArgumentError, match=what):
            fn()
