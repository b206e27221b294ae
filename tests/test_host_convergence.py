"""The host side of convergencediagnostics: the split-R-hat of the traces (K, r, p, loglik, logposterior) against an
independent statement of BDA3 11.4, and the argument errors of the list form, which are raised before any device call."""
import importlib
import math

import numpy as np
import pytest


def bda3_split_rhat(x):
    """Chains as rows; the first and last floor(S / 2) samples of each chain are separate sequences."""
    x = np.asarray(x, dtype=np.float64)
    S = x.shape[1]
    h = S // 2
    seqs = [row[:h] for row in x] + [row[S - h:] for row in x]
    if all(np.ptp(s) == 0 for s in seqs):
        return 1.0 if len({float(s[0]) for s in seqs}) == 1 else math.inf
    m = len(seqs)
    means = np.array([s.sum() / h for s in seqs])
    grand = means.sum() / m
    B = h / (m - 1) * ((means - grand) ** 2).sum()
    W = np.mean([((s - s.sum() / h) ** 2).sum() / (h - 1) for s in seqs])
    return math.sqrt(((h - 1) / h * W + B / h) / W)


@pytest.fixture(scope="module")
def host(pkg):
    return importlib.import_module(pkg.__name__ + ".host")


@pytest.mark.parametrize("C, S", [(1, 4), (1, 9), (4, 100), (4, 101), (16, 37)])
def test_trace_rhat_against_bda3(host, C, S):
    g = np.random.default_rng(C * 1000 + S)
    x = g.normal(size=(C, S)) + np.arange(C)[:, None] * 0.3
    assert math.isclose(host._split_rhat(x), bda3_split_rhat(x), rel_tol=1e-12)
    K = g.integers(5, 9, size=(C, S))                           # integer traces, as K
    assert math.isclose(host._split_rhat(K), bda3_split_rhat(K), rel_tol=1e-12)


def test_trace_rhat_drops_the_middle_sample(host):
    x = np.array([[1.0, 2.0, 100.0, 1.0, 2.0], [2.0, 1.0, -50.0, 2.0, 1.0]])
    assert host._split_rhat(x) == host._split_rhat(np.delete(x, 2, axis=1))


def test_trace_rhat_constant_groups(host):
    same = np.full((3, 8), 0.1)
    assert host._split_rhat(same) == 1.0
    differ = np.repeat(np.array([[0.1], [0.1], [0.2]]), 8, axis=1)
    assert host._split_rhat(differ) == math.inf
    halves = np.concatenate([np.full((2, 4), 1.0), np.full((2, 4), 2.0)], axis=1)   # constant halves that disagree
    assert host._split_rhat(halves) == math.inf == bda3_split_rhat(halves)
    with pytest.raises(host.ArgumentError):
        host._split_rhat(np.zeros((2, 3)))


def fake(pkg, S, n, seed=0):
    g = np.random.default_rng(seed)
    r = pkg.MCMCResult()
    r.clusts = [g.integers(1, 4, size=n) for _ in range(S)]
    for k in ("K", "r", "p", "loglik", "logposterior"):
        setattr(r, k, g.normal(size=S))
    return r


def test_list_argument_errors(pkg):
    a = fake(pkg, 10, 20)
    for bad, what in (([], "at least one"), ([a, None], "slot capacity"), ([a, fake(pkg, 11, 20)], "numbers of samples"),
                      ([a, fake(pkg, 10, 21)], "numbers of points")):
        with pytest.raises(pkg.ArgumentError, match=what):
            pkg.convergencediagnostics(bad)
    with pytest.raises(pkg.ArgumentError):
        pkg.cocl_rhat(np.ones((4, 5), np.int64))
