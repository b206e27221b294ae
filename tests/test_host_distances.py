"""CPU tests of the oracle's Euclidean distance matrix (rco_distm, the operation order of the RCB200_DISTM=exact kernel)
against the difference form in np.longdouble, on data where the Gram form |x_i|^2 + |x_j|^2 - 2 x_i.x_j cancels:
offset points, near-duplicates, coordinates of mixed magnitude.  Entries the Gram form cannot resolve are recomputed
from the differences (rc_math.h), so every off-diagonal entry is within (dim + 4) u / tau of the exact distance."""
import numpy as np
import pytest


@pytest.mark.parametrize("family", ["centred", "offset1e2", "offset1e4", "utm", "planted", "mixed", "collinear"])
def test_distm_within_bound_of_longdouble_reference(orc, family):
    rng = np.random.default_rng(sum(map(ord, family)))
    shapes = ((257, 2), (200, 2)) if family == "utm" else ((2, 3), (257, 100), (129, 17), (64, 1000))
    for n, dim in shapes:
        X = orc.distance_family(family, n, dim, rng)
        D = orc.distm(X)
        assert np.array_equal(D, D.T) and np.all(np.diag(D) == 0)
        assert orc.distm_within_bound(D, orc.distm_longdouble(X), dim) <= 1.0, (family, n, dim)


def test_distm_bound_is_tight_enough_to_see_cancellation(orc):
    """The Gram form alone (no recomputation) misses the bound on these data: the test above is not vacuous."""
    rng = np.random.default_rng(7)
    for family, n, dim in (("planted", 257, 100), ("offset1e4", 129, 17), ("utm", 200, 2)):
        X = orc.distance_family(family, n, dim, rng)
        sq = (X * X).sum(1)
        gram = np.sqrt(np.maximum(sq[:, None] + sq[None, :] - 2 * X @ X.T, 0))
        np.fill_diagonal(gram, 0)
        R = orc.distm_longdouble(X)
        off = ~np.eye(n, dtype=bool)
        rel = np.abs(gram[off] - R[off]) / R[off]
        assert rel.max() > 100 * orc.distm_bound(dim), family


def test_distm_utm_pair_one_centimetre_apart(orc):
    """Two points of projected coordinates (metres, ~5e6) 1 cm apart: the Gram form gives 0 (the log of which MCMCData
    cannot take); the recomputed entry is the distance."""
    rng = np.random.default_rng(3)
    X = 5e6 + 100.0 * rng.normal(size=(50, 2))
    X[1] = X[0] + [0.006, 0.008]
    D = orc.distm(X)
    R = orc.distm_longdouble(X)
    assert abs(D[0, 1] - R[0, 1]) <= orc.distm_bound(2) * R[0, 1] and abs(D[0, 1] - 0.01) < 1e-8
    assert orc.distm_within_bound(D, R, 2) <= 1.0


def test_distm_identical_points_give_zero(orc):
    rng = np.random.default_rng(4)
    for X in (rng.normal(size=(40, 33)), 1e4 + rng.normal(size=(40, 33)), np.zeros((5, 7))):
        X[[3, 17 % len(X)]] = X[1]
        D = orc.distm(X)
        assert D[1, 3] == D[3, 1] == 0.0
        assert orc.distm_within_bound(D, orc.distm_longdouble(X), X.shape[1]) <= 1.0


@pytest.mark.parametrize("n,dim", [(3, 1), (129, 17), (100, 1000)])
def test_distm_integer_points_exact(orc, n, dim):
    """Integer coordinates in [-2^16, 2^16]: every product, sum and difference is exact in fp64, so each entry is the
    correctly rounded square root of the exact squared distance, bit for bit, whichever form computes it."""
    rng = np.random.default_rng(n + dim)
    X = rng.integers(-2 ** 16, 2 ** 16 + 1, size=(n, dim)).astype(np.float64)
    X[1] = X[0] + 1                                                        # a pair the Gram form leaves to the recompute
    Xi = X.astype(np.int64)
    exact = np.stack([((Xi - Xi[i]) ** 2).sum(1) for i in range(n)])
    assert np.array_equal(orc.distm(X), np.sqrt(exact.astype(np.float64)))
