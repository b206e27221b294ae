"""GPU tests of MCMCData(points)'s Euclidean distance matrix on every path (the default 128 x 128-tile DMMA kernel,
RCB200_DISTM=exact and RCB200_DISTM=dmma32), of its row blocks and of crossdistances, against the difference form in
np.longdouble.  The data are those on which the Gram form |x_i|^2 + |x_j|^2 - 2 x_i.x_j cancels (offset points,
projected coordinates, near-duplicates, mixed magnitudes); the shapes sit on both sides of the 32- and 128-point tiles
and of the 16- and 32-coordinate chunks.  Every off-diagonal entry must be within (dim + 4) u / tau of the exact
distance, and on integer points, where every form is exact, equal to it bit for bit."""
import ctypes as C
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = [None, "exact", "dmma32"]
NS = (2, 3, 127, 128, 129, 255, 256, 257, 1000)
# every n and every dim in {1, 2, 15, 16, 17, 33, 130, 1000} appears
SHAPES = ((2, 1000), (3, 1), (127, 16), (128, 17), (129, 15), (255, 130), (256, 33), (257, 2), (257, 1000), (1000, 17), (1000, 130))
FEW = ((3, 2), (129, 17), (257, 130), (1000, 33))
CASES = ([(f, n, d) for f in ("offset1e2", "offset1e4", "planted") for n, d in SHAPES] + [("utm", n, 2) for n in NS] +
         [(f, n, d) for f in ("centred", "mixed", "collinear") for n, d in FEW])


def set_mode(monkeypatch, mode):
    if mode:
        monkeypatch.setenv("RCB200_DISTM", mode)
    else:
        monkeypatch.delenv("RCB200_DISTM", raising=False)


@functools.lru_cache(maxsize=None)
def case(orc, family, n, dim):
    X = orc.distance_family(family, n, dim, np.random.default_rng([sum(map(ord, family)), n, dim]))
    return X, orc.distm_longdouble(X)


@pytest.mark.parametrize("mode", MODES)
def test_from_points_within_bound(pkg, orc, monkeypatch, mode):
    set_mode(monkeypatch, mode)
    worst = {}
    for family, n, dim in CASES:
        X, R = case(orc, family, n, dim)
        D = pkg.MCMCData.from_points(X).D
        assert np.array_equal(D, D.T) and np.all(np.diag(D) == 0), (family, n, dim)
        r = orc.distm_within_bound(D, R, dim)
        assert r <= 1.0, (family, n, dim, r)
        worst[family] = max(worst.get(family, 0.0), r)
        if mode == "exact":
            assert np.array_equal(D, orc.distm(X)), (family, n, dim)       # the oracle's operation order
    print(mode, {k: f"{v:.3g}" for k, v in worst.items()})


@pytest.mark.parametrize("mode", MODES)
def test_from_points_integer_points_bit_exact(pkg, monkeypatch, mode):
    """Integer coordinates in [-2^16, 2^16], dim <= 1000: every product, sum and difference is exact in fp64, so each
    entry is the correctly rounded square root of the exact squared distance whichever form, tile or chunk computes
    it.  A wrong index, padding or mirror in a ragged tile shows here as a wrong bit."""
    set_mode(monkeypatch, mode)
    for n, dim in SHAPES + ((1000, 1000),):
        g = np.random.default_rng([n, dim])
        X = g.integers(-2 ** 16, 2 ** 16 + 1, size=(n, dim)).astype(np.float64)
        X[1] = X[0]
        X[1, -1] += 1                                                      # distance 1: left to the recompute
        sq = (X * X).sum(1)
        exact = sq[:, None] + sq[None, :] - 2 * (X @ X.T)                  # integers below 2^53: exact in any order
        np.fill_diagonal(exact, 0)
        assert np.array_equal(pkg.MCMCData.from_points(X).D, np.sqrt(exact)), (n, dim)


def distm_rows(pkg, X, row0, nrows):
    import torch
    from redclust_jl_b200._lib import check, lib, ptr
    n, dim = X.shape
    buf = torch.full((nrows, n), -1.0, dtype=torch.float64, device="cuda")
    check(lib().rc_distm_rows_dev(ptr(X), dim, n, row0, nrows, 0, C.c_void_p(buf.data_ptr())))
    return buf.cpu().numpy()


@pytest.mark.parametrize("mode", [None, "exact"])
def test_row_blocks_bit_equal_to_whole_matrix(pkg, orc, monkeypatch, mode):
    """rc_distm_rows_dev: the non-symmetric launch with an arbitrary first row and a partial last tile, on offset data
    with planted pairs (entries recomputed on both sides) -- the same rows of from_points bit for bit."""
    set_mode(monkeypatch, mode)
    for n, dim in ((257, 17), (1000, 130)):
        X = 1e3 + orc.distance_family("planted", n, dim, np.random.default_rng([n, dim, 5]))
        full = pkg.MCMCData.from_points(X).D
        assert orc.distm_within_bound(full, orc.distm_longdouble(X), dim) <= 1.0
        for row0, nrows in ((0, 1), (1, 1), (n - 1, 1), (127, 130), (5, n - 5)):
            assert np.array_equal(distm_rows(pkg, X, row0, nrows), full[row0:row0 + nrows]), (n, dim, row0, nrows)
        assert np.array_equal(pkg.MCMCData.from_points_sharded(X).D, full)    # a world of one


@pytest.mark.parametrize("mode", [None, "exact"])
def test_crossdistances_within_bound(pkg, orc, monkeypatch, mode):
    set_mode(monkeypatch, mode)
    g = np.random.default_rng(8)
    X = 1e4 + g.normal(size=(300, 17))
    for Y in (X[7:8] + 1e-6 * g.normal(size=(1, 17)),                     # m = 1, next to a training point
              X[:40] + 1e5,                                                # far from every training point
              5e6 + 100 * g.normal(size=(33, 17))):
        got = pkg.crossdistances(X, Y)
        assert orc.distm_within_bound(got, orc.distm_longdouble(X, Y), 17) <= 1.0
        assert np.array_equal(got, pkg.MCMCData.from_points(np.vstack([X, Y])).D[300:, :300])
    same = pkg.crossdistances(X, X[[4, 250]])                              # identical points: exactly 0
    assert same[0, 4] == 0.0 and same[1, 250] == 0.0
    assert orc.distm_within_bound(same, orc.distm_longdouble(X, X[[4, 250]]), 17) <= 1.0


@pytest.mark.parametrize("mode", MODES)
def test_close_pairs_accepted_duplicates_refused(pkg, orc, monkeypatch, mode):
    """Projected coordinates with two points 1 cm apart are valid data (the Gram form gave them distance 0, refused as
    a zero dissimilarity); a truly duplicated point is still refused with RC_ERR_DOMAIN, also on offset data, where the
    Gram form leaves rounding noise instead of 0."""
    set_mode(monkeypatch, mode)
    g = np.random.default_rng(3)
    X = 5e6 + 100.0 * g.normal(size=(50, 2))
    X[1] = X[0] + [0.006, 0.008]
    D = pkg.MCMCData.from_points(X).D
    R = orc.distm_longdouble(X)
    assert abs(D[0, 1] - R[0, 1]) <= orc.distm_bound(2) * R[0, 1]
    assert orc.distm_within_bound(D, R, 2) <= 1.0
    for Y in (X.copy(), 1e4 + g.normal(size=(200, 33)), g.normal(size=(129, 16))):
        Y[-1] = Y[len(Y) // 2]
        with pytest.raises(pkg.RCError) as e:
            pkg.MCMCData.from_points(Y)
        assert e.value.status == -4
