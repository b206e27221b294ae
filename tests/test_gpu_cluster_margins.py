"""Scans decided as a whole by per-slot margins of the row summaries: a stationary chain's scan tests O(K) slot bounds and
one uniform per row instead of n summaries.  The margins are validated by the chain's change count, survive launches and are
reset with the other caches, so every output stays bit-identical to the oracle's."""
import numpy as np
import pytest

from test_gpu_sampler import assert_same, mixture, oparams, run_both

pytestmark = pytest.mark.gpu


def separated(pkg):
    X, lab = mixture(600, 6, 10, 0.12, 4)
    data = pkg.MCMCData.from_points(X)
    return data.D, lab, pkg.params_from_labels(data.D, lab)


def margin_scans(smp):
    return int(smp.stats()["bulk_reduce"].sum())     # (counts in the default library)


def test_margins_decide_scans_and_change_nothing(pkg, orc):
    D, lab, params = separated(pkg)
    res, smp = run_both(pkg, orc, D, lab, params, 40, 0, 1, 5, 1, seed=9, nchains=2)
    for got, ref, st in res:
        assert_same(got, ref, st)
    assert margin_scans(smp) > 0


def test_margins_in_launch_groups_resumed(pkg, orc, monkeypatch):
    """One chain per launch group (every launch starts with every cache stale), resumed over three calls."""
    monkeypatch.setenv("RCB200_CHAINS_PER_GROUP", "1")
    D, lab, params = separated(pkg)
    iters, nch, seed = 40, 3, 9
    opts = pkg.MCMCOptionsList(numiters=iters, burnin=0, thin=1, numGibbs=5, numMH=1)
    rp = [pkg.init_rp(params, seed, c) for c in range(nch)]
    smp = pkg.Sampler(pkg.MCMCData(np.ascontiguousarray(D)), opts, params, np.tile(lab, (nch, 1)), [x[0] for x in rp],
                      [x[1] for x in rp], seed=seed)
    smp.run(15); smp.run(10); smp.run(-1)
    assert smp.check_sums() == (0, 0)
    for c in range(nch):
        ref = orc.run_chain(D, orc.Options(iters, 0, 1, 5, 1), oparams(orc, params), lab, rp[c][0], rp[c][1], seed=seed, chain=c)
        assert_same(smp.samples(c), ref, smp.state(c))
    assert margin_scans(smp) > 0


def test_no_margin_scans_without_shortcuts(pkg, orc, monkeypatch):
    monkeypatch.setenv("RCB200_SHORTCUTS", "0")
    D, lab, params = separated(pkg)
    res, smp = run_both(pkg, orc, D, lab, params, 40, 0, 1, 5, 1, seed=9, nchains=2)
    for got, ref, st in res:
        assert_same(got, ref, st)
    assert margin_scans(smp) == 0
