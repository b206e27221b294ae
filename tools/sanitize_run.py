"""Small sampler runs for compute-sanitizer (racecheck / synccheck / memcheck): all chains in one launch and one chain per
launch group, on the reference's n = 100 fixture (split-merge, several proposals per iteration, two chains) and an
n = 2500 problem, each checked against the oracle.  usage: compute-sanitizer --tool racecheck python tools/sanitize_run.py [small|large]"""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import __graft_entry__ as g
from test_gpu_sampler import assert_same, mixture, oparams

which = sys.argv[1] if len(sys.argv) > 1 else "small"
pkg, orc = g.load_package(), g.load_oracle()


def run(D, lab, iters, numMH, nch, mode, seed):
    if mode == "grouped":
        os.environ["RCB200_CHAINS_PER_GROUP"] = "1"
    else:
        os.environ.pop("RCB200_CHAINS_PER_GROUP", None)
    params = pkg.params_from_labels(D, lab)
    opts = pkg.MCMCOptionsList(numiters=iters, burnin=0, thin=1, numGibbs=3, numMH=numMH)
    rp = [pkg.init_rp(params, seed, c) for c in range(nch)]
    smp = pkg.Sampler(pkg.MCMCData(np.ascontiguousarray(D)), opts, params, np.tile(lab, (nch, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=seed)
    smp.run(-1)
    for c in range(nch):
        ref = orc.run_chain(D, orc.Options(iters, 0, 1, 3, numMH), oparams(orc, params), lab, rp[c][0], rp[c][1], seed=seed, chain=c)
        assert_same(smp.samples(c), ref, smp.state(c))
    print(f"ok: mode={mode} n={D.shape[0]} iters={iters} numMH={numMH} chains={nch}", flush=True)


if which == "small":
    gd = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "example1.npz"))
    D, lab = gd["distance_matrix"], gd["cluster_labels"]
    for mode in ("resident", "grouped"):
        run(D, lab, 12, 1, 2, mode, 3)
        run(D, np.ones(100, np.int64), 8, 2, 1, mode, 4)
else:
    X, lab = mixture(2500, 12, 20, 0.2, 8)
    D = orc.distm(X)
    for mode in ("resident", "grouped"):
        run(D, lab, 2, 1, 2, mode, 5)
