"""Chains in launch groups against chains in one launch: the bench workload (generatemixture n = 10 000, K = 50, dim = 100,
sigma = 0.1, numGibbs = 5, numMH = 1, true labels) with 512 chains by default, timed as one run(STEPS) call and as STEPS
run(1) calls.  In launch groups every call rebuilds each group's row sums from its labels, so the run(1) pattern pays
that rebuild once per sweep.  RCB200_CHAINS_PER_GROUP=m forces groups of m chains (256: two groups of the 512).
Prints one JSON line: chain-sweeps/s of both patterns (device time of the runs and wall time around them) and a digest of
the recorded outputs of four chains (the first and last chain of each half), which does not depend on how the chains
were launched.
usage: python tools/group_probe.py [chains] [steps]"""
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402
import bench  # noqa: E402

chains = int(sys.argv[1]) if len(sys.argv) > 1 else 512
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
pkg = g.load_package()
X, lab = bench.synth(10000, 50, 100, 0.1, 50, 44)
data = pkg.MCMCData.from_points(X)
params = pkg.params_from_labels(data, lab)
opts = pkg.MCMCOptionsList(numiters=1 + 2 * steps, burnin=0, thin=1, numGibbs=5, numMH=1)
rp = [pkg.init_rp(params, 44, c) for c in range(chains)]
smp = pkg.Sampler(data, opts, params, np.tile(lab, (chains, 1)), [a for a, _ in rp], [b for _, b in rp], seed=44)
smp.run(1)                                             # warm-up: module load, first-use allocations, the chains' first sweep


def timed(calls, iters):
    _, d0 = smp.progress()
    w0 = time.perf_counter()
    for _ in range(calls):
        smp.run(iters)                                 # returns after the device has finished
    w1 = time.perf_counter()
    _, d1 = smp.progress()
    sweeps = chains * calls * iters
    return {"chain_sweeps_per_s_device": sweeps / (d1 - d0), "chain_sweeps_per_s_wall": sweeps / (w1 - w0),
            "device_s": d1 - d0, "wall_s": w1 - w0}


one = timed(1, steps)
many = timed(steps, 1)
h = hashlib.sha256()
for c in sorted({0, chains // 2 - 1, chains // 2, chains - 1}):
    s = smp.samples(c)
    for k in ("labels", "K", "r", "p", "loglik", "logposterior", "r_acc", "sm_acc", "sm_split"):
        h.update(np.ascontiguousarray(s[k]).tobytes())
print(json.dumps({"chains": chains, "steps": steps, "chains_per_group": os.environ.get("RCB200_CHAINS_PER_GROUP"),
                  "run_steps": one, "run_1_x_steps": many, "outputs_sha256": h.hexdigest(),
                  "check_sums": list(smp.check_sums())}), flush=True)
smp.close()
