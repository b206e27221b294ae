"""The sampler at large n (30 000 by default; up to 65 535, the 16-bit point indices): a few sweeps of a few chains, checked by the sums invariant (the maintained
row / block sums against a rebuild from the labels) and by the log-likelihood of the final state recomputed through
rc_loglik-free means (block sums rebuilt).  usage: python tools/large_n_probe.py [n] [chains] [sweeps]"""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g
import bench

n = int(sys.argv[1]) if len(sys.argv) > 1 else 30000
chains = int(sys.argv[2]) if len(sys.argv) > 2 else 8
sweeps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
pkg = g.load_package()
X, lab = bench.synth(n, 50, 100, 0.12, 50, 44)
t = time.perf_counter()
data = pkg.MCMCData.from_points(X)
print(f"MCMCData(points) n={n}: {time.perf_counter() - t:.2f} s", flush=True)
params = pkg.params_from_labels(data, lab)
opts = pkg.MCMCOptionsList(numiters=sweeps, burnin=0, thin=1)
rp = [pkg.init_rp(params, 5, c) for c in range(chains)]
smp = pkg.Sampler(data, opts, params, np.tile(lab, (chains, 1)), [a for a, _ in rp], [b for _, b in rp], seed=5, slot_cap=96)
smp.run(0)
t = time.perf_counter(); smp.run(-1); dt = time.perf_counter() - t
st = smp.stats()
out = smp.samples(0)
print(f"n={n}: {chains} chains x {sweeps} sweeps in {dt:.2f} s ({chains * sweeps / dt:.1f} chain-sweeps/s), moves per sweep {st['moves'].sum() / (chains * sweeps):.1f}, "
      f"K {out['K'].tolist()}, loglik {out['loglik'].tolist()}", flush=True)
print("sums invariant (mismatching words S, W):", smp.check_sums(), flush=True)
