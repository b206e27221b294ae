"""Predictive allocation of new observations (rc_predict.cu) at the bench's sizes: per-kernel device times, the call time
with its copies, bytes and operations from shapes, a host numpy baseline on a smaller case, and an output check.

Workload: the bench mixture (bench.synth, n = 10 000 training points, K = 50, dim = 100) with m = 1 000 extra points of the
same draw, passed through crossdistances; S = 16 chains x 250 recorded samples of a Sampler run from the true labels.  A
second case runs at sigma = 0.25 with maxK = 100 (the bench's `moving` setting), where the per-CTA accumulators hold
about twice as many slots.  Writes one JSON document (--out) and prints it."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g  # noqa: E402
import bench  # noqa: E402

HBM_BPS = 7.7e12                     # HGX B200 data sheet, one GPU
PX = 4                               # rc_predict.cu: new points per CTA


def gpu_env():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else "not available")


def samples_T(K):
    """Samples per k_pred_sums CTA (rc_predict.cu: 96 KB of int64 pairs for PX points)."""
    return max(1, min(64, 96 * 1024 // (PX * K * 16)))


def shape_counts(m, n, S, K):
    T = samples_T(K)
    triples = m * n * S
    sums_bytes = -(-S // T) * m * n * 16 + -(-m // PX) * S * n   # image once per sample block, labels once per point block
    cocl_bytes = -(-m // PX) * S * n + m * n * 16               # labels once per point block, output read + written
    return dict(triples=triples, samples_per_cta=T, int64_adds=2 * triples, gathers=triples, fp64_adds=triples,
                sums_dram_bytes=sums_bytes, cocl_dram_bytes=cocl_bytes, transcendentals=3 * m * S * (K + 1))


def kernel_times(fn, reps):
    """Per-kernel device times (CUDA events recorded by the library with RCB200_VERBOSE, read from its stderr line), median
    over `reps` calls after the warm-up."""
    runs = []
    os.environ["RCB200_VERBOSE"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            for _ in range(reps):
                fn()
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["RCB200_VERBOSE"]
        f.seek(0)
        for line in f.read().splitlines():
            if "rc_predict" in line and "CUDA events" in line:
                toks = line.split("):")[1].split()
                runs.append({toks[k]: float(toks[k + 1]) for k in range(0, len(toks), 2)})
    return {k: float(np.median([r[k] for r in runs])) for k in runs[0]}


def bounds(cnt, kernel_ms, n_sm=148, clock_hz=1.965e9):
    """HBM share of k_pred_sums + k_pred_cocl, and the shared-memory atomics and shuffles pass 1 of k_pred_sums issues per
    SM clock: 2 atomic warp instructions and 18 shuffles per 32 columns x 4 points x 1 sample when the warp shares a label
    (training data stored by cluster), 16 atomic warp instructions when it does not."""
    groups = cnt["triples"] / 128
    cycles = kernel_ms["k_pred_sums"] / 1e3 * n_sm * clock_hz
    return dict(hbm_bound_ms=(cnt["sums_dram_bytes"] + cnt["cocl_dram_bytes"]) / HBM_BPS * 1e3,
                warp_groups=groups, sums_sm_cycles=cycles, sums_cycles_per_warp_group_per_sm=cycles / groups,
                atomic_warp_instr_uniform=2 * groups, shuffle_warp_instr_uniform=18 * groups,
                atomic_warp_instr_scattered=16 * groups)


def case(pkg, args, sigma, maxK, label):
    N = args.n + args.m
    X, lab = bench.synth(N, args.K, args.dim, sigma, args.K, args.seed)
    new = np.sort(np.random.default_rng(args.seed).choice(N, size=args.m, replace=False))
    keep = np.setdiff1d(np.arange(N), new)
    data = pkg.MCMCData.from_points(X[keep])
    t = time.perf_counter(); Dn = pkg.crossdistances(X[keep], X[new]); t_cross = time.perf_counter() - t
    params = pkg.params_from_labels(data, lab[keep], maxK=maxK)
    opts = pkg.MCMCOptionsList(numiters=args.burnin + args.samples, burnin=args.burnin)
    rp = [pkg.init_rp(params, args.seed, c) for c in range(args.chains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab[keep], (args.chains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=args.seed)
    t = time.perf_counter(); smp.run(-1); t_run = time.perf_counter() - t
    K = smp.samples_all()["K"]
    S = K.size
    smp.predict(Dn)                                          # warm-up
    calls = []
    for _ in range(args.reps):
        t = time.perf_counter(); out = smp.predict(Dn); calls.append(time.perf_counter() - t)
    kt = kernel_times(lambda: smp.predict(Dn), args.reps)
    cnt = shape_counts(args.m, args.n, S, int(K.max()))
    dev_ms = sum(kt.values())
    kernel_ms = kt["k_pred_sums"] + kt["k_pred_cocl"]
    bd = bounds(cnt, kt)
    smp.close()
    return dict(case=label, sigma=sigma, maxK=maxK, n=args.n, m=args.m, S=S, chains=args.chains, K_mean=float(K.mean()),
                K_max=int(K.max()), crossdistances_s=t_cross, sampler_run_s=t_run, call_s=calls, call_s_median=float(np.median(calls)),
                kernel_ms_cuda_events=kt, device_ms_total=dev_ms, counts=cnt, bounds=bd,
                hbm_share_of_sums_plus_cocl=bd["hbm_bound_ms"] / kernel_ms,
                triples_per_s=cnt["triples"] / (kernel_ms / 1e3),
                newcluster_mean=float(out["newcluster"].mean()))


def baseline(pkg, args):
    """The ascending-order numpy statement of the averages (tests/test_gpu_predict.py, test 3) against the device."""
    n, m, S = 2000, 200, 200
    X, lab = bench.synth(n + m, args.K, args.dim, args.sigma, args.K, args.seed)
    new = np.sort(np.random.default_rng(1).choice(n + m, size=m, replace=False))
    keep = np.setdiff1d(np.arange(n + m), new)
    data = pkg.MCMCData.from_points(X[keep])
    Dn = pkg.crossdistances(X[keep], X[new])
    params = pkg.params_from_labels(data, lab[keep])
    g0 = np.random.default_rng(2)
    labs = np.tile(lab[keep], (S, 1))
    flip = g0.random(labs.shape) < 0.05
    labs[flip] = g0.integers(1, args.K + 1, size=int(flip.sum()))
    labs = np.stack([pkg.sortlabels(x) for x in labs])
    r = g0.gamma(4.0, size=S); p = g0.uniform(0.2, 0.8, size=S)
    lp = pkg.predictive_from_labels(data, Dn, labs, r, p, params, logprobs=True)["logprobs"]
    pkg.predictive_from_labels(data, Dn, labs, r, p, params)     # warm-up
    t = time.perf_counter(); dev = pkg.predictive_from_labels(data, Dn, labs, r, p, params); t_dev = time.perf_counter() - t
    t = time.perf_counter()
    acc, accn = np.zeros((m, n)), np.zeros(m)
    for s in range(S):
        row = lp[s]
        for x in range(m):
            v = row[x][~np.isnan(row[x])]
            e = np.exp(v - v.max()); P = e / e.sum()
            acc[x] += P[labs[s] - 1]
            accn[x] += P[labs[s].max()] if P.size > labs[s].max() else 0.0
    acc /= S; accn /= S
    t_np = time.perf_counter() - t
    return dict(n=n, m=m, S=S, numpy_s=t_np, device_call_s=t_dev, speedup=t_np / t_dev,
                max_abs_diff_coclustering=float(np.abs(dev["coclustering"] - acc).max()),
                max_abs_diff_newcluster=float(np.abs(dev["newcluster"] - accn).max()),
                note="the numpy statement starts from the kernel's log-probabilities; the device call includes the relabelling, "
                     "the copies and the log-probabilities themselves")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--m", type=int, default=1000)
    ap.add_argument("--K", type=int, default=50)
    ap.add_argument("--dim", type=int, default=100)
    ap.add_argument("--sigma", type=float, default=0.1)
    ap.add_argument("--chains", type=int, default=16)
    ap.add_argument("--samples", type=int, default=250)
    ap.add_argument("--burnin", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = g.load_package()
    res = dict(env=gpu_env(), bench_mixture=case(pkg, args, args.sigma, 0, "bench mixture"),
               large_K=case(pkg, args, 0.25, 100, "moving setting"), baseline=baseline(pkg, args))
    res["env_after"] = gpu_env()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
