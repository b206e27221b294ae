"""Distances from a given partition to pooled samples (rc_sampler_partition_dists, the k_pair_loss launch mode of
reference rows) at the size they exist for, and the credible ball built on them.  Kernel times are CUDA events inside the
library (printed with RCB200_VERBOSE), the whole call is a host clock around separate calls; medians of 3 after a warm-up.
Beside each case, rc_mpel's pair rate at the same n and K in the same process: the pairwise search over the first 2 000
samples, and the new path over the same 2 000 host label vectors.  Writes one JSON document (--out) and prints it.

Cases (n = 10 000, 256 chains x 1 000 recorded samples, from the sampler's device-resident samples; the estimate is the
simulation's true partition):
  stationary  the bench mixture (bench.synth: K = 50, dim = 100, sigma = 0.1)
  moving      bench's `moving` setting: sigma = 0.25 with maxK = 100, chains that keep moving points"""
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


def gpu_env():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else "not available")


def verbose_call(fn, key):
    """fn() with RCB200_VERBOSE=1; returns (result, host seconds, the library's last line that contains key)."""
    os.environ["RCB200_VERBOSE"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            t = time.perf_counter()
            out = fn()
            dt = time.perf_counter() - t
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["RCB200_VERBOSE"]
        f.seek(0)
        line = [x for x in f.read().splitlines() if key in x][-1]
    return out, dt, line


def kernel_ms(line):
    return float(line.split("k_pair_loss ")[1].split()[0])


def mpel_rate(line):
    return float(line.split("(")[-1].split()[0])


def ball_summary(b):
    return dict(radius=b["radius"], inball=b["inball"], expectedloss=b["expectedloss"],
                **{k: dict(dist=b[k]["dist"], K=b[k]["K"], count=int(b[k]["indices"].size), first=int(b[k]["indices"][0]))
                   for k in ("horizontal", "upper", "lower")})


def case(pkg, args, name, sigma, maxK):
    from redclust_jl_b200._lib import lib, check, ptr
    X, lab = bench.synth(args.n, 50, 100, sigma, 50, args.seed)
    data = pkg.MCMCData.from_points(X)
    params = pkg.params_from_labels(data.D, lab, maxK=maxK)
    opts = pkg.MCMCOptionsList(numiters=args.samples, burnin=0)
    rp = [pkg.init_rp(params, args.seed, c) for c in range(args.chains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (args.chains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=args.seed)
    t = time.perf_counter(); smp.run(-1); t_run = time.perf_counter() - t
    S = args.chains * args.samples
    res = dict(case=name, sigma=sigma, maxK=maxK, n=args.n, chains=args.chains, samples_per_chain=args.samples, sampler_run_s=t_run)
    for loss in ("VI", "binder"):
        first = smp.credibleball(lab, loss=loss)                       # warm-up of every shape the timed calls use
        ks, calls = [], []
        for _ in range(args.reps):
            _, _, line = verbose_call(lambda: smp.credibleball(lab, loss=loss), "partition dists:")
            ks.append(kernel_ms(line))
            t = time.perf_counter(); again = smp.credibleball(lab, loss=loss); calls.append(time.perf_counter() - t)
            assert np.array_equal(again["dist"], first["dist"])
        K = smp._partition_dists(lab, 0, smp.nchains, loss)["K"]
        ms = float(np.median(ks))
        # the same launch without the exact Binder counts (pairs_out = NULL): what the integer sums cost
        P, d = np.ascontiguousarray(lab[None, :], dtype=np.int64), np.empty(S)
        code = {"binder": 0, "VI": 2}[loss]
        nop = [kernel_ms(verbose_call(lambda: check(lib().rc_sampler_partition_dists(smp._h, ptr(P), 1, 0, smp.nchains, code, ptr(d), None, None)),
                                      "partition dists:")[2]) for _ in range(args.reps)]
        assert np.array_equal(d, first["dist"])
        res[loss + "_without_pairs"] = dict(kernel_ms=nop, kernel_ms_median=float(np.median(nop)))
        res[loss] = dict(kernel_ms=ks, kernel_ms_median=ms, pairs_per_s=S / (ms * 1e-3), whole_call_s=calls,
                         whole_call_s_median=float(np.median(calls)), samples_K_min=int(K.min()), samples_K_max=int(K.max()),
                         ball=ball_summary(first))
    # rc_mpel at the same n and K, in the same process: the pairwise search over the first args.mpel_samples samples, and
    # the new path over the same host label vectors (reference = the first of them)
    per = args.samples
    L = np.concatenate([smp.samples(c)["labels"] for c in range((args.mpel_samples + per - 1) // per)])[:args.mpel_samples]
    smp.close()
    for loss in ("VI", "binder"):
        pkg.mpel_loss_sums(L[:64], loss)
        pkg.partitiondistances(L[0], L, loss)
        mp = [mpel_rate(verbose_call(lambda: pkg.mpel_loss_sums(L, loss), "rc_mpel:")[2]) for _ in range(args.reps)]
        nw = [kernel_ms(verbose_call(lambda: pkg.partitiondistances(L[0], L, loss), "partition dists:")[2]) for _ in range(args.reps)]
        res[loss]["same_labels"] = dict(samples=int(L.shape[0]), K_max=int(max(len(np.unique(x)) for x in L)),
                                        rc_mpel_pairs_per_s=mp, rc_mpel_pairs_per_s_median=float(np.median(mp)),
                                        rc_mpel_timer="host clock from the launch of k_pair_loss to the read-back of the column sums",
                                        new_path_kernel_ms=nw,
                                        new_path_pairs_per_s_median=float(L.shape[0] / (np.median(nw) * 1e-3)))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--mpel-samples", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = g.load_package()
    res = dict(env=gpu_env(), stationary=case(pkg, args, "stationary: bench mixture", 0.1, 0),
               moving=case(pkg, args, "moving: sigma 0.25, maxK 100", 0.25, 100))
    res["env_after"] = gpu_env()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
