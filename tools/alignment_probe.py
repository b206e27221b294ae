"""Allocation probabilities to the clusters of a point estimate over pooled samples (rc_sampler_aligned_alloc) at the size
they exist for.  Kernel times are CUDA events inside the library (printed with RCB200_VERBOSE), the whole call is a host
clock around separate calls; medians of 3 after a warm-up.  Beside each case: k_pair_loss<true> over the same samples
(the same K^ x K_t tables without the assignment: the floor of the table half of k_align_match), and a numpy + scipy
baseline on the first --cpu-samples samples with a check that its outputs agree, and the counts of the first --check-chains
chains against a numpy bincount through the returned maps.  Writes one JSON document (--out) and prints it.

Cases (n = 10 000, 256 chains x 1 000 recorded samples, from the sampler's device-resident samples; the estimate is the
simulation's true partition):
  stationary  the bench mixture (bench.synth: K = 50, dim = 100, sigma = 0.1)
  moving      bench's `moving` setting: sigma = 0.25 with maxK = 100, chains that keep moving points
The algorithmic bytes are the 2 S n label bytes (k_align_match and k_align_count each read every label once)."""
import argparse
import json
import os
import sys
import time

import numpy as np
from scipy.optimize import linear_sum_assignment

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from credibleball_probe import gpu_env, verbose_call, kernel_ms, g, bench  # noqa: E402

HBM_TBPS = 7.7                                                      # HGX B200 data sheet, one GPU


def align_ms(line):
    return float(line.split("k_align_match ")[1].split()[0]), float(line.split("k_align_count ")[1].split()[0])


def numpy_scipy(est, L):
    """counts, matched and sigma from a numpy table, scipy's assignment and numpy counting, one sample at a time."""
    e = np.unique(est, return_inverse=True)[1]
    first = np.sort(np.unique(est, return_index=True)[1])
    col_of = np.argsort(e[first])                                     # sorted label index -> first-appearance column
    e = col_of[e]
    kh, n = first.size, est.size
    counts = np.zeros((n, kh + 1), np.int64)
    matched, maps = np.zeros(L.shape[0], np.int64), np.zeros((L.shape[0], 255), np.uint8)
    for t in range(L.shape[0]):
        u, fi, c = np.unique(L[t], return_index=True, return_inverse=True)
        rank = np.empty(u.size, np.int64)
        rank[np.argsort(fi)] = np.arange(u.size)
        c = rank[c]
        T = np.zeros((kh, u.size), np.int64)
        np.add.at(T, (e, c), 1)
        r, cc = linear_sum_assignment(T, maximize=True)
        sig = np.full(u.size, kh)
        keep = T[r, cc] > 0
        sig[cc[keep]] = r[keep]
        matched[t] = T[r, cc].sum()
        maps[t, :u.size] = np.where(sig == kh, 0, sig + 1)
        counts[np.arange(n), sig[c]] += 1
    return counts, matched, maps


def case(pkg, args, name, sigma, maxK):
    X, lab = bench.synth(args.n, 50, 100, sigma, 50, args.seed)
    data = pkg.MCMCData.from_points(X)
    params = pkg.params_from_labels(data.D, lab, maxK=maxK)
    opts = pkg.MCMCOptionsList(numiters=args.samples, burnin=0)
    rp = [pkg.init_rp(params, args.seed, c) for c in range(args.chains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (args.chains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=args.seed)
    t = time.perf_counter(); smp.run(-1); t_run = time.perf_counter() - t
    S, n = args.chains * args.samples, args.n
    res = dict(case=name, sigma=sigma, maxK=maxK, n=n, chains=args.chains, samples_per_chain=args.samples, sampler_run_s=t_run)
    first = smp.alignedallocation(lab)                               # warm-up of every shape the timed calls use
    match, count, calls = [], [], []
    for _ in range(args.reps):
        _, _, line = verbose_call(lambda: smp.alignedallocation(lab), "aligned allocation:")
        m, c = align_ms(line)
        match.append(m); count.append(c)
        t = time.perf_counter(); again = smp.alignedallocation(lab); calls.append(time.perf_counter() - t)
        assert np.array_equal(again["counts"], first["counts"]) and np.array_equal(again["matched"], first["matched"])
    # the counts of the first --check-chains chains against a bincount through the returned maps: sample slices of
    # k_align_count far above its 64-sample sigma chunk (the device samples are already 1..K in first-appearance order)
    part = smp.alignedallocation(lab, 0, args.check_chains, maps=True)
    kh, bins = part["clusters"].size, np.zeros(n * (part["clusters"].size + 1), np.int64)
    for c in range(args.check_chains):
        Lc = smp.samples(c)["labels"]
        m = np.take_along_axis(part["maps"][c * args.samples:(c + 1) * args.samples].astype(np.int64), Lc - 1, axis=1)
        bins += np.bincount((np.arange(n)[None, :] * (kh + 1) + np.where(m == 0, kh, m - 1)).ravel(), minlength=bins.size)
    assert np.array_equal(part["counts"], bins.reshape(n, kh + 1))
    res["counts_equal_bincount_through_maps"] = dict(samples=args.check_chains * args.samples, equal=True)
    smp.credibleball(lab)
    tables = [kernel_ms(verbose_call(lambda: smp.credibleball(lab), "partition dists:")[2]) for _ in range(args.reps)]
    mm, cm = float(np.median(match)), float(np.median(count))
    res.update(line=line, k_align_match_ms=match, k_align_match_ms_median=mm, k_align_count_ms=count, k_align_count_ms_median=cm,
               whole_call_s=calls, whole_call_s_median=float(np.median(calls)),
               k_pair_loss_same_tables_ms=tables, k_pair_loss_same_tables_ms_median=float(np.median(tables)),
               label_bytes=2 * S * n,
               label_bytes_share_of_hbm=(2 * S * n) / ((mm + cm) * 1e-3) / (HBM_TBPS * 1e12),
               k_align_count_bytes_share_of_hbm=(S * n) / (cm * 1e-3) / (HBM_TBPS * 1e12),
               samples_K_min=int(first["K"].min()), samples_K_max=int(first["K"].max()), estimate_K=int(first["clusters"].size),
               transfer_distance_mean=float(n - first["matched"].mean()), transfer_distance_max=int(n - first["matched"].min()),
               self_min=float(first["self"].min()), points_self_below_0_9=int((first["self"] < 0.9).sum()),
               unmatched_share=float(first["prob"][:, -1].mean()))
    # numpy + scipy on the first cpu_samples samples of chain 0: the same outputs, one host thread
    L = smp.samples(0)["labels"][:args.cpu_samples]
    smp.close()
    dev = pkg.alignedallocation(lab, L, maps=True)
    t = time.perf_counter(); counts, matched, maps = numpy_scipy(lab, L); dt = time.perf_counter() - t
    same_maps = int((dev["maps"] == maps).all(axis=1).sum())
    assert np.array_equal(dev["matched"], matched)
    if same_maps == L.shape[0]:
        assert np.array_equal(dev["counts"], counts)
    res["numpy_scipy"] = dict(samples=int(L.shape[0]), seconds=dt, ms_per_sample=dt / L.shape[0] * 1e3,
                              pool_seconds_at_that_rate=dt / L.shape[0] * S, matched_equal=True,
                              samples_with_equal_maps=same_maps, counts_equal=bool(np.array_equal(dev["counts"], counts)))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--cpu-samples", type=int, default=200)
    ap.add_argument("--check-chains", type=int, default=8)
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
