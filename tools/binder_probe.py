"""Posterior expected Binder loss over pooled samples (k_binder_w / k_binder_pairs of rc_post.cu) at the sizes it exists for:
the counts time, the W kernel's time (CUDA events, printed by the library with RCB200_VERBOSE), the whole call, and
pair-samples per second.  Writes one JSON document (--out) and prints it.

Cases:
  pooled   256 chains x 1 000 recorded samples of the bench mixture (bench.synth, n = 10 000, K = 50, dim = 100, sigma = 0.1),
           from the sampler's device-resident samples (Sampler.binder_pointestimate): S = 256 000
  configs4 n = 50 000 and S = 10 000 host label vectors (80 base clusters, 10 % of the labels redrawn), where the pairwise
           search rc_mpel (binder) is timed on the same labels and its argmin compared
  tc_check the tensor-core co-clustering counts at S = 256 000 (n = 512) against the byte-compare kernel and against a direct
           numpy count of sampled rows"""
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


def verbose_call(fn):
    """fn() with RCB200_VERBOSE=1; returns (result, host seconds, library stderr lines)."""
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
        lines = [x for x in f.read().splitlines() if x.startswith("[rcb200]")]
    return out, dt, lines


def parse(lines):
    """counts kernel (psm counts line) and W kernel (binder mpel line) times in ms."""
    out = {}
    for x in lines:
        if "psm counts:" in x:                                   # "... kernel=<name> <ms> ms ..."
            out["counts_kernel"], ms = x.split("kernel=")[1].split()[:2]
            out["counts_kernel_ms"] = float(ms)
        if "binder mpel:" in x:
            out["counts_call_ms"] = float(x.split("counts ")[1].split(" ms")[0])
            out["w_kernel_ms"] = float(x.split("W kernel ")[1].split(" ms")[0])
    return out


def pooled(pkg, args):
    X, lab = bench.synth(args.n, 50, 100, 0.1, 50, args.seed)
    data = pkg.MCMCData.from_points(X)
    params = pkg.params_from_labels(data, lab)
    opts = pkg.MCMCOptionsList(numiters=args.samples, burnin=0)
    rp = [pkg.init_rp(params, args.seed, c) for c in range(args.chains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (args.chains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=args.seed)
    t = time.perf_counter(); smp.run(-1); t_run = time.perf_counter() - t
    S = args.chains * args.samples
    smp.binder_pointestimate(0, 1)                               # warm-up: module load, one chain
    reps = []
    for _ in range(args.reps):
        out, dt, lines = verbose_call(smp.binder_pointestimate)
        reps.append(dict(call_s=dt, **parse(lines)))
    w = float(np.median([r["w_kernel_ms"] for r in reps]))
    ps = args.n * (args.n - 1) / 2 * S
    K = smp.samples(out["chain"])["K"]
    smp.close()
    return dict(case="256 chains x 1000 samples, bench mixture", n=args.n, S=S, chains=args.chains, sampler_run_s=t_run, reps=reps,
                w_kernel_ms_median=w, pair_samples=ps, pair_samples_per_s=ps / (w / 1e3),
                call_s_median=float(np.median([r["call_s"] for r in reps])), best_chain=int(out["chain"]), best_index=int(out["index"]),
                best_sum=float(out["sums"].min()), K_of_best_chain_mean=float(K.mean()))


def configs4(pkg, args):
    n, S = 50000, 10000
    gb = np.random.default_rng(9)
    base = np.sort(gb.integers(1, 81, size=n))
    L = np.tile(base, (S, 1))
    flip = gb.random(L.shape) < 0.1
    L[flip] = gb.integers(1, 91, size=int(flip.sum()))
    pkg.binder_loss_sums(L[:64, :2000])                          # warm-up
    reps = []
    for _ in range(args.reps):
        (sums, best, totals), dt, lines = verbose_call(lambda: pkg.binder_loss_sums(L))
        reps.append(dict(call_s=dt, **parse(lines)))
    w = float(np.median([r["w_kernel_ms"] for r in reps]))
    ps = n * (n - 1) / 2 * S
    res = dict(case="configs[4] size", n=n, S=S, reps=reps, w_kernel_ms_median=w, pair_samples=ps, pair_samples_per_s=ps / (w / 1e3),
               call_s_median=float(np.median([r["call_s"] for r in reps])), best=best)
    if not args.skip_mpel:
        t = time.perf_counter(); rs, rb = pkg.mpel_loss_sums(L, "binder"); t_m = time.perf_counter() - t
        res.update(rc_mpel_binder_s=t_m, rc_mpel_best=rb, same_best=rb == best,
                   max_rel_diff_vs_rc_mpel=float(np.max(np.abs(rs - sums) / np.abs(rs))))
    return res


def tc_check(pkg):
    import torch
    n, S = 512, 256000
    gt = np.random.default_rng(3)
    base = np.sort(gt.integers(1, 41, size=n))
    L = np.tile(base, (S, 1))
    flip = gt.random(L.shape) < 0.2
    L[flip] = gt.integers(1, 61, size=int(flip.sum()))
    cnt = torch.zeros((n, n), dtype=torch.int32, device="cuda")
    _, _, lines = verbose_call(lambda: pkg.psm_counts_dev(L, cnt.data_ptr()))
    tc = cnt.cpu().numpy()
    os.environ["RCB200_PSM"] = "compare"
    cnt.zero_()
    _, _, lines2 = verbose_call(lambda: pkg.psm_counts_dev(L, cnt.data_ptr()))
    del os.environ["RCB200_PSM"]
    cmp_ = cnt.cpu().numpy()
    rows = gt.choice(n, size=8, replace=False)
    direct = np.stack([(L == L[:, [i]]).sum(0) for i in rows])
    return dict(n=n, S=S, kernels=[parse(lines).get("counts_kernel"), parse(lines2).get("counts_kernel")],
                tc_equals_compare=bool(np.array_equal(tc, cmp_)), tc_rows_equal_direct_count=bool(np.array_equal(tc[rows], direct)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--skip-mpel", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = g.load_package()
    res = dict(env=gpu_env(), tc_check=tc_check(pkg), pooled=pooled(pkg, args), configs4=configs4(pkg, args))
    res["env_after"] = gpu_env()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
