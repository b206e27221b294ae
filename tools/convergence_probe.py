"""Convergence diagnostics across chains (rc_rhat.cu) at the size they exist for: the pass-1 counts, the pass-2 counts, the
k_rhat_acc and k_rhat_finish kernels (CUDA events inside the library, printed with RCB200_VERBOSE) and the whole call, median
of 3 after a warm-up, plus a numpy statement at a small size whose outputs must equal the device's bit for bit.  Writes one
JSON document (--out) and prints it.

Cases (n = 10 000, 256 chains x 1 000 recorded samples, from the sampler's device-resident samples):
  stationary  the bench mixture (bench.synth: K = 50, dim = 100, sigma = 0.1), every sample the true partition
  moving      bench's `moving` setting: sigma = 0.25 with maxK = 100, chains that keep moving points
  numpy       n = 2 000, 16 chains x 100 samples of random labels with chain structure: one-hot counts in numpy against
              rc_cocl_rhat (host labels)"""
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
    """fn() with RCB200_VERBOSE=1; returns (result, host seconds, the library's `cocl rhat` line parsed)."""
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
        line = [x for x in f.read().splitlines() if "cocl rhat:" in x][-1]
    num = lambda key: float(line.split(key)[1].split()[0])                # noqa: E731
    return out, dt, dict(pass1_ms=num("pass1 "), pass2_counts_ms=num("pass2 counts "), acc_ms=num("k_rhat_acc "),
                         acc_bytes=num("ms ("), acc_share_of_7_7_TBs_pct=float(line.split("B, ")[1].split(" %")[0]),
                         finish_ms=num("k_rhat_finish "))


def summary(d):
    return dict(rhat_max=d["rhat_max"], rhat_pair=list(d["rhat_pair"]), pairs_above=d["pairs_above"],
                chain_meandev_max=float(np.max(d["chain_meandev"])), chain_meandev_argmax=int(np.argmax(d["chain_meandev"])),
                chain_maxdev_max=float(np.max(d["chain_maxdev"])), traces=d["traces"])


def case(pkg, args, name, sigma, maxK):
    X, lab = bench.synth(args.n, 50, 100, sigma, 50, args.seed)
    data = pkg.MCMCData.from_points(X)
    params = pkg.params_from_labels(data.D, lab, maxK=maxK)
    opts = pkg.MCMCOptionsList(numiters=args.samples, burnin=0)
    rp = [pkg.init_rp(params, args.seed, c) for c in range(args.chains)]
    smp = pkg.Sampler(data, opts, params, np.tile(lab, (args.chains, 1)), [x[0] for x in rp], [x[1] for x in rp], seed=args.seed)
    t = time.perf_counter(); smp.run(-1); t_run = time.perf_counter() - t
    first = smp.convergencediagnostics()                               # warm-up of every shape the timed calls use
    reps, calls = [], []
    for _ in range(args.reps):
        out, _, parts = verbose_call(smp.convergencediagnostics)
        reps.append(parts)
        t = time.perf_counter(); again = smp.convergencediagnostics(); calls.append(time.perf_counter() - t)
        assert again["rhat_max"] == first["rhat_max"] and np.array_equal(again["chain_meandev"], first["chain_meandev"])
    med = {k: float(np.median([r[k] for r in reps])) for k in reps[0]}
    smp.close()
    return dict(case=name, sigma=sigma, maxK=maxK, n=args.n, chains=args.chains, samples_per_chain=args.samples, sampler_run_s=t_run,
                reps=reps, median=med, acc_bytes_per_pair=28, whole_call_s=calls, whole_call_s_median=float(np.median(calls)),
                result=summary(first))


def numpy_reference(L):
    C, S, n = L.shape
    h, m = S // 2, 2 * C
    Ng = []
    for c in range(C):
        for part in (L[c, :h], L[c, S - h:]):
            codes = np.unique(part, return_inverse=True)[1].reshape(part.shape)
            K = int(codes.max()) + 1
            Y = np.zeros((n, h * K))
            Y[np.tile(np.arange(n), h), (np.arange(h)[:, None] * K + codes).ravel()] = 1.0
            Ng.append(np.rint(Y @ Y.T).astype(np.int64))
    Ng = np.stack(Ng)
    N, Q = Ng.sum(0), (Ng * Ng).sum(0)
    Wn, Bn = h * N - Q, m * Q - N * N
    f = np.float64
    with np.errstate(divide="ignore", invalid="ignore"):
        R = np.sqrt(f(h - 1) / f(h) + (f(h - 1) * Bn.astype(f)) / (f(m - 1) * f(h) * Wn.astype(f)))
    R = np.where(Wn > 0, R, np.where(Bn == 0, 1.0, np.inf))
    np.fill_diagonal(R, 1.0)
    iu = np.triu_indices(n, 1)
    d = np.abs(m * (Ng[0::2] + Ng[1::2]) - 2 * N)[:, iu[0], iu[1]]
    meandev = np.array([f(int(x)) / (f(2 * m * h) * f(n * (n - 1) // 2)) for x in d.sum(1)])
    maxdev = np.array([f(int(x)) / f(2 * m * h) for x in d.max(1)])
    return R, meandev, maxdev


def numpy_case(pkg):
    C, S, n, K = 16, 100, 2000, 20
    gr = np.random.default_rng(6)
    base = gr.integers(1, K + 1, size=n)
    L = np.empty((C, S, n), np.int64)
    for c in range(C):
        cb = base.copy()
        mv = gr.random(n) < 0.05
        cb[mv] = gr.integers(1, K + 1, size=int(mv.sum()))
        x = np.tile(cb, (S, 1))
        fl = gr.random(x.shape) < 0.1
        x[fl] = gr.integers(1, K + 1, size=int(fl.sum()))
        L[c] = x
    t = time.perf_counter(); R, md, xd = numpy_reference(L); t_np = time.perf_counter() - t
    pkg.cocl_rhat(L[:2, :8, :64])                                      # warm-up
    t = time.perf_counter(); dev = pkg.cocl_rhat(L, matrix=True); t_dev = time.perf_counter() - t
    same = (np.array_equal(R.view(np.int64), dev["rhat"].view(np.int64)) and np.array_equal(md.view(np.int64), dev["chain_meandev"].view(np.int64))
            and np.array_equal(xd.view(np.int64), dev["chain_maxdev"].view(np.int64)))
    return dict(case="numpy baseline", n=n, chains=C, samples_per_chain=S, numpy_s=t_np, device_call_s_with_matrix=t_dev,
                bit_identical=bool(same), rhat_max=dev["rhat_max"], pairs_above=dev["pairs_above"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = g.load_package()
    res = dict(env=gpu_env(), numpy=numpy_case(pkg), stationary=case(pkg, args, "stationary: bench mixture", 0.1, 0),
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
