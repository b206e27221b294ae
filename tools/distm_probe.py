"""Cost of recomputing the distance entries the Gram form cannot resolve (rc_dist_unresolved, rc_math.h) in
MCMCData(points) on the default path (k_gram128), against a build without the rule (--parent-lib: librcb200.so of the
previous commit).

Workloads, n = 10 000 points of dim 100 (bench.synth, seed 44):
  bench    bench.py's headline mixture (sigma = 0.1): no entry is recomputed, so D must be bit-equal to the parent's
  moving   bench.py's `moving` mixture (sigma = 0.25): likewise
  offset   the bench points + 1e3 in every coordinate: nearly every entry is recomputed from the differences
Each (library, workload) runs in a subprocess of its own (one library per process), the two libraries alternate within
every round, and the order of the two flips from round to round.  A subprocess makes two untimed calls, then --reps
timed calls (host clock around from_points, which ends in a device synchronise: upload, distances, checks, log D and
the fixed-point images, as bench.py's distm_s), then one call with RCB200_VERBOSE for the kernel's CUDA-event time.
The share of entries the rule recomputes is counted on the host with numpy's Gram form (not the kernel's bits).
Writes one JSON document (--out) and prints it."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
TAU = 2.0 ** -6


def points(name):
    import bench
    X, _ = bench.synth(10000, 50, 100, 0.25 if name == "moving" else 0.1, 50, 44)
    return X + 1e3 if name == "offset" else X


def worker(name, reps):
    import __graft_entry__ as g
    pkg = g.load_package()
    X = points(name)
    for _ in range(2):
        pkg.MCMCData.from_points(X)
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        d = pkg.MCMCData.from_points(X)
        ts.append(time.perf_counter() - t)
        del d
    D = pkg.MCMCData.from_points(X).D
    os.environ["RCB200_VERBOSE"] = "1"
    pkg.MCMCData.from_points(X)                                          # the kernel's line goes to stderr
    print(json.dumps(dict(seconds=ts, sha256=hashlib.sha256(D.tobytes()).hexdigest())), flush=True)


def recomputed_share(X):
    """(share of off-diagonal entries with v < tau s, smallest v / s) of numpy's Gram form, in blocks of rows."""
    sq = (X * X).sum(1)
    hit, lo = 0, np.inf
    for i0 in range(0, X.shape[0], 1000):
        s = sq[i0:i0 + 1000, None] + sq[None, :]
        ratio = (s - 2 * X[i0:i0 + 1000] @ X.T) / s
        ratio[np.arange(ratio.shape[0]), np.arange(i0, i0 + ratio.shape[0])] = np.inf
        hit += int((ratio < TAU).sum()); lo = min(lo, float(ratio.min()))
    n = X.shape[0]
    return hit / (n * (n - 1)), lo


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="librcb200.so built from the previous commit")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker, args.reps)
    from credibleball_probe import gpu_env
    libs = dict(parent=os.path.abspath(args.parent_lib), this=os.path.join(ROOT, "redclust.jl_b200", "librcb200.so"))
    res = {w: {k: dict(seconds=[], kernel_ms=[], sha256=set()) for k in libs} for w in ("bench", "moving", "offset")}
    for r in range(args.rounds):
        for k in (("parent", "this") if r % 2 == 0 else ("this", "parent")):
            for w in res:
                env = dict(os.environ, RCB200_LIB=libs[k])
                env.pop("RCB200_DISTM", None)
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--parent-lib", libs["parent"], "--reps", str(args.reps),
                                    "--worker", w], env=env, capture_output=True, text=True, check=True)
                out = json.loads(p.stdout.strip().splitlines()[-1])
                line = [l for l in p.stderr.splitlines() if "k_gram128 (distances)" in l][-1]
                res[w][k]["seconds"] += out["seconds"]
                res[w][k]["sha256"].add(out["sha256"])
                res[w][k]["kernel_ms"].append(float(line.split(": ")[1].split(" ms")[0]))
    doc = dict(env=gpu_env(), tau=TAU, rounds=args.rounds, reps=args.reps, workloads={})
    for w, by in res.items():
        share, lo = recomputed_share(points(w))
        e = dict(recomputed_share_numpy=share, min_v_over_s_numpy=lo)
        for k, v in by.items():
            e[k] = dict(from_points_median_s=float(np.median(v["seconds"])), from_points_min_s=min(v["seconds"]),
                        from_points_max_s=max(v["seconds"]), k_gram128_ms=v["kernel_ms"], sha256=sorted(v["sha256"]))
        e["D_bit_equal_to_parent"] = by["parent"]["sha256"] == by["this"]["sha256"] and len(by["this"]["sha256"]) == 1
        e["median_ratio_this_over_parent"] = e["this"]["from_points_median_s"] / e["parent"]["from_points_median_s"]
        e["kernel_ratio_this_over_parent"] = float(np.median(by["this"]["kernel_ms"]) / np.median(by["parent"]["kernel_ms"]))
        doc["workloads"][w] = e
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
