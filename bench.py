#!/usr/bin/env python
"""bench.py -- headline benchmark of the sampler hot path (BASELINE.json: "Gibbs+SM sweeps/sec x chains at n=10k").

One *step* = one iteration of runsampler's loop (sample_r, sample_p, one split-merge proposal with 5 restricted
Gibbs scans, one full Gibbs scan, record) for EVERY chain on the GPU.  The K timed steps are ONE launch of the
persistent chain kernel (every chain advances K iterations on the device, exactly what runsampler does); the W
warm-up steps are separate launches.  Workload at N=1: BASELINE configs[2] "generatemixture n=10,000 K~50 dim=100, fp64 distM (800 MB),
256 chains".  The headline `value` keeps round 1's definition (sigma = 0.1, 256 chains PER GPU: independent chains
shard with no data-path collective -> weak scaling) so the rounds compare; the same JSON line also carries
  "strong"  configs[2] taken literally: 256 chains in TOTAL, sharded over the N GPUs (strong scaling),
  "moving"  the same sizes at sigma = 0.25 with the reference's own cluster cap maxK = 100: a chain that keeps
            moving points (moves_per_sweep is reported for every workload; the sigma = 0.1 chain is stationary),
  "post"    the other half of BASELINE's metric: distance build, PSM and point-estimate seconds (rank 0, N = 1).
Prints ONE JSON line (see the task contract).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...        (N > 1)

--dump-outputs DIR writes what the headline run's last timed step recorded (see write_outputs) as DIR/<name>.npy:
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402


def synth(n, K, dim, sigma, alpha, seed):
    """Point generator of generatemixture (utils.jl:113-128) without the oracle co-clustering loop."""
    g = np.random.default_rng(seed)
    probs = g.dirichlet(np.full(K, float(alpha)))
    lab = np.sort(g.choice(K, size=n, p=probs))
    lab = (np.unique(lab, return_inverse=True)[1] + 1).astype(np.int64)
    X = g.normal(0.0, sigma, size=(n, dim))
    X[np.arange(n), lab - 1] += 1.0
    return X, lab


class ClockSampler(threading.Thread):
    """nvidia-smi-equivalent clock / throttle-reason samples during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def profile_numbers():
    """Per-launch numbers of the dominant kernel from the committed ncu capture of this workload (profiles/traffic.json:
    dram bytes, fp64-pipe activity, the launch duration under ncu), or {}."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def cpu_reference(args, X, lab, params_fields, steps, warmup, cores, D=None):
    """The CPU restatement of RedClust.jl (oracle/rc_oracle.cpp) on the host cores: `cores` independent chains,
    one per thread, each running one sweep per step.  Returns (chain-sweeps/s, ms per step, description)."""
    orc = graft.load_oracle()
    if D is None:
        D = orc.distm(X)
    P = orc.make_params(**params_fields)
    r0 = [1.5] * cores
    p0 = [0.9] * cores
    if warmup > 0:
        orc.time_chains(D, orc.Options(min(warmup, 1), 0, 1, args.numGibbs, args.numMH), P, lab, r0, p0, seed=args.seed, nthreads=cores)
    secs, _ = orc.time_chains(D, orc.Options(steps, 0, 1, args.numGibbs, args.numMH), P, lab, r0, p0, seed=args.seed, nthreads=cores)
    return cores * steps / secs, secs / steps * 1e3, f"{cores} independent chains x {steps} sweeps of the n={args.n} workload, one chain per host thread"


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly one JSON line: everything else that libraries print to fd 1 (NCCL's version banner,
    for one) is sent to stderr from here on; emit() writes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_BYTES = 48 << 20      # label rows written by --dump-outputs; more chains than fit are sampled (seeded)


def write_outputs(smp, chain0, out_dir):
    """The sample every chain recorded in the last step, as samples(c) returns it for that step: labels (float32, exact
    below 2^24), K, r, p, loglik, logposterior (float64), and that iteration's r / split-merge acceptances (float32).
    `chain` holds the global chain ids of the rows; when the label rows of all chains exceed DUMP_BYTES a fixed, seeded
    subset of the chains is written."""
    n, iters, numMH = smp.data.n, smp.options.numiters, smp.options.numMH
    keep = np.arange(smp.nchains)
    if smp.nchains * n * 4 > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(smp.nchains, max(DUMP_BYTES // (n * 4), 1), replace=False))
    cols = {k: [] for k in ("labels", "K", "r", "p", "loglik", "logposterior", "r_acc", "sm_acc", "sm_split")}
    for c in keep:
        s = smp.samples(int(c))
        for k in ("labels", "K", "r", "p", "loglik", "logposterior", "r_acc"):
            cols[k].append(s[k][-1])
        for k in ("sm_acc", "sm_split"):
            cols[k].append(s[k].reshape(iters, numMH)[-1])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "chain.npy"), (chain0 + keep).astype(np.float64))
    for k, v in cols.items():
        dt = np.float64 if k in ("K", "r", "p", "loglik", "logposterior") else np.float32
        np.save(os.path.join(out_dir, f"{k}.npy"), np.stack(v).astype(dt))


def timed_sampler(pkg, torch, dist, world, data, params, lab, chains, chain0, args, warm, steps, local_rank, dump=None):
    """`warm` untimed sweeps then `steps` timed ones (one kernel launch each) of `chains` chains on this rank; with `dump`
    a directory, write_outputs() then writes what the last timed step recorded.
    Returns (device seconds max over ranks, wall seconds max over ranks, moves per chain-sweep, K of chain 0, clock summary)."""
    opts = pkg.MCMCOptionsList(numiters=warm + steps, burnin=0, thin=1, numGibbs=args.numGibbs, numMH=args.numMH)
    rp = [pkg.init_rp(params, args.seed, chain0 + c) for c in range(chains)]
    r0 = np.array([x[0] for x in rp]); p0 = np.array([x[1] for x in rp])
    labs = np.tile(lab, (chains, 1))
    smp = pkg.Sampler(data, opts, params, labs, r0, p0, seed=args.seed, chain_offset=chain0, slot_cap=args.slot_cap)
    smp.run(0)                       # builds the per-chain sums (setup, like MCMCData construction)
    for _ in range(warm):
        smp.run(1)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clk = ClockSampler(local_rank)
    barrier()
    clk.start()
    m0 = smp.stats()["moves"].sum()
    _, t0 = smp.progress()
    w0 = time.perf_counter()
    smp.run(steps)                   # the K timed steps: ONE launch of the persistent chain kernel (as runsampler does)
    barrier()
    w1 = time.perf_counter()
    _, t1 = smp.progress()
    clk.stop_flag = True
    moves = float(smp.stats()["moves"].sum() - m0) / (chains * steps)
    tt = torch.tensor([t1 - t0, w1 - w0, moves], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tt.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        tt = torch.stack([mx[0], mx[1], sm[2] / world])
    Kfinal = int(smp.samples(0)["K"][-1])
    if dump:
        write_outputs(smp, chain0, dump)
    smp.close()
    return float(tt[0]), float(tt[1]), float(tt[2]), Kfinal, clk.summary(), (labs, r0, p0)


def post_block(pkg, args, data, lab):
    """PSM + point-estimate seconds (the second half of BASELINE's metric) through the host API, rank 0 at N = 1:
    synthetic label samples around the truth (15 % of the entries re-drawn), sizes named in the output."""
    import torch
    out = {}
    g = np.random.default_rng(args.seed)

    def samples(S, n, K):
        base = np.sort(g.integers(1, K + 1, size=n))
        L = np.tile(base, (S, 1))
        flip = g.random((S, n)) < 0.15
        L[flip] = g.integers(1, K + 11, size=int(flip.sum()))
        return np.ascontiguousarray(L, dtype=np.int64)

    # distance build (MCMCData(points), types.jl:159-162) at the bench size
    X, _ = synth(args.n, args.K, args.dim, args.sigma, args.K, args.seed)
    for _ in range(2):                               # warm: first-use allocations of the pool stay out of the timing
        d0 = pkg.MCMCData.from_points(X); del d0
    ts = []
    for _ in range(5):
        t = time.perf_counter(); d0 = pkg.MCMCData.from_points(X); ts.append(time.perf_counter() - t); del d0
    out["distm_s"] = min(ts); out["distm_median_s"] = sorted(ts)[2]
    out["distm"] = f"MCMCData(points) n={args.n} dim={args.dim}: upload, Euclidean distances, checks, logD and fixed-point images"
    # PSM of host label vectors into a host fp64 matrix (mcmc.jl:560)
    n1, S1 = 10000, 2000
    L = samples(S1, n1, 50)
    pkg.psm(L[:50])
    t = time.perf_counter(); pkg.psm(L); out["psm_s"] = time.perf_counter() - t
    out["psm"] = f"psm(labels) n={n1} S={S1}: host int64 labels -> host fp64 n x n"
    # configs[4]-shaped PSM: exact int32 counts left on the device (the all-reduce input of the multi-GPU path)
    n2, S2 = 50000, 10000
    try:
        L2 = samples(S2, n2, 90)
        cnt = torch.empty((n2, n2), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ts = []
        for _ in range(2):                           # the first call pays the staging buffers' first allocation
            t = time.perf_counter(); pkg.psm_counts_dev(L2, cnt.data_ptr()); torch.cuda.synchronize()
            ts.append(time.perf_counter() - t)
        out["psm_c4_s"] = ts[1]; out["psm_c4_first_s"] = ts[0]
        out["psm_c4"] = f"psm_counts_dev n={n2} S={S2} (BASELINE configs[4]): host labels -> device int32 counts (relabel, upload, transpose, tcgen05 one-hot counts)"
        del cnt
        # MPEL search over candidate samples (pointestimate.jl:34-59)
        S3 = 2000
        for loss in ("binder", "VI"):
            t = time.perf_counter(); pkg.mpel_loss_sums(L2[:S3], loss); out[f"mpel_{loss}_s"] = time.perf_counter() - t
        out["mpel"] = f"getpointestimate(method=MPEL) search, n={n2}, {S3} candidate samples ({S3 * (S3 - 1) // 2} pairs)"
    except Exception as e:  # noqa: BLE001
        out["psm_c4_error"] = str(e)[:200]
    return out


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--K", type=int, default=50)
    ap.add_argument("--dim", type=int, default=100)
    ap.add_argument("--sigma", type=float, default=0.1)
    ap.add_argument("--maxK", type=int, default=0)
    ap.add_argument("--chains", type=int, default=256, help="chains per GPU (headline, weak scaling) / in total (the strong block)")
    ap.add_argument("--numGibbs", type=int, default=5)
    ap.add_argument("--numMH", type=int, default=1)
    ap.add_argument("--seed", type=int, default=44)
    ap.add_argument("--slot-cap", type=int, default=0, help="cluster slots per chain (0: library default, 128)")
    ap.add_argument("--moving-sigma", type=float, default=0.25)
    ap.add_argument("--moving-maxK", type=int, default=100)
    ap.add_argument("--moving-warmup", type=int, default=5)
    ap.add_argument("--moving-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-moving", action="store_true")
    ap.add_argument("--no-noshort", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-post", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline run's last timed step recorded as DIR/<name>.npy (rank 0's chains)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    W = max(args.warmup, 0)
    steps = args.steps
    workload = (f"generatemixture(N={args.n}, K={args.K}; alpha={args.K}, sigma={args.sigma}, dim={args.dim}) seed {args.seed}, "
                f"{args.chains} chains per GPU, numGibbs={args.numGibbs}, numMH={args.numMH}, every sweep recorded")
    config = {"workload": workload, "n": args.n, "chains_per_gpu": args.chains, "hyperparameters": "from true labels as prior.jl:73-110",
              "init": "true labels, r/p from their priors",
              "l2": f"inputs larger than L2 (DL = {16 * args.n * args.n / 1e9:.2f} GB, per-chain row sums {16 * 128 * args.n * args.chains / 1e9:.2f} GB)"}
    X, lab = synth(args.n, args.K, args.dim, args.sigma, args.K, args.seed)

    if args.impl == "reference":
        if rank != 0:
            return
        orc = graft.load_oracle()
        D = orc.distm(X)
        pkg = graft.load_package()
        params = pkg.params_from_labels(D, lab, maxK=args.maxK)
        fields = {k: getattr(params, k) for k in params._fields}
        cores = os.cpu_count() or 1
        val, ms, sample = cpu_reference(args, X, lab, fields, steps, W, cores, D=D)
        line = {"impl": "reference", "metric": "Gibbs+SM chain-sweeps/sec", "value": val, "unit": "chain-sweeps/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 (exact i64 fixed-point cluster sums)", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "chain-sweeps/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "chain-sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "CPU restatement of RedClust.jl v1.2.2 (Julia is not installed; the reference itself is single-threaded)"}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = graft.load_package()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup (untimed): distance matrix on the GPU, hyperparameters ----
    data = pkg.MCMCData.from_points(X, device=local_rank)
    Dh = data.D
    params = pkg.params_from_labels(Dh, lab, maxK=args.maxK)
    chain0 = rank * args.chains

    # ---- headline: `chains` chains per GPU (weak scaling, round 1's definition) ----
    dev_s, wall_s, moves, Kfinal, clocks, (labs, r0, p0) = timed_sampler(pkg, torch, dist, world, data, params, lab, args.chains, chain0,
                                                                        args, W, steps, local_rank,
                                                                        dump=args.dump_outputs if rank == 0 else None)
    value = world * args.chains * steps / dev_s

    # ---- configs[2] literally: `chains` chains in total over the N GPUs (strong scaling) ----
    strong = None
    if not args.no_strong:
        per = max(args.chains // world, 1)
        if world == 1:
            strong = {"value": value, "unit": "chain-sweeps/s", "ms_per_step": dev_s / steps * 1e3, "chains_total": args.chains, "chains_per_gpu": per,
                      "note": "N = 1: the headline run"}
        else:
            d2, w2, mv2, _, _, _ = timed_sampler(pkg, torch, dist, world, data, params, lab, per, rank * per, args, W, steps, local_rank)
            strong = {"value": world * per * steps / d2, "unit": "chain-sweeps/s", "ms_per_step": d2 / steps * 1e3, "chains_total": world * per,
                      "chains_per_gpu": per, "moves_per_sweep": mv2,
                      "note": "256 chains sharded over the GPUs: a sweep of one chain is sequential in the points, so fewer chains per GPU leave SMs idle"}

    # ---- the same headline run with the exact shortcuts off (RCB200_SHORTCUTS=0): every row evaluated, every merge proposal's
    #      restricted scans run -- what the kernel costs when nothing can be skipped ----
    noshort = None
    if not args.no_noshort:
        os.environ["RCB200_SHORTCUTS"] = "0"
        try:
            d4, w4, mv4, _, _, _ = timed_sampler(pkg, torch, dist, world, data, params, lab, args.chains, chain0, args, W, steps, local_rank)
        finally:
            os.environ.pop("RCB200_SHORTCUTS", None)
        noshort = {"value": world * args.chains * steps / d4, "unit": "chain-sweeps/s", "ms_per_step": d4 / steps * 1e3, "moves_per_sweep": mv4,
                   "note": "RCB200_SHORTCUTS=0: row summaries and the merge-proposal bound disabled (results are identical either way)"}

    # ---- a chain that moves: sigma = 0.25, the reference's own cap maxK (PriorHyperparamsList.maxK, src/types.jl:107) ----
    moving = None
    if not args.no_moving:
        X2, lab2 = synth(args.n, args.K, args.dim, args.moving_sigma, args.K, args.seed)
        data2 = pkg.MCMCData.from_points(X2, device=local_rank)
        params2 = pkg.params_from_labels(data2.D, lab2, maxK=args.moving_maxK)
        d3, w3, mv3, K3, clk3, _ = timed_sampler(pkg, torch, dist, world, data2, params2, lab2, args.chains, chain0, args,
                                                 max(args.moving_warmup, 0), max(args.moving_steps, 1), local_rank)
        moving = {"value": world * args.chains * args.moving_steps / d3, "unit": "chain-sweeps/s", "ms_per_step": d3 / args.moving_steps * 1e3,
                  "moves_per_sweep": mv3, "K_final_chain0": K3, "steps": args.moving_steps, "warmup": args.moving_warmup, "clocks": clk3,
                  "config": {"workload": f"generatemixture(N={args.n}, K={args.K}; alpha={args.K}, sigma={args.moving_sigma}, dim={args.dim}) seed {args.seed}, "
                                         f"maxK={args.moving_maxK}, {args.chains} chains per GPU, init true labels, {args.moving_warmup} untimed sweeps first",
                             "why_maxK": "at sigma = 0.25 the model opens several hundred clusters at this n; the sampler holds at most 255 live "
                                         "clusters per chain, so the run uses the reference's own cap parameter"},
                  "note": "per sweep the chain moves ~2 % of the points (every move invalidates the row summaries) and its split-merge proposals "
                          "involve clusters of thousands of points; most merge proposals are rejected by their bound, the splits' restricted "
                          "Gibbs scans (sequential, O(members) per move) and the full scan's move updates dominate"}
        del data2

    # ---- end-to-end through the public API with HOST buffers (upload D, build, run, read results back) ----
    e2e = None
    if not args.no_e2e:
        Dp = torch.from_numpy(Dh).pin_memory()
        o2 = pkg.MCMCOptionsList(numiters=steps, burnin=0, thin=1, numGibbs=args.numGibbs, numMH=args.numMH)

        def one_pass():
            """host D -> MCMCData -> Sampler -> run -> every chain's samples back on the host"""
            t = [time.perf_counter()]
            d2 = pkg.MCMCData(Dp.numpy(), device=local_rank); t.append(time.perf_counter())
            s2 = pkg.Sampler(d2, o2, params, labs, r0, p0, seed=args.seed, chain_offset=chain0, slot_cap=args.slot_cap); t.append(time.perf_counter())
            s2.run(-1); t.append(time.perf_counter())
            outs = [s2.samples_all()]                      # every chain's samples, traces and acceptances on the host
            barrier(); t.append(time.perf_counter())
            dev = s2.progress()[1]
            s2.close()
            del d2
            return t, dev, outs

        tw, devw, _ = one_pass()     # untimed warm-up of the whole path (first-use kernel loading, pinned staging buffers)
        if rank == 0:
            print("[bench] e2e warm-up pass (s): data %.3f, sampler %.3f, run %.3f (device %.3f), readback %.3f" %
                  (tw[1] - tw[0], tw[2] - tw[1], tw[3] - tw[2], devw, tw[4] - tw[3]), file=sys.stderr)
        passes = []
        for _ in range(3):           # three timed passes, the median is reported (host-side allocation and page-fault noise is +-30 %)
            barrier()
            t, dev, outs = one_pass()
            if rank == 0:
                print("[bench] e2e phases (s): data %.3f, sampler %.3f, run %.3f (device %.3f), readback %.3f" %
                      (t[1] - t[0], t[2] - t[1], t[3] - t[2], dev, t[4] - t[3]), file=sys.stderr)
            e1 = torch.tensor([t[4] - t[0]], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(e1, op=dist.ReduceOp.MAX)
            passes.append(float(e1[0]))
        et = torch.tensor([sorted(passes)[1]], dtype=torch.float64, device="cuda")
        h2d = Dh.nbytes + labs.nbytes + r0.nbytes + p0.nbytes
        d2h = sum(sum(v.nbytes for v in o.values()) for o in outs)
        e2e = {"value": world * args.chains * steps / float(et[0]), "unit": "chain-sweeps/s",
               "h2d_bytes_per_step": int(h2d / steps), "d2h_bytes_per_step": int(d2h / steps),
               "passes_s": passes,
               "includes": "upload of D from pinned host memory, logD / fixed-point build, per-chain sum initialisation, sampling, readback of all samples; one untimed warm-up pass of the same path first, then three timed passes of which the median is reported"}
        del outs

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peaks()
    b_scan = 16.0 * args.n * (args.n - 1)                         # algorithmic bytes per chain-sweep (SURVEY 8d)
    step_s = dev_s / steps
    per_launch_bytes = b_scan * args.chains * steps               # the timed launch advances every chain by K sweeps
    achieved = per_launch_bytes / dev_s / 1e9
    prof = profile_numbers().get(f"k_chain_inc:{args.n}:{args.chains}", {})
    traffic = prof["dram_bytes_per_sweep"] * steps if "dram_bytes_per_sweep" in prof else None     # per launch = K sweeps
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "k_chain_inc", "peak_source": peak_src + " (of measured)",
                "algorithmic_bytes_per_launch": per_launch_bytes,
                "dram_frac": (traffic / steps / step_s / 1e9 / peak) if traffic else None,
                "fp64_pipe_frac": prof.get("fp64_pipe_frac"), "issue_active_frac": prof.get("issue_active_frac"),
                "note": "algorithmic bytes = chains x 16 n (n-1) per sweep: what a scan that reads every row costs (SURVEY 8d).  This kernel does "
                        "not read the rows: each chain keeps the sums of every row by cluster (exact integers) and a Gibbs step reads one 16-byte "
                        "entry per live cluster; only a move streams a row; a row whose stored leader margin already proves the outcome is not "
                        "evaluated at all, and a merge proposal whose prior + likelihood ratio already lies below log U is rejected without its "
                        "restricted scans (both exact; no_shortcuts gives the rate with them off).  frac > 1 therefore measures the work avoided, "
                        "dram_frac is the real DRAM utilisation (ncu bytes / step time / peak); the kernel is bound by latency, not by a pipe: "
                        "fp64_pipe_frac and issue_active_frac are ncu's (profiles/r02_kchaininc_summary.md)"}
    cpu = None
    if not args.no_cpu and world == 1:
        cores = os.cpu_count() or 1
        fields = {k: getattr(params, k) for k in params._fields}
        v, ms, sample = cpu_reference(args, X, lab, fields, args.cpu_steps, 0, cores, D=Dh)
        cpu = {"value": v, "unit": "chain-sweeps/s", "cores": cores, "kind": "port", "sample": sample}
    post = None
    if not args.no_post and world == 1:
        post = post_block(pkg, args, data, lab)
    line = {"metric": "Gibbs+SM chain-sweeps/sec", "value": value, "unit": "chain-sweeps/s", "n_gpus": world, "steps": steps, "warmup": W,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 (exact i64 fixed-point cluster sums)", "data": "synthetic", "config": config,
            "clocks": clocks, "e2e": e2e, "gpu_launches": 1, "roofline": roofline, "cpu_baseline": cpu,
            "moves_per_sweep": moves, "strong": strong, "no_shortcuts": noshort, "moving": moving, "post": post,
            "wall_ms_per_step": wall_s / steps * 1e3, "K_final_chain0": Kfinal}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
