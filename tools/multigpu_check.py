"""N-rank check of the sharded paths of SURVEY 8e over NCCL: distance build by row blocks + all_gather, chains sharded
across GPUs with per-rank int32 PSM counts + one all_reduce of the n x n matrix, MPEL candidates sharded + all_gather,
the convergence diagnostics, the credible ball and the aligned allocation over the chains of every rank.
torchrun --nproc-per-node N tools/multigpu_check.py [n] [chains_per_rank] [iters]
Rank 0 compares each with the single-process result (all three are bit-equal) and prints timings."""
import os, sys, time
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g
import bench

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
cpr = int(sys.argv[2]) if len(sys.argv) > 2 else 4
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 50
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = g.load_package()
X, lab = bench.synth(n, 20, 50, 0.1, 20, 3)
torch.cuda.synchronize(); dist.barrier()
t = time.perf_counter()
data = pkg.MCMCData.from_points_sharded(X)
torch.cuda.synchronize(); dist.barrier()
dt_d = time.perf_counter() - t
if rank == 0:
    ref = pkg.MCMCData.from_points(X, device=local)
    same = np.array_equal(ref.D, data.D) and np.array_equal(ref.logD, data.logD)
    print(f"world={world} n={n}: sharded distance build + all_gather {dt_d * 1e3:.1f} ms; equal to the single-GPU matrix: {same}", flush=True)
    assert same
    del ref
params = pkg.params_from_labels(data.D, lab)
opts = pkg.MCMCOptionsList(numiters=iters, burnin=0, thin=1, numGibbs=5, numMH=1)

def make(chain0, nch, dev_data):
    rp = [pkg.init_rp(params, 7, chain0 + c) for c in range(nch)]
    s = pkg.Sampler(dev_data, opts, params, np.tile(lab, (nch, 1)), [a for a, _ in rp], [b for _, b in rp], seed=7, chain_offset=chain0)
    s.run()
    return s

smp = make(rank * cpr, cpr, data)
torch.cuda.synchronize(); dist.barrier()
t = time.perf_counter()
psm = smp.psm_allreduce()
torch.cuda.synchronize(); dist.barrier()
dt = time.perf_counter() - t
if rank == 0:
    ref = make(0, cpr * world, data).psm()
    print(f"world={world} n={n} chains={cpr * world} samples/chain={iters}: psm_allreduce {dt * 1e3:.1f} ms; "
          f"equal to the single-process PSM of the same chains: {np.array_equal(psm, ref)}", flush=True)
    assert np.array_equal(psm, ref)
# Binder MPEL over the chains of every rank: all-reduced counts, per-rank W and P, one all_gather of the int64 totals
torch.cuda.synchronize(); dist.barrier()
t = time.perf_counter()
bp = smp.binder_pointestimate_allreduce()
torch.cuda.synchronize(); dist.barrier()
dt = time.perf_counter() - t
if rank == 0:
    one = make(0, cpr * world, data).binder_pointestimate()
    okb = (np.array_equal(bp["totals"], one["totals"]) and np.array_equal(bp["sums"], one["sums"])
           and bp["best"] == one["chain"] * opts.numsamples + one["index"])
    print(f"world={world} n={n} chains={cpr * world}: binder_pointestimate_allreduce over {bp['totals'].size} samples {dt * 1e3:.1f} ms; "
          f"equal to one process over the same chains: {okb}", flush=True)
    assert okb
# convergence across the chains of every rank: all-reduced counts N, one all_reduce of Q, one all_gather of the deviations
torch.cuda.synchronize(); dist.barrier()
t = time.perf_counter()
cd = smp.convergencediagnostics_allreduce(matrix=True)
torch.cuda.synchronize(); dist.barrier()
dt = time.perf_counter() - t
if rank == 0:
    one = make(0, cpr * world, data).convergencediagnostics(matrix=True)
    okc = (np.array_equal(cd["rhat"], one["rhat"]) and cd["rhat_max"] == one["rhat_max"] and cd["rhat_pair"] == one["rhat_pair"]
           and cd["pairs_above"] == one["pairs_above"] and np.array_equal(cd["chain_meandev"], one["chain_meandev"])
           and np.array_equal(cd["chain_maxdev"], one["chain_maxdev"]) and cd["traces"] == one["traces"])
    print(f"world={world} n={n} chains={cpr * world}: convergencediagnostics_allreduce {dt * 1e3:.1f} ms; "
          f"equal to one process over the same chains: {okc}", flush=True)
    assert okc
# credible ball over the chains of every rank: each rank's distances to the estimate, one all_gather of {dist, pairs, K}
for loss in ("VI", "binder"):
    torch.cuda.synchronize(); dist.barrier()
    t = time.perf_counter()
    cb = smp.credibleball_allreduce(lab, loss=loss)
    torch.cuda.synchronize(); dist.barrier()
    dt = time.perf_counter() - t
    if rank == 0:
        one = make(0, cpr * world, data).credibleball(lab, loss=loss)
        okb = (np.array_equal(cb["dist"], one["dist"]) and cb["radius"] == one["radius"] and cb["inball"] == one["inball"]
               and cb["expectedloss"] == one["expectedloss"]
               and all(np.array_equal(cb[k]["indices"], one[k]["indices"]) and cb[k]["dist"] == one[k]["dist"] and cb[k]["K"] == one[k]["K"]
                       for k in ("horizontal", "upper", "lower")))
        print(f"world={world} n={n} chains={cpr * world}: credibleball_allreduce ({loss}) over {cb['dist'].size} samples {dt * 1e3:.1f} ms; "
              f"equal to one process over the same chains: {okb}", flush=True)
        assert okb
# allocation probabilities to the estimate's clusters over the chains of every rank: one all_reduce of the counts, one
# all_gather of {matched, K, maps}
torch.cuda.synchronize(); dist.barrier()
t = time.perf_counter()
al = smp.alignedallocation_allreduce(lab, maps=True)
torch.cuda.synchronize(); dist.barrier()
dt = time.perf_counter() - t
if rank == 0:
    one = make(0, cpr * world, data).alignedallocation(lab, maps=True)
    oka = all(np.array_equal(al[k], one[k]) for k in one) and set(al) == set(one)
    print(f"world={world} n={n} chains={cpr * world}: alignedallocation_allreduce over {al['matched'].size} samples {dt * 1e3:.1f} ms; "
          f"equal to one process over the same chains: {oka}", flush=True)
    assert oka
# one common set of label vectors on every rank: rank 0's samples, broadcast, then 5 % of the labels reshuffled with a
# fixed seed so that the samples differ from each other
S = np.ascontiguousarray(smp.samples(0)["labels"])
tS = torch.from_numpy(S).cuda(); dist.broadcast(tS, 0); S = tS.cpu().numpy()
g5 = np.random.default_rng(5)
flip = g5.random(S.shape) < 0.05
S[flip] = g5.integers(1, 21, size=int(flip.sum()))
S = np.concatenate([S, S[::-1][:23] % 3 + 1])          # and a few coarse clusterings
# PSM of host label vectors sharded by sample: per-rank counts + all_reduce
P = pkg.psm_sharded(S[rank::world])
if rank == 0:
    okp = np.array_equal(P, pkg.psm(S, device=local))
    print(f"world={world} PSM of {S.shape[0]} host label vectors sharded by sample: equal to one GPU: {okp}", flush=True)
    assert okp
# MPEL: candidates sharded (cyclic rows of the pairwise loss matrix) + all_gather
for loss in ("binder", "VI"):
    torch.cuda.synchronize(); dist.barrier()
    t = time.perf_counter()
    sums, best = pkg.mpel_loss_sums_sharded(S, loss)
    torch.cuda.synchronize(); dist.barrier()
    dt = time.perf_counter() - t
    if rank == 0:
        s1, b1 = pkg.mpel_loss_sums(S, loss, device=local)
        ok = np.array_equal(s1, sums) and b1 == best
        print(f"world={world} MPEL {loss} over {S.shape[0]} samples: sharded {dt * 1e3:.1f} ms; equal to one GPU: {ok}", flush=True)
        assert ok
# BASELINE configs[4]-shaped PSM: n x n int32 counts of S samples sharded over the ranks, one ncclAllReduce (10 GB at
# n = 50 000).  RCB200_VERBOSE=1 prints the all-reduce time and bandwidth from inside the library.
if len(sys.argv) > 4:
    nb, Sb = int(sys.argv[4]), int(sys.argv[5]) if len(sys.argv) > 5 else 2000
    gb = np.random.default_rng(9)
    base = np.sort(gb.integers(1, 81, size=nb))
    mine = np.tile(base, (Sb // world, 1))
    gr = np.random.default_rng(100 + rank)
    flip = gr.random(mine.shape) < 0.1
    mine[flip] = gr.integers(1, 91, size=int(flip.sum()))
    comm = pkg.Comm.from_torch()
    cnt = torch.zeros((nb, nb), dtype=torch.int32, device="cuda")
    from redclust_jl_b200._lib import lib, check, ptr
    import ctypes as C
    for rep in range(2):
        torch.cuda.synchronize(); dist.barrier()
        t = time.perf_counter()
        check(lib().rc_comm_psm(comm._h, ptr(np.ascontiguousarray(mine)), mine.shape[0], nb, None, C.c_void_p(cnt.data_ptr())))
        torch.cuda.synchronize(); dist.barrier()
        dt = time.perf_counter() - t
    # bit-equality: rows of the reduced counts against a direct comparison over ALL ranks' samples
    allS = [None] * world
    dist.all_gather_object(allS, mine[:, :0].shape[0])
    rows = np.random.default_rng(1).choice(nb, size=8, replace=False)
    part = np.stack([(mine == mine[:, [i]]).sum(0) for i in rows]).astype(np.int64)
    tp = torch.from_numpy(part).cuda(); dist.all_reduce(tp)
    ok = bool((cnt[torch.from_numpy(rows).cuda()].to(torch.int64) == tp).all())
    if rank == 0:
        print(f"world={world} configs[4]-shaped PSM n={nb} S={mine.shape[0] * world} (sharded): counts + all-reduce {dt * 1e3:.1f} ms; "
              f"8 sampled rows equal to direct label comparison over all ranks: {ok}", flush=True)
    assert ok
dist.barrier()
dist.destroy_process_group()
