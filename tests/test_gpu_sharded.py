"""The sharded rc_comm_* entry points at world sizes 2 and 3, every rank a process on device 0.

Real NCCL refuses two ranks on one GPU, so the library loads a stand-in (RCB200_NCCL_LIB) built from the C source below:
each collective synchronises the stream, copies the send buffer to the host, exchanges it through files in the directory
its unique id names, and copies the result back to the device.  Every wait is bounded and ends in an NCCL error, so a
rank that is left waiting fails instead of hanging.  The ranks hold unequal numbers of chains, so the padded blocks and
the rank-ordered unpacking of the gathers are used on ranks that are not last."""
import multiprocessing as mp
import os
import pickle
import subprocess
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLDS = {2: (1, 3), 3: (2, 1, 3)}                # chains per rank
ITERS = 24

STANDIN_NCCL = r"""
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

typedef struct { char internal[128]; } ncclUniqueId;        /* the directory of the exchange files */
typedef struct ncclComm { char dir[128]; int rank, world; long seq; } *ncclComm_t;
enum { OK = 0, CUDA_ERR = 1, SYS_ERR = 2, BAD_ARG = 4, TIMEOUT = 6 };

const char* ncclGetErrorString(int r) {
  return r == TIMEOUT ? "stand-in NCCL: another rank did not reach the collective within 60 s"
       : r == BAD_ARG ? "stand-in NCCL: the ranks passed different sizes or an unsupported type"
       : r == CUDA_ERR ? "stand-in NCCL: CUDA error" : "stand-in NCCL: file error";
}

int ncclGetUniqueId(ncclUniqueId* id) {
  const char* base = getenv("STANDIN_NCCL_DIR");
  memset(id, 0, sizeof *id);
  snprintf(id->internal, sizeof id->internal, "%s/idXXXXXX", base ? base : "/tmp");
  return mkdtemp(id->internal) ? OK : SYS_ERR;
}

int ncclCommInitRank(ncclComm_t* comm, int world, ncclUniqueId id, int rank) {
  ncclComm_t c = (ncclComm_t)calloc(1, sizeof *c);
  memcpy(c->dir, id.internal, sizeof c->dir);
  c->dir[sizeof c->dir - 1] = 0;
  c->rank = rank;
  c->world = world;
  *comm = c;
  return OK;
}

int ncclCommDestroy(ncclComm_t c) { free(c); return OK; }

/* this rank's `bytes` at send (device) to its file of the next collective; every rank's file into *all (host, world x
   bytes, rank order).  The send buffer is on the host before anything is written, so it may overlap the receive buffer. */
static int exchange(ncclComm_t c, const void* send, size_t bytes, cudaStream_t s, char** all) {
  char path[300], tmp[310];
  const long seq = c->seq++;
  char* mine = (char*)malloc(bytes + 1);
  *all = (char*)malloc(bytes * c->world + 1);
  if (cudaStreamSynchronize(s) != cudaSuccess || (bytes && cudaMemcpy(mine, send, bytes, cudaMemcpyDeviceToHost) != cudaSuccess)) {
    free(mine); free(*all); return CUDA_ERR;
  }
  snprintf(path, sizeof path, "%s/%ld.%d", c->dir, seq, c->rank);
  snprintf(tmp, sizeof tmp, "%s.part", path);
  FILE* f = fopen(tmp, "wb");
  const int written = f && fwrite(mine, 1, bytes, f) == bytes;
  free(mine);
  if (!f || fclose(f) != 0 || !written || rename(tmp, path) != 0) { free(*all); return SYS_ERR; }
  for (int r = 0; r < c->world; ++r) {
    struct stat st;
    const time_t t0 = time(NULL);
    snprintf(path, sizeof path, "%s/%ld.%d", c->dir, seq, r);
    while (stat(path, &st) != 0) {
      if (time(NULL) - t0 > 60) { free(*all); return TIMEOUT; }
      usleep(1000);
    }
    if ((size_t)st.st_size != bytes) { free(*all); return BAD_ARG; }
    f = fopen(path, "rb");
    const int got = f && fread(*all + r * bytes, 1, bytes, f) == bytes;
    if (f) fclose(f);
    if (!got) { free(*all); return SYS_ERR; }
  }
  return OK;
}

static size_t word(int type) { return type == 2 ? 4 : (type == 4 || type == 8) ? 8 : 0; }   /* int32, int64, float64 */

int ncclAllReduce(const void* send, void* recv, size_t count, int type, int op, ncclComm_t c, cudaStream_t s) {
  const size_t w = word(type);
  char* all;
  if (op != 0 || type == 8) return BAD_ARG;                    /* sum of integers only */
  int r = exchange(c, send, count * w, s, &all);
  if (r) return r;
  for (int q = 1; q < c->world; ++q)
    for (size_t i = 0; i < count; ++i) {
      if (w == 4) ((uint32_t*)all)[i] += ((const uint32_t*)(all + q * count * w))[i];
      else ((uint64_t*)all)[i] += ((const uint64_t*)(all + q * count * w))[i];
    }
  r = count && cudaMemcpy(recv, all, count * w, cudaMemcpyHostToDevice) != cudaSuccess ? CUDA_ERR : OK;
  free(all);
  return r;
}

int ncclAllGather(const void* send, void* recv, size_t count, int type, ncclComm_t c, cudaStream_t s) {
  const size_t w = word(type);
  char* all;
  if (!w) return BAD_ARG;
  int r = exchange(c, send, count * w, s, &all);
  if (r) return r;
  r = count && cudaMemcpy(recv, all, c->world * count * w, cudaMemcpyHostToDevice) != cudaSuccess ? CUDA_ERR : OK;
  free(all);
  return r;
}
"""


def _outcome(fn, *args, **kw):
    try:
        return ("ok", fn(*args, **kw))
    except Exception as e:                         # an RCError, or what a wrong result leads to on the host
        return ("err", getattr(e, "status", None), str(e))


def _make(pkg, data, lab, chain0, nch, numiters=ITERS):
    """nch chains from global chain chain0 on, as tools/multigpu_check.py's make; run to the end."""
    params = pkg.params_from_labels(data.D, lab)
    opts = pkg.MCMCOptionsList(numiters=numiters, burnin=0, thin=1, numGibbs=5, numMH=1)
    rp = [pkg.init_rp(params, 7, chain0 + c) for c in range(nch)]
    return pkg.Sampler(data, opts, params, np.tile(lab, (nch, 1)), [a for a, _ in rp], [b for _, b in rp], seed=7,
                       chain_offset=chain0)


def _host_labels(rng, n):
    return np.stack([rng.integers(1, 6, size=n) for _ in range(13)])


def _worker(rank, world, port, nccl_lib, iddir, out):
    os.environ.update(RCB200_NCCL_LIB=nccl_lib, STANDIN_NCCL_DIR=iddir, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import __graft_entry__ as g
    pkg = g.load_package()
    dist.init_process_group("gloo", rank=rank, world_size=world)
    gd = np.load(os.path.join(ROOT, "tests", "golden", "example1.npz"))
    X, D, lab = gd["points"], gd["distance_matrix"], gd["cluster_labels"]
    chains = WORLDS[world]
    last = world - 1
    comm = pkg.Comm.from_torch(device=0)
    res = {}
    try:
        data = pkg.MCMCData(D)
        smp = _make(pkg, data, lab, sum(chains[:rank]), chains[rank])
        smp.run()
        # equal to one sampler over the same global chains
        res["psm"] = smp.psm_allreduce(comm=comm)
        res["binder"] = smp.binder_pointestimate_allreduce(comm=comm)
        res["conv"] = smp.convergencediagnostics_allreduce(comm=comm, matrix=True)
        res["ball"] = {loss: smp.credibleball_allreduce(lab, loss=loss, comm=comm) for loss in ("VI", "binder")}
        res["align"] = smp.alignedallocation_allreduce(lab, maps=True, comm=comm)
        res["D"] = pkg.MCMCData.from_points_sharded(X, comm=comm).D
        L = _host_labels(np.random.default_rng(5), D.shape[0])
        res["psm_sharded"] = pkg.psm_sharded(L[rank::world], comm=comm)
        res["mpel"] = {loss: pkg.mpel_loss_sums_sharded(L, loss, comm=comm) for loss in ("binder", "VI")}
        # one rank's sampler has not finished its run: every rank returns, and the communicator then serves a complete call
        part = _make(pkg, data, lab, sum(chains[:rank]), chains[rank])
        part.run(ITERS // 2 if rank == last else -1)
        res["refused"] = {name: _outcome(getattr(part, name), comm=comm) for name in (
            "psm_allreduce", "binder_pointestimate_allreduce", "convergencediagnostics_allreduce")}
        res["refused"]["credibleball_allreduce"] = _outcome(part.credibleball_allreduce, lab, comm=comm)
        res["refused"]["alignedallocation_allreduce"] = _outcome(part.alignedallocation_allreduce, lab, comm=comm)
        res["after_refusal"] = smp.psm_allreduce(comm=comm)
        # ranks that disagree: another n on the last rank, another number of samples per chain on the last rank
        m = 60 if rank == last else D.shape[0]
        small = pkg.MCMCData(np.ascontiguousarray(D[:m, :m]))
        other_n = _make(pkg, small, lab[:m], sum(chains[:rank]), chains[rank])
        other_n.run()
        res["disagree"] = {
            "sampler_psm": _outcome(other_n.psm_allreduce, comm=comm),
            "data_from_points": _outcome(pkg.MCMCData.from_points_sharded, X[:m], comm=comm),
            "psm": _outcome(pkg.psm_sharded, L[rank::world, :m], comm=comm),
        }
        other_S = _make(pkg, data, lab, sum(chains[:rank]), chains[rank], numiters=ITERS + 2 * (rank == last))
        other_S.run()
        res["disagree"]["cocl_rhat"] = _outcome(other_S.convergencediagnostics_allreduce, comm=comm)
        # rc_comm_psm with more than 255 clusters in the first rank's labels (last: a rank refusing before any
        # collective leaves a library without the status exchange one collective behind)
        wide = np.tile(np.arange(300) % (256 if rank == 0 else 5) + 1, (2, 1))
        res["psm_slots"] = _outcome(pkg.psm_sharded, wide, comm=comm)
    finally:
        with open(os.path.join(out, f"rank{rank}.pkl"), "wb") as f:
            pickle.dump(res, f)
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """world -> the results of every rank, each world run once for the module."""
    base = tmp_path_factory.mktemp("sharded")
    lib = str(base / "libstandin_nccl.so")
    (base / "standin_nccl.c").write_text(STANDIN_NCCL)
    subprocess.check_call(["nvcc", "-shared", "-Xcompiler", "-fPIC", "-O2", "-Wno-deprecated-gpu-targets", "-o", lib, str(base / "standin_nccl.c")])
    ctx = mp.get_context("spawn")
    got = {}
    for world, port in ((2, 29541), (3, 29543)):
        out = base / f"world{world}"
        out.mkdir()
        procs = [ctx.Process(target=_worker, args=(r, world, port, lib, str(base), str(out))) for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=600)
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
        got[world] = [p.exitcode for p in procs], []
        for r in range(world):
            with open(out / f"rank{r}.pkl", "rb") as f:
                got[world][1].append(pickle.load(f))
    return got


def _ranks(runs, world):
    codes, res = runs[world]
    assert codes == [0] * world
    return res


@pytest.fixture(scope="module")
def one(pkg, golden):
    """One sampler over the global chains of each world, and the single-GPU results of the sharded host calls."""
    X, D, lab = golden[1]["points"], golden[1]["distance_matrix"], golden[1]["cluster_labels"]
    data = pkg.MCMCData(D)
    ref = {}
    for world, chains in WORLDS.items():
        smp = _make(pkg, data, lab, 0, sum(chains))
        smp.run()
        ref[world] = dict(psm=smp.psm(), binder=smp.binder_pointestimate(), conv=smp.convergencediagnostics(matrix=True),
                          ball={loss: smp.credibleball(lab, loss=loss) for loss in ("VI", "binder")},
                          align=smp.alignedallocation(lab, maps=True), S=smp.options.numsamples)
        smp.close()
    L = _host_labels(np.random.default_rng(5), D.shape[0])
    host = dict(D=pkg.MCMCData.from_points(X).D, psm_sharded=pkg.psm(L),
                mpel={loss: pkg.mpel_loss_sums(L, loss) for loss in ("binder", "VI")})
    return ref, host


def _same_values(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("world", sorted(WORLDS))
def test_equal_to_one_sampler(runs, one, world):
    ref, host = one
    r1 = ref[world]
    S = r1["S"]
    owners = 0
    for rank, got in enumerate(_ranks(runs, world)):
        assert np.array_equal(got["psm"], r1["psm"])
        b, b1 = got["binder"], r1["binder"]
        assert np.array_equal(b["sums"], b1["sums"]) and np.array_equal(b["totals"], b1["totals"])
        assert b["best"] == b1["chain"] * S + b1["index"]
        if b["clust"] is not None:
            owners += 1
            assert np.array_equal(b["clust"], b1["clust"])
        c, c1 = got["conv"], r1["conv"]
        assert np.array_equal(c["rhat"], c1["rhat"], equal_nan=True)
        assert _same_values(c["rhat_max"], c1["rhat_max"]) and c["rhat_pair"] == c1["rhat_pair"]
        assert c["pairs_above"] == c1["pairs_above"]
        assert np.array_equal(c["chain_meandev"], c1["chain_meandev"]) and np.array_equal(c["chain_maxdev"], c1["chain_maxdev"])
        assert c["traces"].keys() == c1["traces"].keys()
        assert all(_same_values(c["traces"][k], c1["traces"][k]) for k in c1["traces"])
        for loss, cb1 in r1["ball"].items():
            cb = got["ball"][loss]
            assert np.array_equal(cb["dist"], cb1["dist"]) and cb["radius"] == cb1["radius"] and cb["inball"] == cb1["inball"]
            assert cb["expectedloss"] == cb1["expectedloss"]
            for k in ("horizontal", "upper", "lower"):
                assert np.array_equal(cb[k]["indices"], cb1[k]["indices"]) and cb[k]["dist"] == cb1[k]["dist"]
                assert cb[k]["K"] == cb1[k]["K"]
        assert set(got["align"]) == set(r1["align"])
        for k in r1["align"]:
            assert np.array_equal(got["align"][k], r1["align"][k]), k
        assert np.array_equal(got["D"], host["D"])
        assert np.array_equal(got["psm_sharded"], host["psm_sharded"])
        for loss, (s1, b1) in host["mpel"].items():
            assert np.array_equal(got["mpel"][loss][0], s1) and got["mpel"][loss][1] == b1
    assert owners == 1


@pytest.mark.gpu
@pytest.mark.parametrize("world", sorted(WORLDS))
def test_refusal_does_not_leave_ranks_waiting(runs, one, world):
    last = world - 1
    for rank, got in enumerate(_ranks(runs, world)):
        for name, o in got["refused"].items():
            assert o[0] == "err" and o[1] == -6, (rank, name, o)
            if rank != last:
                assert f"rank {last} refused (status -6)" in o[2], (rank, name, o)
            else:
                assert "refused" not in o[2], (rank, name, o)
        assert np.array_equal(got["after_refusal"], one[0][world]["psm"])
        o = got["psm_slots"]
        assert o[0] == "err" and o[1] == -5, (rank, o)
        assert ("more than 255 clusters" in o[2]) if rank == 0 else ("rank 0 refused (status -5)" in o[2]), (rank, o)


@pytest.mark.gpu
@pytest.mark.parametrize("world", sorted(WORLDS))
def test_disagreement_is_refused_on_every_rank(runs, world):
    for rank, got in enumerate(_ranks(runs, world)):
        for case, o in got["disagree"].items():
            assert o[0] == "err" and o[1] == -1, (rank, case, o)
            want = "samples per chain" if case == "cocl_rhat" else "disagree on n "
            assert want in o[2], (rank, case, o)
