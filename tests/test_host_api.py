"""CPU tests: the C-ABI library loads and exports every symbol include/rcb200.h declares (no compute calls
without a GPU), the host-side mirror validates arguments like the reference (src/types.jl:40-54,
src/pointestimate.jl:19-26, src/utils.jl:103-108), and the oracle's numpy restatements agree with each other."""
import ctypes
import os
import re
import struct
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "rcb200.h")).read()
    declared = set(re.findall(r"\b(rc_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"rc_status"}
    assert len(declared) >= 25
    assert os.path.exists(pkg.LIB_PATH), "librcb200.so is not built: run __graft_entry__.build()"
    lib = ctypes.CDLL(pkg.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    from redclust_jl_b200 import _lib
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib.rc_version.restype = ctypes.c_int32
    assert lib.rc_version() == 100


def test_no_cpu_fallback_without_device(pkg):
    """The product path fails loudly when there is no CUDA device."""
    from redclust_jl_b200._lib import lib
    if lib().rc_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(pkg.RCError) as e:
        pkg.MCMCData(np.zeros((3, 3)))
    assert "no CUDA device" in str(e.value) or "CUDA" in str(e.value)


def test_options_validation_matches_reference_messages(pkg):
    o = pkg.MCMCOptionsList()
    assert (o.numiters, o.burnin, o.thin, o.numGibbs, o.numMH, o.numsamples) == (5000, 1000, 1, 5, 1, 4000)
    assert pkg.MCMCOptionsList(numiters=10, burnin=3, thin=2).numsamples == 3
    for kw, msg in ((dict(numiters=0), "numiters must be ≥ 1."), (dict(numiters=5, burnin=6), "burnin must be < numiters"),
                    (dict(thin=0), "thin must be positive."), (dict(numGibbs=-1), "numGibbs must be non-negative."),
                    (dict(numMH=-1), "numMH must be non-negative.")):
        with pytest.raises(pkg.RCError) as e:
            pkg.MCMCOptionsList(**kw)
        assert str(e.value) == msg


def test_hyperparameter_defaults(pkg):
    p = pkg.PriorHyperparamsList(eta=4.0, sigma=2.0)
    assert p.proposalsd_r == 1.0 and p.repulsion is True and p.maxK == 0 and p.K_initial == 1      # types.jl:93-108
    q = pkg.PriorHyperparamsList(**{"δ1": 2.0, "α": 3.0})
    assert q.delta1 == 2.0 and q.alpha == 3.0
    c = q._c()
    assert ctypes.sizeof(c) == 11 * 8 + 8 + 8 + 4 + 4


def test_label_utilities(pkg, orc):
    rng = np.random.default_rng(0)
    for _ in range(20):
        x = rng.integers(1, 9, size=50)
        y = pkg.sortlabels(x)
        assert np.array_equal(y, orc.sortlabels(x))
        assert np.array_equal(pkg.adjacencymatrix(x), pkg.adjacencymatrix(y))            # test/test_utils.jl:23-29
        first = [np.where(y == k)[0][0] for k in range(1, y.max() + 1)]
        assert first == sorted(first)
    m = pkg.makematrix([[1.0, 2.0], [3.0, 4.0], [5.0, 6.0]])
    assert m.shape == (2, 3) and m[1, 2] == 6.0                                          # test/test_utils.jl:1-8
    M = np.arange(16.0).reshape(4, 4)
    assert list(pkg.uppertriangle(M)) == [1, 2, 3, 6, 7, 11]


def test_getpointestimate_argument_errors(pkg):
    class R:
        logposterior = np.array([0.0, 2.0, 1.0]); loglik = np.array([3.0, 1.0, 2.0]); clusts = [np.array([1, 1]), np.array([1, 2]), np.array([2, 1])]
    assert pkg.getpointestimate(R, method="MAP")[1] == 1 and pkg.getpointestimate(R, method="MLE")[1] == 0
    with pytest.raises(pkg.ArgumentError, match="Invalid method specifier."):
        pkg.getpointestimate(R, method="foo")
    with pytest.raises(pkg.ArgumentError, match="Invalid loss function specifier."):
        pkg.getpointestimate(R, method="MPEL", loss="foo")
    with pytest.raises(pkg.ArgumentError, match="Length of the input vectors must be equal."):
        pkg.binderloss([1, 2], [1, 2, 3])
    with pytest.raises(pkg.ArgumentError, match="Length of the input vectors must be equal."):
        pkg.infodist([1, 2], [1, 2, 3])


def test_generatemixture_argument_errors(pkg):
    for args, kw in (((0, 1), {}), ((10, 11), {}), ((10, 2), dict(alpha=0)), ((10, 5), dict(dim=3)), ((10, 2), dict(radius=0)), ((10, 2), dict(sigma=0))):
        with pytest.raises(pkg.ArgumentError):
            pkg.generatemixture(*args, **kw)


def test_oracle_losses_consistency(orc):
    """binder = Mirkin / C(n,2); VI = H(a) + H(b) - 2 I; ID = max(H) - I; identities of test/test_pointestimates.jl:3-8."""
    rng = np.random.default_rng(4)
    a = rng.integers(1, 5, 60); b = rng.integers(1, 7, 60)
    assert abs(orc.binderloss(a, a)) < 1e-9 and abs(orc.infodist(a, a)) < 1e-9
    n = 60
    dis = sum((a[i] == a[j]) != (b[i] == b[j]) for i in range(n) for j in range(i + 1, n))
    assert abs(orc.binderloss(a, b) - dis / (n * (n - 1) / 2)) < 1e-12
    assert abs(orc.binderloss(a, b, normalised=False) - dis) < 1e-9
    S = rng.integers(1, 5, size=(7, 30))
    sums = orc.mpel_loss_sums(S, "binder")
    cnt = orc.psm_counts(S)
    # Binder column sums collapse onto the PSM counts (SURVEY 8a row 15)
    for i in range(7):
        A = orc.adjacencymatrix(S[i])
        iu = np.triu_indices(30, 1)
        tot = (7 * A[iu].sum() + cnt[iu].sum() - 2 * (A[iu] * cnt[iu]).sum()) / (30 * 29 / 2)
        assert abs(sums[i] - tot) < 1e-12


def test_fitprior_host_pieces(pkg, golden):
    from redclust_jl_b200.prior import detectknee, gamma_mle_shape, sampleK, sampledist
    assert detectknee([1, 2, 3, 4, 5], [10, 4, 2, 1.5, 1.2])[0] == 2
    x = np.random.default_rng(0).gamma(5.0, 2.0, 20000)
    assert abs(gamma_mle_shape(x) - 5.0) < 0.2
    p = pkg.PriorHyperparamsList(eta=4.0, sigma=2.0, u=2.0, v=20.0, alpha=10.0, beta=5.0, delta1=3.0)
    assert sampleK(p, 5, 30).shape == (5,) and sampledist(p, "intracluster", 4).shape == (4,)
    with pytest.raises(ValueError):
        sampledist(p, "foo")


def test_reference_utils_cases(pkg):
    """test/test_utils.jl:1-61 case by case (makematrix, adjacencymatrix, sortlabels, prettytime)."""
    rng = np.random.default_rng(0)
    m, n = 50, 100
    temp = [rng.random(m) for _ in range(n)]
    M = pkg.makematrix(temp)
    assert M.shape == (m, n) and sum(int((M[:, i] == temp[i]).sum()) for i in range(n)) == m * n
    K, n = 20, 500
    lab = rng.integers(1, K + 1, size=n)
    A = pkg.adjacencymatrix(lab)
    assert int((A == (lab[:, None] == lab[None, :])).sum()) == n * n
    assert int((pkg.adjacencymatrix(lab) == pkg.adjacencymatrix(pkg.sortlabels(lab))).sum()) == n * n
    cases = {1e-9: "1.00 ns", 999e-9: "999.00 ns", 1e-6: "1.00 μs", 999e-6: "999.00 μs", 1e-3: "1.00 ms", 999e-3: "999.00 ms",
             1: "1.00 s", 5: "5.00 s", 60: "1 min", 120: "2 mins", 65: "1 min 5 s", 125: "2 mins 5 s", 3600: "1 hr", 7200: "2 hrs",
             7205: "2 hrs 5 s", 7265: "2 hrs 1 min 5 s", 7325: "2 hrs 2 mins 5 s", 24 * 3600: "1 day", 2 * 24 * 3600: "2 days"}
    for t, want in cases.items():
        assert pkg.prettytime(t) == want, (t, pkg.prettytime(t), want)


_UNDEF = 0xFFFFFFFFFFFFFFFF


def _q(v):
    return struct.pack("<Q", v)


def _write_h5(path, groups):
    """A small HDF5 file of the layout h5min.py reads (that of RedClust.jl's data/example_datasets.h5): superblock
    version 0, an old-style root group (symbol-table B-tree + local heap) holding compact new-style groups (link
    messages) of contiguous little-endian int64 / float64 datasets.  groups: {group: {dataset: array}}."""
    buf = bytearray(96)                                              # superblock + root symbol-table entry, written last

    def put(b):
        buf.extend(b"\0" * (-len(buf) % 8))
        addr = len(buf)
        buf.extend(b)
        return addr

    def msg(mtype, payload):
        payload += b"\0" * (-len(payload) % 8)
        return struct.pack("<HHB3x", mtype, len(payload), 0) + payload

    def ohdr(msgs):                                                  # version-1 object header
        body = b"".join(msgs)
        return put(struct.pack("<BBHII4x", 1, 0, len(msgs), 1, len(body)) + body)

    def entry(name_off, addr, cache=0, scratch=b"\0" * 16):          # symbol-table entry
        return _q(name_off) + _q(addr) + struct.pack("<I4x", cache) + scratch

    def dataset(a):
        a = np.ascontiguousarray(a)
        assert a.dtype in (np.int64, np.float64)
        data = put(a.tobytes())
        space = struct.pack("<BBB5x", 1, a.ndim, 0) + b"".join(_q(d) for d in a.shape)
        if a.dtype == np.int64:                                      # fixed-point, signed
            dtype = struct.pack("<BBBBIHH", 0x10, 0x08, 0, 0, 8, 0, 64)
        else:                                                        # IEEE binary64
            dtype = struct.pack("<BBBBIHHBBBBI", 0x11, 0x20, 63, 0, 8, 0, 64, 52, 11, 0, 52, 1023)
        return ohdr([msg(0x01, space), msg(0x03, dtype), msg(0x08, struct.pack("<BB", 3, 1) + _q(data) + _q(a.nbytes))])

    def group(members):                                              # link info, group info, one link message per member
        links = [msg(0x02, struct.pack("<BB", 0, 0) + _q(_UNDEF) + _q(_UNDEF)), msg(0x0A, struct.pack("<BB", 0, 0))]
        for name, addr in members.items():
            links.append(msg(0x06, struct.pack("<BBB", 1, 0, len(name)) + name.encode() + _q(addr)))
        return ohdr(links)

    gaddr = {g: group({k: dataset(v) for k, v in ds.items()}) for g, ds in groups.items()}
    names = sorted(gaddr)
    heapdata, offs = bytearray(8), {}                                # offset 0: the empty name
    for g in names:
        offs[g] = len(heapdata)
        heapdata += g.encode() + b"\0" * (8 - len(g) % 8)
    heap = put(b"HEAP" + struct.pack("<B3x", 0) + _q(len(heapdata)) + _q(_UNDEF) + _q(put(bytes(heapdata))))
    snod = put(b"SNOD" + struct.pack("<BBH", 1, 0, len(names)) + b"".join(entry(offs[g], gaddr[g]) for g in names)
               + bytes(40 * (8 - len(names))))                      # 2 x group leaf K (4) entries per node
    btree = put(b"TREE" + struct.pack("<BBH", 0, 0, 1) + _q(_UNDEF) + _q(_UNDEF) + _q(0) + _q(snod) + _q(offs[names[-1]]))
    root = ohdr([msg(0x11, _q(btree) + _q(heap))])
    buf[:96] = (b"\x89HDF\r\n\x1a\n" + bytes([0, 0, 0, 0, 0, 8, 8, 0]) + struct.pack("<HHI", 4, 16, 0)
                + _q(0) + _q(_UNDEF) + _q(len(buf)) + _q(_UNDEF) + entry(0, root, 1, _q(btree) + _q(heap)))
    with open(path, "wb") as f:
        f.write(buf)


def test_example_dataset_reader(pkg, golden, tmp_path):
    """example_dataset(n) / example_datasets() (example_data.jl:33-71): the package copy, and the same arrays through the
    minimal HDF5 reader from a file of the reference's layout.  The golden arrays are RedClust.jl's own
    data/example_datasets.h5 (tests/golden/make_golden.py); here they are written back into such a file."""
    for n in (1, 2, 3):
        d = pkg.example_dataset(n)
        assert len(d["points"]) == 100 and d["points"][0].shape == golden[n]["points"][0].shape
        assert np.array_equal(np.stack(d["points"]), golden[n]["points"])
        assert np.array_equal(d["distmatrix"], golden[n]["distance_matrix"])
        assert np.array_equal(d["clusts"], golden[n]["cluster_labels"]) and d["clusts"].dtype == np.int64
        assert abs(d["probs"].sum() - 1) < 1e-12
        assert np.array_equal(d["oracle_coclustering"], golden[n]["oracle_coclustering_probabilities"])
    with pytest.raises(pkg.ArgumentError):
        pkg.example_dataset(4)
    f = pkg.example_datasets()
    assert f.keys() == ["example1", "example2", "example3"]
    assert "distance_matrix" in f["example2"].keys()
    f.close()
    ref = str(tmp_path / "example_datasets.h5")
    _write_h5(ref, {f"example{n}": golden[n] for n in (1, 2, 3)})
    h = pkg.example_datasets(ref)
    assert h.keys() == ["example1", "example2", "example3"]
    for n in (1, 2, 3):
        assert h[f"example{n}"].keys() == sorted(golden[n])
        for name in golden[n]:
            assert np.array_equal(h[f"example{n}"][name], golden[n][name]), (n, name)
    h.close()
    assert np.array_equal(pkg.example_dataset(3, path=ref)["distmatrix"], golden[3]["distance_matrix"])
