"""ctypes binding of librcb200.so (include/rcb200.h).  This is the Python twin of the Julia `ccall`
layer in julia/RedClustB200.jl: same entry points, same argument order.  There is no CPU fallback --
if the shared library is missing or has no CUDA device, calls raise."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RCB200_LIB") or os.path.join(_HERE, "librcb200.so")   # RCB200_LIB: experiment builds

RC_OK, RC_ERR_ARG, RC_ERR_CUDA, RC_ERR_NOTSYM, RC_ERR_DOMAIN, RC_ERR_SLOTS, RC_ERR_STATE = 0, -1, -2, -3, -4, -5, -6


class rc_options(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("numiters", "burnin", "thin", "numGibbs", "numMH")]


class rc_params(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("delta1", "delta2", "alpha", "beta", "zeta", "gamma", "eta", "sigma",
                                         "proposalsd_r", "u", "v")] + [
        ("K_initial", C.c_int64), ("maxK", C.c_int64), ("repulsion", C.c_int32), ("_pad", C.c_int32)]


class rc_rhat_summary(C.Structure):
    _fields_ = [("max", C.c_double), ("a", C.c_int64), ("b", C.c_int64), ("above", C.c_int64)]


class RCError(RuntimeError):
    """ErrorException of the Julia API (error(...) in src/types.jl)."""

    def __init__(self, status, msg):
        super().__init__(msg)
        self.status = status


_lib = None
_P = C.POINTER
_vp = C.c_void_p

# name -> (restype, argtypes): every symbol include/rcb200.h declares
SIGNATURES = {
    "rc_version": (C.c_int32, []),
    "rc_last_error": (C.c_char_p, []),
    "rc_device_count": (C.c_int32, []),
    "rc_data_from_dist": (C.c_int32, [_vp, C.c_int64, C.c_int32, _P(_vp)]),
    "rc_data_from_points": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, _P(_vp)]),
    "rc_distm_rows_dev": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _vp]),
    "rc_data_from_dist_dev": (C.c_int32, [_vp, C.c_int64, C.c_int32, _P(_vp)]),
    "rc_oracle_coclustering": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_double, _vp, C.c_int64, C.c_int32, _vp]),
    "rc_data_n": (C.c_int64, [_vp]),
    "rc_data_copy_dist": (C.c_int32, [_vp, _vp]),
    "rc_data_copy_logdist": (C.c_int32, [_vp, _vp]),
    "rc_data_scales": (C.c_int32, [_vp, _P(C.c_int32), _P(C.c_int32)]),
    "rc_data_copy_row": (C.c_int32, [_vp, C.c_int64, _vp]),
    "rc_kmeans": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, _vp, C.c_int64, C.c_double, C.c_int32, _vp, _vp, _P(C.c_double), _P(C.c_int32), _P(C.c_int64)]),
    "rc_kmedoids_seed": (C.c_int32, [_vp, C.c_int64, _vp, _vp]),
    "rc_kmedoids": (C.c_int32, [_vp, C.c_int64, _vp, C.c_int64, _vp, _vp, _P(C.c_double), _P(C.c_int32), _P(C.c_int64)]),
    "rc_pair_stats": (C.c_int32, [_vp, _vp, _vp]),
    "rc_sample_rp": (C.c_int32, [_vp, C.c_int64, _P(rc_options), _P(rc_params), C.c_uint64, C.c_int32, _vp, _vp, _vp]),
    "rc_data_destroy": (None, [_vp]),
    "rc_init_rp": (C.c_int32, [_P(rc_params), C.c_uint64, C.c_int64, _P(C.c_double), _P(C.c_double)]),
    "rc_sampler_create": (C.c_int32, [_vp, _P(rc_options), _P(rc_params), C.c_int64, C.c_int64, _vp, _vp, _vp,
                                      C.c_uint64, C.c_int32, _P(_vp)]),
    "rc_sampler_run": (C.c_int32, [_vp, C.c_int64]),
    "rc_sampler_progress": (C.c_int32, [_vp, _P(C.c_int64), _P(C.c_double)]),
    "rc_sampler_numsamples": (C.c_int64, [_vp]),
    "rc_sampler_n": (C.c_int64, [_vp]),
    "rc_sampler_nchains": (C.c_int64, [_vp]),
    "rc_sampler_copy_samples": (C.c_int32, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rc_sampler_copy_all": (C.c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rc_sampler_copy_acceptances": (C.c_int32, [_vp, C.c_int64, _vp, _vp, _vp]),
    "rc_sampler_copy_state": (C.c_int32, [_vp, C.c_int64, _vp, _P(C.c_double), _P(C.c_double)]),
    "rc_sampler_chain_status": (C.c_int32, [_vp, C.c_int64]),
    "rc_sampler_overflowed": (C.c_int64, [_vp]),
    "rc_sampler_check_sums": (C.c_int32, [_vp, _P(C.c_int64), _P(C.c_int64)]),
    "rc_sampler_copy_stats": (C.c_int32, [_vp, _vp]),
    "rc_sampler_psm_counts_dev": (C.c_int32, [_vp, C.c_int64, C.c_int64, _vp]),
    "rc_sampler_psm": (C.c_int32, [_vp, C.c_int64, C.c_int64, _vp]),
    "rc_sampler_destroy": (None, [_vp]),
    "rc_predict": (C.c_int32, [_vp, _P(rc_params), _vp, C.c_int64, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp]),
    "rc_sampler_predict": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, _vp, _vp]),
    "rc_crossdist": (C.c_int32, [_vp, C.c_int64, _vp, C.c_int64, C.c_int64, C.c_int32, _vp]),
    "rc_loglik": (C.c_int32, [_vp, _P(rc_params), _vp, _P(C.c_double)]),
    "rc_psm": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, _vp]),
    "rc_psm_counts_dev": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, _vp]),
    "rc_mpel": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _vp, _P(C.c_int64)]),
    "rc_mpel_rows_dev": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, _vp]),
    "rc_mpel_finish_dev": (C.c_int32, [_vp, C.c_int64, C.c_int32, _vp, _P(C.c_int64)]),
    "rc_binder_mpel": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int32, _vp, _P(C.c_int64), _vp]),
    "rc_sampler_binder_mpel": (C.c_int32, [_vp, C.c_int64, C.c_int64, _vp, _P(C.c_int64), _vp]),
    "rc_cocl_rhat": (C.c_int32, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _P(rc_rhat_summary), _vp, _vp, _vp]),
    "rc_sampler_cocl_rhat": (C.c_int32, [_vp, C.c_int64, C.c_int64, _P(rc_rhat_summary), _vp, _vp, _vp]),
    "rc_partition_dists": (C.c_int32, [_vp, C.c_int64, _vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp]),
    "rc_sampler_partition_dists": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _vp, _vp, _vp]),
    "rc_aligned_alloc": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp]),
    "rc_sampler_aligned_alloc": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp]),
    "rc_comm_unique_id": (C.c_int32, [_vp]),
    "rc_comm_init": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _P(_vp)]),
    "rc_comm_info": (C.c_int32, [_vp, _P(C.c_int32), _P(C.c_int32)]),
    "rc_comm_destroy": (None, [_vp]),
    "rc_comm_allreduce_i32": (C.c_int32, [_vp, _vp, C.c_int64]),
    "rc_comm_data_from_points": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, _P(_vp)]),
    "rc_comm_sampler_psm": (C.c_int32, [_vp, _vp, _vp, _vp]),
    "rc_comm_psm": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "rc_comm_mpel": (C.c_int32, [_vp, _vp, C.c_int64, C.c_int64, C.c_int32, _vp, _P(C.c_int64)]),
    "rc_comm_sampler_binder_mpel": (C.c_int32, [_vp, _vp, _vp, _P(C.c_int64), _vp]),
    "rc_comm_sampler_cocl_rhat": (C.c_int32, [_vp, _vp, _P(rc_rhat_summary), _vp, _vp, _vp]),
    "rc_comm_sampler_partition_dists": (C.c_int32, [_vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, _vp]),
    "rc_comm_sampler_aligned_alloc": (C.c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RCError(RC_ERR_CUDA, f"{LIB_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                                       "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != RC_OK:
        raise RCError(status, lib().rc_last_error().decode("utf-8", "replace"))


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
