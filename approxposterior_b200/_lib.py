"""ctypes binding of libapgp.so (the C-ABI declared in include/apgp.h).

The library is built in-tree by ``__graft_entry__.build()`` (``make -C approxposterior_b200/csrc``).
There is deliberately no fallback: if the shared object is missing, or no B200 is visible,
every entry point raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("APGP_LIB") or os.path.join(_HERE, "libapgp.so")     # APGP_LIB: debug/profiling builds

APGP_OK, APGP_NOT_POSDEF, APGP_NOT_COMPUTED, APGP_NEEDS_REFACTOR, APGP_NEEDS_HOST = 0, 1, 2, 3, 4
MAX_DIM = 32
UTIL_KINDS = {None: 0, "none": 0, "agp": 1, "bape": 2, "jones": 3, "negmean": 4}
OPT_METHODS = {"nelder-mead": 0, "powell": 1}
OPT_INF = 1 << 62


class PredictOpts(C.Structure):
    _fields_ = [("want_var", C.c_int), ("utility", C.c_int), ("has_box", C.c_int),
                ("lo", C.c_double * MAX_DIM), ("hi", C.c_double * MAX_DIM),
                ("ybest", C.c_double), ("zeta", C.c_double)]


class SamplerOpts(C.Structure):
    _fields_ = [("nens", C.c_int), ("nwalkers", C.c_int), ("nsteps", C.c_int), ("thin", C.c_int),
                ("a", C.c_double), ("seed", C.c_ulonglong),
                ("lo", C.c_double * MAX_DIM), ("hi", C.c_double * MAX_DIM),
                ("lnprior_const", C.c_double),
                ("replay_inds", C.c_void_p), ("replay_zz", C.c_void_p),
                ("replay_rint", C.c_void_p), ("replay_logu", C.c_void_p)]


class OptOpts(C.Structure):
    _fields_ = [("method", C.c_int), ("adaptive", C.c_int), ("xtol", C.c_double), ("ftol", C.c_double),
                ("maxiter", C.c_longlong), ("maxfev", C.c_longlong)]


_SIGNATURES = {
    "apgp_last_error": (C.c_char_p, []),
    "apgp_version": (C.c_int, []),
    "apgp_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "apgp_destroy": (C.c_int, [C.c_void_p]),
    "apgp_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "apgp_reset": (C.c_int, [C.c_void_p]),
    "apgp_synchronize": (C.c_int, [C.c_void_p]),
    "apgp_launch_count": (C.c_longlong, [C.c_void_p]),
    "apgp_set_training": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "apgp_set_hyper": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_double]),
    "apgp_factorize": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "apgp_append_point": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "apgp_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.POINTER(PredictOpts), C.c_int]),
    "apgp_grad_log_likelihood": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "apgp_loglik_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p,
                                    C.c_void_p]),
    "apgp_sampler_run": (C.c_int, [C.c_void_p, C.POINTER(SamplerOpts), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int]),
    "apgp_comm_unique_id": (C.c_int, [C.c_char_p]),
    "apgp_comm_init": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int]),
    "apgp_comm_destroy": (C.c_int, [C.c_void_p]),
    "apgp_comm_group_start": (C.c_int, []),
    "apgp_comm_group_end": (C.c_int, []),
    "apgp_comm_broadcast_factor": (C.c_int, [C.c_void_p, C.c_int]),
    "apgp_comm_allgather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int]),
    "apgp_integrated_time": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_int,
                                       C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    "apgp_minimize_utility": (C.c_int, [C.c_void_p, C.POINTER(PredictOpts), C.POINTER(OptOpts), C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "apgp_minimize_nll": (C.c_int, [C.c_void_p, C.POINTER(OptOpts), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double,
                                    C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "apgp_minimize_nll_fits": (C.c_int, [C.c_void_p, C.c_int]),
    "apgp_get_alpha": (C.c_int, [C.c_void_p, C.c_void_p]),
    "apgp_get_linv": (C.c_int, [C.c_void_p, C.c_void_p]),
    "apgp_get_chol": (C.c_int, [C.c_void_p, C.c_void_p]),
    "apgp_set_group": (C.c_int, [C.c_void_p, C.c_int]),
    "apgp_set_var_engine": (C.c_int, [C.c_void_p, C.c_int]),
    "apgp_set_predict_few": (C.c_int, [C.c_void_p, C.c_int]),
    "apgp_debug_exp_neg": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "apgp_debug_exp_neg256": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "apgp_debug_read_prof": (C.c_int, [C.c_void_p]),
    "apgp_debug_group_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "apgp_debug_last_var_path": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "apgp_debug_last_loglik_path": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "apgp_debug_i8_operands": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "apgp_debug_pack_linv_i8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class ApgpError(RuntimeError):
    pass


def load():
    """Load libapgp.so (once).  Raises if it has not been built -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ApgpError("libapgp.so not found at %s: build it with `python -c 'import __graft_entry__ as g; "
                        "g.build()'` (make -C approxposterior_b200/csrc). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().apgp_last_error().decode()


def check(status, what):
    """Raise on library/CUDA errors (status < 0); data conditions (> 0) are returned to the caller."""
    if status < 0:
        raise ApgpError("%s failed (%d): %s" % (what, status, last_error()))
    return status


def ptr(a):
    """Raw address of a NumPy array or torch tensor (device or host)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()          # torch.Tensor


def fill_bounds(dst_lo, dst_hi, bounds, d):
    for i in range(d):
        dst_lo[i] = float(bounds[i][0])
        dst_hi[i] = float(bounds[i][1])
