"""ctypes binding of libsbd.so - exactly the symbols declared in include/sbd.h.

This is the stand-in, inside this image, for the MEX gateway a MATLAB/Octave
host would use (mex/sbd_mex.c binds the same symbols).  It never computes
anything itself and never falls back to a CPU path: if the shared library is
missing, `load_library()` raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsbd.so")

SBD_N_PHASES = 8
SBD_N_GEOM = 10
SBD_NCCL_ID_BYTES = 128

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class SbdError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libsbd error {code}: {msg}")
        self.code = code
        self.msg = msg


class sbd_params(C.Structure):
    _fields_ = [
        ("samples", C.c_int32), ("warmup", C.c_int32), ("burnIn", C.c_int32), ("n_chains", C.c_int32),
        ("gam", C.c_double), ("lamb", C.c_double), ("prox_lambda", C.c_double),
        ("chambolle_maxiter", C.c_int32), ("pad0", C.c_int32),
        ("chambolle_tol", C.c_double), ("chambolle_tau", C.c_double),
        ("th_init", C.c_double), ("min_th", C.c_double), ("max_th", C.c_double), ("c_theta", C.c_double),
        ("psi_init", C.c_double * 2), ("psi_min", C.c_double * 2), ("psi_max", C.c_double * 2),
        ("c_psi", C.c_double * 2), ("psi_fixed", C.c_double * 2), ("psi_true", C.c_double * 2),
        ("fix_psi", C.c_int32 * 2),
        ("sigma2_init", C.c_double), ("sigma2_min", C.c_double), ("sigma2_max", C.c_double),
        ("c_sigma2", C.c_double), ("sigma2_fixed", C.c_double),
        ("fix_sigma", C.c_int32), ("err_psf_lag", C.c_int32),
        ("d_scale", C.c_double), ("d_exp", C.c_double),
        ("seed", C.c_uint64), ("chain_offset", C.c_int32), ("total_chains", C.c_int32),
        ("post_mean", C.c_int32), ("use_graph", C.c_int32),
    ]


TRACE_DOUBLE_FIELDS = [
    "logPiTrace_WU", "thetas", "sigmas", "psi0", "psi1", "grad_theta", "grad_psi0", "grad_psi1",
    "grad_sigma", "logPiTraceX", "gXTrace", "err_psf", "err_sample", "tol_theta", "tol_psi0",
    "tol_psi1", "tol_sigma", "mean_theta", "mean_psi0", "mean_psi1", "mean_sigma",
]


class sbd_traces(C.Structure):
    _fields_ = ([(n, c_double_p) for n in TRACE_DOUBLE_FIELDS] +
                [("chambolle_iters", C.POINTER(C.c_int32)),
                 ("X_warm", c_double_p), ("X_last", c_double_p), ("X_mean", c_double_p),
                 ("EB", C.c_double * 4), ("err_warm0", C.c_double), ("seconds", C.c_double),
                 ("seconds_main", C.c_double), ("launches_main", C.c_longlong),
                 ("last_samp", C.c_int32), ("pad1", C.c_int32)])


# name -> (restype, argtypes); mirrors include/sbd.h one to one
SIGNATURES = {
    "sbd_version": (C.c_int, []),
    "sbd_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int]),
    "sbd_destroy": (C.c_int, [C.c_void_p]),
    "sbd_last_error": (C.c_char_p, [C.c_void_p]),
    "sbd_launch_count": (C.c_longlong, [C.c_void_p]),
    "sbd_synchronize": (C.c_int, [C.c_void_p]),
    "sbd_psf_taps": (C.c_int, [C.c_void_p, c_double_p, C.c_int, c_double_p]),
    "sbd_psf_spectrum": (C.c_int, [C.c_void_p, c_double_p, C.c_int, c_double_p, c_double_p]),
    "sbd_blur": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_int, c_double_p, C.c_int]),
    "sbd_blur_dev": (C.c_int, [C.c_void_p, C.c_void_p, c_double_p, C.c_int, C.c_void_p, C.c_int]),
    "sbd_tvnorm": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_int]),
    "sbd_diff": (C.c_int, [C.c_void_p, c_double_p, C.c_int, c_double_p, C.c_int]),
    "sbd_tvprox": (C.c_int, [C.c_void_p, c_double_p, C.c_double, C.c_int, C.c_double, C.c_double,
                             c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_int_p, c_double_p, C.c_int]),
    "sbd_tvprox_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double,
                                 C.c_void_p, c_int_p, c_double_p, C.c_int]),
    "sbd_likelihood": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_double_p, C.c_double, C.c_double,
                                 c_double_p, c_double_p]),
    "sbd_max_eigenval": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_double, C.c_int, C.c_uint64,
                                   c_double_p, c_int_p]),
    "sbd_observe": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_double, c_double_p, C.c_uint64,
                              c_double_p, c_double_p, c_double_p]),
    "sbd_salsa_tv": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int,
                               c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_int_p]),
    "sbd_sapg_run": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_double_p, C.POINTER(sbd_params),
                               c_double_p, C.POINTER(sbd_traces)]),
    "sbd_sapg_run_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(sbd_params), C.POINTER(sbd_traces)]),
    "sbd_comm_unique_id": (C.c_int, [C.c_char_p]),
    "sbd_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "sbd_comm_destroy": (C.c_int, [C.c_void_p]),
    "sbd_phase_times": (C.c_int, [C.c_void_p, c_double_p, C.POINTER(C.c_longlong)]),
    "sbd_set_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "sbd_phase_name": (C.c_char_p, [C.c_int]),
    "sbd_set_posterior": (C.c_int, [C.c_void_p, C.c_int]),
    "sbd_posterior_stats": (C.c_int, [C.c_void_p, C.c_int, c_double_p, c_double_p, c_double_p, c_int_p, c_int_p]),
    "sbd_set_posterior_diagnostics": (C.c_int, [C.c_void_p, C.c_int]),
    "sbd_posterior_diagnostics": (C.c_int, [C.c_void_p, C.c_int] + [c_double_p] * 6 + [c_int_p] * 3),
    "sbd_set_posterior_quantiles": (C.c_int, [C.c_void_p, C.c_double]),
    "sbd_posterior_quantiles": (C.c_int, [C.c_void_p, C.c_int] + [c_double_p] * 4 + [C.POINTER(C.c_longlong)]),
    "sbd_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "sbd_get_geometry": (C.c_int, [C.c_void_p, C.c_int, c_int_p]),
}

_lib = None


def load_library(path=None):
    """Load libsbd.so and declare every prototype.  Raises if it is missing -
    there is deliberately no fallback implementation."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  sbd_b200 has no CPU fallback.")
    handle = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)       # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = handle
    return handle


class _LazyLib:
    def __getattr__(self, name):
        return getattr(load_library(), name)


lib = _LazyLib()
