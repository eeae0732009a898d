"""ctypes binding of libcocons_b200.so (the C ABI declared in include/cocons_b200.h).

The library is the product; this module only marshals numpy arrays to the
plain-pointer entry points an R `.Call` glue would bind (INTEGRATION.md).
There is no fallback: if the shared object is missing, or no sm_100 device is
usable, the calls raise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcocons_b200.so")

ML, PROFILE, REML = 0, 1, 2
PAR_DIFF, PAR_CLASSIC = 0, 1

ASPECTS = ("std.dev", "scale", "aniso", "tilt", "smooth", "nugget")

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_lp = ctypes.POINTER(ctypes.c_int64)
_i32p = ctypes.POINTER(ctypes.c_int32)
_i64 = ctypes.c_int64
_vp = ctypes.c_void_p

# every symbol include/cocons_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "cocons_version": (ctypes.c_int, []),
    "cocons_last_error": (ctypes.c_char_p, []),
    "cocons_device_count": (ctypes.c_int, []),
    "cocons_launch_count": (ctypes.c_longlong, []),
    "cocons_cov_rns": (ctypes.c_int, [_i64, _i64, _dp, _dp, _dp, _dp, _dp]),
    "cocons_cov_rns_pred": (ctypes.c_int, [_i64, _i64, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "cocons_cov_rns_classic": (ctypes.c_int, [_i64, _i64, _dp, _dp, _dp, _dp]),
    "cocons_sumsmoothlone": (ctypes.c_double, [_dp, _i64, ctypes.c_double, ctypes.c_double]),
    "cocons_qr_rank": (ctypes.c_int, [_dp, _i64, _i64, ctypes.c_double]),
    "cocons_ctx_create": (ctypes.c_int, [ctypes.c_int, _i64, _i64, _i64, _dp, _dp, _dp, _vp, ctypes.POINTER(_vp)]),
    "cocons_ctx_destroy": (None, [_vp]),
    "cocons_ctx_set_z": (ctypes.c_int, [_vp, _dp]),
    "cocons_ctx_set_xbetas": (ctypes.c_int, [_vp, _i64, _dp]),
    "cocons_n2ll": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _ip]),
    "cocons_ctx_create_batch": (ctypes.c_int, [ctypes.c_int, _i64, _i64, _i64, _dp, _dp, _dp, _i64, _vp,
                                               ctypes.POINTER(_vp)]),
    "cocons_n2ll_batch": (ctypes.c_int, [_vp, ctypes.c_int, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip]),
    "cocons_cov_rns_taper": (ctypes.c_int, [_i64, _i64, _dp, _dp, _dp, _dp, _i32p, _i32p, _i64, _dp]),
    "cocons_cov_rns_taper_pred": (ctypes.c_int, [_i64, _i64, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _i32p, _i32p, _i64,
                                                 _dp]),
    "cocons_ctx_set_taper": (ctypes.c_int, [_vp, _i32p, _i32p, _dp, _i64]),
    "cocons_ctx_create_taper_tiled": (ctypes.c_int, [ctypes.c_int, _i64, _i64, _i64, _dp, _dp, _dp, _i32p, _i32p, _dp,
                                                     _i64, _vp, ctypes.POINTER(_vp)]),
    "cocons_ctx_tile_stats": (ctypes.c_int, [_vp, _lp]),
    "cocons_n2ll_taper": (ctypes.c_int, [_vp, _dp, _dp, _dp, _dp, _dp]),
    "cocons_factor_taper": (ctypes.c_int, [_vp, _dp, _dp]),
    "cocons_predict_taper": (ctypes.c_int, [_vp, _i64, _dp, _dp, _i32p, _i32p, _dp, _i64, _dp, _dp, _dp]),
    "cocons_profile_betas": (ctypes.c_int, [_vp, ctypes.c_int, _dp]),
    "cocons_factor": (ctypes.c_int, [_vp, ctypes.c_int, _dp, _dp]),
    "cocons_predict": (ctypes.c_int, [_vp, _i64, _dp, _dp, _dp, _dp, _dp]),
    "cocons_sim": (ctypes.c_int, [_vp, _i64, _dp, _dp]),
    "cocons_sim_taper": (ctypes.c_int, [_vp, _i64, _dp, _dp]),
    "cocons_sim_cond": (ctypes.c_int, [_vp, _i64, _dp, _dp, _i64, _dp, _dp]),
    "cocons_ctx_get_factor": (ctypes.c_int, [_vp, _dp, _lp]),
    "cocons_ctx_factor_rows": (ctypes.c_int, [_vp, _lp, _i64, _dp, _lp]),
    "cocons_debug_solve_units": (ctypes.c_int64, [_i64, _i32p, _i64]),
    "cocons_ctx_dims": (ctypes.c_int, [_vp, _vp]),
    "cocons_ctx_timings": (ctypes.c_int, [_vp, _dp]),
    "cocons_ctx_debug_checksums": (ctypes.c_int, [_vp, _dp]),
    "cocons_ctx_kernel_timing": (ctypes.c_int, [_vp, _dp, _dp]),
    "cocons_neg2loglik_dense": (ctypes.c_int, [ctypes.c_int, _i64, _i64, _i64, _i64, _dp, _dp, _dp, _dp, _dp, _dp,
                                               _dp, _dp, _dp, _dp, _ip]),
    "cocons_release_workspace": (None, []),
    "cocons_dist_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _i64, _i64, _i64, _dp, _dp, _dp, _vp,
                                          ctypes.POINTER(_vp)]),
    "cocons_dist_destroy": (None, [_vp]),
    "cocons_dist_set_xbetas": (ctypes.c_int, [_vp, _i64, _dp]),
    "cocons_dist_npanels": (_i64, [_vp]),
    "cocons_dist_npad": (_i64, [_vp]),
    "cocons_dist_panel_elems": (_i64, [_vp, _i64]),
    "cocons_dist_assemble": (ctypes.c_int, [_vp, _dp, _dp, _dp]),
    "cocons_dist_side_stream": (_vp, [_vp]),
    "cocons_dist_factor_panel": (ctypes.c_int, [_vp, _i64, ctypes.c_int]),
    "cocons_dist_pack_panel": (ctypes.c_int, [_vp, _i64, _vp, ctypes.c_int]),
    "cocons_dist_update": (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64]),
    "cocons_dist_fill_rhs": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _ip]),
    "cocons_dist_solve_block": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, ctypes.c_int]),
    "cocons_dist_reduce_local": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp]),
    "cocons_dist_perm": (ctypes.c_int, [_vp, _lp]),
    "cocons_bench_syrk": (ctypes.c_int, [ctypes.c_int, _i64, _i64, ctypes.c_int, _dp]),
    "cocons_trailing_update": (ctypes.c_int, [ctypes.c_int, _i64, _dp, _dp, ctypes.c_int, ctypes.c_int, _dp]),
}

_lib = None


class CoconsError(RuntimeError):
    """A negative status from the C ABI (CUDA / argument / state error)."""


class NotPositiveDefinite(ArithmeticError):
    """Status k > 0: the leading minor of order k is not positive definite."""

    def __init__(self, k):
        super().__init__("the leading minor of order %d is not positive definite" % k)
        self.k = k


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CoconsError(
                "%s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(cocons_b200 has no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def check(status):
    if status < 0:
        raise CoconsError("cocons_b200 error %d: %s" % (status, lib().cocons_last_error().decode()))
    if status > 0:
        raise NotPositiveDefinite(status)


def fmat(a, rows=None):
    """float64, column-major copy/view of a vector or matrix (R's storage)."""
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 1:
        a = a.reshape(-1, 1) if rows is None else a.reshape(rows, -1)
    return np.asfortranarray(a)


def ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def iptr(a):
    return a.ctypes.data_as(_i32p)


def pack_theta(theta, p):
    """Named list of aspect vectors -> (6, p) block in ASPECTS order; lookup by name,
    extra names (e.g. "mean") ignored, missing ones an error (src/cocons_full.cpp:47-54)."""
    rows = []
    for name in ASPECTS:
        if name not in theta:
            raise KeyError("Index out of bounds: [index='%s']." % name)
        v = np.atleast_1d(np.asarray(theta[name], dtype=np.float64))
        if v.shape[0] != p:
            raise ValueError("theta$%s has length %d, expected %d" % (name, v.shape[0], p))
        rows.append(v)
    return np.ascontiguousarray(np.stack(rows))
