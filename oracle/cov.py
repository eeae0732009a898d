"""TEST INFRASTRUCTURE ONLY (oracle/): ctypes access to the CPU checkers.

Two libraries, same call shapes:
  * ``restatement`` - oracle/liboracle.so, built from oracle/cov_oracle.cpp
    (plain-array restatement of src/cocons_full.cpp:40-594 and src/cocons_taper.cpp:17-433);
  * ``reference``   - oracle/_ref/libcocons_ref.so, the reference's own
    src/cocons_full.cpp and src/cocons_taper.cpp compiled against the Rcpp/BH stand-ins (oracle/shim/).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import
this module.  Matrices are numpy float64, column-major (Fortran order), as R
holds them.
"""
import ctypes
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ASPECTS = ("std.dev", "scale", "aniso", "tilt", "smooth", "nugget")


def _reference_path():
    """Source tree of the reference R package (cocons 0.1.5), which this repository does not ship: $COCONS_REFERENCE,
    else BASELINE.json's reference_path.  oracle/Makefile asks this module for it."""
    if os.environ.get("COCONS_REFERENCE"):
        return os.environ["COCONS_REFERENCE"]
    with open(os.path.join(os.path.dirname(_HERE), "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


REFERENCE = _reference_path()

_dp = ctypes.POINTER(ctypes.c_double)
_libs = {}


def _reference_source_present():
    return os.path.exists(os.path.join(REFERENCE, "src", "cocons_full.cpp"))


def build(force=False):
    """Compile liboracle.so (and _ref when REFERENCE holds the reference's source)."""
    so = os.path.join(_HERE, "liboracle.so")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(_HERE, "cov_oracle.cpp")):
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle.so"])
    ref = os.path.join(_HERE, "_ref", "libcocons_ref.so")
    if _reference_source_present() and (force or not os.path.exists(ref)):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref", "REFERENCE=" + REFERENCE])


def _load(kind):
    if kind in _libs:
        return _libs[kind]
    if kind == "restatement":
        build()
        path, prefix = os.path.join(_HERE, "liboracle.so"), "oracle_"
    elif kind == "reference":
        path, prefix = os.path.join(_HERE, "_ref", "libcocons_ref.so"), "ref_"
        if not os.path.exists(path):
            build()
    else:
        raise ValueError(kind)
    lib = ctypes.CDLL(path)
    L = ctypes.c_long
    f = getattr(lib, prefix + "cov_rns")
    f.argtypes, f.restype = [L, L, _dp, _dp, _dp, _dp, _dp], ctypes.c_int
    f = getattr(lib, prefix + "cov_rns_pred")
    f.argtypes, f.restype = [L, L, L, _dp, _dp, _dp, _dp, _dp, _dp, _dp], ctypes.c_int
    f = getattr(lib, prefix + "cov_rns_classic")
    f.argtypes, f.restype = [L, L, _dp, _dp, _dp, _dp], ctypes.c_int
    f = getattr(lib, prefix + "sumsmoothlone")
    f.argtypes, f.restype = [_dp, L, ctypes.c_double, ctypes.c_double], ctypes.c_double
    f = getattr(lib, prefix + "cov_rns_taper")
    f.argtypes, f.restype = [L, L, _dp, _dp, _dp, _dp, _dp, _dp, L, _dp], ctypes.c_int
    f = getattr(lib, prefix + "cov_rns_taper_pred")
    f.argtypes, f.restype = [L, L, L, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, L, _dp], ctypes.c_int
    if kind == "restatement":
        lib.oracle_bessel_k.argtypes, lib.oracle_bessel_k.restype = [ctypes.c_double, ctypes.c_double], ctypes.c_double
    _libs[kind] = (lib, prefix)
    return _libs[kind]


def have_reference():
    return os.path.exists(os.path.join(_HERE, "_ref", "libcocons_ref.so")) or _reference_source_present()


def _f(a):
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def _p(a):
    return a.ctypes.data_as(_dp)


def pack_theta(theta, p=None):
    """R named list (dict) of aspect vectors -> (6, p) C-contiguous block in ASPECTS order.

    Lookup is by name and extra entries such as "mean" are ignored, as in
    src/cocons_full.cpp:47-54; a missing aspect is an error.
    """
    rows = []
    for name in ASPECTS:
        if name not in theta:
            raise KeyError("theta has no element named '%s'" % name)
        rows.append(np.atleast_1d(np.asarray(theta[name], dtype=np.float64)))
    p = p or len(rows[0])
    return np.ascontiguousarray(np.stack([r.reshape(p) for r in rows]))


def cov_rns(theta, locs, x_covariates, smooth_limits, kind="restatement"):
    lib, pre = _load(kind)
    locs, X = _f(locs), _f(x_covariates)
    n, p = X.shape
    th, lim = pack_theta(theta, p), _f(smooth_limits)
    out = np.empty((n, n), order="F")
    rc = getattr(lib, pre + "cov_rns")(n, p, _p(locs), _p(X), _p(th), _p(lim), _p(out))
    assert rc == 0
    return out


def cov_rns_pred(theta, locs, locs_pred, x_covariates, x_covariates_pred, smooth_limits, kind="restatement"):
    lib, pre = _load(kind)
    locs, lp, X, Xp = _f(locs), _f(locs_pred), _f(x_covariates), _f(x_covariates_pred)
    n, p = X.shape
    m = Xp.shape[0]
    th, lim = pack_theta(theta, p), _f(smooth_limits)
    out = np.empty((m, n), order="F")
    rc = getattr(lib, pre + "cov_rns_pred")(n, m, p, _p(locs), _p(lp), _p(X), _p(Xp), _p(th), _p(lim), _p(out))
    assert rc == 0
    return out


def cov_rns_classic(theta, locs, x_covariates, kind="restatement"):
    lib, pre = _load(kind)
    locs, X = _f(locs), _f(x_covariates)
    n, p = X.shape
    th = pack_theta(theta, p)
    out = np.empty((n, n), order="F")
    rc = getattr(lib, pre + "cov_rns_classic")(n, p, _p(locs), _p(X), _p(th), _p(out))
    assert rc == 0
    return out


def cov_rns_taper(theta, locs, x_covariates, colindices, rowpointers, smooth_limits, kind="restatement"):
    """src/cocons_taper.cpp:151-433; colindices / rowpointers are spam's 1-based CSR slots."""
    lib, pre = _load(kind)
    locs, X = _f(locs), _f(x_covariates)
    n, p = X.shape
    th, lim = pack_theta(theta, p), _f(smooth_limits)
    ci, rp = _f(colindices), _f(rowpointers)
    assert len(rp) == n + 1 and int(rp[-1]) - 1 == len(ci)
    out = np.empty(len(ci))
    rc = getattr(lib, pre + "cov_rns_taper")(n, p, _p(locs), _p(X), _p(th), _p(lim), _p(ci), _p(rp), len(ci), _p(out))
    assert rc == 0
    return out


def cov_rns_taper_pred(theta, locs, locs_pred, x_covariates, x_covariates_pred, colindices, rowpointers,
                       smooth_limits, kind="restatement"):
    """src/cocons_taper.cpp:17-139; the pattern's rows are the prediction sites."""
    lib, pre = _load(kind)
    locs, lp, X, Xp = _f(locs), _f(locs_pred), _f(x_covariates), _f(x_covariates_pred)
    n, p = X.shape
    m = Xp.shape[0]
    th, lim = pack_theta(theta, p), _f(smooth_limits)
    ci, rp = _f(colindices), _f(rowpointers)
    assert len(rp) == m + 1 and int(rp[-1]) - 1 == len(ci)
    out = np.empty(len(ci))
    rc = getattr(lib, pre + "cov_rns_taper_pred")(n, m, p, _p(locs), _p(lp), _p(X), _p(Xp), _p(th), _p(lim), _p(ci),
                                                  _p(rp), len(ci), _p(out))
    assert rc == 0
    return out


def sumsmoothlone(x, lam, alpha=1e6, kind="restatement"):
    lib, pre = _load(kind)
    x = np.ascontiguousarray(np.atleast_1d(np.asarray(x, dtype=np.float64)))
    return getattr(lib, pre + "sumsmoothlone")(_p(x), len(x), float(lam), float(alpha))


def bessel_k(nu, x):
    lib, _ = _load("restatement")
    return lib.oracle_bessel_k(float(nu), float(x))
