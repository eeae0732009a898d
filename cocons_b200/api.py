"""Host-side mirror of the reference's R interface for the dense-likelihood path.

The reference's host language is R, which is not installed here; the R glue a
maintainer would drop into the package is in cocons_b200/rglue/ (see
INTEGRATION.md).  This module offers the same functions, names and argument
order in Python on top of the same C ABI so that the path can be driven and
tested without R.  Everything numeric of order n^2 or n^3 happens in
libcocons_b200.so on the GPU; what stays here is what stays in R in the
reference: parameter packing (getModelLists), standardisation (getScale), the
penalty (.cocons.getPen), the `safe`/1e6 logic and the n log(2 pi) constant.

Reference lines are cited per function.  R lists become dicts, formulas become
strings such as "~ 1 + cov_x + cov_y", data.frames become dicts of columns (or
pandas DataFrames).
"""
import copy

import numpy as np

from . import _lib
from ._lib import NotPositiveDefinite, CoconsError  # noqa: F401  (re-exported)

DICTIONARY = ("mean", "std.dev", "scale", "aniso", "tilt", "smooth", "nugget")  # R/profile.R:5-7


# --------------------------------------------------------------------------
# FFI-level functions (R/RcppExports.R:10-46)
# --------------------------------------------------------------------------
def sumsmoothlone(x, lambda_, alpha=1e6):
    """R/RcppExports.R:10-12 -> src/cocons_full.cpp:12-30."""
    x = np.ascontiguousarray(np.atleast_1d(np.asarray(x, dtype=np.float64)))
    return _lib.lib().cocons_sumsmoothlone(_lib.ptr(x), x.shape[0], float(lambda_), float(alpha))


def cov_rns(theta, locs, x_covariates, smooth_limits):
    """R/RcppExports.R:21-23 -> src/cocons_full.cpp:40-321.  Returns the n x n matrix."""
    locs, X = _lib.fmat(locs), _lib.fmat(x_covariates)
    n, p = X.shape
    th = _lib.pack_theta(theta, p)
    lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
    out = np.empty((n, n), order="F")
    _lib.check(_lib.lib().cocons_cov_rns(n, p, _lib.ptr(locs), _lib.ptr(X), _lib.ptr(th), _lib.ptr(lim),
                                         _lib.ptr(out)))
    return out


def cov_rns_pred(theta, locs, locs_pred, x_covariates, x_covariates_pred, smooth_limits):
    """R/RcppExports.R:34-36 -> src/cocons_full.cpp:334-471.  Returns m x n (prediction sites are rows)."""
    locs, lp = _lib.fmat(locs), _lib.fmat(locs_pred)
    X, Xp = _lib.fmat(x_covariates), _lib.fmat(x_covariates_pred)
    n, p = X.shape
    m = Xp.shape[0]
    th = _lib.pack_theta(theta, p)
    lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
    out = np.empty((m, n), order="F")
    _lib.check(_lib.lib().cocons_cov_rns_pred(n, m, p, _lib.ptr(locs), _lib.ptr(lp), _lib.ptr(X), _lib.ptr(Xp),
                                              _lib.ptr(th), _lib.ptr(lim), _lib.ptr(out)))
    return out


def cov_rns_classic(theta, locs, x_covariates):
    """R/RcppExports.R:44-46 -> src/cocons_full.cpp:480-594."""
    locs, X = _lib.fmat(locs), _lib.fmat(x_covariates)
    n, p = X.shape
    th = _lib.pack_theta(theta, p)
    out = np.empty((n, n), order="F")
    _lib.check(_lib.lib().cocons_cov_rns_classic(n, p, _lib.ptr(locs), _lib.ptr(X), _lib.ptr(th), _lib.ptr(out)))
    return out


def _pattern(colindices, rowpointers):
    """spam's 1-based CSR slots as contiguous int32 (what INTEGER() of the slots points at)."""
    ci = np.ascontiguousarray(np.asarray(colindices).astype(np.int32, copy=False))
    rp = np.ascontiguousarray(np.asarray(rowpointers).astype(np.int32, copy=False))
    return ci, rp


def cov_rns_taper(theta, locs, x_covariates, colindices, rowpointers, smooth_limits):
    """R/RcppExports.R:72-74 -> src/cocons_taper.cpp:151-433.  Returns the covariance entries on the pattern."""
    locs, X = _lib.fmat(locs), _lib.fmat(x_covariates)
    n, p = X.shape
    th = _lib.pack_theta(theta, p)
    lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
    ci, rp = _pattern(colindices, rowpointers)
    out = np.empty(ci.shape[0])
    _lib.check(_lib.lib().cocons_cov_rns_taper(n, p, _lib.ptr(locs), _lib.ptr(X), _lib.ptr(th), _lib.ptr(lim),
                                               _lib.iptr(ci), _lib.iptr(rp), ci.shape[0], _lib.ptr(out)))
    return out


def cov_rns_taper_pred(theta, locs, locs_pred, x_covariates, x_covariates_pred, colindices, rowpointers,
                       smooth_limits):
    """R/RcppExports.R:59-61 -> src/cocons_taper.cpp:17-139.  The pattern's rows are the prediction sites."""
    locs, lp = _lib.fmat(locs), _lib.fmat(locs_pred)
    X, Xp = _lib.fmat(x_covariates), _lib.fmat(x_covariates_pred)
    n, p = X.shape
    m = Xp.shape[0]
    th = _lib.pack_theta(theta, p)
    lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
    ci, rp = _pattern(colindices, rowpointers)
    out = np.empty(ci.shape[0])
    _lib.check(_lib.lib().cocons_cov_rns_taper_pred(n, m, p, _lib.ptr(locs), _lib.ptr(lp), _lib.ptr(X), _lib.ptr(Xp),
                                                    _lib.ptr(th), _lib.ptr(lim), _lib.iptr(ci), _lib.iptr(rp),
                                                    ci.shape[0], _lib.ptr(out)))
    return out


# --------------------------------------------------------------------------
# the pieces of `spam` the sparse path touches (third-party in the reference:
# spam >= 2.9.1, DESCRIPTION:21; absent here, restated from its documentation)
# --------------------------------------------------------------------------
class spam:
    """The slots of a spam matrix the path reads: `entries`, 1-based `colindices` / `rowpointers`
    (CSR, columns ascending within a row) and `dimension`."""

    def __init__(self, entries, colindices, rowpointers, dimension):
        self.entries = np.ascontiguousarray(np.asarray(entries, dtype=np.float64))
        self.colindices, self.rowpointers = _pattern(colindices, rowpointers)
        self.dimension = (int(dimension[0]), int(dimension[1]))

    def copy(self):
        return spam(self.entries.copy(), self.colindices, self.rowpointers, self.dimension)

    def density(self):
        return self.entries.shape[0] / (self.dimension[0] * self.dimension[1])

    def toarray(self):
        out = np.zeros(self.dimension)
        rows = np.repeat(np.arange(self.dimension[0]), np.diff(self.rowpointers))
        out[rows, self.colindices - 1] = self.entries
        return out


def nearest_dist(x, y=None, delta=1.0, upper=None):
    """spam::nearest.dist(x, y, method = "euclidean", delta, upper = NULL) as the reference calls it
    (R/optim.R:377, R/predict.R:219,233): the Euclidean distances not exceeding `delta`, rows = sites
    of x, columns = sites of y (or x).  Coincident pairs and the diagonal are kept - the reference's
    pair loop expects them (`ii == jj`, src/cocons_taper.cpp:227; coordinate equality, :89)."""
    from scipy.spatial import cKDTree

    if upper is not None:
        raise NotImplementedError("only upper = NULL (the whole matrix) is used on this path")
    x = np.asarray(x, dtype=np.float64)
    yy = x if y is None else np.asarray(y, dtype=np.float64)
    tx = cKDTree(x)
    ty = tx if y is None else cKDTree(yy)
    trip = tx.sparse_distance_matrix(ty, float(delta), output_type="ndarray")
    order = np.lexsort((trip["j"], trip["i"]))
    i, j, v = trip["i"][order], trip["j"][order], trip["v"][order]
    rowpointers = np.concatenate([[0], np.cumsum(np.bincount(i, minlength=x.shape[0]))]) + 1
    return spam(v, j + 1, rowpointers, (x.shape[0], yy.shape[0]))


def _apply_on_entries(h, fun):
    if isinstance(h, spam):
        return spam(fun(h.entries), h.colindices, h.rowpointers, h.dimension)
    return fun(np.asarray(h, dtype=np.float64))


def cov_wend1(h, theta):
    """spam::cov.wend1: theta = c(range, sill[, nugget]); sill (1 - d)^4_+ (1 + 4 d), d = h / range."""
    rng, sill = float(theta[0]), float(theta[1]) if len(theta) > 1 else 1.0

    def f(d):
        d = d / rng
        return sill * np.where(d < 1, (1 - d) ** 4 * (1 + 4 * d), 0.0)
    return _apply_on_entries(h, f)


def cov_wend2(h, theta):
    """spam::cov.wend2: sill (1 - d)^6_+ (1 + 6 d + 35 d^2 / 3), d = h / range."""
    rng, sill = float(theta[0]), float(theta[1]) if len(theta) > 1 else 1.0

    def f(d):
        d = d / rng
        return sill * np.where(d < 1, (1 - d) ** 6 * (1 + 6 * d + 35 * d * d / 3), 0.0)
    return _apply_on_entries(h, f)


# --------------------------------------------------------------------------
# parameter packing that stays on the host (R/getFunctions.R)
# --------------------------------------------------------------------------
def is_formula(x):
    """R/isFunctions.R:10-12."""
    return isinstance(x, str) and x.strip().startswith("~")


def _terms(formula):
    rhs = formula.strip()[1:]
    intercept, labels = True, []
    for tok in rhs.replace("-", "+-").split("+"):
        tok = tok.strip()
        if tok in ("", "1"):
            continue
        if tok in ("0", "-1"):
            intercept = False
            continue
        labels.append(tok)
    return intercept, labels


def _columns(data):
    if hasattr(data, "columns") and hasattr(data, "__getitem__") and not isinstance(data, dict):
        return {c: np.asarray(data[c], dtype=np.float64) for c in data.columns}
    return {k: np.asarray(v, dtype=np.float64) for k, v in data.items()}


def getDesignMatrix(model_list, data):
    """R/getFunctions.R:450-555 for main-effect formulas: the union model matrix (intercept +
    covariates in order of first appearance) and, per aspect, a logical index (free) or the
    fixed value."""
    cols = _columns(data)
    n = len(next(iter(cols.values())))
    formulas = [(k, v) for k, v in model_list.items() if is_formula(v)]
    if not formulas:
        raise ValueError("No formula detected")
    labels, any_intercept = [], False
    for _, f in formulas:
        ic, ls = _terms(f)
        any_intercept = any_intercept or ic
        for l in ls:
            if l not in labels:
                labels.append(l)
    names = (["(Intercept)"] if (any_intercept or not labels) else []) + labels
    mm = np.empty((n, len(names)), order="F")
    for j, nm in enumerate(names):
        mm[:, j] = 1.0 if nm == "(Intercept)" else cols[nm]
    par_pos = {}
    for k, v in model_list.items():
        if not is_formula(v):
            par_pos[k] = float(np.atleast_1d(v)[0])
            continue
        ic, ls = _terms(v)
        pos = np.array([nm in ls for nm in names], dtype=bool)
        if ic and names[0] == "(Intercept)":
            pos[0] = True
        par_pos[k] = pos
    return {"model.matrix": mm, "par.pos": par_pos, "colnames": names}


def getScale(x, mean_vector=None, sd_vector=None):
    """R/getFunctions.R:376-436: centre and scale columns 2..p (sd with n-1); column 1 untouched."""
    if isinstance(x, coco):
        x = getDesignMatrix(x.model_list, x.data)["model.matrix"]
    x = np.array(x, dtype=np.float64, order="F", copy=True)
    if mean_vector is None:
        mean_vector = x.mean(axis=0)
        mean_vector[0] = 0.0
    if sd_vector is None:
        sd_vector = x.std(axis=0, ddof=1)
        sd_vector[0] = 1.0
    for k in range(1, x.shape[1]):
        x[:, k] = (x[:, k] - mean_vector[k]) / sd_vector[k]
    return {"std.covs": x, "mean.vector": np.asarray(mean_vector), "sd.vector": np.asarray(sd_vector)}


def getModelLists(theta, par_pos, type="diff"):
    """R/getFunctions.R:570-616: theta vector -> one length-p vector per aspect; fixed aspects put
    their constant in slot 1; with type "diff", where std.dev and scale are both free at column k,
    std.dev_k = (a+b)/2 and scale_k = (a-b)/2."""
    theta = np.atleast_1d(np.asarray(theta, dtype=np.float64))
    free = {k: isinstance(v, np.ndarray) and v.dtype == bool for k, v in par_pos.items()}
    length = max((len(v) if free[k] else 1) for k, v in par_pos.items())
    pars, used = {}, 0
    for name, pos in par_pos.items():
        vec = np.zeros(length)
        if free[name]:
            k = int(pos.sum())
            vec[np.flatnonzero(pos)] = theta[used:used + k]
            used += k
        else:
            vec[0] = float(np.atleast_1d(pos)[0])
        pars[name] = vec
    if type == "classic":
        return pars
    out = {k: v.copy() for k, v in pars.items()}
    if free.get("std.dev") and free.get("scale"):
        both = par_pos["std.dev"] & par_pos["scale"]
        out["std.dev"][both] = (pars["std.dev"][both] + pars["scale"][both]) / 2
        out["scale"][both] = (pars["std.dev"][both] - pars["scale"][both]) / 2
    return out


def _getPen(n, lambda_, theta_list, smooth_limits):
    """.cocons.getPen, R/checkFunctions.R:474-492."""
    names = list(theta_list.keys())
    summ = lambda_[2] * np.exp(theta_list["scale"][0]) * np.sqrt(
        (smooth_limits[1] - smooth_limits[0]) / (1 + np.exp(-theta_list["smooth"][0])) + smooth_limits[0]
    ) + sumsmoothlone(theta_list[names[0]][1:], lambda_[1])
    for ii in range(1, 6):
        summ = summ + sumsmoothlone(theta_list[names[ii]][1:], lambda_[0])
    return 2 * n * summ


# --------------------------------------------------------------------------
# device-resident likelihood context
# --------------------------------------------------------------------------
class DenseLikelihood:
    """locs / x_covariates / z resident on one GPU; evaluates the three objectives and keeps the
    Cholesky factor for prediction and simulation.  Wraps cocons_ctx_* (include/cocons_b200.h)."""

    def __init__(self, locs, x_covariates, z, device=0, stream=None):
        self.locs, self.X = _lib.fmat(locs), _lib.fmat(x_covariates)
        self.n, self.p = self.X.shape
        self.z = _lib.fmat(z, rows=self.n)
        self.r = self.z.shape[1]
        self._h = _lib._vp()
        _lib.check(_lib.lib().cocons_ctx_create(int(device), self.n, self.p, self.r, _lib.ptr(self.locs),
                                                _lib.ptr(self.X), _lib.ptr(self.z), stream, self._h))
        self.q = 0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().cocons_ctx_destroy(self._h)
            self._h = _lib._vp()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_z(self, z):
        z = _lib.fmat(z, rows=self.n)
        assert z.shape == (self.n, self.r)
        _lib.check(_lib.lib().cocons_ctx_set_z(self._h, _lib.ptr(z)))

    def set_xbetas(self, x_betas):
        xb = _lib.fmat(x_betas, rows=self.n)
        self.q = xb.shape[1]
        _lib.check(_lib.lib().cocons_ctx_set_xbetas(self._h, self.q, _lib.ptr(xb)))

    def terms(self, kind, theta_list, smooth_limits, mean=None):
        """One evaluation; returns dict(logdet, quad[r], logdet_w, rank).  Raises NotPositiveDefinite."""
        th = _lib.pack_theta(theta_list, self.p)
        lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
        mean_v = None if mean is None else np.ascontiguousarray(np.asarray(mean, dtype=np.float64))
        logdet, ldw = _lib.ctypes.c_double(), _lib.ctypes.c_double()
        rank = _lib.ctypes.c_int()
        quad = np.empty(self.r)
        _lib.check(_lib.lib().cocons_n2ll(self._h, int(kind), _lib.ptr(th), _lib.ptr(lim), _lib.ptr(mean_v),
                                          _lib.ctypes.byref(logdet), _lib.ptr(quad), _lib.ctypes.byref(ldw),
                                          _lib.ctypes.byref(rank)))
        return {"logdet": logdet.value, "quad": quad, "logdet_w": ldw.value, "rank": rank.value}

    def set_taper(self, ref_taper):
        """Attach the taper of a sparse coco object (a `spam`: pattern + taper values, R/optim.R:376-379)."""
        assert ref_taper.dimension == (self.n, self.n)
        _lib.check(_lib.lib().cocons_ctx_set_taper(self._h, _lib.iptr(ref_taper.colindices),
                                                   _lib.iptr(ref_taper.rowpointers), _lib.ptr(ref_taper.entries),
                                                   ref_taper.entries.shape[0]))

    def terms_taper(self, theta_list, smooth_limits, mean=None):
        """One evaluation of the tapered model; returns dict(logdet, quad[r])."""
        th = _lib.pack_theta(theta_list, self.p)
        lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
        mean_v = None if mean is None else np.ascontiguousarray(np.asarray(mean, dtype=np.float64))
        logdet = _lib.ctypes.c_double()
        quad = np.empty(self.r)
        _lib.check(_lib.lib().cocons_n2ll_taper(self._h, _lib.ptr(th), _lib.ptr(lim), _lib.ptr(mean_v),
                                                _lib.ctypes.byref(logdet), _lib.ptr(quad)))
        return {"logdet": logdet.value, "quad": quad}

    def factor_taper(self, theta_list, smooth_limits):
        th = _lib.pack_theta(theta_list, self.p)
        lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
        _lib.check(_lib.lib().cocons_factor_taper(self._h, _lib.ptr(th), _lib.ptr(lim)))

    def predict_taper(self, locs_pred, x_covariates_pred, pred_taper, resid, want_explained=True):
        """`pred_taper`: the taper on the prediction pattern (m x n `spam`), before the covariance is multiplied in."""
        lp, Xp = _lib.fmat(locs_pred), _lib.fmat(x_covariates_pred)
        m = Xp.shape[0]
        assert pred_taper.dimension == (m, self.n)
        resid = np.ascontiguousarray(np.asarray(resid, dtype=np.float64))
        sto = np.empty(m)
        expl = np.empty(m) if want_explained else None
        _lib.check(_lib.lib().cocons_predict_taper(self._h, m, _lib.ptr(lp), _lib.ptr(Xp),
                                                   _lib.iptr(pred_taper.colindices), _lib.iptr(pred_taper.rowpointers),
                                                   _lib.ptr(pred_taper.entries), pred_taper.entries.shape[0],
                                                   _lib.ptr(resid), _lib.ptr(sto), _lib.ptr(expl)))
        return sto, expl

    def profile_betas(self, kind):
        k = self.q if kind == _lib.PROFILE else self.p
        out = np.empty(k)
        _lib.check(_lib.lib().cocons_profile_betas(self._h, int(kind), _lib.ptr(out)))
        return out

    def factor(self, theta_list, smooth_limits=None, type="diff"):
        th = _lib.pack_theta(theta_list, self.p)
        lim = None if smooth_limits is None else np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
        par = _lib.PAR_CLASSIC if type == "classic" else _lib.PAR_DIFF
        _lib.check(_lib.lib().cocons_factor(self._h, par, _lib.ptr(th), _lib.ptr(lim)))

    def predict(self, locs_pred, x_covariates_pred, resid, want_explained=True):
        lp, Xp = _lib.fmat(locs_pred), _lib.fmat(x_covariates_pred)
        m = Xp.shape[0]
        resid = np.ascontiguousarray(np.asarray(resid, dtype=np.float64))
        sto = np.empty(m)
        expl = np.empty(m) if want_explained else None
        _lib.check(_lib.lib().cocons_predict(self._h, m, _lib.ptr(lp), _lib.ptr(Xp), _lib.ptr(resid), _lib.ptr(sto),
                                             _lib.ptr(expl)))
        return sto, expl

    def sim(self, eps):
        eps = _lib.fmat(eps, rows=self.n)
        out = np.empty_like(eps, order="F")
        _lib.check(_lib.lib().cocons_sim(self._h, eps.shape[1], _lib.ptr(eps), _lib.ptr(out)))
        return out

    def sim_taper(self, eps):
        """L eps with the tapered factor kept by factor_taper / terms_taper (cocons_sim_taper); on a dense context
        the same bits as sim()."""
        eps = _lib.fmat(eps, rows=self.n)
        out = np.empty_like(eps, order="F")
        _lib.check(_lib.lib().cocons_sim_taper(self._h, eps.shape[1], _lib.ptr(eps), _lib.ptr(out)))
        return out

    def sim_cond(self, locs_pred, x_covariates_pred, eps):
        lp, Xp = _lib.fmat(locs_pred), _lib.fmat(x_covariates_pred)
        m = Xp.shape[0]
        eps = _lib.fmat(eps, rows=m)
        out = np.empty_like(eps, order="F")
        _lib.check(_lib.lib().cocons_sim_cond(self._h, m, _lib.ptr(lp), _lib.ptr(Xp), eps.shape[1], _lib.ptr(eps),
                                              _lib.ptr(out)))
        return out

    def get_factor(self):
        L = np.empty((self.n, self.n), order="F")
        perm = np.empty(self.n, dtype=np.int64)
        _lib.check(_lib.lib().cocons_ctx_get_factor(self._h, _lib.ptr(L), perm.ctypes.data_as(_lib._lp)))
        return L, perm

    def factor_rows(self, sites):
        """Rows of the kept factor for the given caller-order sites: (rows [m x n], pos [m]); the covariance of
        sites a, b is rows[a] @ rows[b] (see cocons_ctx_factor_rows)."""
        sites = np.ascontiguousarray(np.asarray(sites, dtype=np.int64))
        rows = np.empty((len(sites), self.n))
        pos = np.empty(len(sites), dtype=np.int64)
        _lib.check(_lib.lib().cocons_ctx_factor_rows(self._h, sites.ctypes.data_as(_lib._lp), len(sites),
                                                     _lib.ptr(rows), pos.ctypes.data_as(_lib._lp)))
        return rows, pos

    def timings(self):
        ms = np.empty(4)
        _lib.lib().cocons_ctx_timings(self._h, _lib.ptr(ms))
        kms, kfl = _lib.ctypes.c_double(), _lib.ctypes.c_double()
        _lib.lib().cocons_ctx_kernel_timing(self._h, _lib.ctypes.byref(kms), _lib.ctypes.byref(kfl))
        return {"assembly_ms": ms[0], "factor_ms": ms[1], "solve_ms": ms[2], "total_ms": ms[3],
                "kernel_ms": kms.value, "kernel_flops": kfl.value}


class DenseLikelihoodBatch:
    """`batch` matrices over the same data on one GPU (cocons_ctx_create_batch): terms_batch evaluates many points per
    call, up to `batch` of them with one launch per step of the assembly and the factorisation.  Each point's terms are
    bit for bit those of DenseLikelihood.terms.  For n_pad = ceil(n / 128) * 128 < 16 384 only (CoconsError above)."""

    def __init__(self, locs, x_covariates, z, batch, device=0, stream=None):
        self.locs, self.X = _lib.fmat(locs), _lib.fmat(x_covariates)
        self.n, self.p = self.X.shape
        self.z = _lib.fmat(z, rows=self.n)
        self.r = self.z.shape[1]
        self.batch = int(batch)
        self._h = _lib._vp()
        _lib.check(_lib.lib().cocons_ctx_create_batch(int(device), self.n, self.p, self.r, _lib.ptr(self.locs),
                                                      _lib.ptr(self.X), _lib.ptr(self.z), self.batch, stream, self._h))
        self.q = 0

    close = DenseLikelihood.close
    __del__ = close
    __enter__ = DenseLikelihood.__enter__
    __exit__ = DenseLikelihood.__exit__
    set_z = DenseLikelihood.set_z
    set_xbetas = DenseLikelihood.set_xbetas

    def terms_batch(self, kind, theta_lists, smooth_limits, means=None):
        """[terms of point i] for the named theta lists: per point the dict DenseLikelihood.terms returns, or that
        point's NotPositiveDefinite (returned, not raised).  `means`: one mean vector per point, or None."""
        k = len(theta_lists)
        th = np.asfortranarray(np.stack([_lib.pack_theta(t, self.p).reshape(-1) for t in theta_lists], axis=1))
        lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
        mean_m = None if means is None else np.asfortranarray(
            np.stack([np.asarray(m, dtype=np.float64).reshape(self.p) for m in means], axis=1))
        logdet, ldw = np.zeros(k), np.zeros(k)
        quad = np.zeros((self.r, k), order="F")
        rank = _lib.ctypes.c_int()
        status = np.zeros(k, dtype=np.int32)
        _lib.check(_lib.lib().cocons_n2ll_batch(self._h, int(kind), k, _lib.ptr(th), _lib.ptr(lim), _lib.ptr(mean_m),
                                                _lib.ptr(logdet), _lib.ptr(quad), _lib.ptr(ldw),
                                                _lib.ctypes.byref(rank),
                                                status.ctypes.data_as(_lib.ctypes.POINTER(_lib.ctypes.c_int))))
        out = []
        for i in range(k):
            if status[i] > 0:
                out.append(NotPositiveDefinite(int(status[i])))
            else:
                _lib.check(int(status[i]))
                out.append({"logdet": float(logdet[i]), "quad": quad[:, i].copy(), "logdet_w": float(ldw[i]),
                            "rank": rank.value})
        return out

    def timings(self):
        """phase times of the last terms_batch call, added up over its groups of `batch` points"""
        ms = np.empty(4)
        _lib.check(_lib.lib().cocons_ctx_timings(self._h, _lib.ptr(ms)))
        return {"assembly_ms": ms[0], "factor_ms": ms[1], "solve_ms": ms[2], "total_ms": ms[3]}


class TaperedLikelihood(DenseLikelihood):
    """A context for the tapered model only (cocons_ctx_create_taper_tiled): the pattern of `ref_taper` (a `spam`,
    n x n) is fixed at creation and only the tiles of the Cholesky factor that can be nonzero are stored on the
    device - so n is bounded by the factor's fill, not by n^2.  terms_taper / factor_taper / predict_taper /
    sim_taper / get_factor / factor_rows / set_z / timings work as on a DenseLikelihood (and so do
    GetNeg2loglikelihoodTaper{,Profile} with ctx=); the dense objectives, set_taper, predict, sim and sim_cond raise
    CoconsError.  At most 128 columns of z."""

    def __init__(self, locs, x_covariates, z, ref_taper, device=0, stream=None):
        self.locs, self.X = _lib.fmat(locs), _lib.fmat(x_covariates)
        self.n, self.p = self.X.shape
        self.z = _lib.fmat(z, rows=self.n)
        self.r = self.z.shape[1]
        assert ref_taper.dimension == (self.n, self.n)
        self._h = _lib._vp()
        _lib.check(_lib.lib().cocons_ctx_create_taper_tiled(
            int(device), self.n, self.p, self.r, _lib.ptr(self.locs), _lib.ptr(self.X), _lib.ptr(self.z),
            _lib.iptr(ref_taper.colindices), _lib.iptr(ref_taper.rowpointers), _lib.ptr(ref_taper.entries),
            ref_taper.entries.shape[0], stream, self._h))
        self.q = 0

    def tile_stats(self):
        """dict(tile_columns, stored_tiles, fill_tiles, tile_products) - see cocons_ctx_tile_stats."""
        out = np.empty(4, dtype=np.int64)
        _lib.check(_lib.lib().cocons_ctx_tile_stats(self._h, out.ctypes.data_as(_lib._lp)))
        return dict(zip(("tile_columns", "stored_tiles", "fill_tiles", "tile_products"), (int(v) for v in out)))


# --------------------------------------------------------------------------
# objectives (R/neg2loglikelihood.R), one-shot: host buffers in, scalar out
# --------------------------------------------------------------------------
def _one_shot(kind, theta_list, locs, x_covariates, smooth_limits, z, n, x_betas=None):
    locs, X = _lib.fmat(locs), _lib.fmat(x_covariates)
    z = _lib.fmat(z, rows=n)
    p, r = X.shape[1], z.shape[1]
    xb = None if x_betas is None else _lib.fmat(x_betas, rows=n)
    q = 0 if xb is None else xb.shape[1]
    th = _lib.pack_theta(theta_list, p)
    lim = np.ascontiguousarray(np.asarray(smooth_limits, dtype=np.float64))
    mean = np.ascontiguousarray(np.asarray(theta_list["mean"], dtype=np.float64))
    logdet, ldw = _lib.ctypes.c_double(), _lib.ctypes.c_double()
    rank = _lib.ctypes.c_int()
    quad = np.empty(r)
    _lib.check(_lib.lib().cocons_neg2loglik_dense(int(kind), n, p, r, q, _lib.ptr(locs), _lib.ptr(X), _lib.ptr(z),
                                                  _lib.ptr(xb), _lib.ptr(th), _lib.ptr(lim), _lib.ptr(mean),
                                                  _lib.ctypes.byref(logdet), _lib.ptr(quad), _lib.ctypes.byref(ldw),
                                                  _lib.ctypes.byref(rank)))
    return {"logdet": logdet.value, "quad": quad, "logdet_w": ldw.value, "rank": rank.value}


def _combine(kind, t, n, r, lambda_, theta_list, smooth_limits):
    if kind == _lib.REML:  # R/neg2loglikelihood.R:283-289
        p = t["rank"]
        total = sum((n - p) * np.log(2 * np.pi) + 2 * t["logdet"] + 2 * t["logdet_w"] + qd for qd in t["quad"])
        return total + _getPen((n - p) * r, lambda_, theta_list, smooth_limits)
    total = sum(n * np.log(2 * np.pi) + 2 * t["logdet"] + qd for qd in t["quad"])  # :155-160, :212-218
    return total + _getPen(n * r, lambda_, theta_list, smooth_limits)


def _objective(kind, theta, par_pos, locs, x_covariates, smooth_limits, z, n, lambda_, safe, x_betas=None, ctx=None):
    theta_list = getModelLists(theta, par_pos, "diff")
    try:
        if ctx is not None:
            t = ctx.terms(kind, theta_list, smooth_limits, theta_list["mean"])
            r = ctx.r
        else:
            t = _one_shot(kind, theta_list, locs, x_covariates, smooth_limits, z, n, x_betas)
            r = len(t["quad"])
    except NotPositiveDefinite:
        if safe:
            return 1e6  # R/neg2loglikelihood.R:138-142, 202-206, 261-265
        raise ArithmeticError("Cholesky error")
    return _combine(kind, t, n, r, lambda_, theta_list, smooth_limits)


def _objectives_batch(kind, thetas, par_pos, smooth_limits, n, lambda_, safe, bctx):
    """_objective at every point of `thetas` through one DenseLikelihoodBatch.terms_batch call: the same values, bit for
    bit; with safe=False the first point that is not PD, in point order, raises"""
    lists = [getModelLists(t, par_pos, "diff") for t in thetas]
    out = []
    for tl, t in zip(lists, bctx.terms_batch(kind, lists, smooth_limits, [tl["mean"] for tl in lists])):
        if isinstance(t, NotPositiveDefinite):
            if not safe:
                raise ArithmeticError("Cholesky error")
            out.append(1e6)
        else:
            out.append(_combine(kind, t, n, bctx.r, lambda_, tl, smooth_limits))
    return out


def GetNeg2loglikelihood(theta, par_pos, locs, x_covariates, smooth_limits, z, n, lambda_, safe=True, ctx=None):
    """R/neg2loglikelihood.R:183-222.  `ctx` (a DenseLikelihood) keeps the data on the device between
    calls; without it every call uploads locs / x_covariates / z, as the R closure would."""
    return _objective(_lib.ML, theta, par_pos, locs, x_covariates, smooth_limits, z, n, lambda_, safe, None, ctx)


def GetNeg2loglikelihoodProfile(theta, par_pos, locs, x_covariates, smooth_limits, z, n, x_betas, lambda_, safe=True,
                                ctx=None):
    """R/neg2loglikelihood.R:127-165."""
    return _objective(_lib.PROFILE, theta, par_pos, locs, x_covariates, smooth_limits, z, n, lambda_, safe, x_betas,
                      ctx)


def GetNeg2loglikelihoodREML(theta, par_pos, locs, x_covariates, x_betas, smooth_limits, z, n, lambda_, safe=True,
                             ctx=None):
    """R/neg2loglikelihood.R:241-291 (x_betas is accepted and unused there too; z are the contrasts of
    R/optim.R:311, see reml_contrasts())."""
    return _objective(_lib.REML, theta, par_pos, locs, x_covariates, smooth_limits, z, n, lambda_, safe, None, ctx)


def reml_contrasts(mod_DM, z):
    """R/optim.R:311 without forming the n x n projector: z - X (X'X)^-1 X' z."""
    X = np.asarray(mod_DM, dtype=np.float64)
    z = np.asarray(z, dtype=np.float64).reshape(X.shape[0], -1)
    return z - X @ np.linalg.solve(X.T @ X, X.T @ z)


def _taper_terms(theta_list, ref_taper, locs, x_covariates, smooth_limits, z, n, safe, ctx):
    try:
        if ctx is not None:
            return ctx.terms_taper(theta_list, smooth_limits, theta_list["mean"])
        with DenseLikelihood(locs, x_covariates, _lib.fmat(z, rows=n)) as tmp:
            tmp.set_taper(ref_taper)
            return tmp.terms_taper(theta_list, smooth_limits, theta_list["mean"])
    except NotPositiveDefinite:
        if safe:
            return None
        raise ArithmeticError("Cholesky error")


def GetNeg2loglikelihoodTaper(theta, par_pos, ref_taper, locs, x_covariates, smooth_limits, cholS, z, n, lambda_,
                              safe=True, ctx=None):
    """R/neg2loglikelihood.R:20-53.  `ref_taper` is the taper as a `spam`; `cholS` (spam's symbolic
    Cholesky object there) is accepted and unused: the tapered matrix is factored densely on the GPU.
    `ctx`: a DenseLikelihood that already had set_taper(ref_taper)."""
    theta_list = getModelLists(theta, par_pos, "diff")
    t = _taper_terms(theta_list, ref_taper, locs, x_covariates, smooth_limits, z, n, safe, ctx)
    if t is None:
        return 1e6  # :35-39
    r = len(t["quad"])
    sumlogs = sum(n * np.log(2 * np.pi) + 2 * t["logdet"] + qd for qd in t["quad"])  # :43-49
    return sumlogs + _getPen(n * r, lambda_, theta_list, smooth_limits)


def GetNeg2loglikelihoodTaperProfile(theta, par_pos, ref_taper, locs, x_covariates, smooth_limits, cholS, z, n,
                                     lambda_, safe=True, ctx=None):
    """R/neg2loglikelihood.R:73-108: the global variance profiled out (std.dev intercept set to 0, :78)."""
    theta_list = getModelLists(theta, par_pos, "diff")
    theta_list["std.dev"] = np.array(theta_list["std.dev"], dtype=np.float64)
    theta_list["std.dev"][0] = 0.0
    t = _taper_terms(theta_list, ref_taper, locs, x_covariates, smooth_limits, z, n, safe, ctx)
    if t is None:
        return 1e6
    r = len(t["quad"])
    sum_in = float(np.sum(t["quad"]))
    return (r * n * np.log(2 * np.pi) + r * n + r * 2 * t["logdet"] + r * n * np.log(sum_in / (r * n)) +
            _getPen(n * r, lambda_, theta_list, smooth_limits))  # :101-105


# --------------------------------------------------------------------------
# coco objects and the user-facing verbs
# --------------------------------------------------------------------------
class coco:
    """S4 class `coco` (R/methods.R:17-25) built by coco() (R/cocons.R:84-175)."""

    def __init__(self, type, data, locs, z, model_list, info=None, output=None):
        if type not in ("dense", "sparse"):
            raise ValueError("type must be 'dense' or 'sparse'")
        self.type = type
        self.data = _columns(data)
        self.locs = np.asfortranarray(np.asarray(locs, dtype=np.float64))
        z = np.asarray(z, dtype=np.float64)
        self.z = np.asfortranarray(z.reshape(-1, 1) if z.ndim == 1 else z)
        ml = dict(model_list)
        ml.setdefault("mean", 0)
        ml.setdefault("aniso", 0)
        ml.setdefault("tilt", 0)
        ml.setdefault("smooth", 0.5)
        ml.setdefault("nugget", -np.inf)
        self.model_list = {k: ml[k] for k in DICTIONARY}  # :132
        info = dict(info or {})
        info.setdefault("lambda.reg", 0)
        info.setdefault("lambda.betas", 0)
        info.setdefault("lambda.Sigma", 0)
        if not is_formula(self.model_list["smooth"]):  # :157-162
            s = float(np.atleast_1d(self.model_list["smooth"])[0])
            info["smooth.limits"] = np.array([s, s])
        if "smooth.limits" not in info:
            raise ValueError("info['smooth.limits'] is required when smooth is a formula")
        info["smooth.limits"] = np.asarray(info["smooth.limits"], dtype=np.float64)
        if type == "sparse":  # .cocons.check.info, R/checkFunctions.R:316-331
            if not callable(info.get("taper")):
                raise ValueError("taper must be one compact supported function from package spam")
            if info.get("delta") is None:
                raise ValueError("taper type requires specifying a delta > 0")
            if info["delta"] < 0:
                raise ValueError("taper argument must be non-negative")
        elif info.get("taper") is not None or info.get("delta") is not None:  # :334-339
            raise ValueError("if type is dense taper / delta should not be specified")
        self.info = info
        self.output = dict(output or {})


def getCovMatrix(coco_object):
    """R/getFunctions.R:35-80 (type 'global'; dense: the n x n matrix, sparse: a `spam`)."""
    x_covs = getScale(coco_object)["std.covs"]
    par_pos = getDesignMatrix(coco_object.model_list, coco_object.data)["par.pos"]
    theta_list = getModelLists(coco_object.output["par"], par_pos, "diff")
    if coco_object.type == "sparse":  # :60-78: the tapered matrix, as a spam
        ref_taper = _ref_taper(coco_object)
        ref_taper.entries = ref_taper.entries * cov_rns_taper(theta_list, coco_object.locs, x_covs,
                                                              ref_taper.colindices, ref_taper.rowpointers,
                                                              coco_object.info["smooth.limits"])
        return ref_taper
    return cov_rns(theta_list, coco_object.locs, x_covs, coco_object.info["smooth.limits"])


def getDensityFromDelta(coco_object, delta):
    """R/getFunctions.R:133-146: density of the tapered covariance matrix for a taper range `delta` (the
    fraction of stored entries, which depends on the pattern only)."""
    if coco_object.type != "sparse":
        raise ValueError("only for sparse coco objects.")
    return nearest_dist(coco_object.locs, delta=delta).density()


def _ref_taper(coco_object, rows=None):
    """info$taper(spam::nearest.dist(locs, delta = info$delta, upper = NULL), theta = c(delta, 1)),
    R/optim.R:376-379; with `rows`, the prediction pattern of R/predict.R:233-235."""
    d = coco_object.info["delta"]
    dist = nearest_dist(coco_object.locs, delta=d) if rows is None else nearest_dist(rows, coco_object.locs, delta=d)
    return coco_object.info["taper"](dist, (d, 1))


def fd_value_and_grad(fn, theta, lower, upper, ndeps, forward=False, group=None, batch=None):
    """What optimParallel does per L-BFGS-B iteration (R/optim.R:157,256,321; options at
    R/profile.R:9-16): fn(theta) and its finite-difference neighbours (2p central, or p forward)
    evaluated as ONE batch of independent points.  With torch.distributed initialised (one process
    per GPU) the batch is dealt to the ranks by distributed.fan_out(); every rank gets every value,
    so all ranks take the same optimiser step."""
    from .distributed import fan_out
    theta = np.asarray(theta, dtype=np.float64)
    p = theta.shape[0]
    pts, spans = [theta.copy()], []
    for i in range(p):
        up, dn = theta.copy(), theta.copy()
        up[i] = min(theta[i] + ndeps, upper[i])
        dn[i] = theta[i] if forward else max(theta[i] - ndeps, lower[i])
        if up[i] == dn[i]:  # pinned at a degenerate bound
            dn[i] = max(theta[i] - ndeps, lower[i])
        pts.append(up)
        if not forward:
            pts.append(dn)
        spans.append((up[i], dn[i]))
    if batch is not None:  # several evaluations in flight on this GPU (DenseLikelihoodPool.map)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            world, rank = dist.get_world_size(group), dist.get_rank(group)
            mine = batch(pts[rank::world])
            it = iter(mine)
            vals = fan_out(pts, lambda _pt: next(it), group=group)
        else:
            vals = batch(pts)
    else:
        vals = fan_out(pts, fn, group=group)
    f0 = vals[0]
    grad = np.empty(p)
    for i in range(p):
        up_i, dn_i = spans[i]
        if forward:
            grad[i] = (vals[1 + i] - f0) / (up_i - dn_i) if up_i != dn_i else 0.0
        else:
            grad[i] = (vals[1 + 2 * i] - vals[2 + 2 * i]) / (up_i - dn_i) if up_i != dn_i else 0.0
    return f0, grad


def getEstims(coco_object):
    """R/getFunctions.R:357-363."""
    par_pos = getDesignMatrix(coco_object.model_list, coco_object.data)["par.pos"]
    return getModelLists(coco_object.output["par"], par_pos, "diff")


def _update_coco_first_step(coco_object, output, boundaries):
    """.cocons.update.coco.first.step, R/checkFunctions.R:515-603: after the penalised first fit, coefficients
    with |estimate| <= sparse.point leave their aspect's formula (an aspect left with at most one coefficient
    becomes "~1"; a lone intercept is never dropped) and the matching entries leave the boundaries.  Mirrored
    statement by statement, including the way the boundaries are pruned independently of the formulas."""
    par_pos = getDesignMatrix(coco_object.model_list, coco_object.data)["par.pos"]
    free = {k: isinstance(v, np.ndarray) and v.dtype == bool for k, v in par_pos.items()}
    nparams = {k: int(par_pos[k].sum()) if free[k] else 0 for k in par_pos}
    fitted = copy.copy(coco_object)
    fitted.info = dict(coco_object.info)
    fitted.output = dict(output)
    parss = getEstims(fitted)
    cut = fitted.info["sparse.point"]
    new_formulas = dict(coco_object.model_list)
    columns = ["(Intercept)"] + _union_labels(coco_object.model_list)

    def small(name):  # 1-based positions among the aspect's own coefficients, as R's which()
        est = parss[name][par_pos[name]]
        return [i + 1 for i, v in enumerate(est) if abs(v) <= cut]

    for name in DICTIONARY:
        if not is_formula(coco_object.model_list[name]):
            continue
        to_zero = small(name)
        if not to_zero:
            continue
        if len(to_zero) in (nparams[name] - 1, nparams[name]):
            new_formulas[name] = "~1"
            continue
        if to_zero == [1]:
            continue
        # drop.terms(terms(formula), dropx = to_zero - 1): term k of the formula is the aspect's coefficient k + 1
        own = [columns[j] for j in np.flatnonzero(par_pos[name])]
        intercept, labels = _terms(coco_object.model_list[name])
        drop = {own[k - 1] for k in to_zero if k - 1 >= (1 if intercept else 0)}
        keep = [l for l in labels if l not in drop]
        new_formulas[name] = "~" + " + ".join((["1"] if intercept and keep else []) + keep) if keep else "~1"
    npar = len(output["par"])
    gone = np.zeros(npar, dtype=bool)
    where = 0
    for name in DICTIONARY:
        if not is_formula(coco_object.model_list[name]):
            continue
        to_zero = small(name)
        if 1 in to_zero and len(to_zero) > 1:
            to_zero = to_zero[1:]
        if to_zero == [1]:
            where += nparams[name]
            continue
        for k in to_zero:
            gone[where + k - 1] = True
        where += nparams[name]
    pruned = {k: np.asarray(v, dtype=np.float64)[~gone] for k, v in boundaries.items()}
    out = copy.copy(coco_object)
    out.info = dict(coco_object.info, boundaries=pruned)
    out.model_list = new_formulas
    out.output = dict(output)
    return out


def _union_labels(model_list):
    labels = []
    for v in model_list.values():
        if is_formula(v):
            for l in _terms(v)[1]:
                if l not in labels:
                    labels.append(l)
    return labels


def _cocoOptim_two_step(coco_object, boundaries, ncores, safe, optim_control, device, forward):
    """R/optim.R:127-230: penalised first fit (lambda.Sigma, lambda.betas, lambda.reg), model pruning at
    sparse.point, second fit of the pruned model with lambda = (0, 0, lambda.reg) from the pruned boundaries."""
    obj = copy.copy(coco_object)
    obj.info = dict(coco_object.info)
    if obj.info.get("sparse.point") is None:
        obj.info["sparse.point"] = 1e-4  # getOption("cocons.sparse.point"), R/cocons.R:32
    first = cocoOptim(copy.copy(obj), boundaries, ncores, safe, "ml", optim_control, device, forward, _first_step=True)
    pen = _update_coco_first_step(obj, first.output, boundaries)
    b2 = pen.info["boundaries"]
    second = cocoOptim(pen, b2, ncores, safe, "ml", optim_control, device, forward, _first_step=False)
    second.info["first.step"] = {"par": first.output["par"], "value": first.output["value"]}
    return second


def cocoOptim(coco_object, boundaries, ncores="auto", safe=True, optim_type="ml", optim_control=None, device=0,
              forward=False, _first_step=None, tiled=False):
    """R/optim.R:65-365 (dense) and :366-690 (sparse, see _cocoOptim_sparse).  L-BFGS-B (scipy) stands in for optimParallel's optimiser; its
    gradient is the same batched finite-difference scheme (fd_value_and_grad), whose independent
    objective evaluations run on the device-resident context of each rank - across all GPUs when
    launched with one process per GPU - instead of on forked R workers.
    `boundaries` = dict(theta_init, theta_lower, theta_upper).  `tiled` (sparse objects only): evaluate on
    TaperedLikelihood contexts, which store only the factor's nonzero tiles, instead of dense ones."""
    from scipy.optimize import minimize

    dm = getDesignMatrix(coco_object.model_list, coco_object.data)
    sc = getScale(dm["model.matrix"])
    mod_DM = sc["std.covs"]
    n = coco_object.z.shape[0]
    lim = coco_object.info["smooth.limits"]
    optim_type = optim_type.lower()  # R/optim.R:113
    # every dense branch optimises with lambda = c(0, 0, lambda.reg) (R/optim.R:248, 287, 316) except the first
    # step of the penalised two-step "ml" fit (:127-223): lambda.Sigma / lambda.betas > 0, then the model is pruned
    # at sparse.point and refitted without those two penalties
    lam = (0.0, 0.0, coco_object.info["lambda.reg"])
    if _first_step is None and optim_type == "ml" and coco_object.type == "dense" and (
            coco_object.info.get("lambda.Sigma", 0) > 0 or coco_object.info.get("lambda.betas", 0) > 0):
        return _cocoOptim_two_step(coco_object, boundaries, ncores, safe, optim_control, device, forward)
    if _first_step:
        lam = (coco_object.info["lambda.Sigma"], coco_object.info["lambda.betas"], coco_object.info["lambda.reg"])
    ctrl = {"maxiter": 500, "ftol": 1e-8, "maxcor": 100}  # R/profile.R:9-16 (factr, maxit, lmm)
    ctrl.update(optim_control or {})
    ndeps = ctrl.pop("ndeps", np.finfo(float).eps ** 0.25)
    init = np.asarray(boundaries["theta_init"], dtype=np.float64)
    lower = np.asarray(boundaries["theta_lower"], dtype=np.float64)
    upper = np.asarray(boundaries["theta_upper"], dtype=np.float64)
    par_pos = dm["par.pos"]
    z = coco_object.z
    x_betas = None
    if coco_object.type == "sparse":
        nc = max(1, min(8, int(4e9 // (8 * n * n)))) if ncores == "auto" else int(ncores)
        return _cocoOptim_sparse(coco_object, boundaries, dm, sc, mod_DM, init, lower, upper, ctrl, ndeps, forward,
                                 nc, safe, optim_type, device, tiled)
    if optim_type in ("pml", "reml"):
        if not isinstance(par_pos["mean"], np.ndarray):
            raise ValueError("Profile ML or Restricted ML only available when considering covariates in the mean.")
        x_betas = mod_DM[:, par_pos["mean"]]
        nb = int(par_pos["mean"].sum())
        init, lower, upper = init[nb:], lower[nb:], upper[nb:]
        par_pos = dict(par_pos)
        par_pos["mean"] = np.zeros_like(dm["par.pos"]["mean"])
        if optim_type == "reml":
            z = reml_contrasts(mod_DM, z)
    # `ncores` keeps its meaning of "objective evaluations in flight" (R/optim.R:80-86): here they are
    # contexts on one GPU; "auto" = as many as fit comfortably, none extra once one evaluation fills the GPU
    if ncores == "auto":
        ncores = max(1, min(8, int(4e9 // (8 * n * n))))
    with DenseLikelihoodPool(coco_object.locs, mod_DM, z, size=int(ncores), device=device) as pool:
        ctx = pool.ctxs[0]
        if optim_type == "pml":
            pool.set_xbetas(x_betas)
        kind = {"ml": _lib.ML, "pml": _lib.PROFILE, "reml": _lib.REML}[optim_type]

        def fn_on(c, theta):
            return _objective(kind, theta, par_pos, None, None, lim, None, n, lam, safe, ctx=c)

        def fn(theta):
            return fn_on(ctx, theta)

        res = minimize(lambda th: fd_value_and_grad(fn, th, lower, upper, ndeps, forward=forward,
                                                    batch=lambda pts: pool.map(fn_on, pts)),
                       init, jac=True, method="L-BFGS-B", bounds=list(zip(lower, upper)), options=ctrl)
        par = res.x
        if optim_type in ("pml", "reml"):  # R/optim.R:326-345
            theta_list = getModelLists(par, par_pos, "diff")
            ctx.set_z(coco_object.z)
            ctx.set_xbetas(x_betas)
            ctx.factor(theta_list, lim)
            betas = ctx.profile_betas(_lib.PROFILE)
            par = np.concatenate([betas, par])
    coco_object.output = {"par": par, "value": res.fun, "counts": res.nfev, "convergence": res.status,
                          "message": res.message}
    coco_object.info.update({"mean.vector": sc["mean.vector"], "sd.vector": sc["sd.vector"],
                             "optim.type": optim_type, "safe": safe, "boundaries": boundaries})
    return coco_object


def _cocoOptim_sparse(coco_object, boundaries, dm, sc, mod_DM, init, lower, upper, ctrl, ndeps, forward, ncores, safe,
                      optim_type, device, tiled=False):
    """R/optim.R:366-690: the tapered model.  "ml" (:480-531) and "pml" (:533-688, global variance profiled
    out and recovered after the fit).  The penalised two-step fit (:368-478) prunes the model through
    .cocons.update.coco.first.step - validation/UI code outside this path - and is not mirrored."""
    from scipy.optimize import minimize

    if optim_type == "ml" and (coco_object.info["lambda.betas"] > 0 or coco_object.info["lambda.Sigma"] > 0):
        raise NotImplementedError("penalised sparse fits (R/optim.R:368-478) are outside this build's scope")
    if optim_type not in ("ml", "pml"):
        raise ValueError("sparse coco objects support optim.type 'ml' and 'pml'")
    n = coco_object.z.shape[0]
    r = coco_object.z.shape[1]
    lim = coco_object.info["smooth.limits"]
    lam = (0.0, 0.0, coco_object.info["lambda.reg"])
    ref_taper = _ref_taper(coco_object)
    par_pos = dm["par.pos"]
    is_free = {k: isinstance(v, np.ndarray) for k, v in par_pos.items()}
    fn_ref = GetNeg2loglikelihoodTaper
    if optim_type == "pml":
        if not is_free["std.dev"]:
            raise ValueError("at least a global sigma needs to be estimated for sparse pml coco objects.")
        par_pos = dict(par_pos)
        par_pos["std.dev"] = par_pos["std.dev"].copy()
        par_pos["std.dev"][0] = False  # :566
        first_sigma = int(dm["par.pos"]["mean"].sum()) if is_free["mean"] else 0  # 0-based :570-572
        keep = np.arange(init.shape[0]) != first_sigma
        init, lower, upper = init[keep], lower[keep], upper[keep]
        fn_ref = GetNeg2loglikelihoodTaperProfile
    kw = {"ctx_class": TaperedLikelihood, "ref_taper": ref_taper} if tiled else {}
    with DenseLikelihoodPool(coco_object.locs, mod_DM, coco_object.z, size=ncores, device=device, **kw) as pool:
        if not tiled:
            pool.set_taper(ref_taper)
        ctx = pool.ctxs[0]

        def fn_on(c, theta):
            return fn_ref(theta, par_pos, ref_taper, None, None, lim, None, None, n, lam, safe, ctx=c)

        res = minimize(lambda th: fd_value_and_grad(lambda t: fn_on(ctx, t), th, lower, upper, ndeps,
                                                    forward=forward, batch=lambda pts: pool.map(fn_on, pts)),
                       init, jac=True, method="L-BFGS-B", bounds=list(zip(lower, upper)), options=ctrl)
        par = res.x
        if optim_type == "pml":  # :590-662
            theta_list = getModelLists(par, par_pos, "diff")
            t = ctx.terms_taper(theta_list, lim, theta_list["mean"])  # resid' Sigma^-1 resid per column (:599-603)
            sigma_0 = float(np.sum(t["quad"])) / (n * r)
            nm = int(par_pos["mean"].sum()) if is_free["mean"] else 0
            nsd = int(par_pos["std.dev"].sum())
            first_scale = nm + nsd  # 0-based
            g = par[first_scale] if is_free["scale"] else float(np.atleast_1d(par_pos["scale"])[0])
            first_par, second_par = np.log(sigma_0) + g, np.log(sigma_0) - g
            new = list(par[:nm]) + [first_par] + list(par[nm:nm + nsd])
            pos = first_scale
            if is_free["scale"]:
                ns = int(par_pos["scale"].sum())
                new += [second_par] + list(par[first_scale + 1:first_scale + ns])
                pos = first_scale + ns
            for k in ("smooth", "nugget"):
                if is_free[k]:
                    cnt = int(par_pos[k].sum())
                    new += list(par[pos:pos + cnt])
                    pos += cnt
            par = np.asarray(new, dtype=np.float64)
    coco_object.output = {"par": par, "value": res.fun, "counts": res.nfev, "convergence": res.status,
                          "message": res.message}
    coco_object.info.update({"mean.vector": sc["mean.vector"], "sd.vector": sc["sd.vector"],
                             "optim.type": optim_type, "safe": safe, "boundaries": boundaries})
    return coco_object


def getHessian(coco_object, ncores="auto", eps=np.finfo(float).eps ** 0.25, device=0):
    """R/getFunctions.R:925-1034, dense branch: forward-difference Hessian of the NEGATIVE log-likelihood
    at the fitted parameters, H[j,i] = 0.5 (f11 - f01 - f10 + f00) / eps^2 with f = -2 loglik (for "pml"
    fits on the full likelihood, as there).  The reference farms three evaluations per index pair over a
    PSOCK cluster; here the p + p(p+1)/2 distinct points are evaluated as one batch on the GPU(s)."""
    if coco_object.info.get("optim.type") == "reml":
        raise NotImplementedError("reml hessian not implemented yet.")  # as the reference
    par = np.asarray(coco_object.output["par"], dtype=np.float64)
    p = par.shape[0]
    dm = getDesignMatrix(coco_object.model_list, coco_object.data)
    X = getScale(dm["model.matrix"], coco_object.info["mean.vector"], coco_object.info["sd.vector"])["std.covs"]
    n = coco_object.z.shape[0]
    lim = coco_object.info["smooth.limits"]
    lam = (coco_object.info["lambda.Sigma"], coco_object.info["lambda.betas"], coco_object.info["lambda.reg"])
    if ncores == "auto":
        ncores = max(1, min(8, int(4e9 // (8 * n * n))))
    singles = [par + eps * np.eye(p)[j] for j in range(p)]
    pairs = [(j, i) for j in range(p) for i in range(j, p)]
    doubles = [par + eps * (np.eye(p)[j] + np.eye(p)[i]) for j, i in pairs]
    with DenseLikelihoodPool(coco_object.locs, X, coco_object.z, size=int(ncores), device=device) as pool:
        def fn_on(c, theta):
            return _objective(_lib.ML, theta, dm["par.pos"], None, None, lim, None, n, lam, True, ctx=c)
        vals = pool.map(fn_on, [par] + singles + doubles)
    f00 = vals[0] if coco_object.info.get("optim.type") == "pml" else coco_object.output["value"]
    f1 = vals[1:1 + p]
    H = np.zeros((p, p))
    for (j, i), f11 in zip(pairs, vals[1 + p:]):
        H[j, i] = 0.5 * ((f11 - f1[j] - f1[i] + f00) / (eps * eps))
    H = H + H.T
    H[np.diag_indices(p)] /= 2
    return H


def cocoPredict(coco_object, newdataset, newlocs, type="mean", index_pred=0, device=0, tiled=False):
    """R/predict.R:84-288: kriging mean and (type "pred") standard deviation, dense and sparse (tapered)
    branches.  The reference solves with LU (`solve`) / spam's sparse solve; here the Cholesky factor on the
    device is used.  `tiled` (sparse objects only): factor and solve on a TaperedLikelihood, which stores only the
    factor's nonzero tiles - for sizes whose dense matrix does not fit the device."""
    if not coco_object.output:
        raise ValueError("coco object has not yet been fitted.")
    if tiled and coco_object.type != "sparse":
        raise ValueError("tiled = True is for sparse coco objects.")
    dm = getDesignMatrix(coco_object.model_list, coco_object.data)
    eff = getModelLists(coco_object.output["par"], dm["par.pos"], "diff")
    X_std = getScale(dm["model.matrix"], coco_object.info["mean.vector"], coco_object.info["sd.vector"])["std.covs"]
    dmp = getDesignMatrix(coco_object.model_list, newdataset)
    X_pred = getScale(dmp["model.matrix"], coco_object.info["mean.vector"], coco_object.info["sd.vector"])["std.covs"]
    systematic = X_pred @ eff["mean"]
    resid = coco_object.z[:, index_pred] - X_std @ eff["mean"]
    if tiled:
        ctx = TaperedLikelihood(coco_object.locs, X_std, coco_object.z, _ref_taper(coco_object), device=device)
    else:
        ctx = DenseLikelihood(coco_object.locs, X_std, coco_object.z, device=device)
    with ctx:
        if coco_object.type == "sparse":  # R/predict.R:190-288: tapered Sigma and tapered cross-covariance
            if not tiled:
                ctx.set_taper(_ref_taper(coco_object))
            ctx.factor_taper(eff, coco_object.info["smooth.limits"])
            sto, expl = ctx.predict_taper(newlocs, X_pred, _ref_taper(coco_object, rows=newlocs), resid,
                                          want_explained=(type == "pred"))
        else:
            ctx.factor(eff, coco_object.info["smooth.limits"])
            sto, expl = ctx.predict(newlocs, X_pred, resid, want_explained=(type == "pred"))
    out = {"systematic": systematic, "stochastic": sto}
    if type == "pred":  # :170-183
        u = 1 / np.exp(-(X_pred @ eff["std.dev"])) + np.exp(X_pred @ eff["nugget"]) - expl
        neg = u < 1e-10
        u[neg] = np.abs(u[neg])
        out["sd.pred"] = np.sqrt(u)
    return out


def cocoSim(coco_object, pars=None, n=1, seed=None, standardize=True, type="classic", sim_type=None, cond_info=None,
            device=0, eps=None, tiled=False):
    """R/sim.R:52-218, dense and sparse branches.  The N(0,1) draws come from numpy's legacy generator seeded
    with `seed` (R's come from set.seed/rnorm; pass `eps` to supply R's own draws).  `tiled` (sparse objects,
    marginal draws only): factor and draw on a TaperedLikelihood, which stores only the factor's nonzero tiles."""
    if tiled and (coco_object.type != "sparse" or sim_type == "cond"):
        raise ValueError("tiled = True is for the marginal draws of sparse coco objects.")
    if pars is None:
        pars, type = coco_object.output["par"], "diff"
    dm = getDesignMatrix(coco_object.model_list, coco_object.data)
    rng = np.random.RandomState(seed)
    if sim_type == "cond":
        std_coco = getScale(dm["model.matrix"])["std.covs"]  # freshly standardised, as at :76
        dmp = getDesignMatrix(coco_object.model_list, cond_info["newdataset"])
        std_pred = getScale(dmp["model.matrix"], coco_object.info["mean.vector"],
                            coco_object.info["sd.vector"])["std.covs"]
        to_pass = getModelLists(coco_object.output["par"], dmp["par.pos"], "diff")
        newlocs = np.asarray(cond_info["newlocs"], dtype=np.float64)
        m = newlocs.shape[0]
        if eps is None:
            eps = rng.standard_normal((m, n))
        with DenseLikelihood(coco_object.locs, std_coco, coco_object.z, device=device) as ctx:
            ctx.factor(to_pass, coco_object.info["smooth.limits"])
            draws = ctx.sim_cond(newlocs, std_pred, eps)
        step_one = cocoPredict(coco_object, cond_info["newdataset"], newlocs, "mean", device=device)
        return draws + (step_one["systematic"] + step_one["stochastic"])[:, None]
    if standardize:
        std_coco = getScale(dm["model.matrix"])["std.covs"]
    else:
        k = dm["model.matrix"].shape[1]
        std_coco = getScale(dm["model.matrix"], np.zeros(k), np.ones(k))["std.covs"]
    theta_to_fit = getModelLists(pars, dm["par.pos"], type)
    if not is_formula(coco_object.model_list["smooth"]):  # :141-145
        theta_to_fit["smooth"][0] = np.log(coco_object.info["smooth.limits"][0])
    nsites = std_coco.shape[0]
    if eps is None:
        eps = rng.standard_normal((nsites, n))
    if tiled:
        with TaperedLikelihood(coco_object.locs, std_coco, coco_object.z, _ref_taper(coco_object),
                               device=device) as ctx:
            ctx.factor_taper(theta_to_fit, coco_object.info["smooth.limits"])
            draws = ctx.sim_taper(eps)
        return draws + (std_coco @ theta_to_fit["mean"])[:, None]
    with DenseLikelihood(coco_object.locs, std_coco, coco_object.z, device=device) as ctx:
        if coco_object.type == "sparse":
            # R/sim.R:176-218.  The reference draws t(eps) %*% chol_spam(P Sigma P') un-permuted; any factor of
            # Sigma gives the same distribution, and the draw here is L eps with the device's own factor.
            ctx.set_taper(_ref_taper(coco_object))
            ctx.factor_taper(theta_to_fit, coco_object.info["smooth.limits"])
        else:
            ctx.factor(theta_to_fit, coco_object.info["smooth.limits"], type=type)
        draws = ctx.sim(eps)
    return draws + (std_coco @ theta_to_fit["mean"])[:, None]


# --------------------------------------------------------------------------
# several evaluations in flight on ONE GPU
# --------------------------------------------------------------------------
class DenseLikelihoodPool:
    """`size` device-resident contexts over the same data, each with its own streams, driven by host
    threads (the C ABI releases the GIL): the shape of the optimiser's independent finite-difference points
    (R/optim.R:157,256,321).  Their kernel chains overlap on the device - below n ~ 10 000 one evaluation
    cannot fill a B200 (holes: 156 evaluations/s one at a time, 321 with 8 in flight) - and every value is
    bit-identical to a single context's (tests/test_gpu_repro.py); across GPUs use distributed.fan_out."""

    def __init__(self, locs, x_covariates, z, size=4, device=0, ctx_class=None, **ctx_kw):
        """`ctx_class` (default DenseLikelihood) and `ctx_kw` make the contexts, e.g. TaperedLikelihood with
        ref_taper=..."""
        from concurrent.futures import ThreadPoolExecutor
        ctx_class = ctx_class or DenseLikelihood
        self.ctxs = [ctx_class(locs, x_covariates, z, device=device, **ctx_kw) for _ in range(int(size))]
        self.exec = ThreadPoolExecutor(max_workers=len(self.ctxs))
        self.n, self.p, self.r = self.ctxs[0].n, self.ctxs[0].p, self.ctxs[0].r

    def close(self):
        self.exec.shutdown(wait=True)
        for c in self.ctxs:
            c.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_xbetas(self, xb):
        for c in self.ctxs:
            c.set_xbetas(xb)

    def set_z(self, z):
        for c in self.ctxs:
            c.set_z(z)

    def set_taper(self, ref_taper):
        for c in self.ctxs:
            c.set_taper(ref_taper)

    def map(self, fn, points):
        """[fn(ctx, point) for point in points], evaluated len(ctxs) at a time."""
        import queue
        free = queue.SimpleQueue()
        for c in self.ctxs:
            free.put(c)

        def run(pt):
            c = free.get()
            try:
                return fn(c, pt)
            finally:
                free.put(c)

        return list(self.exec.map(run, points))
