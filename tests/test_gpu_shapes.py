"""The objective, prediction and simulation paths at the blocking edges of their kernels, output by output, against a
plain float64 LAPACK reference on the oracle's covariance.

Every dimension of the C ABI besides n is cut into blocks somewhere: the columns of z go through the forward
substitution 8 at a time and through cocons_n2ll in passes of 16 - q columns; the mean design (PROFILE's x_betas,
REML's X) is solved once in 8-column launches; predictions run in blocks of 4 096 rows (the tapered variant picks
each block's pattern entries at rowpointers[i0]); draws go through the triangular product 4 columns at a time; the
conditional draw pads its Schur complement to a multiple of 128; the distributed path works in 512-wide panels and
8-column slices.  The cases below sit on both sides of those cuts.  The model is well conditioned (nugget ~ e^-2 of
the sill), so the reference is good to ~1e-13 and each output is held on its own, not only their sum; the columns
of z have scales spread over 1 .. 1e3, so a lost, swapped or duplicated column misses by orders of magnitude.

The `gpu` tests run the device build.  The other tests call the same case functions at small n on the host build of
the same sources (fixture `product_on_host`), so the CPU suite executes these loops too."""
import ctypes
import functools

import numpy as np
import pytest
import scipy.linalg as sla

import cocons_b200 as cb
from cocons_b200 import _lib, api
from conftest import relerr
from oracle import cov, rmirror

KIND = "reference" if cov.have_reference() else "restatement"
TOL = 1e-10     # quad[j], logdet, logdet_w, betas, stochastic, draws
TOL_SD = 1e-7   # sd.pred, as tests/test_gpu_predict_sim.py
LIM = [0.5, 2.5]
LIM_FIXED = [1.5, 1.5]
NAN_BITS = {"nan": 0x7FF8000000000000, "r_na": 0x7FF00000000007A2, "all_ones": 0xFFFFFFFFFFFFFFFF}


# ---- model and data ---------------------------------------------------------------------------------------------------
def theta(p, fixed=False):
    """the covariance model of tests/test_gpu_predict_sim.py with a nugget of ~ e^-2 of the sill, for p columns"""
    base = {"mean": [0.1, 0.3, -0.2], "std.dev": [0.2, 0.15, 0.1], "scale": [-1.6, 0.2, -0.15],
            "aniso": [0.1, 0.2, -0.1], "tilt": [0.3, -0.2, 0.1], "smooth": [0.2, 0.3, -0.2], "nugget": [-1.8, 0.1, 0.1]}
    if fixed:  # as test_predict_after_fixed_smoothness_factor
        base.update(aniso=[0, 0, 0], tilt=[0, 0, 0], smooth=[0, 0, 0], nugget=[-1.8, 0, 0])
    out = {}
    for k, v in base.items():  # columns past the third: small coefficients of alternating sign
        small = 0.02 if k in ("std.dev", "scale", "nugget") and not fixed else 0.0
        out[k] = np.array((v + [small * (-1) ** j for j in range(3, p)])[:p], dtype=np.float64)
    return out


def covariates(locs, p, seed=0):
    """intercept, two smooth functions of the location, then seeded N(0, 1) columns (no data-dependent scaling:
    n = 1 has no standard deviation)"""
    n = locs.shape[0]
    cols = [np.ones(n), np.sin(3 * locs[:, 0]) + 0.2, np.cos(2 * locs[:, 1]) - 0.5][:p]
    if p > 3:
        cols += list(np.random.default_rng(1000 + seed).standard_normal((p - 3, n)))
    return np.asfortranarray(np.column_stack(cols))


def sites(n, seed):
    return np.random.default_rng(seed).uniform(0, 1, (n, 2))


def observations(n, r, seed):
    """n x r, column scales spread over 1 .. 1e3 in shuffled order"""
    rng = np.random.default_rng(seed + 77)
    scale = 10.0 ** (3.0 * rng.permutation(r) / max(r - 1, 1))
    return np.asfortranarray(rng.standard_normal((n, r)) * scale)


def other_design(n, q, seed):
    """a mean design of its own (x_betas), not tied to the covariance design"""
    rng = np.random.default_rng(seed + 5)
    return np.asfortranarray(np.column_stack([np.ones(n)] + list(rng.standard_normal((q - 1, n)))))


# ---- float64 reference -----------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=6)
def _factor(n, p, seed, fixed=False):
    locs = sites(n, seed)
    X = covariates(locs, p, seed)
    tl = theta(p, fixed)
    S = cov.cov_rns(tl, locs, X, LIM_FIXED if fixed else LIM, kind=KIND)
    return locs, X, tl, S, sla.cholesky(S, lower=True)


def _fwd(L, B):
    return sla.solve_triangular(L, B, lower=True)


def ref_terms(L, z, Xmean=None, Xb=None):
    """logdet = sum log diag chol(S); ML: quad_j = |L^-1 (z_j - X beta)|^2;  PROFILE / REML:
    quad_j = |y_j|^2 - b_j' W^-1 b_j with y = L^-1 z, Yx = L^-1 Xb, W = Yx'Yx, b = Yx'y; logdet_w = log det chol(W)"""
    out = {"logdet": float(np.sum(np.log(np.diag(L)))), "logdet_w": 0.0}
    if Xb is None:
        y = _fwd(L, z - Xmean[:, None])
        out["quad"] = np.sum(y * y, axis=0)
        return out
    y, Yx = _fwd(L, z), _fwd(L, Xb)
    Lw = np.linalg.cholesky(Yx.T @ Yx)
    t = _fwd(Lw, Yx.T @ y)
    out["quad"] = np.sum(y * y, axis=0) - np.sum(t * t, axis=0)
    out["logdet_w"] = float(np.sum(np.log(np.diag(Lw))))
    return out


def ref_gls(L, Xb, z):
    """GLS betas on rowSums(z) / r (R/optim.R:326-343)"""
    zbar = z.sum(axis=1) / z.shape[1]
    Yx, y = _fwd(L, Xb), _fwd(L, zbar)
    return np.linalg.solve(Yx.T @ Yx, Yx.T @ y)


def normerr(a, b):
    """max |a - b| / max |b| per column (entries that may cross zero: stochastic, draws, betas)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    a, b = a.reshape(a.shape[0], -1), b.reshape(b.shape[0], -1)
    return float(np.max(np.max(np.abs(a - b), axis=0) / np.max(np.abs(b), axis=0)))


def _check_terms(what, got, want, with_w=False):
    errs = {"logdet": abs(got["logdet"] - want["logdet"]) / abs(want["logdet"]),
            "quad": relerr(got["quad"], want["quad"])}
    if with_w:
        errs["logdet_w"] = abs(got["logdet_w"] - want["logdet_w"]) / max(abs(want["logdet_w"]), 1.0)
    print(what, {k: "%.2e" % v for k, v in errs.items()})
    assert got["quad"].shape == want["quad"].shape
    assert all(v < TOL for v in errs.values()), (what, errs)


# ---- 1. ML: the columns of z -----------------------------------------------------------------------------------------
def case_ml_columns(n, r, seed=1, one_shot=True):
    """passes of 16 columns through n2ll_impl, 8-column launches of the substitution, and every NR instance"""
    locs, X, tl, _, L = _factor(n, 3, seed)
    z = observations(n, r, seed)
    want = ref_terms(L, z, Xmean=X @ tl["mean"])
    with cb.DenseLikelihood(locs, X, z) as ctx:
        got = ctx.terms(_lib.ML, tl, LIM, tl["mean"])
    _check_terms("ml n=%d r=%d" % (n, r), got, want)
    if not one_shot:
        return
    one = api._one_shot(_lib.ML, tl, locs, X, LIM, z, n)  # the one-shot entry point: same kernels, same bits
    assert one["logdet"] == got["logdet"] and np.array_equal(one["quad"], got["quad"])


# ---- 2. PROFILE: the width of x_betas --------------------------------------------------------------------------------
def case_profile(n, q, r, seed=1, one_shot=True):
    locs, X, tl, _, L = _factor(n, 3, seed)
    z = observations(n, r, seed + q)
    xb = other_design(n, q, seed)
    want = ref_terms(L, z, Xb=xb)
    with cb.DenseLikelihood(locs, X, z) as ctx:
        ctx.set_xbetas(xb)
        got = ctx.terms(_lib.PROFILE, tl, LIM)
    _check_terms("profile n=%d q=%d r=%d" % (n, q, r), got, want, with_w=True)
    if not one_shot:
        return
    one = api._one_shot(_lib.PROFILE, tl, locs, X, LIM, z, n, x_betas=xb)
    assert np.array_equal(one["quad"], got["quad"]) and one["logdet_w"] == got["logdet_w"]


# ---- 3. REML: the width of the design ----------------------------------------------------------------------------------
def case_reml(n, p, r, seed=2):
    locs, X, tl, _, L = _factor(n, p, seed)
    zc = cb.reml_contrasts(X, observations(n, r, seed + p))  # as test_gpu_n2ll._values
    want = ref_terms(L, zc, Xb=X)
    with cb.DenseLikelihood(locs, X, zc) as ctx:
        got = ctx.terms(_lib.REML, tl, LIM)
    _check_terms("reml n=%d p=%d r=%d" % (n, p, r), got, want, with_w=True)
    assert got["rank"] == rmirror.r_qr_rank(X) == p


# ---- 4. limits are argument errors -------------------------------------------------------------------------------------
def _expect_arg_error(status, message):
    assert status == -1, status  # COCONS_ERR_ARG
    assert message in _lib.lib().cocons_last_error().decode()


def case_limits(n=130):
    locs = sites(n, 3)
    X = covariates(locs, 3)
    z = observations(n, 2, 3)
    with cb.DenseLikelihood(locs, X, z) as ctx:
        with pytest.raises(cb.CoconsError, match=r"error -1: ctx_set_xbetas: bad argument \(q must be in 1\.\.15\)"):
            ctx.set_xbetas(other_design(n, 16, 3))
        ctx.set_xbetas(other_design(n, 15, 3))  # the widest that fits
    X16 = covariates(locs, 16)
    with cb.DenseLikelihood(locs, X16, z) as ctx:
        with pytest.raises(cb.CoconsError, match="error -1: n2ll: REML supports at most 15 design columns"):
            ctx.terms(_lib.REML, theta(16), LIM)
    # the distributed path: nr = q + r <= 16 right-hand sides, r itself <= 15
    L = _lib.lib()
    h = _lib._vp()
    z16 = observations(n, 16, 3)
    _expect_arg_error(L.cocons_dist_create(0, 0, 1, n, 3, 16, _lib.ptr(locs), _lib.ptr(X), _lib.ptr(z16), None,
                                           ctypes.byref(h)), "dist_create: bad argument")
    assert not h.value
    X8 = covariates(locs, 8)
    z9 = observations(n, 9, 3)
    _lib.check(L.cocons_dist_create(0, 0, 1, n, 8, 9, _lib.ptr(locs), _lib.ptr(X8), _lib.ptr(z9), None,
                                    ctypes.byref(h)))
    try:
        xb = other_design(n, 8, 3)
        _expect_arg_error(L.cocons_dist_set_xbetas(h, 8, _lib.ptr(xb)), "dist_set_xbetas: bad argument")
        nr = ctypes.c_int(-1)
        unused = np.zeros(1)
        _expect_arg_error(L.cocons_dist_fill_rhs(h, _lib.REML, unused.ctypes.data, ctypes.byref(nr)),
                          "dist_fill_rhs: too many right-hand sides")
        assert nr.value == -1
        _lib.check(L.cocons_dist_set_xbetas(h, 7, _lib.ptr(xb)))  # q + r = 16 fits
    finally:
        L.cocons_dist_destroy(h)


# ---- 5. profile_betas ---------------------------------------------------------------------------------------------------
def case_profile_betas(n, kind, width, r, seed=4):
    p = width if kind == _lib.REML else 3
    locs, X, tl, _, L = _factor(n, p, seed)
    xb = X if kind == _lib.REML else other_design(n, width, seed)
    beta = np.linspace(1.0, -2.0, width)
    z = np.asfortranarray(xb @ beta[:, None] + 0.3 * np.random.default_rng(seed + r).standard_normal((n, r)))
    want = ref_gls(L, xb, z)
    with cb.DenseLikelihood(locs, X, z) as ctx:
        if kind == _lib.PROFILE:
            ctx.set_xbetas(xb)
        ctx.factor(tl, LIM)
        got = ctx.profile_betas(kind)
    err = normerr(got, want)
    print("profile_betas n=%d kind=%d width=%d r=%d: %.2e" % (n, kind, width, r, err))
    assert got.shape == (width,) and err < TOL


# ---- 7. dense prediction blocks ----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=2)
def _pred_reference(n, m_max, seed):
    """S^-1 C' for the first m_max prediction sites; rows of C are independent, so smaller m take a prefix"""
    locs, X, tl, _, L = _factor(n, 3, seed)
    lp = sites(m_max, seed + 100)
    Xp = covariates(lp, 3)
    C = cov.cov_rns_pred(tl, locs, lp, X, Xp, LIM, kind=KIND)
    V = sla.cho_solve((L, True), C.T)
    return lp, Xp, C, V


def _sd_pred(tl, Xp, expl):
    u = np.exp(Xp @ tl["std.dev"]) + np.exp(Xp @ tl["nugget"]) - expl
    neg = u < 1e-10
    u[neg] = np.abs(u[neg])
    return np.sqrt(u)


def case_predict(n, m, explained, m_max, seed=5):
    locs, X, tl, _, L = _factor(n, 3, seed)
    lp, Xp, C, V = _pred_reference(n, m_max, seed)
    lp, Xp, C, V = lp[:m], Xp[:m], C[:m], V[:, :m]
    resid = observations(n, 1, seed)[:, 0] - X @ tl["mean"]
    want_sto = resid @ V
    want_expl = np.sum(C * V.T, axis=1)
    with cb.DenseLikelihood(locs, X, resid) as ctx:
        ctx.factor(tl, LIM)
        sto, expl = ctx.predict(lp, Xp, resid, want_explained=explained)
        sub = slice(4090, 4100)
        if m > sub.start:  # rows of the second block (and the end of the first) asked for on their own
            s2, e2 = ctx.predict(lp[sub], Xp[sub], resid, want_explained=explained)
            assert np.array_equal(s2, sto[sub])
            assert not explained or np.array_equal(e2, expl[sub])
    errs = {"stochastic": normerr(sto, want_sto)}
    if explained:
        errs["explained"] = relerr(expl, want_expl)
        errs["sd.pred"] = relerr(_sd_pred(tl, Xp, expl), _sd_pred(tl, Xp, want_expl))
    else:
        assert expl is None
    print("predict n=%d m=%d" % (n, m), {k: "%.2e" % v for k, v in errs.items()})
    assert sto.shape == (m,)
    assert errs["stochastic"] < TOL and errs.get("explained", 0) < TOL and errs.get("sd.pred", 0) < TOL_SD, errs


# ---- 8. tapered prediction blocks ---------------------------------------------------------------------------------------
def case_predict_taper(n, m, seed=6, delta=0.35):
    locs, X, tl, _, _ = _factor(n, 3, seed)
    lp = sites(m, seed + 100)
    Xp = covariates(lp, 3)
    z = observations(n, 1, seed)[:, 0]
    ref = rmirror.predict_taper(tl, delta, locs, lp, X, Xp, LIM, z, type="pred", cov_kind=KIND)
    with cb.DenseLikelihood(locs, X, z) as ctx:
        ctx.set_taper(cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1)))
        ctx.factor_taper(tl, LIM)
        sto, expl = ctx.predict_taper(lp, Xp, cb.cov_wend1(cb.nearest_dist(lp, locs, delta=delta), (delta, 1)),
                                      z - X @ tl["mean"])
    errs = {"stochastic": normerr(sto, ref["stochastic"]), "sd.pred": relerr(_sd_pred(tl, Xp, expl), ref["sd.pred"])}
    print("predict_taper n=%d m=%d" % (n, m), {k: "%.2e" % v for k, v in errs.items()})
    assert errs["stochastic"] < TOL and errs["sd.pred"] < TOL_SD, errs


# ---- 9. draws ---------------------------------------------------------------------------------------------------------
def case_sim(n, k, seed=7):
    """L eps, entry by entry in the context's order (test_marginal_simulation_entrywise_in_sorted_order)"""
    locs, X, tl, S, _ = _factor(n, 3, seed)
    eps = np.random.default_rng(seed + k).standard_normal((n, k)) * 10.0 ** np.arange(k)
    with cb.DenseLikelihood(locs, X, eps[:, 0]) as ctx:
        ctx.factor(tl, LIM)
        Lf, perm = ctx.get_factor()
        got = ctx.sim(eps)
    rec = np.max(np.abs(Lf @ Lf.T - S[np.ix_(perm, perm)])) / np.max(S)
    want = np.empty_like(got)
    want[perm] = Lf @ eps[perm]
    err = normerr(got, want)
    print("sim n=%d k=%d: draws %.2e, factor %.2e" % (n, k, err, rec))
    assert got.shape == (n, k) and err < TOL and rec < 1e-13


def case_sim_cond(n, m, k, fixed, seed=8):
    """chol(S_pp - C S^-1 C') eps, with S_pp padded to a multiple of 128 inside"""
    lim = LIM_FIXED if fixed else LIM
    locs, X, tl, _, L = _factor(n, 3, seed, fixed)
    lp = sites(m, seed + 200)
    Xp = covariates(lp, 3)
    C = cov.cov_rns_pred(tl, locs, lp, X, Xp, lim, kind=KIND)
    Spp = cov.cov_rns(tl, lp, Xp, lim, kind=KIND)
    T = _fwd(L, C.T)
    eps = np.random.default_rng(seed + m).standard_normal((m, k)) * 10.0 ** np.arange(k)
    want = np.linalg.cholesky(Spp - T.T @ T) @ eps
    with cb.DenseLikelihood(locs, X, observations(n, 1, seed)) as ctx:
        ctx.factor(tl, lim)
        got = ctx.sim_cond(lp, Xp, eps)
    err = normerr(got, want)
    print("sim_cond n=%d m=%d k=%d fixed=%s: %.2e" % (n, m, k, fixed, err))
    assert got.shape == (m, k) and err < TOL


# ---- 10. distributed path, one rank ----------------------------------------------------------------------------------
def case_distributed(n, q, r, seed=9):
    from cocons_b200.distributed import DistributedDenseLikelihood
    locs, X, tl, _, L = _factor(n, 3, seed)
    z = observations(n, r, seed + r)
    kinds = [_lib.ML] if q == 0 else [_lib.PROFILE]
    xb = other_design(n, q, seed) if q else None
    with cb.DenseLikelihood(locs, X, z) as ctx:
        if q:
            ctx.set_xbetas(xb)
        res = {k: ctx.terms(k, tl, LIM, tl["mean"]) for k in kinds}
    with DistributedDenseLikelihood(locs, X, z) as d:
        if q:
            d.set_xbetas(xb)
        for kind in kinds:
            got = d.terms(kind, tl, LIM, tl["mean"])
            assert np.allclose(got["quad"], res[kind]["quad"], rtol=1e-10, atol=0)
            assert abs(got["logdet"] - res[kind]["logdet"]) < 1e-11 * abs(res[kind]["logdet"])
            want = ref_terms(L, z, Xmean=X @ tl["mean"]) if kind == _lib.ML else ref_terms(L, z, Xb=xb)
            _check_terms("distributed n=%d q=%d r=%d" % (n, q, r), got, want, with_w=bool(q))


# ---- 11. not positive definite: position and recovery ----------------------------------------------------------------
def case_not_pd_position(n, pos, seed=10):
    """a NaN covariate at the site the context puts at `pos`: status pos + 1 (dpotrf's info, context order); the
    same one-shot workspace then gives, for the clean design, the bits of a fresh context"""
    locs, X, tl, _, _ = _factor(n, 3, seed)
    z = observations(n, 2, seed)
    with cb.DenseLikelihood(locs, X, z) as ctx:
        ctx.factor(tl, LIM)
        _, perm = ctx.get_factor()
        site = int(perm[pos])
        _, where = ctx.factor_rows(np.array([site]))
        assert where[0] == pos
        clean = ctx.terms(_lib.ML, tl, LIM, tl["mean"])
    Xn = X.copy()
    Xn[site, 1] = np.nan
    with pytest.raises(cb.NotPositiveDefinite) as e:
        api._one_shot(_lib.ML, tl, locs, Xn, LIM, z, n)
    assert e.value.k == pos + 1, (e.value.k, pos + 1)
    again = api._one_shot(_lib.ML, tl, locs, X, LIM, z, n)
    assert again["logdet"] == clean["logdet"] and np.array_equal(again["quad"], clean["quad"])


# ---- 12. NaN in z and resid ---------------------------------------------------------------------------------------------
def _nan(pattern):
    return np.array([NAN_BITS[pattern]], dtype=np.uint64).view(np.float64)[0]


def case_nan_in_z(n, pattern, seed=11):
    """a NaN (whatever its bits) in one column of z makes that column's quad NaN and nothing else; status 0"""
    locs, X, tl, _, L = _factor(n, 3, seed)
    z = observations(n, 3, seed)
    zn = z.copy()
    zn[n // 2, 1] = _nan(pattern)
    assert zn.view(np.uint64)[n // 2, 1] == NAN_BITS[pattern]
    xb = other_design(n, 2, seed)
    want = {_lib.ML: ref_terms(L, z, Xmean=X @ tl["mean"]), _lib.PROFILE: ref_terms(L, z, Xb=xb)}
    with cb.DenseLikelihood(locs, X, zn) as ctx, cb.DenseLikelihood(locs, X, z) as fresh:
        ctx.set_xbetas(xb)
        fresh.set_xbetas(xb)
        for kind in (_lib.ML, _lib.PROFILE):
            got = ctx.terms(kind, tl, LIM, tl["mean"])
            assert np.isnan(got["quad"][1]) and not np.isnan(got["quad"][[0, 2]]).any(), got["quad"]
            assert relerr(got["quad"][[0, 2]], want[kind]["quad"][[0, 2]]) < TOL
            assert abs(got["logdet"] - want[kind]["logdet"]) < TOL * abs(want[kind]["logdet"])
        betas = ctx.profile_betas(_lib.PROFILE)
        assert np.isnan(betas).all()
        ctx.set_z(z)  # the next clean evaluation on the same context: the bits of a fresh one
        for kind in (_lib.ML, _lib.PROFILE):
            a, b = ctx.terms(kind, tl, LIM, tl["mean"]), fresh.terms(kind, tl, LIM, tl["mean"])
            assert a["logdet"] == b["logdet"] and np.array_equal(a["quad"], b["quad"])
        assert np.array_equal(ctx.profile_betas(_lib.PROFILE), fresh.profile_betas(_lib.PROFILE))


def case_nan_in_resid(n, m, pattern, seed=12):
    locs, X, tl, _, _ = _factor(n, 3, seed)
    lp = sites(m, seed + 100)
    Xp = covariates(lp, 3)
    resid = observations(n, 1, seed)[:, 0]
    rn = resid.copy()
    rn[n // 3] = _nan(pattern)
    with cb.DenseLikelihood(locs, X, resid) as ctx, cb.DenseLikelihood(locs, X, resid) as fresh:
        ctx.factor(tl, LIM)
        fresh.factor(tl, LIM)
        sto, expl = ctx.predict(lp, Xp, rn)
        assert np.isnan(sto).all()
        s_clean, e_clean = ctx.predict(lp, Xp, resid)
        s_fresh, e_fresh = fresh.predict(lp, Xp, resid)
    assert np.array_equal(expl, e_clean)  # explained does not read resid
    assert np.array_equal(s_clean, s_fresh) and np.array_equal(e_clean, e_fresh)


# =======================================================================================================================
# on a B200
# =======================================================================================================================
R_VALUES = [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 33]
PROFILE_QR = [(1, 16), (7, 9), (8, 8), (8, 9), (9, 1), (15, 1), (15, 3)]
REML_PR = [(p, r) for p in (1, 2, 8, 15) for r in sorted({1, 16 - p, 17 - p})]
BETAS = [(_lib.PROFILE, q, r) for q in (1, 8, 15) for r in (1, 5)] + [(_lib.REML, p, r) for p in (3, 15) for r in (1, 5)]
M_PRED = [1, 129, 4096, 4097, 9000]


@pytest.mark.gpu
@pytest.mark.parametrize("r", R_VALUES)
def test_ml_columns_of_z(r):
    case_ml_columns(1000, r)


@pytest.mark.gpu
@pytest.mark.parametrize("q,r", PROFILE_QR)
def test_profile_width_of_x_betas(q, r):
    case_profile(1000, q, r)


@pytest.mark.gpu
@pytest.mark.parametrize("p,r", REML_PR)
def test_reml_width_of_the_design(p, r):
    case_reml(1000, p, r)


@pytest.mark.gpu
def test_limits_are_argument_errors():
    case_limits(1000)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,width,r", BETAS)
def test_profile_betas_against_gls(kind, width, r):
    case_profile_betas(1000, kind, width, r)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 127, 129, 2049, 2177, 8193])
def test_ml_at_the_factorisation_and_solve_edges(n):
    """2 049: 17 tile rows, every row's solve one chunk; 2 177: row 17 is the first cut into two chunks
    (kSolveChunk = 16); 8 193: n_pad = 8 320, four-tile outer panels and a last outer panel one tile wide"""
    case_ml_columns(n, 3, seed=20)


@pytest.mark.gpu
@pytest.mark.parametrize("m", M_PRED)
@pytest.mark.parametrize("explained", [True, False])
def test_predict_blocks(m, explained):
    case_predict(700, m, explained, max(M_PRED))


@pytest.mark.gpu
@pytest.mark.parametrize("m", [4097, 9000])
def test_predict_taper_blocks(m):
    case_predict_taper(700, m)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 4, 5, 9])
def test_sim_columns(k):
    case_sim(700, k)


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 100, 129, 300])
@pytest.mark.parametrize("k", [1, 5])
@pytest.mark.parametrize("fixed", [False, True])
def test_sim_cond_padding(m, k, fixed):
    case_sim_cond(700, m, k, fixed)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 1100])
@pytest.mark.parametrize("q,r", [(0, 9), (0, 15), (3, 13)])
def test_distributed_single_rank_columns(n, q, r):
    case_distributed(n, q, r)


@pytest.mark.gpu
def test_not_positive_definite_position_in_the_last_outer_panel():
    # n = 3 000: n_pad = 3 072, outer panels of two tiles, the last one (tiles 22, 23) factored on the side stream
    case_not_pd_position(3000, 2900)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", sorted(NAN_BITS))
def test_nan_in_z(pattern):
    case_nan_in_z(1000, pattern)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", sorted(NAN_BITS))
def test_nan_in_resid(pattern):
    case_nan_in_resid(1000, 300, pattern)


# =======================================================================================================================
# the same cases on the host build (n_pad = 256: two tile rows)
# =======================================================================================================================
NH = 130
# The emulated Gram kernel costs ~0.05 s per column pair, so the host takes the cheapest values that still cross each
# cut: two and three passes of n2ll_impl, partial and full 8-column launches, a two-launch mean block.


@pytest.mark.parametrize("r", [1, 2, 5, 9, 17])
def test_host_ml_columns_of_z(product_on_host, r):
    case_ml_columns(NH, r, one_shot=(r <= 5))


@pytest.mark.parametrize("q,r", [(1, 16), (9, 1)])
def test_host_profile_width_of_x_betas(product_on_host, q, r):
    case_profile(NH, q, r, one_shot=(r == 1))


def test_host_reml_width_of_the_design(product_on_host):
    case_reml(NH, 9, 1)


def test_host_limits_are_argument_errors(product_on_host):
    case_limits(NH)


def test_host_profile_betas_against_gls(product_on_host):
    case_profile_betas(NH, _lib.PROFILE, 9, 5)


@pytest.mark.parametrize("n", [1, 2, 127, 129])
def test_host_ml_at_the_factorisation_and_solve_edges(product_on_host, n):
    case_ml_columns(n, 3, seed=20)


def test_host_predict_blocks(product_on_host):
    for m, explained in [(1, True), (129, False), (4097, True)]:
        case_predict(NH, m, explained, 4097)


def test_host_predict_taper_blocks(product_on_host):
    case_predict_taper(NH, 4097)


def test_host_draws(product_on_host):
    for k in (1, 5, 9):
        case_sim(NH, k)
    for m, k, fixed in [(1, 5, False), (129, 1, True), (300, 5, False)]:
        case_sim_cond(NH, m, k, fixed)


def test_host_not_positive_definite_position(product_on_host):
    case_not_pd_position(NH, 129)  # the second tile row


@pytest.mark.parametrize("pattern", sorted(NAN_BITS))
def test_host_nan_in_z_and_resid(product_on_host, pattern):
    case_nan_in_z(NH, pattern)
    case_nan_in_resid(NH, 20, pattern)
