"""The split-int8 trailing update (csrc/syrk_i8.cu) where an int8 split can go wrong, held to exact references.

Kernel (cocons_trailing_update, m = 1024): on the adversarial panels of tests/exact_syrk.py (17 decades, maxima at
and just below the split's powers of two, one dominant entry, alternating signs, 2^+-500, subnormal row maxima) the
int8 path is the numpy model bit for bit, and both paths stay within their own bounds of C - P P^T computed exactly;
a NaN, +Inf, -Inf or NaN row in the panel makes every entry of that row and column NaN, wherever the DMMA path gives
a non-finite one.  Objectives at 17 500 sites (the first trailing update runs on the int8 path): a NaN taper entry or
a NaN location is not positive definite on both paths; on an ill-conditioned covariance (nugget 1e-8, smoothness at
its upper limit) the int8 error of 1/2 logdet stays within the envelope of tests/test_ozaki_model.py against LAPACK
at 17 500 sites, and within 1e-9 of the DMMA path at 50 000."""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

import bench
import cocons_b200 as cb
import exact_syrk
from cocons_b200 import _lib

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ozaki_model  # noqa: E402

pytestmark = pytest.mark.gpu
K, SLICES, M = 768, 8, 1024
ENVELOPE_C = 16.0  # tests/test_ozaki_model.py::ENVELOPE_C


def _update(P, C, path):
    P = np.asfortranarray(P, dtype=np.float64)
    out = np.array(C, dtype=np.float64, order="F")
    _lib.check(_lib.lib().cocons_trailing_update(0, P.shape[0], P.ctypes.data_as(_lib._dp),
                                                 out.ctypes.data_as(_lib._dp), path, 0, None))
    return out


def _lower_tiles(m):
    r = np.arange(m) // 128
    return r[:, None] >= r[None, :]


@pytest.mark.parametrize("kind", exact_syrk.PANELS)
def test_int8_update_is_the_model_bit_for_bit_on_adversarial_panels(kind):
    P, C = exact_syrk.adversarial_panel(kind, M, 21)
    got = _update(P, C, 1)
    want = C - ozaki_model.emulated_product(P, P, SLICES)
    low = _lower_tiles(M)
    bad = np.flatnonzero(got[low].view(np.int64) != want[low].view(np.int64))
    assert bad.size == 0, (kind, bad.size, got[low][bad[:4]], want[low][bad[:4]])
    assert np.array_equal(got[~low], C[~low])


@pytest.mark.parametrize("kind", exact_syrk.PANELS)
def test_both_paths_within_their_bounds_of_the_exact_update(kind):
    """int8: |got - exact| <= 1152 2^-55 s_i s_j + the roundings of the product and of the subtraction (with half the
    least subnormal for each scaling by s_i, s_j that underflows).  DMMA: <= 768 2^-53 sum_k |P_ik P_jk| (FP64 sums
    of 768 products, in any order) + the rounding of the subtraction, + 768 halves of the least subnormal for the
    products and partial sums that underflow."""
    P, C = exact_syrk.adversarial_panel(kind, M, 22)
    i8, dm = _update(P, C, 1), _update(P, C, 0)
    y = ozaki_model.emulated_product(P, P, SLICES)
    s = ozaki_model.row_scale(P)
    ii, jj = exact_syrk.sample_lower(M, np.random.default_rng(23), blocks=((0, 64), (-64, 64)), count=2000)
    R = exact_syrk.ExactRows(P)
    tiny = exact_syrk.TINY
    worst = [0.0, 0.0]
    for i, j in zip(ii, jj):
        exact = Fraction(float(C[i, j])) - R.dot(i, j)
        si, sj = Fraction(float(s[i])), Fraction(float(s[j]))
        b8 = (1152 * si * sj / 2 ** 55 + exact_syrk.ulp(y[i, j]) / 2 + tiny / 2 * (1 + sj)
              + exact_syrk.ulp(i8[i, j]) / 2)
        bd = 768 * (1 + Fraction(1, 2 ** 40)) * R.abs_dot(i, j) / 2 ** 53 + exact_syrk.ulp(dm[i, j]) / 2 + 384 * tiny
        e8, ed = abs(Fraction(float(i8[i, j])) - exact), abs(Fraction(float(dm[i, j])) - exact)
        assert e8 <= b8, ("int8", kind, i, j, float(e8), float(b8))
        assert ed <= bd, ("DMMA", kind, i, j, float(ed), float(bd))
        worst = [max(worst[0], float(e8 / b8)), max(worst[1], float(ed / bd))]
    print("%s: max error / bound: int8 %.3f, DMMA %.3f" % (kind, worst[0], worst[1]))


def test_non_finite_panel_rows_make_their_rows_and_columns_nan():
    """a NaN, +Inf, -Inf entry and a NaN row: int8 is NaN in every entry of those rows and columns - non-finite at
    least wherever DMMA is - the rest is the model bit for bit, and the tiles above the diagonal blocks are untouched"""
    P, C, bad = exact_syrk.nonfinite_panel(M, 24)
    with np.errstate(invalid="ignore"):
        i8, dm = _update(P, C, 1), _update(P, C, 0)
        want = C - ozaki_model.emulated_product(P, P, SLICES)
    low = _lower_tiles(M)
    touch = np.zeros(M, dtype=bool)
    touch[bad] = True
    touch2 = (touch[:, None] | touch[None, :]) & low
    assert np.all(~np.isfinite(dm[low]) <= ~np.isfinite(i8[low]))
    assert np.all(np.isnan(i8[touch2]))
    rest = low & ~touch2
    assert np.array_equal(i8[rest], want[rest])
    assert np.array_equal(i8[~low], C[~low])


# ---- objectives at 17 500 sites: the first trailing update (16 768 rows) is the only one on the int8 path --------

N_I8 = 17500


def _par_pos(p=5):
    return {k: np.ones(p, dtype=bool) for k in ("mean", "std.dev", "scale", "aniso", "tilt", "smooth", "nugget")}


def _not_pd_on_both_paths(evaluate, objective, monkeypatch):
    for flag in ("0", "1"):
        monkeypatch.setenv("COCONS_SYRK_I8", flag)
        with pytest.raises(cb.NotPositiveDefinite):
            evaluate()
        assert objective() == 1e6, flag


def test_nan_taper_entry_is_not_positive_definite_on_both_paths(monkeypatch):
    """a NaN taper entry between a site among the first 768 of the context's order and one beyond: the NaN enters
    the first panel's rows below its diagonal block, and so reaches the int8 update, not the panel's own pivots"""
    locs, X, z = bench.synthetic(N_I8)
    tl = bench.theta_at(0, 0)
    delta = 0.15
    taper = cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))
    near = np.argsort(locs[:, 0] + locs[:, 1])[:600]  # the corner where Morton order starts
    theta = bench.theta_vec(tl, _par_pos())
    with cb.DenseLikelihood(locs, X, z) as ctx:
        ctx.set_taper(taper)
        for flag in ("0", "1"):
            monkeypatch.setenv("COCONS_SYRK_I8", flag)
            assert np.isfinite(ctx.terms_taper(tl, bench.LIMITS, tl["mean"])["logdet"])
        _, pos = ctx.factor_rows(near)
        a = int(near[np.argmax(np.where(pos < 768, pos, -1))])  # the last of the first panel among them
        rp, ci = taper.rowpointers - 1, taper.colindices - 1
        nbr = ci[rp[a]:rp[a + 1]]
        _, npos = ctx.factor_rows(nbr)
        assert np.any(npos >= 768), "site %d has no taper neighbour beyond the first panel" % a
        b = int(nbr[np.argmax(npos)])
        bad = taper.copy()
        for r, c in ((a, b), (b, a)):
            bad.entries[rp[r] + np.searchsorted(ci[rp[r]:rp[r + 1]], c)] = np.nan
        ctx.set_taper(bad)
        _not_pd_on_both_paths(
            lambda: ctx.terms_taper(tl, bench.LIMITS, tl["mean"]),
            lambda: cb.GetNeg2loglikelihoodTaper(theta, _par_pos(), bad, None, None, bench.LIMITS, None, None, N_I8,
                                                 (0, 0, 0), ctx=ctx), monkeypatch)


@pytest.mark.parametrize("coords", ["x", "xy"])
def test_nan_location_is_not_positive_definite_on_both_paths(coords, monkeypatch):
    """a NaN location makes its row of the covariance NaN.  x: the site with the largest y, its x NaN - the Morton
    order places it past the first panel; xy: both coordinates NaN - it comes first, in the first panel"""
    locs, X, z = bench.synthetic(N_I8)
    site = int(np.argmax(locs[:, 1]))
    locs = np.array(locs, order="F")
    locs[site, 0] = np.nan
    if coords == "xy":
        locs[site, 1] = np.nan
    tl = bench.theta_at(0, 0)
    theta = bench.theta_vec(tl, _par_pos())
    with cb.DenseLikelihood(locs, X, z) as ctx:
        _not_pd_on_both_paths(
            lambda: ctx.terms(_lib.ML, tl, bench.LIMITS, tl["mean"]),
            lambda: cb.GetNeg2loglikelihood(theta, _par_pos(), None, None, bench.LIMITS, None, N_I8, (0, 0, 0),
                                            ctx=ctx), monkeypatch)


def _ill_conditioned_theta():
    """bench.py's model with the nugget intercept at log 1e-8, the smoothness at its upper limit (2.5) and a
    longer scale"""
    th = {k: v.copy() for k, v in bench.THETA.items()}
    th["nugget"][0] = np.log(1e-8)
    th["smooth"][:] = 0.0
    th["smooth"][0] = 30.0
    th["scale"][0] = -0.6
    return th


def _sampled_backward_error(ctx, S_sites, sites):
    rows, _ = ctx.factor_rows(sites)
    d = np.sqrt(np.diag(S_sites))
    return float(np.max(np.abs(rows @ rows.T - S_sites) / np.outer(d, d)))


def _both_paths(n, monkeypatch, S_of_sites):
    locs, X, z = bench.synthetic(n)
    th = _ill_conditioned_theta()
    sites = bench.sampled_sites(n, m=64)
    out = {}
    with cb.DenseLikelihood(locs, X, z) as ctx:
        for flag in ("0", "1"):
            monkeypatch.setenv("COCONS_SYRK_I8", flag)
            t = ctx.terms(_lib.ML, th, bench.LIMITS, th["mean"])
            out[flag] = (t["logdet"], _sampled_backward_error(ctx, S_of_sites(locs, X, th, sites), sites))
    return out


def test_ill_conditioned_sweep_at_17500_sites_against_lapack(monkeypatch):
    """errors of 1/2 logdet against LAPACK on the device-assembled covariance (so that assembly rounding cancels):
    int8 <= ENVELOPE_C x DMMA + 1e-13 |1/2 logdet|; sampled backward errors of both factors below 1e-13 (measured
    on B200: DMMA -2.9e-6, int8 +3.6e-7 of 1.1e5; backward errors 1.2e-15 and 1.3e-15)"""
    locs, X, _ = bench.synthetic(N_I8)
    th = _ill_conditioned_theta()
    S = cb.cov_rns(th, locs, X, bench.LIMITS)
    S = np.tril(S) + np.tril(S, -1).T
    ref = float(np.sum(np.log(np.diag(np.linalg.cholesky(S)))))
    out = _both_paths(N_I8, monkeypatch, lambda locs, X, th, sites: S[np.ix_(sites, sites)])
    del S
    e_dm, e_i8 = abs(out["0"][0] - ref), abs(out["1"][0] - ref)
    print("\nn=%d nugget 1e-8: 1/2 logdet (LAPACK) %.6f | DMMA - ref %+.2e | int8 - ref %+.2e | ratio %.1f | "
          "backward error DMMA %.2e int8 %.2e" % (N_I8, ref, out["0"][0] - ref, out["1"][0] - ref, e_i8 / e_dm,
                                                  out["0"][1], out["1"][1]))
    assert e_i8 <= ENVELOPE_C * e_dm + 1e-13 * abs(ref), (e_i8, e_dm)
    assert out["0"][1] < 1e-13 and out["1"][1] < 1e-13, out


def test_ill_conditioned_int8_against_dmma_at_50000_sites(monkeypatch):
    """no CPU reference at this size, so the two paths against each other: |int8 - DMMA| of 1/2 logdet, the sum of
    both errors, within 1e-9 relative (measured on B200: 2.9e-10, where the FP64 error alone is not known), and
    sampled backward errors of both factors below 1e-13 (measured: 1.4e-15 and 1.3e-15)"""
    n = 50000
    out = _both_paths(n, monkeypatch, lambda locs, X, th, sites: cb.cov_rns(th, locs[sites], X[sites], bench.LIMITS))
    diff = abs(out["1"][0] - out["0"][0])
    print("\nn=%d nugget 1e-8: 1/2 logdet (DMMA) %.6f | int8 - DMMA %+.2e (rel %.2e) | backward error DMMA %.2e "
          "int8 %.2e" % (n, out["0"][0], out["1"][0] - out["0"][0], diff / abs(out["0"][0]), out["0"][1],
                         out["1"][1]))
    assert diff <= 1e-9 * abs(out["0"][0]), out
    assert out["0"][1] < 1e-13 and out["1"][1] < 1e-13, out
