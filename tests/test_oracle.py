"""Pins the oracle (CPU restatement under oracle/) before anything is compared with it.

The reference's own tests hold no numeric goldens for this path (tests/coco_test.R only
asserts shapes / positive eigenvalues / absence of NA, SURVEY.md §4), so the pins are:
  * bit equality with the reference's own src/cocons_full.cpp compiled here (oracle/_ref),
    live when that library is present and through the committed tests/golden/cov_cases.npz
    it generated otherwise;
  * 40-digit mpmath evaluations of the mathematical formula;
  * closed forms, the stationary textbook Matern limit and the Profile/REML identities.
"""
import os

import mpmath as mp
import numpy as np
import pytest

from conftest import relerr, theta_dict
from oracle import cov, fresh_inputs, rmirror


def _run_square(case, kind):
    th = theta_dict(case["theta6"])
    if "limits" in case:
        return cov.cov_rns(th, case["locs"], case["X"], case["limits"], kind=kind)
    return cov.cov_rns_classic(th, case["locs"], case["X"], kind=kind)


def _run_case(case, kind):
    if "locs_pred" in case:
        return cov.cov_rns_pred(theta_dict(case["theta6"]), case["locs"], case["locs_pred"], case["X"],
                                case["X_pred"], case["limits"], kind=kind)
    return _run_square(case, kind)


def test_restatement_reproduces_reference_goldens_bit_for_bit(cov_cases):
    assert len(cov_cases) >= 18
    for name, case in cov_cases.items():
        got = _run_case(case, "restatement")
        assert np.array_equal(got, case["out"]), name


@pytest.mark.skipif(not cov.have_reference(), reason="needs the reference's source (COCONS_REFERENCE)")
def test_compiled_reference_reproduces_its_goldens(cov_cases):
    for name, case in cov_cases.items():
        assert np.array_equal(_run_case(case, "reference"), case["out"]), name


@pytest.mark.skipif(not cov.have_reference(), reason="needs the reference's source (COCONS_REFERENCE)")
def test_restatement_equals_compiled_reference_on_fresh_inputs():
    for call in fresh_inputs.dense_calls():
        assert np.array_equal(fresh_inputs.run(call, "restatement"), fresh_inputs.run(call, "reference")), call[0]


FRESH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fresh_cases.npz")


@pytest.mark.skipif(not os.path.exists(FRESH), reason="tests/golden/fresh_cases.npz not generated "
                                                      "(python -m oracle.make_golden --only fresh, needs the reference)")
def test_restatement_reproduces_the_stored_reference_results_on_fresh_inputs():
    stored = np.load(FRESH)
    for call in list(fresh_inputs.dense_calls()) + list(fresh_inputs.taper_calls()):
        assert np.array_equal(fresh_inputs.run(call, "restatement"), stored[call[0]]), call[0]


def test_bessel_stand_in_against_mpmath():
    mp.mp.dps = 40
    worst = 0.0
    for nu in (0.3, 0.5, 1.0, 1.7, 2.5, 3.3):
        for x in (1e-6, 1e-3, 0.1, 1.0, 1.999, 2.001, 5.0, 16.5, 25.0, 100.0, 700.0):
            ref = mp.besselk(mp.mpf(nu), mp.mpf(x))
            worst = max(worst, float(abs((mp.mpf(cov.bessel_k(nu, x)) - ref) / ref)))
    assert worst < 5e-15


def _mp_entry(th, xi, xj, li, lj, lim):
    """Mathematical formula (Paciorek-Schervish kernel with effective-range scaling), SURVEY App. A."""
    mp.mp.dps = 50
    f = lambda v: mp.mpf(float(v))
    dot = lambda b, x: mp.fsum(f(bk) * f(xk) for bk, xk in zip(b, x))
    gr = mp.exp(2 * f(th["scale"][0]))
    sje = np.array(th["scale"], dtype=float).copy()
    sje[0] = 0.0

    def site(x):
        t = mp.pi / (1 + mp.exp(-dot(th["tilt"], x)))
        r = mp.exp(2 * dot(sje, x))
        a = mp.exp(dot(th["aniso"], x))
        nu = (f(lim[1]) - f(lim[0])) / (1 + mp.exp(-dot(th["smooth"], x))) + f(lim[0])
        return t, r, a, mp.exp(dot(th["std.dev"], x) / 2), nu

    ti, ri, ai, si, nui = site(xi)
    tj, rj, aj, sj, nuj = site(xj)
    s11 = (ri + rj) / 2
    s22 = (ri * ai ** 2 + rj * aj ** 2) / 2
    s12 = (ri * ai * mp.cos(ti) + rj * aj * mp.cos(tj)) / 2
    det = s11 * s22 - s12 ** 2
    dx, dy = f(li[0]) - f(lj[0]), f(li[1]) - f(lj[1])
    nu = mp.sqrt(nui * nuj)
    Q = mp.sqrt(8 * nu / (gr * det)) * mp.sqrt(s22 * dx ** 2 + s11 * dy ** 2 - 2 * s12 * dx * dy)
    corr = 2 ** (1 - nu) / mp.gamma(nu) * Q ** nu * mp.besselk(nu, Q)
    pre = si * sj * mp.sqrt(ri * ai * mp.sin(ti) * rj * aj * mp.sin(tj)) / mp.sqrt(det)
    return corr * pre, Q


def test_general_branch_against_mpmath(cov_cases):
    case = cov_cases["general_all_aspects"]
    th = theta_dict(case["theta6"])
    S = case["out"]
    rng = np.random.default_rng(3)
    worst = 0.0
    for _ in range(40):
        i, j = rng.choice(S.shape[0], 2, replace=False)
        ref, Q = _mp_entry(th, case["X"][i], case["X"][j], case["locs"][i], case["locs"][j], case["limits"])
        # the entry is ~exp(-Q): a 1-ulp change of a site quantity moves it by ~Q ulp
        worst = max(worst, float(abs((mp.mpf(S[i, j]) - ref) / ref)) / max(1.0, float(Q)))
    assert worst < 2e-15


def test_closed_forms_equal_bessel_branch(cov_cases):
    for name, nu in (("nu05_fixed", 0.5), ("nu15_vignette", 1.5), ("nu25_fixed", 2.5)):
        case = cov_cases[name]
        th = theta_dict(case["theta6"])
        # same model forced through the general branch: limits a hair apart, constant logistic
        eps = 1e-13
        th2 = dict(th)
        th2["smooth"] = th["smooth"].copy()
        g = cov.cov_rns(th2, case["locs"], case["X"], [nu - eps, nu + eps], "restatement")
        assert relerr(g, case["out"]) < 5e-12, name


def test_stationary_limit_is_textbook_matern():
    rng = np.random.default_rng(11)
    n, p = 50, 3
    locs = rng.uniform(-1, 1, (n, 2))
    X = np.column_stack([np.ones(n), rng.standard_normal((n, p - 1))])
    th = {k: np.zeros(p) for k in cov.ASPECTS}
    sigma2, rho, nu = 1.7, 0.4, 1.5
    th["std.dev"][0] = np.log(sigma2)
    th["scale"][0] = np.log(rho)
    th["nugget"][0] = -np.inf
    S = cov.cov_rns(th, locs, X, [nu, nu], "restatement")
    d = np.linalg.norm(locs[:, None, :] - locs[None, :, :], axis=2)
    Q = np.sqrt(8 * nu) * d / rho
    M = sigma2 * (1 + Q) * np.exp(-Q)
    assert relerr(S, M) < 1e-12
    assert np.array_equal(S, S.T)
    assert np.all(np.linalg.eigvalsh(S) > 0)


def test_quirks_are_preserved(cov_cases):
    # App. B-1: fixed non-half-integer smoothness -> every off-diagonal equals the row's variance
    S = cov_cases["degenerate_nu1_fixed"]["out"]
    i, j = 3, 50
    assert S[i, j] == S[i, i] and S[j, i] == S[i, i]
    # App. B-2: duplicated locations get variance + nugget of the lower index
    S = cov_cases["general_duplicates"]["out"]
    assert S[5, 90] == S[5, 5] and S[90, 5] == S[5, 5]
    assert S[17, 100] == S[17, 17]
    # cov_rns_pred: a prediction site on a training site takes its OWN variance + nugget
    case = cov_cases["pred_general"]
    th = theta_dict(case["theta6"])
    own = np.exp(case["X_pred"] @ th["std.dev"]) + np.exp(case["X_pred"] @ th["nugget"])
    assert abs(case["out"][3, 10] - own[3]) < 1e-14 * own[3]
    # App. B-4: cov_rns_pred never takes the closed forms
    a = cov.cov_rns(theta_dict(cov_cases["nu15_vignette"]["theta6"]), case["locs"], case["X"], [1.5, 1.5])
    b = cov.cov_rns_pred(theta_dict(cov_cases["nu15_vignette"]["theta6"]), case["locs"], case["locs"], case["X"],
                         case["X"], [1.5, 1.5])
    off = ~np.eye(a.shape[0], dtype=bool)
    assert relerr(b[off], a[off]) < 1e-12


def test_objective_golden_values_and_identities(n2ll_cases, datasets):
    from conftest import case_design
    for name in ("holes777_ragged", "holes1500_nu15"):
        c = n2ll_cases[name]
        locs, X, z = case_design(c, datasets)
        n, p = c["n"], c["p"]
        lam = c["lambda"]
        v = rmirror.neg2loglik(c["theta"], c["par_pos"], locs, X, c["limits"], z, n, lam)
        assert abs(v - c["values"]["ml"]) <= 1e-12 * abs(v)
        # Profile / REML identities of SURVEY.md §8c(v): z'Pz = |y|^2 - b'W^-1 b
        ppm = dict(c["par_pos"])
        ppm["mean"] = np.zeros(p, dtype=bool)
        tl = rmirror.get_model_lists(c["theta"][p:], ppm, "diff")
        S = cov.cov_rns(tl, locs, X, c["limits"])
        R = rmirror.r_chol(S)
        Yx = rmirror._fwd(R, X)
        yz = rmirror._fwd(R, z[:, 0])
        W, b = Yx.T @ Yx, Yx.T @ yz
        quad = yz @ yz - b @ np.linalg.solve(W, b)
        logdet = np.sum(np.log(np.diag(R)))
        prof = n * np.log(2 * np.pi) + 2 * logdet + quad
        assert abs(prof - c["values"]["profile"]) <= 1e-10 * abs(prof)


def test_host_helpers():
    par_pos = {"mean": np.array([True, True, False]), "std.dev": np.array([True, False, True]),
               "scale": np.array([True, True, True]), "aniso": 0.0, "tilt": 0.0, "smooth": 1.5, "nugget": -np.inf}
    theta = np.arange(1.0, 9.0)
    tl = rmirror.get_model_lists(theta, par_pos, "diff")
    assert np.array_equal(tl["mean"], [1, 2, 0])
    # std.dev free at columns 0,2 ; scale free at 0,1,2: 'diff' applies where both are free
    assert np.allclose(tl["std.dev"], [(3 + 5) / 2, 0, (4 + 7) / 2])
    assert np.allclose(tl["scale"], [(3 - 5) / 2, 6, (4 - 7) / 2])
    assert tl["smooth"][0] == 1.5 and np.isneginf(tl["nugget"][0])
    X = np.column_stack([np.ones(5), np.arange(5.0), np.arange(5.0) ** 2])
    sc = rmirror.get_scale(X)
    assert np.allclose(sc["std.covs"][:, 1].std(ddof=1), 1.0) and np.allclose(sc["std.covs"][:, 0], 1.0)
    assert rmirror.r_qr_rank(X) == 3
    assert rmirror.r_qr_rank(np.column_stack([X, X[:, 1] * 2])) == 3


def test_sigma_sample_fixture_matches_the_oracle():
    """The fixture bench.py checks its n = 100 000 factor against is what the oracle gives for those sites."""
    import bench
    from conftest import GOLD
    fx = np.load(os.path.join(GOLD, "sigma_samples.npz"))
    n = 100000
    locs, X, _, _, _, th = bench.north_star_problem(n)
    sites = bench.sampled_sites(n)
    assert np.array_equal(fx["sites_n%d" % n], sites)
    kind = "reference" if cov.have_reference() else "restatement"
    S = cov.cov_rns(th, np.asfortranarray(locs[sites]), np.asfortranarray(X[sites]), bench.LIMITS, kind=kind)
    assert np.array_equal(S, fx["sigma_n%d" % n])
