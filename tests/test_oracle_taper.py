"""Pins the oracle of the sparse (tapered) model (SURVEY.md §8f N3) before the CUDA path is compared with
it: the plain-array restatement of src/cocons_taper.cpp must be bit-equal to the reference's own source
compiled here (oracle/_ref) - live when that library is present, through the committed
tests/golden/taper_cases.npz otherwise - and the host-side `spam` stand-ins must agree with the brute-force
ones the goldens were generated with."""
import numpy as np
import pytest

import cocons_b200 as cb
from conftest import theta_dict
from oracle import cov, fresh_inputs, rmirror


def _entries(case, kind):
    th = theta_dict(case["theta6"])
    if "locs_pred" in case:
        return cov.cov_rns_taper_pred(th, case["locs"], case["locs_pred"], case["X"], case["X_pred"],
                                      case["colindices"], case["rowpointers"], case["limits"], kind=kind)
    return cov.cov_rns_taper(th, case["locs"], case["X"], case["colindices"], case["rowpointers"], case["limits"],
                             kind=kind)


def _cov_cases(taper_cases):
    return {k: v for k, v in taper_cases.items() if k != "obj"}


def test_restatement_reproduces_reference_goldens_bit_for_bit(taper_cases):
    cases = _cov_cases(taper_cases)
    assert len(cases) >= 11
    for name, case in cases.items():
        assert np.array_equal(_entries(case, "restatement"), case["out"]), name


@pytest.mark.skipif(not cov.have_reference(), reason="needs the reference's source (COCONS_REFERENCE)")
def test_compiled_reference_reproduces_its_goldens(taper_cases):
    for name, case in _cov_cases(taper_cases).items():
        assert np.array_equal(_entries(case, "reference"), case["out"]), name


@pytest.mark.skipif(not cov.have_reference(), reason="needs the reference's source (COCONS_REFERENCE)")
def test_restatement_equals_compiled_reference_on_fresh_inputs():
    for call in fresh_inputs.taper_calls():
        assert np.array_equal(fresh_inputs.run(call, "restatement"), fresh_inputs.run(call, "reference")), call[0]


def test_tapered_family_is_the_isotropic_member_of_the_dense_one(taper_cases):
    """With aniso = tilt = 0 the dense kernel (src/cocons_full.cpp) and the tapered one (src/cocons_taper.cpp)
    are the same function written twice; their entries agree to rounding."""
    c = taper_cases["taper_general"]
    th = theta_dict(c["theta6"])
    dense = cov.cov_rns(th, c["locs"], c["X"], c["limits"])
    rows = np.repeat(np.arange(len(c["rowpointers"]) - 1), np.diff(c["rowpointers"].astype(np.int64)))
    cols = c["colindices"].astype(np.int64) - 1
    assert np.allclose(dense[rows, cols], c["out"], rtol=1e-12, atol=0)


def test_quirks_are_preserved(taper_cases):
    # fixed non-half-integer smoothness: every stored entry is the ROW site's variance + nugget
    c = taper_cases["taper_degenerate_nu1"]
    rp = c["rowpointers"].astype(np.int64)
    for i in (0, 17, 499):
        row = c["out"][rp[i] - 1:rp[i + 1] - 1]
        assert np.all(row == row[0])
    # duplicated locations: the coincident entry equals the row's diagonal value
    c = taper_cases["taper_duplicates"]
    rp, ci = c["rowpointers"].astype(np.int64), c["colindices"].astype(np.int64)
    def entry(i, j):
        seg = slice(rp[i] - 1, rp[i + 1] - 1)
        return c["out"][seg][np.flatnonzero(ci[seg] == j + 1)[0]]
    assert entry(90, 5) == entry(90, 90) and entry(5, 90) == entry(5, 5)
    # a prediction site sitting on a training site: sigma_pred^2 + nugget_pred, not the Matern value
    c = taper_cases["taper_pred_general"]
    assert np.array_equal(c["locs_pred"][3], c["locs"][10])


def test_spam_stand_ins_match_the_brute_force_ones(taper_cases):
    c = taper_cases["taper_general"]
    delta = float(taper_cases["obj"]["delta"])
    d, ci, rp = rmirror.nearest_dist(c["locs"], delta=delta)
    assert np.array_equal(ci, c["colindices"]) and np.array_equal(rp, c["rowpointers"])
    sp = cb.nearest_dist(c["locs"], delta=delta)
    assert np.array_equal(sp.colindices, ci) and np.array_equal(sp.rowpointers, rp)
    assert np.allclose(sp.entries, d, rtol=0, atol=1e-15)
    w = cb.cov_wend1(sp, (delta, 1))
    assert isinstance(w, cb.spam) and np.allclose(w.entries, rmirror.cov_wend1(d, (delta, 1)), rtol=0, atol=1e-15)
    assert w.entries.max() == 1.0 and w.entries.min() >= 0.0 and 0 < w.density() < 1
    # rectangular (prediction) pattern
    p = taper_cases["taper_pred_general"]
    sp2 = cb.nearest_dist(p["locs_pred"], p["locs"], delta=delta)
    assert np.array_equal(sp2.colindices, p["colindices"]) and np.array_equal(sp2.rowpointers, p["rowpointers"])
    assert sp2.dimension == (len(p["locs_pred"]), len(p["locs"]))
    # Wendland-2 at a few points of its documented formula
    assert np.allclose(cb.cov_wend2(np.array([0.0, 0.5, 1.0, 2.0]), (1.0, 1.0)),
                       [1.0, 0.5 ** 6 * (1 + 3 + 35 / 12), 0.0, 0.0])


def test_objective_goldens_are_reproduced_by_the_restatement(taper_cases):
    """The committed objective values were computed with the compiled reference's entries; the restatement
    (bit-equal entries) must give the same numbers on this machine's LAPACK to rounding."""
    o, c = taper_cases["obj"], taper_cases["taper_general"]
    n = len(c["locs"])
    pp = {k: np.ones(3, dtype=bool) for k in rmirror.ASPECT_ORDER}
    pp["aniso"], pp["tilt"] = 0.0, 0.0
    d, ci, rp = rmirror.nearest_dist(c["locs"], delta=float(o["delta"]))
    taper = rmirror.cov_wend1(d, (float(o["delta"]), 1))
    v = rmirror.neg2loglik_taper(o["theta"], pp, taper, ci, rp, c["locs"], c["X"], [0.5, 2.5], o["z"], n, (0, 0, 0))
    assert abs(v - float(o["ml"])) < 1e-11 * abs(v)
    ppp = dict(pp)
    ppp["std.dev"] = np.array([False, True, True])
    v = rmirror.neg2loglik_taper_profile(o["theta_profile"], ppp, taper, ci, rp, c["locs"], c["X"], [0.5, 2.5], o["z"],
                                         n, (0, 0, 0))
    assert abs(v - float(o["profile"])) < 1e-11 * abs(v)
    v = rmirror.neg2loglik_taper(o["theta"], pp, o["notpd_taper"], o["notpd_colindices"], o["notpd_rowpointers"],
                                 c["locs"], c["X"], [0.5, 2.5], o["z"], n, (0, 0, 0))
    assert v == 1e6 == float(o["notpd"])
    # profile identity: at the profiled variance the Profile value equals the full value
    tl = rmirror.get_model_lists(o["theta_profile"], ppp, "diff")
    tl["std.dev"][0] = 0.0
    logdet, quads = rmirror._taper_chol_terms(tl, taper, ci, rp, c["locs"], c["X"], [0.5, 2.5], o["z"], n,
                                              "restatement")
    r = len(quads)
    s0 = sum(quads) / (r * n)
    full = sum(n * np.log(2 * np.pi) + 2 * (logdet + 0.5 * n * np.log(s0)) + q / s0 for q in quads)
    assert abs(full - float(o["profile"])) < 1e-12 * abs(full)
