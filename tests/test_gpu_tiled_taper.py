"""The tiled tapered context on a B200: the taper objective goldens through TaperedLikelihood, tiled against dense at
n = 20 000, and at n = 200 000 (whose dense matrix, 320 GB, does not fit one GPU) the properties that need no dense
reference: factor rows against host-computed covariance entries, the diagonal closed form, additivity over two far
apart clusters, reproducible bits and the stored share of the lower triangle."""
import numpy as np
import pytest

import bench
import cocons_b200 as cb
import test_gpu_taper
from oracle import cov

pytestmark = pytest.mark.gpu
PP = test_gpu_taper.PP
N_BIG, DELTA_BIG = 200000, 0.05


def _taper(locs, delta):
    return cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))


def test_objectives_match_goldens_through_the_tiled_context(taper_cases):
    o, c, delta, ref_taper = test_gpu_taper._obj_setup(taper_cases)
    n, lim, z = len(c["locs"]), [0.5, 2.5], o["z"]
    ppp = dict(PP)
    ppp["std.dev"] = np.array([False, True, True])
    with cb.TaperedLikelihood(c["locs"], c["X"], z, ref_taper) as t:
        for _ in range(2):
            v = cb.GetNeg2loglikelihoodTaper(o["theta"], PP, ref_taper, None, None, lim, None, None, n, (0, 0, 0), ctx=t)
            assert abs(v - float(o["ml"])) < 1e-9 * abs(v), (v, float(o["ml"]))
            v = cb.GetNeg2loglikelihoodTaperProfile(o["theta_profile"], ppp, ref_taper, None, None, lim, None, None, n,
                                                    (0, 0, 0), ctx=t)
            assert abs(v - float(o["profile"])) < 1e-9 * abs(v), (v, float(o["profile"]))
    bad = cb.spam(o["notpd_taper"], o["notpd_colindices"], o["notpd_rowpointers"], (n, n))
    with cb.TaperedLikelihood(c["locs"], c["X"], z, bad) as t:
        assert cb.GetNeg2loglikelihoodTaper(o["theta"], PP, bad, None, None, lim, None, None, n, (0, 0, 0),
                                            ctx=t) == 1e6


@pytest.mark.parametrize("delta", [0.11, 0.27])  # about 1 % and 5 % of the pairs
def test_tiled_against_dense_at_20000_sites(delta):
    n = 20000
    locs, X, z1 = bench.synthetic(n)
    z = np.column_stack([z1, 100 * np.roll(z1, 7)])
    sp = _taper(locs, delta)
    tl = dict(bench.THETA)
    with cb.DenseLikelihood(locs, X, z) as d, cb.TaperedLikelihood(locs, X, z, sp) as t:
        d.set_taper(sp)
        want = d.terms_taper(tl, bench.LIMITS, tl["mean"])
        got = t.terms_taper(tl, bench.LIMITS, tl["mean"])
    assert abs(got["logdet"] - want["logdet"]) <= 1e-12 * abs(want["logdet"])
    assert np.all(np.abs(got["quad"] - want["quad"]) <= 1e-12 * np.abs(want["quad"])), (got, want)


@pytest.fixture(scope="module")
def big():
    locs, X, z = bench.synthetic(N_BIG)
    sp = _taper(locs, DELTA_BIG)
    t = cb.TaperedLikelihood(locs, X, z, sp)
    yield locs, X, z, sp, t
    t.close()


def test_factor_rows_reproduce_the_tapered_covariance_at_200000_sites(big):
    locs, X, z, sp, t = big
    tl = dict(bench.THETA)
    t.factor_taper(tl, bench.LIMITS)
    sites = np.random.default_rng(5).choice(N_BIG, 64, replace=False)
    sites[1] = sites[0] + 1  # a few neighbours so that the pattern has entries among them
    rows, pos = t.factor_rows(sites)
    got = rows @ rows.T
    sub = _taper(locs[sites], DELTA_BIG)
    want = np.zeros((64, 64))
    rp = sub.rowpointers.astype(np.int64) - 1
    i = np.repeat(np.arange(64), np.diff(rp))
    j = sub.colindices.astype(np.int64) - 1
    want[i, j] = sub.entries * cov.cov_rns_taper(tl, locs[sites], X[sites], sub.colindices, sub.rowpointers,
                                                 bench.LIMITS)
    scale = np.max(np.abs(want))
    assert np.max(np.abs(got - want)) <= 1e-12 * scale
    st = t.tile_stats()
    T = st["tile_columns"]
    assert st["stored_tiles"] < 0.10 * T * (T + 1) / 2, st


def test_two_evaluations_give_the_same_bits_at_200000_sites(big):
    locs, X, z, sp, t = big
    tl = dict(bench.THETA)
    a = t.terms_taper(tl, bench.LIMITS, tl["mean"])
    b = t.terms_taper(tl, bench.LIMITS, tl["mean"])
    assert a["logdet"] == b["logdet"] and np.array_equal(a["quad"], b["quad"])


def test_diagonal_pattern_at_200000_sites():
    locs, X, z = bench.synthetic(N_BIG)
    tl = dict(bench.THETA)
    sp = cb.nearest_dist(locs, delta=1e-7)
    assert sp.entries.shape[0] == N_BIG
    with cb.TaperedLikelihood(locs, X, z, cb.cov_wend1(sp, (1e-7, 1))) as t:
        st = t.tile_stats()
        assert st["stored_tiles"] == st["tile_columns"] and st["tile_products"] == 0
        r = t.terms_taper(tl, bench.LIMITS, tl["mean"])
    dv = 1 / np.exp(-(X @ tl["std.dev"])) + 1 / np.exp(-(X @ tl["nugget"]))
    resid = z.reshape(-1) - X @ tl["mean"]
    assert abs(r["logdet"] - 0.5 * np.sum(np.log(dv))) < 1e-11 * abs(0.5 * np.sum(np.log(dv)))
    assert abs(r["quad"][0] - np.sum(resid ** 2 / dv)) < 1e-11 * np.sum(resid ** 2 / dv)


def test_two_far_apart_clusters_add_up_at_200000_sites():
    locs, X, z = bench.synthetic(N_BIG)
    h = N_BIG // 2
    locs = locs.copy()
    locs[h:, 0] += 10.0  # beyond any taper radius: the matrix is block diagonal
    tl = dict(bench.THETA)
    parts = []
    for sl in (slice(0, N_BIG), slice(0, h), slice(h, N_BIG)):
        with cb.TaperedLikelihood(locs[sl], X[sl], z[sl], _taper(locs[sl], DELTA_BIG)) as t:
            parts.append(t.terms_taper(tl, bench.LIMITS, tl["mean"]))
    whole, a, b = parts
    assert abs(whole["logdet"] - (a["logdet"] + b["logdet"])) <= 1e-12 * abs(whole["logdet"])
    assert abs(whole["quad"][0] - (a["quad"][0] + b["quad"][0])) <= 1e-12 * whole["quad"][0]


def test_sparse_cocooptim_on_tiled_contexts(taper_cases, datasets):
    obj, o, c = test_gpu_taper._sparse_coco(taper_cases, datasets)
    n = len(c["locs"])
    ref_taper = cb.api._ref_taper(obj)
    dm = cb.getDesignMatrix(obj.model_list, obj.data)
    X = cb.getScale(dm["model.matrix"])["std.covs"]
    rng = np.random.default_rng(1)
    thetas = [o["theta"] + 0.05 * rng.standard_normal(o["theta"].shape) for _ in range(4)]
    with cb.DenseLikelihood(obj.locs, X, obj.z) as d, cb.TaperedLikelihood(obj.locs, X, obj.z, ref_taper) as t:
        d.set_taper(ref_taper)
        for th in thetas:
            vd = cb.GetNeg2loglikelihoodTaper(th, dm["par.pos"], ref_taper, None, None, [0.5, 2.5], None, None, n,
                                              (0, 0, 0), ctx=d)
            vt = cb.GetNeg2loglikelihoodTaper(th, dm["par.pos"], ref_taper, None, None, [0.5, 2.5], None, None, n,
                                              (0, 0, 0), ctx=t)
            assert abs(vt - vd) <= 1e-12 * abs(vd), (vt, vd)
        start = cb.GetNeg2loglikelihoodTaper(o["theta"], dm["par.pos"], ref_taper, None, None, [0.5, 2.5], None, None,
                                             n, (0, 0, 0), ctx=t)
    bounds = {"theta_init": o["theta"], "theta_lower": o["theta"] - 2, "theta_upper": o["theta"] + 2}
    obj.info.update({"lambda.reg": 0.0, "lambda.betas": 0.0, "lambda.Sigma": 0.0})
    out = cb.cocoOptim(obj, bounds, ncores=2, optim_control={"maxiter": 5}, tiled=True)
    assert out.output["value"] <= start
