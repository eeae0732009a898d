"""Prediction and simulation on the tiled tapered context on a B200: tiled against dense at n = 20 000, and at
n = 200 000 (whose dense matrix, 320 GB, does not fit one GPU) the properties that need no dense reference: unit-vector
draws against the factor's rows, additivity of predictions over two far-apart clusters, bounds and reproducible bits,
and the public cocoPredict / cocoSim end to end."""
import numpy as np
import pytest

import bench
import cocons_b200 as cb

pytestmark = pytest.mark.gpu
N_BIG, DELTA_BIG = 200000, 0.05


def _taper(locs, delta):
    return cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))


def _raw(locs):
    """bench.synthetic's covariates before scaling: smooth functions of the location"""
    c1, c2 = (locs[:, 0] + 1) / 2, (locs[:, 1] + 1) / 2
    return np.column_stack([np.ones(len(locs)), c1, c2, c1 * c2,
                            0.5 + 0.5 * np.sin(np.pi * locs[:, 0]) * np.cos(np.pi * locs[:, 1])])


def _pred_sites(m, seed, locs, delta):
    """m sites over the training sites' box, some on training sites, with the training design's covariates scaled as
    the training design is (so that a site's parameters are those of its neighbours)"""
    rng = np.random.default_rng(seed)
    lo, hi = locs.min(axis=0), locs.max(axis=0)
    lp = lo + (hi - lo) * rng.uniform(0, 1, (m, 2))
    lp[:5] = locs[rng.choice(len(locs), 5, replace=False)]
    raw = _raw(locs)
    mean, sd = raw.mean(axis=0), raw.std(axis=0, ddof=1)
    mean[0], sd[0] = 0.0, 1.0
    Xp = (_raw(lp) - mean) / sd
    return lp, Xp, cb.cov_wend1(cb.nearest_dist(lp, locs, delta=delta), (delta, 1))


def _rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


@pytest.mark.parametrize("delta", [0.11, 0.27])
def test_tiled_predict_and_sim_against_dense_at_20000_sites(delta):
    n = 20000
    locs, X, z = bench.synthetic(n)
    sp = _taper(locs, delta)
    tl = dict(bench.THETA)
    lp, Xp, pt = _pred_sites(2000, 1, locs, delta)
    resid = z - X @ tl["mean"]
    eps = np.random.default_rng(2).standard_normal((n, 10))
    with cb.DenseLikelihood(locs, X, z) as d, cb.TaperedLikelihood(locs, X, z, sp) as t:
        d.set_taper(sp)
        d.factor_taper(tl, bench.LIMITS)
        t.factor_taper(tl, bench.LIMITS)
        want_s, want_e = d.predict_taper(lp, Xp, pt, resid)
        got_s, got_e = t.predict_taper(lp, Xp, pt, resid)
        want_d, got_d = d.sim_taper(eps), t.sim_taper(eps)
        assert np.array_equal(want_d, d.sim(eps))
    # the kriging mean is a sum of terms of both signs: relative to its largest value; the explained variance is a sum
    # of squares: relative at every site
    assert np.max(np.abs(got_s - want_s)) <= 1e-12 * np.max(np.abs(want_s)), np.max(np.abs(got_s - want_s))
    assert _rel(got_e, want_e) <= 1e-12, _rel(got_e, want_e)
    assert np.max(np.abs(got_d - want_d)) <= 1e-12 * np.max(np.abs(want_d))


@pytest.fixture(scope="module")
def big():
    locs, X, z = bench.synthetic(N_BIG)
    t = cb.TaperedLikelihood(locs, X, z, _taper(locs, DELTA_BIG))
    tl = dict(bench.THETA)
    t.factor_taper(tl, bench.LIMITS)
    yield locs, X, z, t, tl
    t.close()


def test_unit_vector_draws_are_the_factor_rows_at_200000_sites(big):
    locs, X, z, t, tl = big
    rng = np.random.default_rng(7)
    sites = rng.choice(N_BIG, 8, replace=False)
    d2 = np.sum((locs - locs[sites[0]]) ** 2, axis=1)
    sites[1:4] = np.argsort(d2)[1:4]  # neighbours of the first site
    rows, pos = t.factor_rows(sites)
    eps = np.zeros((N_BIG, 8))
    eps[sites, np.arange(8)] = 1.0
    out = t.sim_taper(eps)
    for a in range(8):
        for j in range(8):
            assert out[sites[a], j] == rows[a, pos[j]], (a, j)


def test_bounds_and_reproducible_bits_at_200000_sites(big):
    locs, X, z, t, tl = big
    lp, Xp, pt = _pred_sites(3000, 3, locs, DELTA_BIG)
    resid = z - X @ tl["mean"]
    s1, e1 = t.predict_taper(lp, Xp, pt, resid)
    s2, e2 = t.predict_taper(lp, Xp, pt, resid)
    assert np.array_equal(s1, s2) and np.array_equal(e1, e2)
    prior = 1 / np.exp(-(Xp @ tl["std.dev"])) + 1 / np.exp(-(Xp @ tl["nugget"]))  # sigma^2 + nugget
    assert np.all(e1 >= 0) and np.all(e1 <= prior * (1 + 1e-12))


def test_two_far_apart_clusters_predict_alone_at_200000_sites():
    locs, X, z = bench.synthetic(N_BIG)
    h = N_BIG // 2
    locs = locs.copy()
    locs[h:, 0] += 10.0  # beyond any taper radius: the matrix is block diagonal
    tl = dict(bench.THETA)
    resid = z - X @ tl["mean"]
    lp, Xp, _ = _pred_sites(2000, 4, locs[:h], DELTA_BIG)  # inside cluster A
    out = []
    for sl in (slice(0, N_BIG), slice(0, h)):
        with cb.TaperedLikelihood(locs[sl], X[sl], z[sl], _taper(locs[sl], DELTA_BIG)) as t:
            t.factor_taper(tl, bench.LIMITS)
            out.append(t.predict_taper(lp, Xp, _taper_pred(lp, locs[sl]), resid[sl]))
    (sw, ew), (sa, ea) = out
    assert np.max(np.abs(sw - sa)) <= 1e-12 * np.max(np.abs(sa))
    assert np.max(np.abs(ew - ea)) <= 1e-12 * np.max(np.abs(ea))


def _taper_pred(lp, locs):
    return cb.cov_wend1(cb.nearest_dist(lp, locs, delta=DELTA_BIG), (DELTA_BIG, 1))


def test_cocopredict_and_cocosim_tiled_end_to_end_at_200000_sites(taper_cases):
    """the model of the sparse golden case (three covariates) on the bench's 200 000 sites"""
    o = taper_cases["obj"]
    locs, _, z = bench.synthetic(N_BIG)
    rng = np.random.default_rng(9)
    data = {"cov_x": (locs[:, 0] + 1) / 2, "cov_y": (locs[:, 1] + 1) / 2}
    f = "~ 1 + cov_x + cov_y"
    obj = cb.coco("sparse", data, locs, z, {"mean": f, "std.dev": f, "scale": f, "smooth": f, "nugget": f},
                  info={"smooth.limits": [0.5, 2.5], "taper": cb.cov_wend1, "delta": DELTA_BIG})
    sc = cb.getScale(cb.getDesignMatrix(obj.model_list, obj.data)["model.matrix"])
    obj.info.update({"mean.vector": sc["mean.vector"], "sd.vector": sc["sd.vector"]})
    obj.output = {"par": o["theta"]}
    m = 20000
    lp = rng.uniform(locs.min(axis=0), locs.max(axis=0), (m, 2))
    new = {"cov_x": rng.uniform(0, 1, m), "cov_y": rng.uniform(0, 1, m)}
    out = cb.cocoPredict(obj, new, lp, type="pred", tiled=True)
    assert out["stochastic"].shape == (m,) and np.all(np.isfinite(out["sd.pred"]))
    sim = cb.cocoSim(obj, n=2, seed=3, tiled=True)
    assert sim.shape == (N_BIG, 2) and np.all(np.isfinite(sim))
