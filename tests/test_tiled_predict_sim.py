"""Prediction and simulation on the tiled tapered context (cocons_predict_taper, cocons_sim_taper) on the CPU, through
the product's API bound to the host build of the library's sources (fixture `product_on_host`): the tile-sparse
substitutions and product against a dense context holding the same tapered factor."""
import numpy as np
import pytest

import cocons_b200 as cb
import test_gpu_taper
import test_tiled_taper
from cocons_b200 import _lib

LIM = test_tiled_taper.LIM
TH = test_gpu_taper.theta_dict(np.array([[0.3, 0.1, -0.1], [-1.5, 0.1, 0.1], [0, 0, 0], [0, 0, 0], [0.2, 0.0, 0.1],
                                         [-2.5, 0.1, 0.0]]))


def _pred_sites(m, seed, delta, locs):
    rng = np.random.default_rng(seed)
    lp = rng.uniform(0, 1, (m, 2))
    lp[: min(m, 3)] = locs[[5, 17, 40]][: min(m, 3)]  # some on training sites
    Xp = np.column_stack([np.ones(m), rng.standard_normal((m, 2))])
    return lp, Xp, cb.cov_wend1(cb.nearest_dist(lp, locs, delta=delta), (delta, 1))


def _contexts(n=600, delta=0.09, seed=11):
    locs, X, z = test_tiled_taper._problem(n, seed)
    sp = test_tiled_taper._taper(locs, delta)
    d, t = test_tiled_taper._pair(locs, X, z, sp)
    return locs, X, z, sp, d, t


def _rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


@pytest.mark.parametrize("m", [1, 129, 700])
def test_tiled_predict_taper_matches_the_dense_context(product_on_host, m):
    """n = 600: 5 tile columns, some tiles empty and some filled; m = 700 spans six blocks of 128 sites"""
    delta = 0.09
    locs, X, z, sp, d, t = _contexts(delta=delta)
    lp, Xp, pt = _pred_sites(m, m, delta, locs)
    resid = z[:, 0] - X @ np.array([0.1, -0.2, 0.3])
    with d, t:
        st = t.tile_stats()
        assert st["stored_tiles"] < st["tile_columns"] * (st["tile_columns"] + 1) // 2
        d.factor_taper(TH, LIM)
        t.factor_taper(TH, LIM)
        want_s, want_e = d.predict_taper(lp, Xp, pt, resid)
        got_s, got_e = t.predict_taper(lp, Xp, pt, resid)
        assert _rel(got_s, want_s) <= 1e-12 and _rel(got_e, want_e) <= 1e-12, (_rel(got_s, want_s), _rel(got_e, want_e))
        again_s, again_e = t.predict_taper(lp, Xp, pt, resid)
        assert np.array_equal(again_s, got_s) and np.array_equal(again_e, got_e)
        mean_s, none = t.predict_taper(lp, Xp, pt, resid, want_explained=False)
        assert none is None and np.array_equal(mean_s, got_s)


def test_sites_without_neighbours_predict_exactly_zero(product_on_host):
    delta = 0.09
    locs, X, z, sp, d, t = _contexts(delta=delta)
    lp = np.vstack([[5.0, 5.0], locs[3], [-4.0, 7.0], [0.5, 0.5]])
    Xp = np.column_stack([np.ones(4), np.zeros((4, 2))])
    pt = cb.cov_wend1(cb.nearest_dist(lp, locs, delta=delta), (delta, 1))
    assert np.diff(pt.rowpointers)[[0, 2]].tolist() == [0, 0]
    with t:
        t.factor_taper(TH, LIM)
        s, e = t.predict_taper(lp, Xp, pt, z[:, 0])
    d.close()
    assert s[0] == 0 and e[0] == 0 and s[2] == 0 and e[2] == 0
    assert e[1] > 0 and e[3] > 0


def test_tiled_sim_taper_is_the_expanded_factor_times_eps(product_on_host):
    locs, X, z, sp, d, t = _contexts()
    eps = np.random.default_rng(2).standard_normal((len(locs), 10))
    with d, t:
        t.factor_taper(TH, LIM)
        L, perm = t.get_factor()
        out = t.sim_taper(eps)
        want = L @ eps[perm]
        assert np.max(np.abs(out[perm] - want)) <= 1e-13 * np.max(np.abs(want))
        assert np.array_equal(t.sim_taper(eps), out)
        # k = 32: the 32-column variant of the product
        eps32 = np.random.default_rng(3).standard_normal((len(locs), 32))
        want = L @ eps32[perm]
        assert np.max(np.abs(t.sim_taper(eps32)[perm] - want)) <= 1e-13 * np.max(np.abs(want))
        # a dense context holding a tapered factor: sim_taper is sim itself
        d.factor_taper(TH, LIM)
        assert np.array_equal(d.sim_taper(eps), d.sim(eps))


def test_refusals_without_a_tapered_factor(product_on_host):
    locs, X, z, sp, d, t = _contexts(n=200, delta=0.1)
    lp, Xp, pt = _pred_sites(5, 1, 0.1, locs)
    eps = np.zeros((200, 1))
    with d, t:
        with pytest.raises(cb.CoconsError, match="no tapered factor kept"):
            t.sim_taper(eps)
        with pytest.raises(cb.CoconsError, match="no factor kept"):
            t.predict_taper(lp, Xp, pt, z[:, 0])
        assert _lib.lib().cocons_sim_taper(t._h, 1, _lib.ptr(eps), _lib.ptr(eps)) == -5  # COCONS_ERR_STATE
        d.factor(TH, LIM)  # a dense factor is not a tapered one
        with pytest.raises(cb.CoconsError, match="no tapered factor kept"):
            d.sim_taper(eps)
        t.factor_taper(TH, LIM)
        assert _lib.lib().cocons_sim_taper(t._h, 0, _lib.ptr(eps), _lib.ptr(eps)) == -1  # COCONS_ERR_ARG
        # the dense-only entries still refuse the tiled context
        with pytest.raises(cb.CoconsError, match="tiled tapered context"):
            t.sim(eps)


def test_a_not_positive_definite_taper_keeps_no_factor(product_on_host, taper_cases):
    o, c, delta, _ = test_gpu_taper._obj_setup(taper_cases)
    n = len(c["locs"])
    bad = cb.spam(o["notpd_taper"], o["notpd_colindices"], o["notpd_rowpointers"], (n, n))
    th = cb.getModelLists(o["theta"], test_gpu_taper.PP, "diff")
    with cb.TaperedLikelihood(c["locs"], c["X"], o["z"], bad) as t:
        with pytest.raises(cb.NotPositiveDefinite):
            t.factor_taper(th, LIM)
        with pytest.raises(cb.CoconsError, match="no tapered factor kept"):
            t.sim_taper(np.zeros((n, 1)))


def test_cocopredict_and_cocosim_tiled_match_the_dense_route(product_on_host, taper_cases, datasets):
    obj, o, c = test_gpu_taper._sparse_coco(taper_cases, datasets)
    p = taper_cases["taper_pred_general"]
    HT = datasets["holes_test"]
    m = len(p["locs_pred"])
    new = {"cov_x": HT[:m, 2], "cov_y": HT[:m, 3]}
    want = cb.cocoPredict(obj, new, p["locs_pred"], type="pred")
    got = cb.cocoPredict(obj, new, p["locs_pred"], type="pred", tiled=True)
    assert _rel(got["stochastic"], want["stochastic"]) <= 1e-12
    assert _rel(got["sd.pred"], want["sd.pred"]) <= 1e-12
    eps = np.random.default_rng(5).standard_normal((len(c["locs"]), 3))
    want = cb.cocoSim(obj, eps=eps)
    got = cb.cocoSim(obj, eps=eps, tiled=True)
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    dense = cb.coco("dense", obj.data, obj.locs, obj.z, obj.model_list, info={"smooth.limits": [0.5, 2.5]})
    dense.output = obj.output
    with pytest.raises(ValueError, match="sparse"):
        cb.cocoPredict(dense, new, p["locs_pred"], tiled=True)
    with pytest.raises(ValueError, match="sparse"):
        cb.cocoSim(dense, eps=eps, tiled=True)


def test_tiled_predict_and_sim_through_dot_call_on_the_host_build(product_on_host, tmp_path):
    """R's view: _cocons_ctx_new_taper_tiled -> _cocons_ctx_factor_taper -> _cocons_ctx_predict_taper and
    _cocons_ctx_sim_taper give the Python results bit for bit"""
    from rmock import RMock, RError
    delta = 0.09
    locs, X, z = test_tiled_taper._problem(600, 11)
    sp = test_tiled_taper._taper(locs, delta)
    lp, Xp, pt = _pred_sites(150, 4, delta, locs)
    resid = z[:, 0]
    eps = np.random.default_rng(6).standard_normal((600, 2))
    with cb.TaperedLikelihood(locs, X, z, sp) as t:
        t.factor_taper(TH, LIM)
        want_s, want_e = t.predict_taper(lp, Xp, pt, resid)
        want_d = t.sim_taper(eps)
    R = RMock(tmp_path, library=product_on_host._name)
    try:
        ctx = R.call("_cocons_ctx_new_taper_tiled", locs, X, z, sp.colindices, sp.rowpointers, sp.entries, 0)
        theta6 = {k: TH[k] for k in _lib.ASPECTS}
        R.call("_cocons_ctx_factor_taper", ctx, theta6, 3, LIM)
        pr = R.call("_cocons_ctx_predict_taper", ctx, lp, Xp, pt.colindices, pt.rowpointers, pt.entries, resid)
        draws = R.call("_cocons_ctx_sim_taper", ctx, eps)
        with pytest.raises(RError, match="n x k"):
            R.call("_cocons_ctx_sim_taper", ctx, eps[:10])
        R.call("_cocons_ctx_free", ctx)
    finally:
        R.release_all()
    assert np.array_equal(np.asarray(pr[0]), want_s) and np.array_equal(np.asarray(pr[1]), want_e)
    assert np.array_equal(draws, want_d)
