"""Batched evaluation of the dense objectives: cocons_ctx_create_batch / cocons_n2ll_batch, DenseLikelihoodBatch and the
.Call glue.  Every point's terms must be bit for bit those of a single DenseLikelihood.terms call (the batch runs the
same arithmetic per matrix, in the same order), whatever the batch size, the point's position and the other points.

CPU tests run against the host build of the library's sources (fixture `product_on_host`); the rest needs a B200."""
import numpy as np
import pytest

import cocons_b200 as cb
from cocons_b200 import _lib
from conftest import case_design

KINDS = (_lib.ML, _lib.PROFILE, _lib.REML)


def _design(datasets, name, n, r):
    """(locs, X, z) of holes / stripes cut to n sites, z with r columns (the data's own first, then seeded draws)"""
    c = {"n": n, "dataset": name}
    locs, X, z = case_design(c, datasets)
    if r > 1:
        z = np.column_stack([z[:, 0], np.random.default_rng(n).standard_normal((n, r - 1))])
    return locs, X, z


def _fd_lists(theta, par_pos, eps=1e-4):
    """theta and its 2p central finite-difference neighbours, as theta lists"""
    pts = [theta]
    for i in range(len(theta)):
        for s in (1, -1):
            t = theta.copy()
            t[i] += s * eps
            pts.append(t)
    return [cb.getModelLists(t, par_pos, "diff") for t in pts]


def _single(ctx, kind, lists, lim):
    out = []
    for tl in lists:
        try:
            out.append(ctx.terms(kind, tl, lim, tl["mean"]))
        except cb.NotPositiveDefinite as e:
            out.append(e)
    return out


def _assert_same(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, cb.NotPositiveDefinite):
            assert isinstance(g, cb.NotPositiveDefinite) and g.k == w.k, (i, g, w)
            continue
        assert isinstance(g, dict), (i, g)
        assert g["logdet"] == w["logdet"] and g["logdet_w"] == w["logdet_w"] and g["rank"] == w["rank"], (i, g, w)
        assert np.array_equal(g["quad"], w["quad"]), (i, g["quad"] - w["quad"])


def _prepare(ctx, kind, X, z):
    """the state a kind needs: PROFILE the mean design, REML the contrasts; returns z as set"""
    if kind == _lib.PROFILE:
        ctx.set_xbetas(X)
    zk = cb.reml_contrasts(X, z) if kind == _lib.REML else z
    ctx.set_z(zk)
    return zk


def _compare(locs, X, z, lists, lim, batch, kinds=KINDS):
    with cb.DenseLikelihood(locs, X, z) as one, cb.DenseLikelihoodBatch(locs, X, z, batch) as many:
        for kind in kinds:
            _prepare(one, kind, X, z)
            _prepare(many, kind, X, z)
            want = _single(one, kind, lists, lim)
            _assert_same(many.terms_batch(kind, lists, lim, [tl["mean"] for tl in lists]), want)


def _case_theta(n2ll_cases, name="holes1500_general"):
    c = n2ll_cases[name]
    return c["theta"], c["par_pos"], c["limits"]


# ---- CPU: the host build ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [301, 645])
def test_batch_is_bit_identical_to_single_contexts_on_the_host(product_on_host, n2ll_cases, datasets, n):
    bad = n2ll_cases["holes300_notpd"]
    theta, par_pos, _ = _case_theta(n2ll_cases)
    lim = bad["limits"]  # equal limits: the non-PD point takes the fixed-smoothness branch, the others the general one
    locs, X, z = _design(datasets, "holes", n, 2)
    lists = _fd_lists(theta, par_pos)[:4]
    lists.insert(2, cb.getModelLists(bad["theta"], bad["par_pos"], "diff"))
    with cb.DenseLikelihood(locs, X, z) as one:
        assert isinstance(_single(one, _lib.ML, lists[2:3], lim)[0], cb.NotPositiveDefinite)
    _compare(locs, X, z, lists, lim, 2)  # 5 points, B = 2: groups of 2, 2, 1 with the non-PD point in the second



def _refusals(datasets):
    """n_pad >= 16 384, entries a batch context does not serve, PROFILE without x_betas, a batch call on a dense
    context"""
    locs, X, z = _design(datasets, "holes", 200, 1)
    L = _lib.lib()
    h = _lib._vp()
    big = np.zeros((16257, 2))
    assert L.cocons_ctx_create_batch(0, 16257, 1, 1, _lib.ptr(big), _lib.ptr(np.ones((16257, 1))),
                                     _lib.ptr(np.zeros(16257)), 2, None, h) == -1  # n_pad = 16 384: COCONS_ERR_ARG
    p = X.shape[1]
    th, lim = _lib.ptr(np.zeros(6 * p)), _lib.ptr(np.array([0.5, 0.5]))
    with cb.DenseLikelihoodBatch(locs, X, z, 2) as b:
        assert L.cocons_factor(b._h, _lib.PAR_DIFF, th, lim) == -5  # COCONS_ERR_STATE
        assert L.cocons_ctx_get_factor(b._h, _lib.ptr(np.zeros(200 * 200)), None) == -5
        assert L.cocons_n2ll(b._h, _lib.ML, th, lim, None, _lib.ptr(np.zeros(1)), _lib.ptr(np.zeros(1)), None,
                             None) == -5
        assert L.cocons_sim(b._h, 1, _lib.ptr(np.zeros(200)), _lib.ptr(np.zeros(200))) == -5
        tl = cb.getModelLists(np.zeros(7 * p), {k: np.ones(p, dtype=bool) for k in ("mean",) + _lib.ASPECTS}, "diff")
        with pytest.raises(cb.CoconsError, match="set_xbetas"):
            b.terms_batch(_lib.PROFILE, [tl], [0.5, 0.5])
    with cb.DenseLikelihood(locs, X, z) as d:
        st = np.zeros(1, dtype=np.int32)
        assert L.cocons_n2ll_batch(d._h, _lib.ML, 1, th, lim, None, _lib.ptr(np.zeros(1)), _lib.ptr(np.zeros(1)), None,
                                   None, st.ctypes.data_as(_lib._ip)) == -5


def test_batch_refusals_on_the_host_build(product_on_host, datasets):
    _refusals(datasets)


def _r_batch(R, locs, X, z, lists, lim, batch):
    """_cocons_ctx_new_batch -> _cocons_ctx_n2ll_batch -> _cocons_ctx_free, ML, as rglue/R/cocons_b200.R calls them"""
    p = X.shape[1]
    ctx = R.call("_cocons_ctx_new_batch", locs, X, z, batch, 0)
    thetas = [{k: tl[k] for k in _lib.ASPECTS} for tl in lists]
    logdet, quad, ldw, rank, status = R.call("_cocons_ctx_n2ll_batch", ctx, 0, thetas, p, z.shape[1], lim,
                                             [tl["mean"] for tl in lists])
    assert R.call("_cocons_ctx_free", ctx) is None
    return logdet, np.asarray(quad).reshape(z.shape[1], -1, order="F"), ldw, status


def _r_matches_python(R, locs, X, z, lists, lim, batch):
    logdet, quad, ldw, status = _r_batch(R, locs, X, z, lists, lim, batch)
    with cb.DenseLikelihoodBatch(locs, X, z, batch) as b:
        want = b.terms_batch(_lib.ML, lists, lim, [tl["mean"] for tl in lists])
    for i, w in enumerate(want):
        if isinstance(w, cb.NotPositiveDefinite):
            assert status[i] == w.k
        else:
            assert status[i] == 0 and logdet[i] == w["logdet"] and np.array_equal(quad[:, i], w["quad"])


@pytest.fixture(scope="module")
def R_host(tmp_path_factory, emu):
    from rmock import RMock
    r = RMock(tmp_path_factory.mktemp("rmock_batch_host"), library=emu._name)
    yield r
    r.release_all()


def test_dot_call_batch_on_the_host_build(R_host, product_on_host, n2ll_cases, datasets):
    theta, par_pos, lim = _case_theta(n2ll_cases)
    locs, X, z = _design(datasets, "holes", 300, 1)
    _r_matches_python(R_host, locs, X, z, _fd_lists(theta, par_pos)[:3], lim, 2)


# ---- GPU --------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
GOLDEN = {"holes": ("holes", 5570, "holes_full_general"), "stripes": ("stripes", 11977, "stripes_full_general"),
          "ragged": ("holes", 3001, "holes1500_general")}


@gpu
@pytest.mark.parametrize("r", [1, 10])
@pytest.mark.parametrize("data", ["holes", "stripes", "ragged"])
def test_fd_points_are_bit_identical_to_single_contexts(datasets, n2ll_cases, data, r):
    name, n, case = GOLDEN[data]
    theta, par_pos, lim = _case_theta(n2ll_cases, case)
    locs, X, z = _design(datasets, name, n, r)
    _compare(locs, X, z, _fd_lists(theta, par_pos), lim, 8)


@gpu
@pytest.mark.parametrize("data", ["holes", "stripes"])
def test_composed_values_match_the_goldens(datasets, n2ll_cases, data):
    """the objectives composed from one batch call (cb.api._objectives_batch) against the reference-made values"""
    name, n, case = GOLDEN[data]
    c = n2ll_cases[case]
    if c["n"] != n:
        pytest.skip("golden value not generated")
    locs, X, z = case_design(c, datasets)
    p, lam = c["p"], c["lambda"]
    ppm = dict(c["par_pos"], mean=np.zeros(p, dtype=bool))
    with cb.DenseLikelihoodBatch(locs, X, z, 4) as b:
        got = {"ml": cb.api._objectives_batch(_lib.ML, [c["theta"]], c["par_pos"], c["limits"], n, lam, True, b)[0]}
        b.set_xbetas(X)
        got["profile"] = cb.api._objectives_batch(_lib.PROFILE, [c["theta"][p:]], ppm, c["limits"], n, lam, True, b)[0]
        b.set_z(cb.reml_contrasts(X, z))
        got["reml"] = cb.api._objectives_batch(_lib.REML, [c["theta"][p:]], ppm, c["limits"], n, lam, True, b)[0]
    for k, v in got.items():
        if k in c["values"]:
            assert abs(v - c["values"][k]) < 1e-9 * abs(c["values"][k]), (k, v, c["values"][k])


@gpu
def test_batch_shapes_give_the_same_bits(datasets, n2ll_cases):
    theta, par_pos, lim = _case_theta(n2ll_cases, "holes_full_general")
    locs, X, z = _design(datasets, "holes", 5570, 1)
    lists = _fd_lists(theta, par_pos)[:11]
    B = 4
    with cb.DenseLikelihood(locs, X, z) as one, cb.DenseLikelihoodBatch(locs, X, z, B) as many:
        want = _single(one, _lib.ML, lists, lim)
        means = [tl["mean"] for tl in lists]
        for k in (3, B, 2 * B + 3):  # npoints < B, = B, groups of B, B, 3
            _assert_same(many.terms_batch(_lib.ML, lists[:k], lim, means[:k]), want[:k])
        _assert_same(many.terms_batch(_lib.ML, lists[::-1], lim, means[::-1]), want[::-1])
        _assert_same(many.terms_batch(_lib.ML, lists, lim, means), want)
        _assert_same(many.terms_batch(_lib.ML, lists, lim, means), want)


@gpu
def test_a_batch_mixing_smoothness_modes(datasets, n2ll_cases):
    """equal limits: a point whose smoothness slopes are all zero takes the closed-form nu = 1.5 branch, its
    neighbours the general one - two assembly launches in one group"""
    theta, par_pos, _ = _case_theta(n2ll_cases, "holes_full_general")
    locs, X, z = _design(datasets, "holes", 5570, 1)
    lists = _fd_lists(theta, par_pos)[:5]
    flat = {k: v.copy() for k, v in lists[0].items()}
    flat["smooth"][1:] = 0.0
    lists = [lists[1], flat, lists[2], lists[3], flat, lists[4]]
    _compare(locs, X, z, lists, [1.5, 1.5], 4, kinds=(_lib.ML,))


@gpu
def test_a_point_that_is_not_pd_leaves_the_others_alone(datasets, n2ll_cases):
    c = n2ll_cases["holes300_notpd"]
    locs, X, z = case_design(c, datasets)
    theta, par_pos, _ = _case_theta(n2ll_cases)
    lim = c["limits"]
    lists = _fd_lists(theta, par_pos)[:4]
    lists.insert(2, cb.getModelLists(c["theta"], c["par_pos"], "diff"))
    with cb.DenseLikelihood(locs, X, z) as one:
        want = _single(one, _lib.ML, lists, lim)
    assert isinstance(want[2], cb.NotPositiveDefinite) and all(isinstance(w, dict) for i, w in enumerate(want) if i != 2)
    _compare(locs, X, z, lists, lim, 8, kinds=(_lib.ML,))


@gpu
def test_refusals_and_a_batch_too_large_for_the_device(datasets, n2ll_cases):
    _refusals(datasets)
    locs, X, z = _design(datasets, "stripes", 11977, 1)
    h = _lib._vp()
    assert _lib.lib().cocons_ctx_create_batch(0, len(locs), X.shape[1], 1, _lib.ptr(_lib.fmat(locs)),
                                              _lib.ptr(_lib.fmat(X)), _lib.ptr(_lib.fmat(z)), 1000, None, h) == -4
    theta, par_pos, lim = _case_theta(n2ll_cases, "stripes_full_general")
    _compare(locs[:2000], X[:2000], z[:2000], _fd_lists(theta, par_pos)[:2], lim, 2, kinds=(_lib.ML,))


@gpu
def test_one_launch_per_step_across_the_batch(datasets, n2ll_cases):
    """B = 8 points at holes: no more launches than one evaluation plus 7 x its per-point solves and reductions"""
    theta, par_pos, lim = _case_theta(n2ll_cases, "holes_full_general")
    locs, X, z = _design(datasets, "holes", 5570, 1)
    lists = _fd_lists(theta, par_pos)[:8]
    L = _lib.lib()
    with cb.DenseLikelihood(locs, X, z) as one, cb.DenseLikelihoodBatch(locs, X, z, 8) as many:
        tl = lists[0]
        l0 = L.cocons_launch_count()
        one.terms(_lib.ML, tl, lim, tl["mean"])
        l1 = L.cocons_launch_count()
        one.factor(tl, lim)
        l2 = L.cocons_launch_count()
        many.terms_batch(_lib.ML, lists, lim, [t["mean"] for t in lists])
        l3 = L.cocons_launch_count()
    single, per_point = l1 - l0, (l1 - l0) - (l2 - l1)
    print("launches: one evaluation %d (solves and reductions %d), batch of 8: %d" % (single, per_point, l3 - l2))
    assert l3 - l2 <= single + 7 * per_point


@gpu
def test_dot_call_batch_matches_python(tmp_path, n2ll_cases, datasets):
    from rmock import RMock
    R = RMock(tmp_path)
    try:
        theta, par_pos, lim = _case_theta(n2ll_cases, "holes_full_general")
        locs, X, z = _design(datasets, "holes", 5570, 1)
        _r_matches_python(R, locs, X, z, _fd_lists(theta, par_pos)[:9], lim, 8)
    finally:
        R.release_all()
