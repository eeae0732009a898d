"""The tiled tapered context (cocons_ctx_create_taper_tiled) on the CPU: the tile-level symbolic analysis against an
independent restatement in numpy, and - through the product's API bound to the host build of the library's sources
(fixture `product_on_host`) - the tiled assembly, factorisation and fused forward substitution against a dense
context's tapered objective on the same data."""
import numpy as np
import pytest

import cocons_b200 as cb
import test_gpu_taper
from cocons_b200 import _lib

PP = test_gpu_taper.PP
LIM = [0.5, 2.5]


def _morton(emu, locs):
    n = len(locs)
    perm = np.empty(n, dtype=np.int64)
    emu.emu_morton(n, _lib.ptr(np.asfortranarray(locs, dtype=np.float64)), perm.ctypes.data_as(_lib._lp))
    return perm


def symbolic_tiles(sp, perm):
    """{tile column J: set of stored tile rows I > J} and the pattern's own lower tiles, by a tile-level symbolic
    Cholesky (each eliminated column adds its rows to those of its parent, the first of them)"""
    n = sp.dimension[0]
    T = (n + 127) // 128
    inv = np.empty(n, dtype=np.int64)
    inv[perm] = np.arange(n)
    rp = sp.rowpointers.astype(np.int64) - 1
    i = np.repeat(np.arange(n), np.diff(rp))
    j = sp.colindices.astype(np.int64) - 1
    keep = i >= j
    ti, tj = inv[i[keep]] // 128, inv[j[keep]] // 128
    lo, hi = np.minimum(ti, tj), np.maximum(ti, tj)
    pattern = {(int(a), int(b)) for a, b in zip(hi, lo) if a != b}
    cols = [set() for _ in range(T)]
    for a, b in pattern:
        cols[b].add(a)
    for J in range(T):
        if cols[J]:
            par = min(cols[J])
            cols[par] |= cols[J] - {par}
    return T, cols, pattern


def expected_stats(sp, perm):
    T, cols, pattern = symbolic_tiles(sp, perm)
    stored = T + sum(len(c) for c in cols)
    return [T, stored, stored - T - len(pattern), sum(len(c) * (len(c) + 1) // 2 for c in cols)]


def _problem(n, seed, r=1):
    rng = np.random.default_rng(seed)
    locs = rng.uniform(0, 1, (n, 2))
    X = np.column_stack([np.ones(n), rng.standard_normal((n, 2))])
    z = rng.standard_normal((n, r)) * np.geomspace(1, 1e3, r)
    return locs, X, z


def _taper(locs, delta):
    return cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))


@pytest.mark.parametrize("n", [1, 127, 129, 700, 3000])
@pytest.mark.parametrize("delta", [1e-9, 0.02, 0.12, 2.0])
def test_tile_stats_match_a_symbolic_elimination_in_numpy(product_on_host, n, delta):
    if delta == 2.0 and n > 700:
        pytest.skip("the full pattern at n = 3000 is 9e6 entries; n = 700 covers it")
    locs, X, z = _problem(n, n)
    sp = _taper(locs, delta)
    with cb.TaperedLikelihood(locs, X, z, sp) as t:
        got = t.tile_stats()
    want = expected_stats(sp, _morton(product_on_host, locs))
    assert [got["tile_columns"], got["stored_tiles"], got["fill_tiles"], got["tile_products"]] == want
    if delta == 1e-9:  # diagonal pattern: no tile below the diagonal, nothing to update
        assert want[1:] == [want[0], 0, 0]
    if delta == 2.0:  # full pattern: the whole lower triangle of tiles
        assert want[1] == want[0] * (want[0] + 1) // 2 and want[2] == 0


def test_every_nonzero_tile_of_the_dense_cholesky_is_stored(product_on_host):
    n, delta = 700, 0.08
    locs, X, z = _problem(n, 3)
    sp = _taper(locs, delta)
    th = test_gpu_taper.theta_dict(np.array([[0.2, 0.1, -0.1], [-1.2, 0.1, 0.1], [0, 0, 0], [0, 0, 0],
                                             [0.1, 0.0, 0.1], [-2.0, 0.1, 0.0]]))
    S = np.zeros((n, n))
    rp = sp.rowpointers.astype(np.int64) - 1
    i = np.repeat(np.arange(n), np.diff(rp))
    j = sp.colindices.astype(np.int64) - 1
    S[i, j] = sp.entries * cb.cov_rns_taper(th, locs, X, sp.colindices, sp.rowpointers, LIM)
    perm = _morton(product_on_host, locs)
    L = np.linalg.cholesky(S[np.ix_(perm, perm)])
    T, cols, _ = symbolic_tiles(sp, perm)
    for I in range(T):
        for J in range(I):
            if np.any(L[128 * I:128 * (I + 1), 128 * J:128 * (J + 1)]):
                assert I in cols[J], (I, J)


def _pair(locs, X, z, sp):
    d = cb.DenseLikelihood(locs, X, z)
    d.set_taper(sp)
    return d, cb.TaperedLikelihood(locs, X, z, sp)


def test_tiled_objective_and_factor_against_the_dense_context(product_on_host):
    """n = 600 (5 tile columns, some off-diagonal tiles empty, some filled), r = 3 columns spread over 1 to 1e3"""
    n = 600
    locs, X, z = _problem(n, 11, r=3)
    sp = _taper(locs, 0.09)
    th = test_gpu_taper.theta_dict(np.array([[0.3, 0.1, -0.1], [-1.5, 0.1, 0.1], [0, 0, 0], [0, 0, 0],
                                             [0.2, 0.0, 0.1], [-2.5, 0.1, 0.0]]))
    mean = np.array([0.1, -0.2, 0.3])
    d, t = _pair(locs, X, z, sp)
    with d, t:
        st = t.tile_stats()
        assert st["stored_tiles"] < st["tile_columns"] * (st["tile_columns"] + 1) // 2  # some tiles are empty
        want = d.terms_taper(th, LIM, mean)
        got = t.terms_taper(th, LIM, mean)
        assert abs(got["logdet"] - want["logdet"]) <= 1e-13 * abs(want["logdet"])
        assert np.all(np.abs(got["quad"] - want["quad"]) <= 1e-13 * np.abs(want["quad"])), (got, want)
        again = t.terms_taper(th, LIM, mean)
        assert again["logdet"] == got["logdet"] and np.array_equal(again["quad"], got["quad"])
        Ld, pd = d.get_factor()
        Lt, pt = t.get_factor()
        assert np.array_equal(pd, pt)
        assert np.max(np.abs(Lt - Ld)) <= 1e-13 * np.max(np.abs(Ld))
        rows, pos = t.factor_rows([0, 5, n - 1])
        assert np.array_equal(rows, Lt[pos]) and np.array_equal(pos, np.argsort(pt)[[0, 5, n - 1]])
        t.factor_taper(th, LIM)  # factor only: the same factor
        assert np.array_equal(t.get_factor()[0], Lt)
        ms = t.timings()
        assert ms["total_ms"] >= 0


def test_golden_objectives_and_not_positive_definite_status(product_on_host, taper_cases):
    o, c, delta, ref_taper = test_gpu_taper._obj_setup(taper_cases)
    n, z = len(c["locs"]), o["z"]
    with cb.TaperedLikelihood(c["locs"], c["X"], z, ref_taper) as t:
        v = cb.GetNeg2loglikelihoodTaper(o["theta"], PP, ref_taper, None, None, LIM, None, None, n, (0, 0, 0), ctx=t)
        assert abs(v - float(o["ml"])) < 1e-9 * abs(v), (v, float(o["ml"]))
    bad = cb.spam(o["notpd_taper"], o["notpd_colindices"], o["notpd_rowpointers"], (n, n))
    th = cb.getModelLists(o["theta"], PP, "diff")
    status = {}
    for cls in ("dense", "tiled"):
        if cls == "dense":
            ctx = cb.DenseLikelihood(c["locs"], c["X"], z)
            ctx.set_taper(bad)
        else:
            ctx = cb.TaperedLikelihood(c["locs"], c["X"], z, bad)
        with ctx:
            with pytest.raises(cb.NotPositiveDefinite) as e:
                ctx.terms_taper(th, LIM, th["mean"])
            status[cls] = e.value.k
    assert status["dense"] == status["tiled"] > 0


def test_dense_only_entries_refuse_a_tiled_context(product_on_host):
    locs, X, z = _problem(200, 5)
    sp = _taper(locs, 0.1)
    th = test_gpu_taper.theta_dict(np.array([[0.3, 0, 0], [-1.5, 0, 0], [0, 0, 0], [0, 0, 0], [0.2, 0, 0],
                                             [-2.5, 0, 0]]))
    with cb.TaperedLikelihood(locs, X, z, sp) as t:
        for call in (lambda: t.terms(_lib.ML, th, LIM, np.zeros(3)), lambda: t.factor(th, LIM),
                     lambda: t.set_taper(sp), lambda: t.predict(locs[:3], X[:3], np.zeros(200)),
                     lambda: t.sim(np.zeros((200, 1))), lambda: t.set_xbetas(X)):
            with pytest.raises(cb.CoconsError, match="tiled tapered context"):
                call()
        kms, kfl = _lib.ctypes.c_double(), _lib.ctypes.c_double()
        assert _lib.lib().cocons_ctx_kernel_timing(t._h, _lib.ctypes.byref(kms), _lib.ctypes.byref(kfl)) == -5
        t.terms_taper(th, LIM, np.zeros(3))  # still usable
    with cb.DenseLikelihood(locs, X, z) as d:
        out = np.empty(4, dtype=np.int64)
        assert _lib.lib().cocons_ctx_tile_stats(d._h, out.ctypes.data_as(_lib._lp)) == -5
        assert b"dense" in _lib.lib().cocons_last_error()
    with pytest.raises(cb.CoconsError, match="bad argument"):
        cb.TaperedLikelihood(locs, X, np.zeros((200, 129)), sp)


def test_tiled_context_through_dot_call_on_the_host_build(product_on_host, taper_cases, tmp_path):
    """R's view: _cocons_ctx_new_taper_tiled gives the external pointer that _cocons_ctx_n2ll_taper takes as it is"""
    from rmock import RMock, RError
    R = RMock(tmp_path, library=product_on_host._name)
    try:
        o, c, delta, ref_taper = test_gpu_taper._obj_setup(taper_cases)
        n, z = len(c["locs"]), o["z"]
        th = cb.getModelLists(o["theta"], PP, "diff")
        col, row = ref_taper.colindices, ref_taper.rowpointers
        with pytest.raises(RError, match="rowpointers"):  # checked before any device call
            R.call("_cocons_ctx_new_taper_tiled", c["locs"], c["X"], z, col, row[:-1], ref_taper.entries, 0)
        ctx = R.call("_cocons_ctx_new_taper_tiled", c["locs"], c["X"], z, col, row, ref_taper.entries, 0)
        theta6 = {k: th[k] for k in _lib.ASPECTS}
        out = R.call("_cocons_ctx_n2ll_taper", ctx, theta6, 3, z.shape[1], LIM, th["mean"])
        with cb.TaperedLikelihood(c["locs"], c["X"], z, ref_taper) as t:
            want = t.terms_taper(th, LIM, th["mean"])
        assert out[0] == 0 and out[1] == want["logdet"] and np.array_equal(out[2:], want["quad"])
        v = n * np.log(2 * np.pi) * z.shape[1] + 2 * z.shape[1] * out[1] + np.sum(out[2:])
        assert abs(v - float(o["ml"])) < 1e-9 * abs(v)
        R.call("_cocons_ctx_free", ctx)
    finally:
        R.release_all()
