"""TEST INFRASTRUCTURE ONLY (oracle/): seeded inputs, beyond the golden cases, on which the restatement must equal the
reference bit for bit (tests/test_oracle.py, tests/test_oracle_taper.py).

Each call is (key, name of the oracle.cov function, positional arguments).  oracle/make_golden.py --only fresh stores
the reference's result of every call in tests/golden/fresh_cases.npz under its key.
"""
import numpy as np

from . import cov, rmirror


def dense_calls():
    rng = np.random.default_rng(7)
    for p, n in ((1, 40), (3, 90), (5, 61)):
        locs = rng.uniform(-1, 1, (n, 2))
        X = np.column_stack([np.ones(n), rng.standard_normal((n, p - 1))])
        th = {k: 0.3 * rng.standard_normal(p) for k in cov.ASPECTS}
        th["scale"][0] = -1.5
        th["nugget"][0] = -3.0
        yield "dense_p%d_cov_rns" % p, "cov_rns", (th, locs, X, [0.5, 2.5])
        yield "dense_p%d_cov_rns_classic" % p, "cov_rns_classic", (th, locs, X)
        lp = rng.uniform(-1, 1, (17, 2))
        Xp = np.column_stack([np.ones(17), rng.standard_normal((17, p - 1))])
        yield "dense_p%d_cov_rns_pred" % p, "cov_rns_pred", (th, locs, lp, X, Xp, [0.5, 2.5])
        x = rng.standard_normal(9) * np.array([1, 1e-5, 1, 1e-6, 0, 1, 1, 1e-4, 1])
        yield "dense_p%d_sumsmoothlone" % p, "sumsmoothlone", (x, 0.3)


def taper_calls():
    rng = np.random.default_rng(11)
    for p, n, delta in ((1, 60, 0.5), (3, 150, 0.3), (5, 97, 0.4)):
        locs = rng.uniform(-1, 1, (n, 2))
        X = np.column_stack([np.ones(n), rng.standard_normal((n, p - 1))])
        th = {k: 0.3 * rng.standard_normal(p) for k in cov.ASPECTS}
        th["scale"][0], th["nugget"][0] = -2.0, -3.0
        _, ci, rp = rmirror.nearest_dist(locs, delta=delta)
        for lim in ([0.5, 2.5], [0.3, 0.9]):
            yield "taper_p%d_lim%g_%g" % (p, *lim), "cov_rns_taper", (th, locs, X, ci, rp, lim)
        th0 = dict(th, smooth=np.zeros(p))
        for lim in ([0.5, 0.5], [1.5, 1.5], [2.5, 2.5], [1.0, 1.0]):
            yield "taper_p%d_fixed_nu%g" % (p, lim[0]), "cov_rns_taper", (th0, locs, X, ci, rp, lim)
        lp = rng.uniform(-1, 1, (23, 2))
        lp[4] = locs[9]
        Xp = np.column_stack([np.ones(23), rng.standard_normal((23, p - 1))])
        _, cip, rpp = rmirror.nearest_dist(lp, locs, delta=delta)
        yield "taper_p%d_pred" % p, "cov_rns_taper_pred", (th, locs, lp, X, Xp, cip, rpp, [0.5, 2.5])


def run(call, kind):
    _, fn, args = call
    return getattr(cov, fn)(*args, kind=kind)
