"""The split-int8 trailing update (csrc/syrk_i8.cu) on a B200: bit for bit what the numpy model of
tools/ozaki_model.py computes, within the model's worst-case bound of the DMMA update on random and real panels,
reproducible, and evaluations with COCONS_SYRK_I8=0 / 1 that agree to 1e-13."""
import ctypes
import os
import sys

import numpy as np
import pytest

import bench
import cocons_b200 as cb
from cocons_b200 import _lib

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ozaki_model  # noqa: E402

pytestmark = pytest.mark.gpu
K, SLICES = 768, 8


def _update(P, C, path):
    P = np.asfortranarray(P, dtype=np.float64)
    out = np.array(C, dtype=np.float64, order="F")
    m = P.shape[0]
    _lib.check(_lib.lib().cocons_trailing_update(0, m, P.ctypes.data_as(_lib._dp), out.ctypes.data_as(_lib._dp), path,
                                                 0, None))
    return out


def _lower_tiles(m):
    """entries the update writes: the 128 x 64 tiles (bi, c) with bi >= c / 2, i.e. the lower 128-blocks"""
    r = np.arange(m) // 128
    return r[:, None] >= r[None, :]


def _random_panel(m, seed):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((m, K)) * np.exp(rng.uniform(-20, 20, m))[:, None]  # rows over 17 decades
    P[5] = 0.0                                                                  # a zero row (padding)
    P[7, :] = 0.0
    P[7, 3] = 1.0                                                               # one entry at the rounding edge
    P[9] = np.ldexp(127.5 / 128, 3) * np.sign(rng.standard_normal(K))           # |P| = 127.5 / 128 2^3 everywhere
    return P


def _real_panel(n=4096):
    """rows below the first 768 columns of the factor of bench.py's covariance (n sites): an actual K = 768 panel"""
    from oracle import cov
    locs, X, _ = bench.synthetic(n)
    S = cov.cov_rns(bench.theta_at(1, 0), locs, X, bench.LIMITS)
    S = np.tril(S) + np.tril(S, -1).T
    L = np.linalg.cholesky(S)
    return L[K:, :K], S[K:, K:]


@pytest.mark.parametrize("panel", ["random", "real"])
def test_int8_update_is_the_model_bit_for_bit(panel):
    if panel == "random":
        P = _random_panel(1024, 1)
        C = np.random.default_rng(2).standard_normal((1024, 1024))
    else:
        P, C = _real_panel()
    got = _update(P, C, 1)
    want = C - ozaki_model.emulated_product(P, P, SLICES)
    low = _lower_tiles(P.shape[0])
    assert np.array_equal(got[low], want[low])
    assert np.array_equal(got[~low], C[~low])  # tiles above the diagonal blocks are not touched


@pytest.mark.parametrize("panel", ["random", "real"])
def test_int8_update_against_dmma_within_the_model_bound(panel):
    if panel == "random":
        P = _random_panel(1280, 3)
        C = np.random.default_rng(4).standard_normal((1280, 1280))
    else:
        P, C = _real_panel()
    i8, dm = _update(P, C, 1), _update(P, C, 0)
    s = ozaki_model.row_scale(P)
    # |emulated - exact| <= 768 (7 2^-58 + 2^-56 + ...) s_i s_j <= 1152 2^-55 s_i s_j (dropped slice pairs and the
    # remainder of the 8th slice), |DMMA - exact| <= 768 2^-53 sum_k |P_ik P_jk| <= 768 2^-53 s_i s_j, plus one
    # rounding of C on each side
    bound = (1152 * 2.0 ** -55 + 768 * 2.0 ** -53) * np.outer(s, s) + 2 * np.spacing(np.abs(dm))
    low = _lower_tiles(P.shape[0])
    err = np.abs(i8 - dm)[low]
    assert np.all(err <= bound[low]), float(np.max(err / bound[low]))
    print("%s panel: max |int8 - DMMA| / bound = %.3f" % (panel, float(np.max(err / bound[low]))))


def test_int8_update_repeats_bit_identically():
    P = _random_panel(2048, 5)
    C = np.random.default_rng(6).standard_normal((2048, 2048))
    first = _update(P, C, 1)
    for _ in range(2):
        assert np.array_equal(_update(P, C, 1), first)


@pytest.mark.parametrize("n", [20000, 50000])
def test_evaluations_with_and_without_the_int8_update(n, monkeypatch):
    locs, X, z1 = bench.synthetic(n)
    z = np.column_stack([z1, 100 * np.roll(z1, 7)])
    tl = bench.theta_at(0, 0)
    out = {}
    with cb.DenseLikelihood(locs, X, z) as d:
        for flag in ("0", "1", "0", "1"):
            monkeypatch.setenv("COCONS_SYRK_I8", flag)
            t = d.terms(_lib.ML, tl, bench.LIMITS, tl["mean"])
            if flag in out:  # each path reproduces itself bit for bit
                assert t["logdet"] == out[flag]["logdet"] and np.array_equal(t["quad"], out[flag]["quad"])
            out[flag] = t
    a, b = out["0"], out["1"]
    assert abs(b["logdet"] - a["logdet"]) <= 1e-13 * abs(a["logdet"]), (a, b)
    assert np.all(np.abs(b["quad"] - a["quad"]) <= 1e-13 * np.abs(a["quad"])), (a, b)
    assert b["logdet"] != a["logdet"] or not np.array_equal(b["quad"], a["quad"])  # the int8 path did run
    print("n=%d: logdet %.3e rel, quad %.3e rel" % (n, abs(b["logdet"] - a["logdet"]) / abs(a["logdet"]),
                                                   float(np.max(np.abs(b["quad"] - a["quad"]) / np.abs(a["quad"])))))


def test_int8_update_is_faster_than_dmma():
    m = 49152
    ms = {}
    for path in (0, 1):
        v = ctypes.c_double()
        _lib.check(_lib.lib().cocons_trailing_update(0, m, None, None, path, 3, ctypes.byref(v)))
        ms[path] = v.value
    flops = (m / 128) * (m / 128 + 1) / 2 * 2 * 128 * 128 * K
    print("m=%d: DMMA %.2f ms (%.1f TFLOP/s), int8 %.2f ms (%.1f TFLOP/s FP64-equivalent)"
          % (m, ms[0], flops / ms[0] / 1e9, ms[1], flops / ms[1] / 1e9))
    assert ms[1] < ms[0]
