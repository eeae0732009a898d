"""The persistent split-int8 update (csrc/syrk_i8.cu) at the edges of its tiling: bit for bit the numpy model of
tools/ozaki_model.py at 1, 2, 3, 9 and 11 tile rows of 128 - fewer tiles than SMs and several per SM, and, in a
build with 2 x 2 clusters, odd and even numbers of tile rows, one and several super-tiles of 256 x 128 and diagonal
super-tiles whose upper-row CTA feeds its cluster and stores nothing - the tiles above the diagonal blocks
untouched, and the same bits on a repeat; evaluations with COCONS_SYRK_I8=0 / 1 just above its threshold."""
import os
import sys

import numpy as np
import pytest

from cocons_b200 import _lib

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ozaki_model  # noqa: E402

pytestmark = pytest.mark.gpu
K, SLICES = 768, 8


def _update(P, C):
    P = np.asfortranarray(P, dtype=np.float64)
    out = np.array(C, dtype=np.float64, order="F")
    _lib.check(_lib.lib().cocons_trailing_update(0, P.shape[0], P.ctypes.data_as(_lib._dp),
                                                 out.ctypes.data_as(_lib._dp), 1, 0, None))
    return out


def _panel(m, seed):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((m, K)) * np.exp(rng.uniform(-8, 8, m))[:, None]
    P[m // 2] = 0.0  # a zero row
    return P


@pytest.mark.parametrize("m", [128, 256, 384, 1152, 1408])
def test_cluster_update_is_the_model_bit_for_bit(m):
    P = _panel(m, m)
    C = np.random.default_rng(m + 1).standard_normal((m, m))
    got = _update(P, C)
    want = C - ozaki_model.emulated_product(P, P, SLICES)
    r = np.arange(m) // 128
    low = r[:, None] >= r[None, :]
    assert np.array_equal(got[low], want[low])
    assert np.array_equal(got[~low], C[~low])
    assert np.array_equal(_update(P, C), got)  # a repeat gives the same bits


def test_evaluations_with_and_without_the_int8_update_just_above_its_threshold(monkeypatch):
    """17 500 sites: the first trailing update (16 768 rows) is the only one that runs on the int8 path"""
    import bench
    import cocons_b200 as cb
    locs, X, z1 = bench.synthetic(17500)
    z = np.column_stack([z1, 100 * np.roll(z1, 7)])
    tl = bench.theta_at(0, 0)
    out = {}
    with cb.DenseLikelihood(locs, X, z) as d:
        for flag in ("0", "1"):
            monkeypatch.setenv("COCONS_SYRK_I8", flag)
            out[flag] = d.terms(_lib.ML, tl, bench.LIMITS, tl["mean"])
    a, b = out["0"], out["1"]
    assert abs(b["logdet"] - a["logdet"]) <= 1e-13 * abs(a["logdet"]), (a, b)
    assert np.all(np.abs(b["quad"] - a["quad"]) <= 1e-13 * np.abs(a["quad"])), (a, b)
    assert b["logdet"] != a["logdet"] or not np.array_equal(b["quad"], a["quad"])  # the int8 path did run
