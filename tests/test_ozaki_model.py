"""The numpy model of the split-int8 trailing update (tools/ozaki_model.py): its integer products are exact, its
slices reassemble the panel, and a blocked Cholesky through it stays within 1e-13 of LAPACK on bench.py's
covariance, plain and tapered."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ozaki_model  # noqa: E402

SLICES = 8


def _panel(m, k, seed):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((m, k)) * np.exp(rng.uniform(-20, 20, m))[:, None]
    P[1] = 0.0
    P[2] = np.ldexp(127.5 / 128, -4)
    return P


def test_slices_are_int8_and_reassemble_the_panel():
    P = _panel(200, 768, 1)
    A, s = ozaki_model.split(P, SLICES)
    assert np.all(np.abs(A[0]) <= 127) and all(np.all(np.abs(a) <= 64) for a in A[1:])
    assert np.array_equal(s, np.ldexp(1.0, np.round(np.log2(s)).astype(int)))  # powers of two
    assert s[2] == np.ldexp(1.0, -3)  # 127.5 / 128 2^-4 would round to 128 at 2^-4: next power
    back = sum(np.ldexp(a, -7 * (t + 1)) for t, a in enumerate(A)) * s[:, None]
    assert np.all(np.abs(back - P) <= np.ldexp(s, -7 * SLICES - 1)[:, None])


def test_weight_sums_are_exact_int64_products():
    P = _panel(96, 768, 2)
    A, _ = ozaki_model.split(P, SLICES)
    S = ozaki_model.weight_sums(A, A, SLICES)
    Ai = [a.astype(np.int64) for a in A]
    for w in range(2, SLICES + 2):
        want = sum(Ai[t - 1] @ Ai[w - t - 1].T for t in range(1, w))
        assert np.array_equal(S[w - 2].astype(np.int64), want)
        assert np.max(np.abs(want)) < 2 ** 31  # int32 accumulators


def test_emulated_product_within_its_bound():
    P = _panel(256, 768, 3)
    got = ozaki_model.emulated_product(P, P, SLICES)
    exact = P @ P.T
    s = ozaki_model.row_scale(P)
    bound = (1152 * 2.0 ** -55 + 768 * 2.0 ** -53) * np.outer(s, s)
    assert np.all(np.abs(got - exact) <= bound)


@pytest.mark.parametrize("taper", [None, 0.27])
def test_blocked_cholesky_through_the_model_against_lapack(taper):
    S, Z = ozaki_model.bench_covariance(2000, taper)
    logdet, quad, residual = ozaki_model.errors(S, ozaki_model.blocked_cholesky(S, SLICES), Z)
    assert logdet < 1e-13 and quad < 1e-13 and residual < 1e-13, (logdet, quad, residual)
