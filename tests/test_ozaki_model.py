"""The numpy model of the split-int8 trailing update (tools/ozaki_model.py): its integer products are exact, its
slices reassemble the panel, and a blocked Cholesky through it stays within 1e-13 of LAPACK on bench.py's
covariance, plain and tapered."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ozaki_model  # noqa: E402

import exact_syrk  # noqa: E402  (tests/exact_syrk.py)

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


# ---- against an exact reference (tests/exact_syrk.py) ----------------------------------------------------------

def test_exact_reference_against_fractions():
    """the integer dot products of exact_syrk against plain Fraction sums, on rows of magnitude 1, 2^500, 2^-500 and
    with subnormal entries, and the one rounding to FP64 against float(Fraction)"""
    from fractions import Fraction
    rng = np.random.default_rng(8)
    P = rng.standard_normal((6, 768))
    P[1] = np.ldexp(P[1], 500)
    P[2] = np.ldexp(P[2], -500)
    P[3] = np.ldexp(P[3], -1060)          # subnormal entries
    P[4, ::2] = np.ldexp(P[4, ::2], -1070)  # normal and subnormal entries in one row
    P[5] = 0.0
    C = rng.standard_normal((6, 6))
    R = exact_syrk.ExactRows(P)
    pairs = [(0, 0), (1, 0), (1, 1), (2, 1), (3, 0), (3, 3), (4, 0), (4, 3), (4, 4), (5, 2)]
    for i, j in pairs:
        want = sum(Fraction(a) * Fraction(b) for a, b in zip(P[i], P[j]))
        assert R.dot(i, j) == want
        assert R.abs_dot(i, j) == sum(abs(Fraction(a) * Fraction(b)) for a, b in zip(P[i], P[j]))
    ii, jj = zip(*pairs)
    ex = exact_syrk.exact_update(C, P, ii, jj)
    assert ex == [Fraction(C[i, j]) - R.dot(i, j) for i, j in pairs]
    got = exact_syrk.rounded(ex)
    assert all(got[t] == float(ex[t]) for t in range(len(pairs)))
    assert float(R.dot(3, 0)) != 0.0 and float(R.dot(3, 3)) == 0.0  # 2^-1060 x 1 survives, 2^-2120 underflows
    assert abs(Fraction(float(R.dot(3, 0))) - R.dot(3, 0)) <= exact_syrk.TINY / 2  # rounded in the subnormal range


def int8_bound(got, s_i, s_j):
    """|emulated - exact| allowed for one entry: 1152 2^-55 s_i s_j (the dropped slice pairs and the remainder of the
    last slice), half an ulp of the result (the one rounding of hi 2^-35 + lo 2^-63; scaling by s_i s_j is exact),
    and, where v s_i or its product with s_j lands below 2^-1022, half the least subnormal for each of those two
    roundings (the first scaled by s_j)"""
    from fractions import Fraction
    si, sj = Fraction(float(s_i)), Fraction(float(s_j))
    return 1152 * si * sj / 2 ** 55 + exact_syrk.ulp(got) / 2 + exact_syrk.TINY / 2 * (1 + sj)


@pytest.mark.parametrize("kind", exact_syrk.PANELS)
def test_emulated_product_within_its_bound_of_the_exact_product(kind):
    """the model's P P^T on adversarial panels against the exact product at sampled entries: within 1152 2^-55
    s_i s_j plus its own rounding (no FP64 product, and so no 768 2^-53 slack, in the reference)"""
    P, _ = exact_syrk.adversarial_panel(kind, 512, 11)
    got = ozaki_model.emulated_product(P, P, SLICES)
    s = ozaki_model.row_scale(P)
    ii, jj = exact_syrk.sample_lower(512, np.random.default_rng(12), blocks=((0, 48), (-48, 48)), count=1500)
    R = exact_syrk.ExactRows(P)
    worst = 0.0
    for i, j in zip(ii, jj):
        from fractions import Fraction
        err = abs(Fraction(float(got[i, j])) - R.dot(i, j))
        b = int8_bound(got[i, j], s[i], s[j])
        assert err <= b, (kind, i, j, float(err), float(b))
        worst = max(worst, float(err / b))
    print("%s: max |emulated - exact| / bound = %.3f" % (kind, worst))


def test_subnormal_row_maxima_split_exactly():
    """a row whose maximum is below 2^-1022 gets s = 2^e with e down to -1073: its slices reassemble the row as for a
    normal row (2^-e overflows there, P 2^-e does not)"""
    P, _ = exact_syrk.adversarial_panel("subnormal", 64, 3)
    A, s = ozaki_model.split(P, SLICES)
    assert s[5] == np.ldexp(1.0, -1073) and np.min(s) < np.ldexp(1.0, -1030)
    assert np.all(np.abs(A[0]) <= 127) and all(np.all(np.abs(a) <= 64) for a in A[1:])
    back = sum(np.ldexp(a, -7 * (t + 1)) for t, a in enumerate(A))  # P / s, exact in FP64
    assert np.all(np.abs(back - np.ldexp(P, -np.round(np.log2(s)).astype(int)[:, None])) <= np.ldexp(1.0, -57))


def test_non_finite_rows_make_their_rows_and_columns_nan():
    """a row with a NaN or infinite entry has the scale NaN: every product in its row and column is NaN - non-finite
    wherever P P^T in FP64 is - and every other entry is what the model gives without those rows"""
    P, _, bad = exact_syrk.nonfinite_panel(256, 5)
    got = ozaki_model.emulated_product(P, P, SLICES)
    touch = np.zeros(256, dtype=bool)
    touch[bad] = True
    touch2 = touch[:, None] | touch[None, :]
    assert np.all(np.isnan(ozaki_model.row_scale(P)[bad]))
    assert np.all(np.isnan(got[touch2]))
    with np.errstate(invalid="ignore"):
        assert np.all(~np.isfinite(P @ P.T)[touch2] <= np.isnan(got[touch2]))
    clean = P.copy()
    clean[bad] = 0.0
    want = ozaki_model.emulated_product(clean, clean, SLICES)
    assert np.array_equal(got[~touch2], want[~touch2])


# ---- accuracy on ill-conditioned covariances ---------------------------------------------------------------------

# int8 error of 1/2 logdet <= ENVELOPE_C x (FP64 error) + 1e-13 |1/2 logdet|.  Measured with the model at 1536 sites
# (below): the int8 error has one sign and is 2.5-9x the FP64 blocked Cholesky's; tests/test_gpu_syrk_i8_edges.py
# holds the kernel to the same envelope at 17 500 and 50 000 sites.
ENVELOPE_C = 16.0


def _cholesky_longdouble(S, b=96):
    """lower Cholesky factor in 80-bit long double (right-looking, blocks of b): the reference of the sweep"""
    A = np.array(S, dtype=np.longdouble)
    n = A.shape[0]
    for j0 in range(0, n, b):
        j1 = min(n, j0 + b)
        D = A[j0:j1, j0:j1]
        for k in range(j1 - j0):
            D[k, k] = np.sqrt(D[k, k] - D[k, :k] @ D[k, :k])
            D[k + 1:, k] = (D[k + 1:, k] - D[k + 1:, :k] @ D[k, :k]) / D[k, k]
        L = np.tril(D)
        A[j0:j1, j0:j1] = L
        if j1 == n:
            break
        X = A[j1:, j0:j1]
        for k in range(j1 - j0):
            X[:, k] = (X[:, k] - X[:, :k] @ L[k, :k]) / L[k, k]
        A[j1:, j1:] -= X @ X.T
    return np.tril(A)


def test_ill_conditioned_sweep_within_the_envelope():
    """Matern 1.5 (range 0.3) on 1536 uniform sites with nuggets 1e-2 .. 1e-8: two 768-wide panels and one int8
    update.  Errors of 1/2 logdet against an 80-bit Cholesky: the int8 model within ENVELOPE_C x the FP64 blocked
    Cholesky's error (+ a 1e-13 relative floor)"""
    from scipy.spatial.distance import cdist
    n = 1536
    x = np.random.default_rng(11).uniform(0, 1, (n, 2))
    d = cdist(x, x) / 0.3
    K = (1 + d) * np.exp(-d)
    print("\n nugget   1/2 logdet     LAPACK-ref  blocked-ref  int8-ref   ratio")
    for nugget in (1e-2, 1e-4, 1e-6, 1e-8):
        S = K + nugget * np.eye(n)
        ref = np.sum(np.log(np.diag(_cholesky_longdouble(S))))
        half = {name: np.sum(np.log(np.diag(L))) - ref for name, L in
                (("lapack", np.linalg.cholesky(S)), ("fp64", ozaki_model.blocked_cholesky(S, None)),
                 ("int8", ozaki_model.blocked_cholesky(S, SLICES)))}
        e64, e8 = abs(float(half["fp64"])), abs(float(half["int8"]))
        print(" %.0e  %.6f  %+.2e  %+.2e  %+.2e  %.1f" % (nugget, float(ref), float(half["lapack"]), float(half["fp64"]),
                                                          float(half["int8"]), e8 / e64))
        assert e8 <= ENVELOPE_C * e64 + 1e-13 * abs(float(ref)), (nugget, e8, e64)
