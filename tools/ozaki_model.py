"""Numpy model of the emulated trailing update of csrc/syrk_i8.cu (C -= P P^T from int8 slices), inside a blocked
right-looking Cholesky with 768-wide panels like chol_factor, compared with LAPACK.

The model follows the kernel operation for operation, so that its errors are the kernel's:
  * row scale: s_i = 2^e_i, the least power of two with max_k |P_ik| 2^(7 - e_i) < 127.5;
  * slices, round to nearest: x = P_ik / s_i; for t = 1..S: y = 128 x, a_t = rint(y), x = y - a_t
    (|a_1| <= 127, |a_t| <= 64 after it; every step is exact in FP64);
  * the products of equal weight w = t + u (t, u = 1..S, w <= S + 1) summed exactly in integers:
    S_w = sum_{t+u=w} A_t A_u^T (|S_w| < 2^28, int32 in the kernel);
  * one FP64 combination per entry: hi = sum_{w=2..5} S_w 2^(7 (5 - w)) and lo = sum_{w=6..S+1} S_w 2^(7 (S+1 - w))
    are exact in int64 (and in FP64), v = hi 2^-35 + lo 2^-7(S+1) is rounded once, C_ij -= (v s_i) s_j once more.

The integer products are taken with FP64 matrix products of the integer slices: every partial sum is an integer below
2^53, so they are exact (tests/test_ozaki_model.py checks them against int64 products).

  python tools/ozaki_model.py --n 10000 --slices 7 8        # bench.py's model at a fresh theta
  python tools/ozaki_model.py --n 10000 --taper 0.27        # the tapered covariance of tests/test_gpu_tiled_taper.py
"""
import argparse
import os
import sys

import numpy as np
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PANEL = 768  # chol_factor's outer panel at n_pad >= 16 384 (6 tiles of 128)
HI_TOP = 5   # weights 2..HI_TOP go to the high int64 word of the combination


def row_scale(P):
    """2^e per row: the least power of two with max |P_i.| 2^(7-e) < 127.5 (1 for a zero row)."""
    m = np.max(np.abs(P), axis=1)
    _, e = np.frexp(m)
    e = e.astype(np.int64)
    bump = np.ldexp(m, 7 - e) >= 127.5
    e = np.where(bump, e + 1, e)
    e = np.where(m > 0, e, 0)
    return np.ldexp(1.0, e)


def split(P, slices):
    """int8-valued slices A_t (as float64 arrays) and the row scales of P (m x K)."""
    s = row_scale(P)
    x = P / s[:, None]
    out = []
    for _ in range(slices):
        y = x * 128.0
        a = np.rint(y)
        x = y - a
        out.append(a)
    return out, s


def weight_sums(A, B, slices):
    """S_w = sum_{t+u=w} A_t B_u^T for w = 2..slices+1 (exact integers held in float64)."""
    S = []
    for w in range(2, slices + 2):
        ts = range(1, w)
        S.append(np.hstack([A[t - 1] for t in ts]) @ np.hstack([B[w - t - 1] for t in ts]).T)
    return S


def combine(S, sa, sb, slices):
    """the FP64 value of P_A P_B^T from the weight sums, as the kernel's epilogue forms it"""
    hi = np.zeros(S[0].shape, dtype=np.int64)
    lo = np.zeros(S[0].shape, dtype=np.int64)
    for w in range(2, slices + 2):
        Sw = S[w - 2].astype(np.int64)
        if w <= HI_TOP:
            hi = hi * 128 + Sw
        else:
            lo = lo * 128 + Sw
    v = np.ldexp(hi.astype(np.float64), -7 * HI_TOP) + np.ldexp(lo.astype(np.float64), -7 * (slices + 1))
    return (v * sa[:, None]) * sb[None, :]


def emulated_product(PA, PB, slices):
    A, sa = split(PA, slices)
    B, sb = split(PB, slices)
    return combine(weight_sums(A, B, slices), sa, sb, slices)


def blocked_cholesky(S, slices, panel=PANEL, min_rows=0):
    """lower Cholesky factor of S: LAPACK on each 768-wide panel, the trailing update C -= P P^T through the
    emulated product (slices=None: FP64) whenever the trailing block has at least min_rows rows"""
    A = np.array(S, dtype=np.float64, order="F")
    n = A.shape[0]
    for j0 in range(0, n, panel):
        j1 = min(n, j0 + panel)
        A[j0:j1, j0:j1] = np.linalg.cholesky(A[j0:j1, j0:j1])
        if j1 == n:
            break
        A[j1:, j0:j1] = scipy.linalg.solve_triangular(A[j0:j1, j0:j1], A[j1:, j0:j1].T, lower=True).T
        P = A[j1:, j0:j1]
        if slices is None or n - j1 < min_rows or j1 - j0 != PANEL:
            A[j1:, j1:] -= P @ P.T
        else:
            A[j1:, j1:] -= emulated_product(P, P, slices)
    return np.tril(A)


def errors(S, L, Z):
    """relative logdet and quad errors against LAPACK, and max |(L L^T - S)_ab| / sqrt(S_aa S_bb)"""
    Lr = np.linalg.cholesky(S)
    ld_ref, ld = 2 * np.sum(np.log(np.diag(Lr))), 2 * np.sum(np.log(np.diag(L)))
    yr = scipy.linalg.solve_triangular(Lr, Z, lower=True)
    y = scipy.linalg.solve_triangular(L, Z, lower=True)
    q_ref, q = np.sum(yr * yr, axis=0), np.sum(y * y, axis=0)
    d = np.sqrt(np.diag(S))
    res = np.max(np.abs(L @ L.T - S) / np.outer(d, d))
    return abs(ld - ld_ref) / abs(ld_ref), float(np.max(np.abs(q - q_ref) / np.abs(q_ref))), float(res)


def bench_covariance(n, taper=None):
    """bench.py's model (its first n sites) at theta_at(1, 0); taper: times a Wendland-1 taper of that range"""
    import bench
    from oracle import cov
    locs, X, z = bench.synthetic(n)
    S = cov.cov_rns(bench.theta_at(1, 0), locs, X, bench.LIMITS)
    S = np.tril(S) + np.tril(S, -1).T
    if taper is not None:
        from scipy.spatial.distance import cdist
        h = cdist(locs, locs) / taper
        S = S * np.where(h < 1, (1 - h) ** 4 * (1 + 4 * h), 0.0)  # Wendland-1 (cov_wend1), range taper
    Z = np.column_stack([z, 100 * np.roll(z, 7)])
    return S, Z


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--slices", type=int, nargs="+", default=[7, 8])
    ap.add_argument("--taper", type=float, default=None, help="taper range (Wendland-1)")
    args = ap.parse_args()
    S, Z = bench_covariance(args.n, args.taper)
    r = errors(S, blocked_cholesky(S, None), Z)
    print("n=%d taper=%s FP64 blocked: logdet %.2e quad %.2e residual %.2e" % ((args.n, args.taper) + r), flush=True)
    for s in args.slices:
        r = errors(S, blocked_cholesky(S, s), Z)
        print("n=%d taper=%s slices=%d: logdet %.2e quad %.2e residual %.2e" % ((args.n, args.taper, s) + r),
              flush=True)


if __name__ == "__main__":
    main()
