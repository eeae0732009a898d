"""Exact reference for entries of C - P P^T (test helper of the split-int8 update tests, not a test module).

Every finite double is an integer times 2^-1074, so a row of P is held as Python integers times one power of two
(the finest unit in the row) and a dot product of two rows is an exact integer times a power of two: no rounding
anywhere, subnormal entries and products included (a Dekker two-product would lose those to underflow).  The exact
value is returned as a Fraction, and rounded to FP64 once by Fraction.__float__ (correctly rounded, to nearest even,
subnormal results included).

Entries are sampled so that a test stays within seconds: whole diagonal blocks, where the diagonal and its
neighbours live, plus random entries of the lower triangle.
"""
from fractions import Fraction
from operator import mul

import numpy as np


def _row_ints(row):
    """(ints, shift): row[k] == ints[k] * 2^shift exactly, for a row of finite doubles"""
    ratios = [float(x).as_integer_ratio() for x in row]  # (numerator, power-of-two denominator)
    den = max(d for _, d in ratios)
    shift = -(den.bit_length() - 1)
    return [n * (den // d) for n, d in ratios], shift


class ExactRows:
    """the rows of P (m x K, finite) as exact integers, for exact dot products of any two of them"""

    def __init__(self, P):
        P = np.asarray(P, dtype=np.float64)
        assert np.all(np.isfinite(P)), "the exact reference takes finite panels"
        self.rows = [_row_ints(r) for r in P]

    def dot(self, i, j):
        """sum_k P_ik P_jk, exactly"""
        (a, ea), (b, eb) = self.rows[i], self.rows[j]
        n, e = sum(map(mul, a, b)), ea + eb
        return Fraction(n * 2 ** e) if e >= 0 else Fraction(n, 2 ** -e)

    def abs_dot(self, i, j):
        """sum_k |P_ik P_jk|, exactly"""
        (a, ea), (b, eb) = self.rows[i], self.rows[j]
        n, e = sum(abs(x * y) for x, y in zip(a, b)), ea + eb
        return Fraction(n * 2 ** e) if e >= 0 else Fraction(n, 2 ** -e)


def exact_update(C, P, ii, jj):
    """C_ij - sum_k P_ik P_jk at the entries (ii[t], jj[t]), exactly (a list of Fractions)"""
    R = ExactRows(P)
    return [Fraction(float(C[i, j])) - R.dot(i, j) for i, j in zip(ii, jj)]


def rounded(values):
    """exact values rounded once to FP64"""
    return np.array([float(v) for v in values])


def sample_lower(m, rng, blocks=((0, 64),), count=2000):
    """(ii, jj) with ii >= jj: every lower entry of the diagonal blocks [b0, b0 + size) in `blocks` (a negative b0
    counts from the end) and `count` random lower entries"""
    ii, jj = [], []
    for b0, size in blocks:
        b0 = b0 % m
        r, c = np.tril_indices(min(size, m - b0))
        ii.append(r + b0), jj.append(c + b0)
    a, b = rng.integers(0, m, count), rng.integers(0, m, count)
    ii.append(np.maximum(a, b)), jj.append(np.minimum(a, b))
    return np.concatenate(ii), np.concatenate(jj)


def ulp(x):
    """the spacing of the doubles at |x|, exactly (2^-1074 in the subnormal range)"""
    return Fraction(float(np.spacing(abs(float(x)))))


TINY = Fraction(1, 2 ** 1074)  # the least subnormal

# panels (m x 768) where a split into int8 slices can go wrong, each with the C it is subtracted from
PANELS = ("decades", "pow2_edges", "dominant", "alternating", "pow500", "subnormal")


def adversarial_panel(kind, m, seed, k=768):
    rng = np.random.default_rng(seed)
    g = rng.standard_normal((m, k))
    C = rng.standard_normal((m, m))
    if kind == "decades":  # row magnitudes over 17 decades, a zero row
        P = g * np.exp(rng.uniform(-20, 20, m))[:, None]
        P[3] = 0.0
    elif kind == "pow2_edges":  # row maxima exactly at 2^e, at 127.5/128 2^e (the split's bump) and just below it
        e = rng.integers(-30, 30, m)
        P = np.ldexp(np.clip(g / 4, -0.99, 0.99), e[:, None])
        top = np.array([1.0, 127.5 / 128, np.nextafter(127.5 / 128, 0), 0.5])[np.arange(m) % 4]
        P[np.arange(m), rng.integers(0, k, m)] = np.ldexp(top, e) * rng.choice([-1.0, 1.0], m)
        P[1::8] = np.ldexp(127.5 / 128, e[1::8])[:, None] * np.sign(g[1::8])  # the edge value in every entry
    elif kind == "dominant":  # one entry per row 2^30 above the others
        P = g * np.exp(rng.uniform(-5, 5, m))[:, None]
        big = rng.integers(0, k, m)
        P[np.arange(m), big] = np.ldexp(rng.uniform(1, 2, m), 30) * np.abs(P).max(axis=1)
    elif kind == "alternating":  # +-1 times the row scale, alternating, and entries at the ties of the first rint
        sgn = np.where(np.arange(k) % 2 == 0, 1.0, -1.0)
        P = np.tile(sgn, (m, 1))
        P[1::2] = (rng.integers(-127, 127, (m // 2, k)) + 0.5) / 128 * sgn
        P *= np.ldexp(1.0, rng.integers(-8, 8, m))[:, None]
    elif kind == "pow500":  # rows at 2^500 and at 2^-500
        P = np.ldexp(g, np.where(np.arange(m) % 2 == 0, 500, -500)[:, None])
        C = np.ldexp(C, 1000)
    elif kind == "subnormal":  # row maxima below 2^-1022, down to 2^-1074, among rows of magnitude 1
        P = g.copy()
        sub = np.arange(m) % 3 != 0
        P[sub] = np.ldexp(g[sub], rng.integers(-1070, -1030, int(sub.sum()))[:, None])
        P[5] = 0.0
        P[5, 7] = 2.0 ** -1074
        C = np.ldexp(C, -1040)  # comparable to the products of a subnormal row and a row of magnitude 1
    else:
        raise ValueError(kind)
    return np.asfortranarray(P), np.asfortranarray(C)


# rows of nonfinite_panel: (row, column or None for the whole row, value)
NONFINITE = ((10, 100, np.nan), (20, 5, np.inf), (30, 767, -np.inf), (40, None, np.nan))


def nonfinite_panel(m, seed):
    """the "decades" panel with, in four rows, one NaN, one +Inf and one -Inf entry and a row of NaN; and those rows"""
    P, C = adversarial_panel("decades", m, seed)
    for r, k, v in NONFINITE:
        P[r, slice(None) if k is None else k] = v
    return P, C, np.array([r for r, _, _ in NONFINITE])
