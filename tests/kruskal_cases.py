"""Exact restatements of the Kruskal-Wallis H test for tests/test_kruskal_twin.py and
tests/test_gpu_kruskal.py: the integer rank terms of a row, H as a fraction, p from mpmath."""
from fractions import Fraction

import numpy as np


def rank_terms(values, labels, k):
    """(D [k], n_g [k], n, T) of one row, NaN cells dropped: D_g = sum over the group's cells of
    (lo + hi + 1) - n_g (n + 1), T = sum over cells of ((hi - lo)^2 - 1), [lo, hi) a cell's tie run."""
    values = np.asarray(values, dtype=np.float64)
    labels = np.asarray(labels, dtype=np.int64)
    ok = ~np.isnan(values)
    v, g = values[ok], labels[ok]
    n = len(v)
    s = np.sort(v)
    lo = np.searchsorted(s, v, "left").astype(np.int64)
    hi = np.searchsorted(s, v, "right").astype(np.int64)
    n_g = np.bincount(g, minlength=k).astype(np.int64)
    twice = np.zeros(k, dtype=np.int64)
    np.add.at(twice, g, lo + hi + 1)
    return twice - n_g * (n + 1), n_g, n, int(((hi - lo) ** 2 - 1).sum())


def exact_h(d, n_g, n, t):
    """H as a Fraction, or None where the kernel reports NaN (an empty group, or every cell tied)."""
    den = n ** 3 - n - t
    if (np.asarray(n_g) == 0).any() or den <= 0:
        return None
    return 3 * (n - 1) * sum(Fraction(int(x) * int(x), int(m)) for x, m in zip(d, n_g)) / den


def mpmath_sf(df, h):
    """chi-square survival function at the double h, 50 digits"""
    import mpmath
    with mpmath.workdps(50):
        return float(mpmath.gammainc(mpmath.mpf(int(df)) / 2, mpmath.mpf(float(h)) / 2, mpmath.inf,
                                     regularized=True))
