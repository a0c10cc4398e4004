"""Exact restatement of the Friedman test for tests/test_friedman_twin.py, tests/test_gpu_friedman.py and
tools/friedman_bench.py: the integer rank terms of one row's blocks, Q as a fraction, scipy on the row."""
import warnings
from fractions import Fraction

import numpy as np


def block_terms(cells):
    """(D [k], n, T) of one row given as cells [n_blocks, k] (float64; NaN = undefined): blocks with a NaN
    cell dropped, n = the complete blocks, and per cell lo / hi = the cells of its block below / at or
    below it; D_c = sum over complete blocks of (lo + hi + 1) - n (k + 1), T = sum over cells of
    ((hi - lo)^2 - 1)."""
    cells = np.asarray(cells, dtype=np.float64)
    k = cells.shape[1]
    v = cells[~np.isnan(cells).any(axis=1)]
    n = len(v)
    lo = (v[:, None, :] < v[:, :, None]).sum(axis=2, dtype=np.int64)     # [b, c]: cells of block b below (b, c)
    hi = (v[:, None, :] <= v[:, :, None]).sum(axis=2, dtype=np.int64)
    d = (lo + hi + 1).sum(axis=0, dtype=np.int64) - n * (k + 1)
    return d, n, int(((hi - lo) ** 2 - 1).sum())


def exact_q(d, n, k, t):
    """Q as a Fraction, or None where the kernel reports NaN (no complete block, or all of them tied)."""
    den = n * (k ** 3 - k) - t
    if n == 0 or den <= 0:
        return None
    return Fraction(3 * (k - 1) * sum(int(x) * int(x) for x in d), den)


def tie_factor(n, k, t):
    """scipy's tie correction 1 - T / (n k (k^2 - 1))"""
    return 1 - t / (n * k * (k * k - 1))


def scipy_q(cells):
    """scipy.stats.friedmanchisquare(*conditions, nan_policy='omit')'s statistic on the float64 cells
    [n_blocks, k]; NaN where scipy raises or returns NaN."""
    from scipy.stats import friedmanchisquare
    cells = np.asarray(cells, dtype=np.float64)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return float(friedmanchisquare(*cells.T, nan_policy="omit")[0])
        except ValueError:
            return np.nan
