"""Row-level restatements of the Wilcoxon signed-rank test for tests/test_signedrank_twin.py and
tests/test_gpu_signedrank.py: the exact integer terms of a row, the (n, c, method, W, p) rule with the
method switch of scipy.stats.wilcoxon(x, y, nan_policy='omit') (scipy 1.18.1 defaults), and scipy itself
run on the differences taken in the PS matrix's precision."""
import warnings

import numpy as np
from scipy import special, stats


def differences(x, y, dtype=np.float64):
    """(n, the differences of the n complete pairs widened to float64); dtype = the PS matrix's (the
    subtraction's) precision"""
    both = ~np.isnan(x) & ~np.isnan(y)
    with np.errstate(invalid="ignore"):                                 # inf - inf
        d = (x[both].astype(dtype) - y[both].astype(dtype)).astype(np.float64)
    return int(both.sum()), d


def terms(x, y, dtype=np.float64):
    """(n, zeros, c, 2 R+, T, doubled ranks) of one row: inf - inf differences count in n only, zeros
    are dropped, the c others are ranked by |d| with average ranks (doubled: lo + hi + 1)."""
    n, d = differences(x, y, dtype)
    d = d[~np.isnan(d)]
    zeros = int((d == 0).sum())
    nz = d[d != 0]
    r2 = np.rint(2 * stats.rankdata(np.abs(nz))).astype(np.int64)
    t = np.unique(np.abs(nz), return_counts=True)[1].astype(np.int64)
    return n, zeros, len(nz), int(r2[nz > 0].sum()), int((t ** 3 - t).sum()), r2


def signed_rank_row(x, y, dtype=np.float64):
    """(n, c, mode, W, p) of one row; dtype = the PS matrix's (the subtraction's) precision.  mode 0 is
    untested (W = p = NaN), 1 the exact count, 2 the normal approximation."""
    n, d = differences(x, y, dtype)           # inf - inf pairs count in n ...
    d = d[~np.isnan(d)]                       # ... but carry no rank
    zeros = int((d == 0).sum())
    nz = d[d != 0]
    c = len(nz)
    if n == 0:
        return 0, 0, 0, np.nan, np.nan
    r2 = np.rint(2 * stats.rankdata(np.abs(nz))).astype(np.int64)
    rp2, tot2 = int(r2[nz > 0].sum()), int(r2.sum())
    W = min(rp2, tot2 - rp2) / 2
    t = np.unique(np.abs(nz), return_counts=True)[1]
    T = int((t ** 3 - t).sum())
    if (n <= 50 and T == 0 and zeros == 0) or n <= 13:
        if n == 1 and zeros == 1:
            return n, c, 0, np.nan, np.nan    # scipy raises
        counts = np.zeros(tot2 + 1, dtype=np.int64)
        counts[0] = 1
        for v in r2:
            counts[v:] = counts[v:] + counts[:len(counts) - v].copy()
        lo = int(counts[:min(rp2, tot2 - rp2) + 1].sum())
        return n, c, 1, W, min(1.0, np.ldexp(float(lo), 1 - c))
    if c == 0:
        return n, c, 0, np.nan, np.nan        # scipy: statistic 0, p NaN
    se = np.sqrt((c * (c + 1.) * (2. * c + 1.) - T / 2) / 24)
    z = (rp2 / 2 - c * (c + 1.) * 0.25) / se
    return n, c, 2, W, 2 * special.ndtr(-abs(z))


def scipy_row(x, y, dtype=np.float64, method="auto"):
    """scipy.stats.wilcoxon(x, y, nan_policy='omit') on the differences taken in `dtype` and widened
    (scipy given float32 arrays would rank, and compute z and p, in float32): (W, p, z), with z only for
    method='asymptotic' and (NaN, NaN, NaN) where scipy raises.  An inf - inf pair stays one: its
    difference is NaN, which scipy counts in n and does not rank."""
    n, d = differences(x, y, dtype)
    inf_inf = np.isnan(d)
    a, b = np.where(inf_inf, np.inf, d), np.where(inf_inf, np.inf, 0.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            r = stats.wilcoxon(a, b, nan_policy="omit", method=method)
        except ValueError:
            return np.nan, np.nan, np.nan
    return float(r.statistic), float(r.pvalue), float(getattr(r, "zstatistic", np.nan))
