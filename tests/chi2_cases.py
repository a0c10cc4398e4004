"""Test vectors and oracles for the Yates-corrected chi-squared test of 2x2 tables
(splicedice_b200/csrc/sd_chi2_math.cuh), shared by the CPU twin test and the GPU kernel test.

Tables are int64 rows (a, b, c, d) = [[a, b], [c, d]]; a and b are inclusion counts (< 2^31), c and d
exclusion sums (< 2^61)."""
import numpy as np

# status codes of sd::chi2::Status
VALUE, ALL_ZERO, REFUSED_00, REFUSED_01, REFUSED_10, REFUSED_ENTRY = range(6)
POSITION = {REFUSED_00: (0, 0), REFUSED_01: (0, 1), REFUSED_10: (1, 0)}


def random_tables(seed=0, per_scale=600):
    """Cells from 3 to 2^30, half uniform and half near independence (moderate statistics, so most
    p-values are neither 1 nor underflowed), plus inclusion counts near 2^31 with exclusion sums near 2^60."""
    rng = np.random.default_rng(seed)
    rows = []
    for scale in (3, 10, 100, 10_000, 1_000_000, 1 << 20, 1 << 25, 1 << 30):
        rows.append(rng.integers(1, scale + 1, size=(per_scale // 2, 4)))
        a = rng.integers(1, scale + 1, size=per_scale // 2)
        b = rng.integers(1, scale + 1, size=per_scale // 2)
        q = rng.uniform(0.2, 5.0, size=per_scale // 2)
        eps = rng.normal(0.0, 2.0, size=per_scale // 2) / np.sqrt(np.minimum(a, b))
        c = np.maximum(1, np.rint(a * q * (1.0 + eps))).astype(np.int64)
        d = np.maximum(1, np.rint(b * q)).astype(np.int64)
        rows.append(np.stack([a, b, c, d], axis=1))
    n = per_scale // 2
    big_a = (1 << 31) - rng.integers(1, 1 << 20, size=n)
    big_b = (1 << 31) - rng.integers(1, 1 << 20, size=n)
    big_c = (1 << 60) - rng.integers(1, 1 << 40, size=n)
    big_d = (big_c.astype(object) * big_b.astype(object) // big_a.astype(object)).astype(np.int64)
    big_d += rng.integers(-(1 << 36), 1 << 36, size=n)           # near independence: moderate statistics
    rows.append(np.stack([big_a, big_b, big_c, big_d], axis=1))
    rows.append(np.stack([big_a, big_b, big_c, (1 << 60) - rng.integers(1, 1 << 40, size=n)], axis=1))
    return np.concatenate(rows).astype(np.int64)


def small_tables(top=8):
    """Every table with cells 0..top: all-zero, every kind of zero margin, p == 1 boundaries."""
    g = np.arange(top + 1)
    return np.stack(np.meshgrid(g, g, g, g, indexing="ij"), axis=-1).reshape(-1, 4).astype(np.int64)


def expected_status(t):
    """Status per table by scipy's rules (first zero of `expected` in row-major order)."""
    a, b, c, d = (t[:, i].astype(object) for i in range(4))
    out = np.full(len(t), VALUE, dtype=np.int32)
    r1, r2, c1, c2 = a + b, c + d, a + c, b + d
    for i in range(len(t)):
        if min(t[i]) < 0 or max(t[i, :2]) >= 1 << 31 or max(t[i, 2:]) >= 1 << 61:
            out[i] = REFUSED_ENTRY
        elif r1[i] + r2[i] == 0:
            out[i] = ALL_ZERO
        elif r1[i] == 0 or c1[i] == 0:
            out[i] = REFUSED_00
        elif c2[i] == 0:
            out[i] = REFUSED_01
        elif r2[i] == 0:
            out[i] = REFUSED_10
    return out


def refused_mask(status):
    return np.asarray(status) >= REFUSED_00


def trivially_one(t):
    """|ad - bc| <= N/2: scipy's clamped Yates step leaves a zero statistic, p == 1 exactly."""
    a, b, c, d = (t[:, i].astype(object) for i in range(4))
    return np.array([2 * abs(x) <= n for x, n in zip(a * d - b * c, a + b + c + d)], dtype=bool)


def mpmath_p(t, dps=50):
    """Exact statistic from the integers, erfc(sqrt(stat / 2)) at ``dps`` digits (non-refused tables)."""
    import mpmath
    out = np.empty(len(t))
    with mpmath.workdps(dps):
        for i, (a, b, c, d) in enumerate(t.tolist()):
            n = a + b + c + d
            x = max(2 * abs(a * d - b * c) - n, 0)
            den = 4 * (a + b) * (c + d) * (a + c) * (b + d)
            stat = mpmath.mpf(x * x * n) / den
            out[i] = float(mpmath.erfc(mpmath.sqrt(stat / 2)))
    return out


def scipy_p(t):
    """scipy.stats.chi2_contingency(table)[1] per table (NaN where it raises)."""
    import warnings
    from scipy.stats import chi2_contingency
    out = np.empty(len(t))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        for i, row in enumerate(t.astype(np.float64).tolist()):
            try:
                out[i] = chi2_contingency([row[:2], row[2:]])[1]
            except ValueError:
                out[i] = np.nan
    return out


def scipy_refusal_position(row):
    """(i, j) of scipy's zero-expected-frequency error for one table, None if it does not raise."""
    import re
    from scipy.stats import chi2_contingency
    try:
        chi2_contingency([[float(row[0]), float(row[1])], [float(row[2]), float(row[3])]])
    except ValueError as e:
        m = re.search(r"zero element at \((?:np\.int64\()?(\d+)\)?, (?:np\.int64\()?(\d+)\)?\)", str(e))
        return (int(m.group(1)), int(m.group(2))) if m else "other"
    return None


def assert_scipy_parity(t, p):
    """rtol 1e-9 against scipy where every cell is below 2^31.  With exclusion sums near 2^60 scipy's
    float64 `expected` is itself inexact (1.3e-9 from the exact value on random_tables(1)), so there the
    bound is 1e-8; mpmath_p holds those tables to 1e-12."""
    want = scipy_p(t)
    small = t.max(axis=1) < (1 << 31)
    np.testing.assert_allclose(p[small], want[small], rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(p[~small], want[~small], rtol=1e-8, atol=1e-300)


def max_rel(got, want, floor=1e-300):
    ok = want > floor
    return float((np.abs(got[ok] - want[ok]) / want[ok]).max(initial=0.0))
