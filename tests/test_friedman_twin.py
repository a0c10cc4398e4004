"""The kernel's Friedman arithmetic (splicedice_b200/csrc/sd_friedman_math.cuh) compiled for the host --
TEST-ONLY build under tests/cpu_twin -- against the exact fraction oracle for Q (bit for bit), scipy's
friedmanchisquare for the statistic it rounds, and scipy.special.chdtrc for p.  tests/test_gpu_friedman.py
runs the real kernel."""
import ctypes
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest
from scipy.special import chdtrc

from tests import friedman_cases as cases

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def twin():
    out_dir = os.path.join(HERE, "cpu_twin", "_build")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "libfriedman_twin.so")
    src = os.path.join(HERE, "cpu_twin", "friedman_twin.cpp")
    deps = [src] + [os.path.join(ROOT, "splicedice_b200", "csrc", h)
                    for h in ("sd_friedman_math.cuh", "sd_kruskal_math.cuh")]
    if not os.path.isfile(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-o", lib, src, "-lm"],
                       check=True)
    return ctypes.CDLL(lib)


def _p(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


def twin_qp(lib, sum_d2, n, k, t):
    a = [np.ascontiguousarray(np.atleast_1d(x), dtype=np.int64) for x in (sum_d2, n, k, t)]
    q, p = np.empty(len(a[0])), np.empty(len(a[0]))
    lib.friedman_twin(ctypes.c_int64(len(q)), *[_p(x, ctypes.c_int64) for x in a], _p(q, ctypes.c_double),
                      _p(p, ctypes.c_double))
    return q, p


def _tables(seed, n_blocks, k, count, levels):
    """`count` random rows [n_blocks, k]: continuous (levels 0) or on `levels` tie levels, some shifted by
    condition, some cells NaN"""
    rng = np.random.default_rng(seed)
    out = []
    for j in range(count):
        v = rng.integers(0, levels, (n_blocks, k)).astype(np.float64) if levels else rng.random((n_blocks, k))
        if j % 3 == 1:
            v += np.arange(k)[None, :] * (0.3 if j % 2 else 0.01) * (levels or 1)
        if j % 4 == 2:
            v[rng.random((n_blocks, k)) < 0.05] = np.nan
        out.append(v)
    return out


def _terms(tables, k):
    rows = [cases.block_terms(v) for v in tables]
    return ([int((d.astype(object) ** 2).sum()) for d, _, _ in rows], [n for _, n, _ in rows], [k] * len(rows),
            [t for _, _, t in rows])


@pytest.mark.parametrize("n_blocks,k,levels", [(1, 3, 0), (2, 3, 2), (9, 3, 3), (39, 8, 0), (39, 8, 4), (250, 4, 0),
                                               (250, 4, 5), (16, 64, 7), (64, 256, 0), (64, 256, 9), (5461, 3, 0),
                                               (5461, 3, 2), (4096, 4, 3)])
def test_q_is_the_exact_fraction_rounded(twin, n_blocks, k, levels):
    tables = _tables(n_blocks * 1000 + k + levels, n_blocks, k, 9, levels)
    s, n, kk, t = _terms(tables, k)
    q, _ = twin_qp(twin, s, n, kk, t)
    for j in range(len(tables)):
        want = cases.exact_q(*cases.block_terms(tables[j])[:2], k, t[j])
        if want is None:
            assert np.isnan(q[j])
        else:
            assert q[j] == float(want), (j, q[j], float(want))          # one correctly rounded division


def test_q_at_the_largest_numerator_and_denominator(twin):
    """Every block ranked the same way maximises sum D^2; n k = 16,384 at k = 256 and k = 3 puts the
    numerator near 2^44 and the denominator near 2^30.  Random large (sum D^2, T) pairs in range too."""
    for n, k in ((64, 256), (5461, 3), (4096, 4), (128, 128)):
        d = n * (2 * np.arange(1, k + 1, dtype=object) - (k + 1))
        s = int(sum(x * x for x in d))
        assert 3 * (k - 1) * s < 2 ** 46 and n * (k ** 3 - k) < 2 ** 31
        q, p = twin_qp(twin, s, n, k, 0)
        assert q[0] == float(cases.exact_q(d, n, k, 0)) == n * (k - 1)
        assert p[0] >= 0
    rng = np.random.default_rng(11)
    for _ in range(2000):
        k = int(rng.integers(3, 257))
        n = int(rng.integers(1, 16384 // k + 1))
        s_max = n * n * (k ** 3 - k) // 3
        s, t = int(rng.integers(0, s_max + 1)), int(rng.integers(0, n * (k ** 3 - k)))
        q, _ = twin_qp(twin, s, n, k, t)
        assert q[0] == float(Fraction(3 * (k - 1) * s, n * (k ** 3 - k) - t))


def test_q_against_scipy(twin):
    """scipy's form cancels; the bound is 1e-13 of its scale 3 n (k + 1) / c, c its tie factor."""
    checked = 0
    for n_blocks, k, levels in ((1, 3, 0), (5, 3, 3), (30, 5, 0), (30, 5, 3), (12, 7, 2), (40, 16, 0)):
        tables = _tables(k * 77 + levels, n_blocks, k, 20, levels)
        s, n, kk, t = _terms(tables, k)
        q, _ = twin_qp(twin, s, n, kk, t)
        for j, v in enumerate(tables):
            want = cases.scipy_q(v)
            if np.isnan(q[j]) or not np.isfinite(want):
                continue
            bound = 1e-13 * 3 * n[j] * (k + 1) / cases.tie_factor(n[j], k, t[j])
            assert abs(q[j] - want) <= bound, (n_blocks, k, j, q[j], want)
            checked += 1
    assert checked > 100


def test_edges(twin):
    # one untied block of three: Q = 2, p = e^-1 (scipy gives the same)
    d, n, t = cases.block_terms([[0.1, 0.5, 0.3]])
    q, p = twin_qp(twin, int((d ** 2).sum()), n, 3, t)
    assert q[0] == 2.0 and abs(p[0] - np.exp(-1.0)) <= 1e-15
    assert abs(cases.scipy_q([[0.1, 0.5, 0.3]]) - 2.0) < 1e-12
    # balanced: Q = 0, p = 1 exactly
    d, n, t = cases.block_terms([[1, 2, 3], [3, 2, 1], [2, 2, 2]])
    assert (d == 0).all()
    q, p = twin_qp(twin, 0, n, 3, t)
    assert q[0] == 0.0 and p[0] == 1.0
    # all tied: the denominator is 0; n = 0: no block
    d, n, t = cases.block_terms(np.full((4, 5), 0.25))
    assert t == n * (5 ** 3 - 5) and cases.exact_q(d, n, 5, t) is None
    q, p = twin_qp(twin, [0, 0], [n, 0], [5, 5], [t, 0])
    assert np.isnan(q).all() and np.isnan(p).all()


@pytest.mark.parametrize("k", [3, 4, 7, 64, 256])
def test_p_against_chdtrc(twin, k):
    rng = np.random.default_rng(k)
    n = max(1, 16384 // k)
    tables = [rng.random((n, k)) + np.arange(k)[None, :] * shift for shift in np.geomspace(1e-5, 1.0, 16) / k]
    s, nn, kk, t = _terms(tables, k)
    q, p = twin_qp(twin, s, nn, kk, t)
    want = chdtrc(k - 1, q)
    keep = want > 1e-300
    assert keep.sum() >= 6
    np.testing.assert_allclose(p[keep], want[keep], rtol=1e-12, atol=0)
    assert (p[~keep] < 1e-299).all()
