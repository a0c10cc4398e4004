"""The kernel's Kruskal-Wallis arithmetic (splicedice_b200/csrc/sd_kruskal_math.cuh) compiled for the
host -- TEST-ONLY build under tests/cpu_twin -- against an exact fraction oracle for H, mpmath at 50
digits and scipy.special.chdtrc for p.  tests/test_gpu_kruskal.py runs the real kernel."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy.special import chdtrc

from tests import kruskal_cases as cases

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def twin():
    out_dir = os.path.join(HERE, "cpu_twin", "_build")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "libkruskal_twin.so")
    src = os.path.join(HERE, "cpu_twin", "kruskal_twin.cpp")
    deps = [src, os.path.join(ROOT, "splicedice_b200", "csrc", "sd_kruskal_math.cuh")]
    if not os.path.isfile(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-o", lib, src, "-lm"],
                       check=True)
    return ctypes.CDLL(lib)


def _p(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


def twin_h(lib, d, n_g, n, t):
    d, n_g = np.ascontiguousarray(d, dtype=np.int64), np.ascontiguousarray(n_g, dtype=np.int64)
    n, t = np.ascontiguousarray(n, dtype=np.int64), np.ascontiguousarray(t, dtype=np.int64)
    out = np.empty(len(n))
    lib.kruskal_twin_h(ctypes.c_int64(len(n)), ctypes.c_int32(d.shape[1]), _p(d, ctypes.c_int64),
                       _p(n_g, ctypes.c_int64), _p(n, ctypes.c_int64), _p(t, ctypes.c_int64), _p(out, ctypes.c_double))
    return out


def twin_sf(lib, df, h):
    df, h = np.ascontiguousarray(df, dtype=np.int32), np.ascontiguousarray(h, dtype=np.float64)
    out = np.empty(len(h))
    lib.kruskal_twin_sf(ctypes.c_int64(len(h)), _p(df, ctypes.c_int32), _p(h, ctypes.c_double), _p(out, ctypes.c_double))
    return out


def _rows(seed, k, n_total, count, tie_levels):
    """rank terms of `count` random rows of n_total cells in k groups (some cells NaN)"""
    rng = np.random.default_rng(seed)
    labels = np.concatenate([np.arange(k), rng.integers(0, k, n_total - k)])
    out = []
    for j in range(count):
        v = rng.integers(0, tie_levels, n_total).astype(np.float64) if tie_levels else rng.random(n_total)
        if j % 3 == 1:
            v += (labels == j % k) * 0.5 * (tie_levels or 1)     # one group shifted: large H
        v[rng.random(n_total) < 0.1] = np.nan
        v[:k][np.isnan(v[:k])] = 0.0                                # every group keeps a cell
        out.append(cases.rank_terms(v, labels, k))
    return out


@pytest.mark.parametrize("k,n_total,tie_levels", [(2, 10, 3), (3, 200, 0), (7, 500, 5), (64, 3000, 40),
                                                  (256, 16384, 0), (256, 16384, 9), (4, 16384, 2)])
def test_h_against_the_exact_fraction(twin, k, n_total, tie_levels):
    rows = _rows(k * 1000 + tie_levels, k, n_total, 12, tie_levels)
    d = np.array([r[0] for r in rows])
    n_g = np.array([r[1] for r in rows])
    n = np.array([r[2] for r in rows])
    t = np.array([r[3] for r in rows])
    h = twin_h(twin, d, n_g, n, t)
    for j, (dj, gj, nj, tj) in enumerate(rows):
        want = cases.exact_h(dj, gj, nj, tj)
        assert want is not None and want > 0
        assert abs(h[j] - float(want)) <= 1e-13 * float(want), (j, h[j], float(want))


def test_h_is_zero_exactly_when_the_rank_sums_balance_and_nan_when_all_tied(twin):
    # balanced: each group holds the same multiset of values
    rng = np.random.default_rng(2)
    rows = []
    for k, per in ((2, 5), (3, 40), (7, 11), (256, 3)):
        base = rng.integers(0, 4, per).astype(np.float64)
        v = np.tile(base, k)
        labels = np.repeat(np.arange(k), per)
        rows.append(cases.rank_terms(v, labels, k))
    for d, n_g, n, t in rows:
        assert cases.exact_h(d, n_g, n, t) == 0
        assert twin_h(twin, d[None], n_g[None], [n], [t])[0] == 0.0
    d, n_g, n, t = cases.rank_terms(np.full(9, 0.25), np.arange(9) % 3, 3)
    assert t == n ** 3 - n and cases.exact_h(d, n_g, n, t) is None
    assert np.isnan(twin_h(twin, d[None], n_g[None], [n], [t])[0])


def _sf_points():
    df = np.arange(1, 256)
    h = np.geomspace(1e-8, 4000.0, 36)
    grid = np.array([(a, x) for a in df for x in np.concatenate([h, [a * np.exp(-6), a, 2.0 * a + 30]])])
    return grid[:, 0].astype(np.int32), grid[:, 1]


def test_p_against_mpmath_at_50_digits(twin):
    df, h = _sf_points()
    p = twin_sf(twin, df, h)
    want = np.array([cases.mpmath_sf(a, x) for a, x in zip(df, h)])
    keep = want >= 1e-300
    deep = keep & (h / 2 > 745)
    assert deep.sum() > 50 and (want[deep] > 0).all()           # x > 745 with p still representable
    assert (keep & (want < 1e-200)).sum() > 20
    rel = np.abs(p[keep] - want[keep]) / want[keep]
    assert rel.max() <= 1e-12, (rel.max(), df[keep][rel.argmax()], h[keep][rel.argmax()])
    assert (p[~keep] < 1e-299).all()


def test_p_against_scipy_chdtrc(twin):
    df, h = _sf_points()
    p = twin_sf(twin, df, h)
    want = chdtrc(df.astype(np.float64), h)
    keep = want > 1e-300
    np.testing.assert_allclose(p[keep], want[keep], rtol=1e-12, atol=0)


def test_p_edges(twin):
    p = twin_sf(twin, [1, 2, 255, 3, 4], [0.0, 0.0, 0.0, np.nan, 1e-300])
    assert p[0] == p[1] == p[2] == 1.0 and np.isnan(p[3]) and 0.0 < p[4] <= 1.0
    assert (twin_sf(twin, np.arange(1, 256), np.full(255, 1e-12)) <= 1.0).all()
