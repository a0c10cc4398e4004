"""The kernel's signed-rank arithmetic (splicedice_b200/csrc/sd_signedrank_math.cuh) compiled for the
host -- TEST-ONLY build under tests/cpu_twin -- against the row rule of tests/signedrank_cases.py and
scipy.stats.wilcoxon: the method switch, the exact count (p bit-identical), and z (bit-identical) and p
(1e-12) of the normal approximation.  tests/test_gpu_signedrank.py runs the real kernel."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import signedrank_cases as cases

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def twin():
    out_dir = os.path.join(HERE, "cpu_twin", "_build")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "libsignedrank_twin.so")
    src = os.path.join(HERE, "cpu_twin", "signedrank_twin.cpp")
    deps = [src, os.path.join(ROOT, "splicedice_b200", "csrc", "sd_signedrank_math.cuh")]
    if not os.path.isfile(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-o", lib, src, "-lm"],
                       check=True)
    return ctypes.CDLL(lib)


def _p(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


def twin_rows(lib, rows, dtype=np.float64):
    """(method, W, z, p) of the twin for a list of (x, y) rows"""
    t = [cases.terms(x, y, dtype) for x, y in rows]
    cols = [np.array([r[k] for r in t], dtype=np.int64) for k in range(5)]
    r2 = np.ascontiguousarray(np.concatenate([r[5] for r in t] + [np.zeros(1, np.int64)]))
    offset = np.concatenate([[0], np.cumsum([len(r[5]) for r in t])[:-1]]).astype(np.int64)
    J = len(rows)
    method = np.empty(J, dtype=np.int32)
    w, z, p = np.empty(J), np.empty(J), np.empty(J)
    lib.signedrank_twin_rows(ctypes.c_int64(J), *(_p(c, ctypes.c_int64) for c in cols), _p(r2, ctypes.c_int64),
                             _p(offset, ctypes.c_int64), _p(method, ctypes.c_int32), _p(w, ctypes.c_double),
                             _p(z, ctypes.c_double), _p(p, ctypes.c_double))
    return method, w, z, p


def make_row(rng, n, ties=False, zeros=0, nan_pairs=0, inf_inf=0):
    """n complete pairs (+ nan_pairs pairs with a NaN cell).  ties: cells on a 1/64 grid with few levels,
    so |d| ties heavily and every difference is exact; otherwise uniform doubles (no ties).  The first
    `zeros` pairs differ by zero (one of them as -0.0 against +0.0), the next `inf_inf` by inf - inf."""
    if ties:
        x = rng.integers(0, 9, n) / 64
        y = rng.integers(0, 9, n) / 64
        y[x == y] += 1 / 64                      # no zeros unless asked for
    else:
        x, y = rng.random(n), rng.random(n)
    y[:zeros] = x[:zeros]
    if zeros:
        x[0], y[0] = 0.0, -0.0
    x[zeros:zeros + inf_inf] = y[zeros:zeros + inf_inf] = np.inf
    if nan_pairs:
        x = np.concatenate([x, np.full(nan_pairs, np.nan)])
        y = np.concatenate([y, rng.random(nan_pairs)])
    return x, y


def assert_rows(lib, rows, dtype=np.float64, scipy_check=True):
    method, w, z, p = twin_rows(lib, rows, dtype)
    for j, (x, y) in enumerate(rows):
        n, c, mode, W, P = cases.signed_rank_row(x, y, dtype)
        assert method[j] == mode, (j, n, c, method[j], mode)
        if mode == 0:
            assert np.isnan(w[j]) and np.isnan(p[j])
            continue
        assert w[j] == W, (j, w[j], W)
        if mode == 1:
            assert p[j] == P, (j, p[j], P)                          # bit-identical
        else:
            assert abs(p[j] - P) <= 1e-12 * P, (j, p[j], P)
        if scipy_check:
            sw, sp, _ = cases.scipy_row(x, y, dtype)
            assert w[j] == sw, (j, w[j], sw)
            if mode == 1:
                assert p[j] == sp, (j, n, c, p[j], sp)
            elif sp > 1e-300:
                assert abs(p[j] - sp) <= 1e-12 * sp, (j, p[j], sp)
            if mode == 2:
                _, _, sz = cases.scipy_row(x, y, dtype, method="asymptotic")
                assert -abs(z[j]) == sz, (j, z[j], sz)              # bit-identical
    return method


@pytest.mark.parametrize("n", [1, 2, 13, 14, 50, 51])
def test_method_switch(twin, n):
    rng = np.random.default_rng(n)
    flavours = {"plain": {}, "ties": {"ties": True}, "zero": {"zeros": 1}, "ties_zeros": {"ties": True, "zeros": 2},
                "nan_pairs": {"nan_pairs": 3}, "inf_inf": {"inf_inf": 1}}
    rows, want = [], []
    for name, kw in flavours.items():
        if n == 1 and name in ("ties_zeros",):
            continue
        for _ in range(4):
            rows.append(make_row(rng, n, **kw))
            if n == 1 and name == "zero":
                want.append(0)                                      # scipy raises
            elif n <= 13:
                want.append(1)                                      # exact or sign-flip enumeration
            elif n <= 50 and name in ("plain", "nan_pairs", "inf_inf"):
                want.append(1)                                      # exact null distribution
            else:
                want.append(2)
    got = assert_rows(twin, rows)
    np.testing.assert_array_equal(got, want)


def test_edges(twin):
    rng = np.random.default_rng(9)
    rows = [(np.full(4, np.nan), rng.random(4)),                    # n = 0
            (np.zeros(5), np.zeros(5)),                             # all zeros, n <= 13: W 0, p 1
            (np.zeros(20), np.zeros(20)),                           # all zeros, n > 13: untested
            (np.array([0.3]), np.array([0.1])),                     # one nonzero difference: p 1
            (np.array([0.3]), np.array([0.3])),                     # one zero: untested
            (np.array([np.inf, np.inf, 1.0]), np.array([np.inf, 0.0, 0.5])),
            (np.array([np.inf, -np.inf, 0.2]), np.array([0.1, 0.3, np.inf]))]
    method, w, z, p = twin_rows(twin, rows)
    np.testing.assert_array_equal(method, [0, 1, 0, 1, 0, 1, 1])
    assert w[1] == 0.0 and p[1] == 1.0 and w[3] == 0.0 and p[3] == 1.0
    assert np.isnan(w[[0, 2, 4]]).all() and np.isnan(p[[0, 2, 4]]).all()
    assert_rows(twin, rows)


@pytest.mark.parametrize("n", [5, 12, 30, 49])
def test_exact_count_of_random_rows(twin, n):
    """many rows through the exact count: untied, and tied at n <= 13; float32 differences too"""
    rng = np.random.default_rng(100 + n)
    rows = [make_row(rng, n, ties=n <= 13 and j % 2 == 0) for j in range(30)]
    assert (assert_rows(twin, rows) == 1).all()
    rows32 = [(x.astype(np.float32), y.astype(np.float32)) for x, y in rows[:10]]
    assert (assert_rows(twin, rows32, np.float32) == 1).all()


@pytest.mark.parametrize("n,levels", [(60, 3), (500, 5), (2000, 40), (8192, 3), (8192, 200), (8192, 0)])
def test_normal_approximation_up_to_the_limit(twin, n, levels):
    """z bit-identical to scipy's and p within 1e-12, for c up to 8,192 with heavy ties"""
    rng = np.random.default_rng(n + levels)
    rows = []
    for j in range(4):
        if levels:
            x = rng.integers(0, levels, n) / 64
            y = rng.integers(0, levels, n) / 64
        else:
            x, y = rng.random(n), rng.random(n)
        if j == 1:
            x = x + 1 / 64                                          # a shifted row: small p
        rows.append((x, y))
    assert (assert_rows(twin, rows) == 2).all()


def test_exact_p_and_bound_helpers(twin):
    """ldexp scaling at the ends: c = 0 and every sign pattern counted give p = 1"""
    rows = [(np.arange(1.0, 51.0), np.zeros(50)), (-np.arange(1.0, 51.0), np.zeros(50)),
            (np.array([np.inf, np.inf]), np.array([np.inf, np.inf]))]
    method, w, _, p = twin_rows(twin, rows)
    np.testing.assert_array_equal(method, [1, 1, 1])
    assert w[0] == 0.0 and p[0] == np.ldexp(1.0, -49) and w[1] == 0.0 and p[1] == p[0]
    assert w[2] == 0.0 and p[2] == 1.0
    assert_rows(twin, rows)
