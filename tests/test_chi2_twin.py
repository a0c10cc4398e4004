"""The kernel's per-table chi-squared arithmetic (splicedice_b200/csrc/sd_chi2_math.cuh) compiled for
the host -- TEST-ONLY build under tests/cpu_twin -- against scipy.stats.chi2_contingency and mpmath.
The GPU suite (tests/test_gpu_chi2.py) runs the same vectors through the real kernel."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import chi2_cases as cases

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def twin():
    out_dir = os.path.join(HERE, "cpu_twin", "_build")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, "libchi2_twin.so")
    src = os.path.join(HERE, "cpu_twin", "chi2_twin.cpp")
    deps = [src, os.path.join(ROOT, "splicedice_b200", "csrc", "sd_chi2_math.cuh")]
    if not os.path.isfile(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-o", lib, src, "-lm"],
                       check=True)
    handle = ctypes.CDLL(lib)
    i64p = ctypes.POINTER(ctypes.c_int64)

    def run(tables):
        t = np.ascontiguousarray(tables, dtype=np.int64)
        cols = [np.ascontiguousarray(t[:, i]) for i in range(4)]
        out = np.empty(len(t))
        status = np.empty(len(t), dtype=np.int32)
        handle.chi2_twin_batch(ctypes.c_int64(len(t)), *[c.ctypes.data_as(i64p) for c in cols],
                               out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                               status.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
        return out, status

    return run


def test_random_tables_against_scipy_and_mpmath(twin):
    t = cases.random_tables(seed=1)
    p, status = twin(t)
    assert (status == cases.VALUE).all()
    exact = cases.mpmath_p(t)
    assert ((exact > 1e-300) & (exact < 0.999)).sum() > len(t) // 4       # the vectors exercise erfc, not just 0 / 1
    assert cases.max_rel(p, exact) < 1e-12
    cases.assert_scipy_parity(t, p)


def test_p_is_exactly_one_inside_the_yates_step(twin):
    t = np.concatenate([cases.small_tables(8)[1:], cases.random_tables(seed=2, per_scale=200)])
    p, status = twin(t)
    one = cases.trivially_one(t) & (status == cases.VALUE)
    assert one.sum() > 500 and (p[one] == 1.0).all()
    assert (p[~one & (status == cases.VALUE)] < 1.0).all()
    # boundary |ad - bc| == N/2 included
    a, b, c, d = t.T
    assert ((2 * np.abs(a * d - b * c) == a + b + c + d) & (status == cases.VALUE)).any()


def test_small_tables_match_scipy_status_and_value(twin):
    """Every table with cells 0..8: value, NaN for the all-zero table, refused with scipy's (i, j)."""
    t = cases.small_tables(8)
    p, status = twin(t)
    np.testing.assert_array_equal(status, cases.expected_status(t))
    want = cases.scipy_p(t)
    val = status == cases.VALUE
    np.testing.assert_allclose(p[val], want[val], rtol=1e-9, atol=0)
    assert np.isnan(p[~val]).all()
    assert status[0] == cases.ALL_ZERO and np.isnan(want[0])            # scipy: NaN, no error
    for kind in (cases.REFUSED_00, cases.REFUSED_01, cases.REFUSED_10):
        rows = t[status == kind]
        assert len(rows)
        for row in rows[:: max(1, len(rows) // 40)]:
            assert cases.scipy_refusal_position(row) == cases.POSITION[kind], row


def test_entries_outside_the_domain_are_refused(twin):
    t = np.array([[-1, 2, 3, 4], [1, -2, 3, 4], [1, 2, -3, 4], [1, 2, 3, -4],
                  [1 << 31, 2, 3, 4], [1, 2, 1 << 61, 4], [(1 << 31) - 1, 2, (1 << 61) - 1, 4]], dtype=np.int64)
    p, status = twin(t)
    assert (status[:-1] == cases.REFUSED_ENTRY).all() and np.isnan(p[:-1]).all()
    assert status[-1] == cases.VALUE and 0.0 <= p[-1] <= 1.0
