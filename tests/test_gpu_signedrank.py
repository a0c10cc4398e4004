"""sd_signedrank_rows on the GPU (Wilcoxon signed-rank test per event between matched sample pairs)
against the row rule of tests/signedrank_cases.py and scipy.stats.wilcoxon(x, y, nan_policy='omit') row
by row, and `compare_paired` end to end on the golden PS tables (TSV, and the NPZ `quant --npz` writes)
against a scipy loop + the numpy BH restatement."""
import argparse
import json
import os

import numpy as np
import pytest

from tests import signedrank_cases as cases

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _dev():
    return torch.device("cuda", 0)


def kernel_rows(ps, cols1, cols2, **kw):
    from splicedice_b200 import ops
    r = ops.signedrank_rows(torch.from_numpy(ps).to(_dev()), cols1, cols2, **kw)
    return {k: v.cpu().numpy() for k, v in r.items()}


def mean_close(a, b):
    """within 1e-12, or the same infinity, or both NaN (no pair, or +inf and -inf in one side)"""
    return a == b or (np.isnan(a) and np.isnan(b)) or abs(a - b) <= 1e-12


def assert_rows_match(got, ps, cols1, cols2, scipy_check=True):
    """n, c, method and W equal to the row rule; method-1 p bit-identical, method-2 p within 1e-12
    relative (p > 1e-300); means within 1e-12; and the same against scipy.  Returns the method codes."""
    dtype = ps.dtype.type
    for j in range(ps.shape[0]):
        x, y = ps[j, cols1], ps[j, cols2]
        n, c, mode, W, P = cases.signed_rank_row(x, y, dtype)
        assert (got["n"][j], got["c"][j], got["method"][j]) == (n, c, mode), (j, got["n"][j], got["c"][j], n, c, mode)
        both = ~np.isnan(x) & ~np.isnan(y)
        for key, v in (("mean1", x), ("mean2", y)):
            assert mean_close(got[key][j], np.mean(v[both].astype(np.float64)) if n else np.nan), (j, key)
        if mode == 0:
            assert np.isnan(got["W"][j]) and np.isnan(got["p"][j]), j
            continue
        assert got["W"][j] == W, (j, got["W"][j], W)
        p = got["p"][j]
        if mode == 1:
            assert p == P, (j, p, P)
        elif P > 1e-300:
            assert abs(p - P) <= 1e-12 * P, (j, p, P)
        if scipy_check:
            sw, sp, _ = cases.scipy_row(x, y, dtype)
            assert got["W"][j] == sw, (j, got["W"][j], sw)
            if mode == 1:
                assert p == sp, (j, p, sp)
            elif sp > 1e-300:
                assert abs(p - sp) <= 1e-12 * sp, (j, p, sp)
    return got["method"]


def paired_matrix(rng, J, P, decimals, extra=3):
    """[J, 2P + extra] float64 and the two column lists (shuffled).  Cells rounded to `decimals` (None:
    untied for most rows), some pairs equal (zeros, some as -0.0 against +0.0), +-inf in either cell,
    NaN in either cell; row j's complete pairs are cut to a target count from a list that crosses
    13 / 14 and 50 / 51 where P allows."""
    S = 2 * P + extra
    perm = rng.permutation(S)
    cols1, cols2 = perm[:P], perm[P:2 * P]
    ps = rng.random((J, S))
    if decimals is not None:
        ps = np.round(ps, decimals)
    targets = [t for t in (0, 1, 2, 5, 12, 13, 14, 15, 49, 50, 51, 52, P) if t <= P]
    for j in range(J):
        x, y = ps[j, cols1], ps[j, cols2]
        kind = j % 5
        if kind == 1:
            eq = rng.random(P) < 0.15
            y[eq] = x[eq]
            z = rng.random(P) < 0.05
            x[z], y[z] = 0.0, -0.0
        elif kind == 2:
            u = rng.random(P)
            x[u < 0.03] = np.inf
            y[(u >= 0.03) & (u < 0.06)] = -np.inf
            y[u < 0.015] = np.inf                                   # inf - inf
        if kind != 4:
            drop = rng.permutation(P)[:P - targets[j % len(targets)]]
            half = drop[: len(drop) // 2]
            x[half] = np.nan
            y[drop[len(drop) // 2:]] = np.nan
        else:
            x[rng.random(P) < 0.1] = np.nan
            y[rng.random(P) < 0.1] = np.nan
        ps[j, cols1], ps[j, cols2] = x, y
    return ps, cols1, cols2


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("P,J,decimals", [(1, 40, 2), (2, 60, 2), (5, 80, 1), (13, 80, 2), (14, 80, 2),
                                          (20, 80, None), (50, 80, None), (50, 60, 3), (51, 80, 3),
                                          (500, 60, 3), (8192, 8, 2)])
def test_rows_against_the_row_rule_and_scipy(P, J, decimals, dtype):
    rng = np.random.default_rng(P * 7 + (decimals or 0))
    ps, c1, c2 = paired_matrix(rng, J, P, decimals)
    ps = ps.astype(dtype)
    method = assert_rows_match(kernel_rows(ps, c1, c2), ps, c1, c2)
    assert (method == 1).any()
    if P >= 14:
        assert (method == 2).any()


def test_n_crosses_the_switch_points_inside_one_matrix():
    rng = np.random.default_rng(11)
    ps, c1, c2 = paired_matrix(rng, 120, 60, None)
    got = kernel_rows(ps, c1, c2)
    assert_rows_match(got, ps, c1, c2, scipy_check=False)
    n, m = got["n"], got["method"]
    for lo, hi in ((13, 14), (50, 51)):
        assert (n == lo).any() and (n == hi).any()
    untied = np.arange(120) % 5 == 0
    assert (m[untied & (n <= 50) & (n > 1)] == 1).all() and (m[untied & (n > 50)] == 2).all()


def test_float32_subtraction_makes_the_tie():
    """(0.152, 0.239) and (0.017, 0.104) in float32 both differ by float32 -0.087, but not as doubles:
    with 18 other untied pairs, the float32 tie sends the row to the normal approximation, while
    differences widened first would stay untied and exact."""
    rng = np.random.default_rng(12)
    x = np.concatenate([[0.152, 0.017], 0.5 + rng.random(18) * 0.4])
    y = np.concatenate([[0.239, 0.104], rng.random(18) * 0.4])
    ps = np.concatenate([x, y])[None, :].astype(np.float32)
    c1, c2 = np.arange(20), np.arange(20, 40)
    xf, yf = ps[0, c1], ps[0, c2]
    assert cases.signed_rank_row(xf, yf, np.float32)[2] == 2
    assert cases.signed_rank_row(xf.astype(np.float64), yf.astype(np.float64))[2] == 1
    got = kernel_rows(ps, c1, c2)
    assert got["method"][0] == 2 and got["c"][0] == 20
    assert_rows_match(got, ps, c1, c2)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_swapping_the_sides_keeps_w_and_p(dtype):
    rng = np.random.default_rng(13)
    ps, c1, c2 = paired_matrix(rng, 200, 40, 2)
    ps = ps.astype(dtype)
    a, b = kernel_rows(ps, c1, c2), kernel_rows(ps, c2, c1)
    for key in ("n", "c", "method"):
        np.testing.assert_array_equal(a[key], b[key])
    for key in ("W", "p"):
        assert np.array_equal(a[key].view(np.uint64), b[key].view(np.uint64)), key
    assert np.array_equal(a["mean1"], b["mean2"], equal_nan=True)


def test_padded_leading_dimensions_row_range_and_out_buffers():
    from splicedice_b200 import ops
    rng = np.random.default_rng(4)
    J, P = 400, 30
    ps, c1, c2 = paired_matrix(rng, J, P, 2)
    S = ps.shape[1]
    buf = torch.full((J, S + 9), 7.0, dtype=torch.float64, device=_dev())
    buf[:, :S] = torch.from_numpy(ps).to(_dev())
    n_buf = torch.full((J, 5), -9, dtype=torch.int32, device=_dev())
    st_buf = torch.full((J, 6), -9.0, dtype=torch.float64, device=_dev())
    r0, r1 = 77, 333
    ops.signedrank_rows(buf[:, :S], c1, c2, row_begin=r0, row_end=r1, out=(n_buf, st_buf))
    n, st = n_buf.cpu().numpy(), st_buf.cpu().numpy()
    for a, w in ((n, 3), (st, 4)):
        assert (a[:r0] == -9).all() and (a[r1:] == -9).all() and (a[:, w:] == -9).all()
    got = dict(n=n[r0:r1, 0], c=n[r0:r1, 1], method=n[r0:r1, 2], mean1=st[r0:r1, 0], mean2=st[r0:r1, 1],
               W=st[r0:r1, 2], p=st[r0:r1, 3])
    assert_rows_match(got, ps[r0:r1], c1, c2, scipy_check=False)
    whole = kernel_rows(ps, c1, c2)
    for key, v in got.items():
        assert np.array_equal(np.ascontiguousarray(whole[key][r0:r1]).view(np.uint8),
                              np.ascontiguousarray(v).view(np.uint8)), key


def _native(ps, cols1, cols2, n_pairs=None):
    """sd_signedrank_rows on device column lists as given (ops checks host lists first)"""
    from splicedice_b200 import native
    J, S = ps.shape
    a = torch.tensor(cols1, dtype=torch.int32, device=_dev())
    b = torch.tensor(cols2, dtype=torch.int32, device=_dev())
    n = torch.zeros((J, 3), dtype=torch.int32, device=_dev())
    st = torch.zeros((J, 4), dtype=torch.float64, device=_dev())
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    native.call("sd_signedrank_rows", J, S, native.ptr(ps), ps.stride(0), kind,
                len(cols1) if n_pairs is None else n_pairs, native.ptr(a), native.ptr(b), 0, J, native.ptr(n),
                n.stride(0), native.ptr(st), st.stride(0), native.stream_ptr())
    return n.cpu().numpy(), st.cpu().numpy()


def test_column_outside_the_matrix_is_never_read():
    ps = torch.rand((50, 10), dtype=torch.float64, device=_dev())
    for cols1, cols2 in (([0, 1, 12], [3, 4, 5]), ([0, 1, 2], [3, -1, 5]), ([0, 1, 2], [3, 4, 10])):
        n, st = _native(ps, cols1, cols2)
        assert (n[:, :2] == -1).all() and (n[:, 2] == 0).all() and np.isnan(st).all()
    n, st = _native(ps, [0, 1, 2], [3, 4, 5])                       # the same call, in range
    assert (n[:, 0] == 3).all() and (n[:, 2] == 1).all() and np.isfinite(st).all()


def test_more_pairs_than_the_limit_are_refused():
    from splicedice_b200 import native, ops
    ps = torch.zeros((2, 16386), dtype=torch.float32, device=_dev())
    with pytest.raises(native.NativeCallError) as e:
        _native(ps, np.arange(8193), np.arange(8193, 16386))
    assert e.value.code == native.SD_ERR_INVALID and "n_pairs = 8193" in str(e.value)
    with pytest.raises(native.NativeCallError) as e:
        _native(ps, [0], [1], n_pairs=0)
    assert e.value.code == native.SD_ERR_INVALID
    with pytest.raises(ValueError, match="8193 pairs"):
        ops.signedrank_rows(ps, np.arange(8193), np.arange(8193, 16386))
    r = ops.signedrank_rows(ps, np.arange(8192), np.arange(8192, 16384))     # the limit itself runs
    torch.cuda.synchronize()
    assert (r["n"] == 8192).all().item() and (r["c"] == 0).all().item() and (r["method"] == 0).all().item()


def test_argument_errors():
    from splicedice_b200 import native, ops
    ps = torch.zeros((4, 10), dtype=torch.float64, device=_dev())
    for c1, c2 in (([0, 1], [2]), ([], []), ([0, 1], [1, 2]), ([0, 0], [1, 2]), ([0], [10]), ([-1], [2]),
                   ([0.5], [1])):
        with pytest.raises(ValueError):
            ops.signedrank_rows(ps, c1, c2)
    with pytest.raises(TypeError):
        ops.signedrank_rows(ps.to(torch.int32), [0], [1])
    with pytest.raises(native.NativeCallError):
        ops.signedrank_rows(ps, [0], [1], row_begin=2, row_end=5)
    n, st = torch.empty((4, 3), dtype=torch.int32, device=_dev()), torch.empty((4, 4), dtype=torch.float64, device=_dev())
    ops.signedrank_rows(ps, [0], [1], out=(n, st))
    for narrow in ((n[:, :2], st), (n, st[:, :3]), (n.to(torch.int64), st)):
        with pytest.raises(TypeError):
            ops.signedrank_rows(ps, [0], [1], out=narrow)


# ---- the CLI -------------------------------------------------------------------------------------
PAIRS = [("s0", "s1"), ("s2", "s3"), ("s4", "s5"), ("s6", "s7")]


def _args(module, argv):
    p = argparse.ArgumentParser()
    module.add_parser(p)
    return p.parse_args(argv)


def _check_file(path, events, samples, ps):
    from oracle import oracle_np
    c1 = np.array([samples.index(a) for a, _ in PAIRS])
    c2 = np.array([samples.index(b) for _, b in PAIRS])
    lines = open(path).read().split("\n")
    assert lines[0] == "event\tn\tmean1\tmean2\tdelta\tW\tpvalue\tcorrected"
    assert lines[-1] == "" and [l.split("\t")[0] for l in lines[1:-1]] == list(events)
    got = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines[1:-1]])
    dtype = ps.dtype.type
    tested = np.zeros(len(events), dtype=bool)
    for j in range(len(events)):
        x, y = ps[j, c1], ps[j, c2]
        n, _, mode, W, _ = cases.signed_rank_row(x, y, dtype)
        sw, sp, _ = cases.scipy_row(x, y, dtype)
        assert got[j, 0] == n
        both = ~np.isnan(x) & ~np.isnan(y)
        if n:
            m1, m2 = np.mean(x[both].astype(np.float64)), np.mean(y[both].astype(np.float64))
            assert mean_close(got[j, 1], m1) and mean_close(got[j, 2], m2)
            assert got[j, 3] == got[j, 1] - got[j, 2]
        else:
            assert np.isnan(got[j, 1:4]).all()
        if mode == 0:
            assert np.isnan(got[j, 4:]).all()
            continue
        tested[j] = True
        assert got[j, 4] == W == sw and got[j, 5] == sp, (j, got[j, 4:6], W, sw, sp)
    corrected = oracle_np.bh_adjust(got[tested, 5])
    np.testing.assert_allclose(got[tested, 6], corrected, rtol=1e-12, atol=0)
    return tested.sum()


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_tsv_equals_a_scipy_loop(case, golden_dir, tmp_path):
    from splicedice_b200 import compare_groups, compare_paired
    tsv = os.path.join(golden_dir, case, "expected", "ref_allPS.tsv")
    samples, events, ps = compare_groups.read_ps(tsv)
    pairs = tmp_path / "pairs.txt"
    pairs.write_text("".join(f"{a}\t{b}\n" for a, b in PAIRS))
    out = tmp_path / "cmp.tsv"
    compare_paired.run_with(_args(compare_paired, ["-p", tsv, "--pairs", str(pairs), "-o", str(out)]))
    assert _check_file(out, events, samples, ps) > 100


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_npz_from_quant(case, golden_dir, tmp_path):
    from splicedice_b200 import compare_paired, quant
    from tests.test_gpu_cli import _manifest
    case_dir = os.path.join(golden_dir, case)
    over = json.load(open(os.path.join(case_dir, "quant_args.json")))
    argv = ["-m", _manifest(case_dir, tmp_path), "-o", str(tmp_path / "out"), "--npz"]
    if over.get("lowCoverageNan"):
        argv.append("--lowCoverageNan")
    if "minUnique" in over:
        argv += ["--minUnique", str(over["minUnique"])]
    quant.run_with(_args(quant, argv))
    npz = str(tmp_path / "out_allPS.npz")
    z = np.load(npz)
    samples, events, ps = [str(s) for s in z["cols"]], [str(e) for e in z["rows"]], z["data"]
    assert ps.dtype == np.float32
    pairs = tmp_path / "pairs.txt"
    pairs.write_text("".join(f"{a}\t{b}\r\n" for a, b in PAIRS))
    out = tmp_path / "cmp.tsv"
    compare_paired.run_with(_args(compare_paired, ["-p", npz, "--pairs", str(pairs), "-o", str(out)]))
    assert _check_file(out, events, samples, ps) > 100
