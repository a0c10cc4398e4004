"""sd_ranksum_rows on the GPU (Wilcoxon rank-sum test per event between two sample groups) against
scipy.stats.ranksums(x, y, nan_policy='omit') row by row, and `compare_groups` end to end on the golden
PS tables (TSV, and the NPZ `quant --npz` writes) against a scipy loop + the numpy BH restatement."""
import argparse
import json
import os

import numpy as np
import pytest
from scipy.stats import ranksums

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _dev():
    return torch.device("cuda", 0)


def scipy_rows(ps, cols1, cols2):
    """Per row: n1, n2, mean1, mean2, z, p as the kernel defines them, from scipy and numpy."""
    J = ps.shape[0]
    n = np.zeros((J, 2), dtype=np.int64)
    st = np.full((J, 4), np.nan)
    for j in range(J):
        x = ps[j, cols1].astype(np.float64)
        y = ps[j, cols2].astype(np.float64)
        xv, yv = x[~np.isnan(x)], y[~np.isnan(y)]
        n[j] = len(xv), len(yv)
        if len(xv):
            st[j, 0] = np.mean(xv)
        if len(yv):
            st[j, 1] = np.mean(yv)
        if len(xv) and len(yv):
            st[j, 2:] = ranksums(x, y, nan_policy="omit")
    return n, st


def kernel_rows(ps, cols1, cols2, **kw):
    from splicedice_b200 import ops
    r = ops.ranksum_rows(torch.from_numpy(ps).to(_dev()), cols1, cols2, **kw)
    n = torch.stack([r["n1"], r["n2"]], 1).cpu().numpy()
    st = torch.stack([r["mean1"], r["mean2"], r["z"], r["p"]], 1).cpu().numpy()
    return n, st


def assert_rows_match(got, want):
    (gn, gs), (wn, ws) = got, want
    np.testing.assert_array_equal(gn, wn)
    assert np.array_equal(np.isnan(gs), np.isnan(ws))
    ok = ~np.isnan(ws)
    for k in (0, 1):
        np.testing.assert_allclose(gs[ok[:, k], k], ws[ok[:, k], k], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gs[ok[:, 2], 2], ws[ok[:, 2], 2], rtol=0, atol=1e-13)
    big = ok[:, 3] & (ws[:, 3] > 1e-300)
    np.testing.assert_allclose(gs[big, 3], ws[big, 3], rtol=1e-12, atol=0)


def interleaved_groups(rng, S, n1, n2):
    """Two disjoint, shuffled column lists drawn from interleaved positions; other columns unused."""
    chosen = np.sort(rng.choice(S, n1 + n2, replace=False))
    k = min(n1, n2)
    rest = chosen[2 * k:]
    c1 = np.concatenate([chosen[0:2 * k:2], rest[:n1 - k]])
    c2 = np.concatenate([chosen[1:2 * k:2], rest[n1 - k:]])
    return rng.permutation(c1), rng.permutation(c2)


def tied_matrix(rng, J, S):
    """Heavy ties: mostly 0 or 1, the rest rounded to 3 decimals; whole-row ties; -0.0 next to +0.0."""
    ps = np.round(rng.random((J, S)), 3)
    u = rng.random((J, S))
    ps[u < 0.35] = 0.0
    ps[(u >= 0.35) & (u < 0.6)] = 1.0
    ps[rng.random((J, S)) < 0.15] = -0.0
    ps[:: 17] = 0.5                                       # whole rows tied
    ps[5:: 19] = rng.choice([0.0, -0.0], size=ps[5:: 19].shape)
    ps[rng.random((J, S)) < 0.1] = np.nan
    return ps


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_heavy_ties_signed_zero_and_unused_columns(dtype):
    rng = np.random.default_rng(1)
    J, S = 300, 1100
    ps = tied_matrix(rng, J, S).astype(dtype)
    c1, c2 = interleaved_groups(rng, S, 500, 500)
    assert len(set(c1) | set(c2)) == 1000
    assert_rows_match(kernel_rows(ps, c1, c2), scipy_rows(ps, c1, c2))


@pytest.mark.parametrize("n1,n2", [(1, 1), (1, 500), (32, 32), (500, 500), (8192, 8192)])
def test_group_sizes(n1, n2):
    rng = np.random.default_rng(n1 * 7 + n2)
    J = 12 if n1 + n2 > 4000 else 200
    S = n1 + n2 + 3
    ps = rng.random((J, S))
    ps[:, :: 3] = np.round(ps[:, :: 3], 2)
    ps[rng.random((J, S)) < 0.2] = np.nan
    ps[1, :] = np.nan                                      # nothing defined
    c1, c2 = interleaved_groups(rng, S, n1, n2)
    assert_rows_match(kernel_rows(ps, c1, c2), scipy_rows(ps, c1, c2))


def test_nan_patterns():
    rng = np.random.default_rng(3)
    S = 80
    c1, c2 = np.arange(0, 64, 2), np.arange(1, 64, 2)
    rows = []
    for pattern in range(8):
        r = rng.random(S)
        if pattern == 0:
            r[c1] = np.nan                                 # group 1 empty
        elif pattern == 1:
            r[c2] = np.nan                                 # group 2 empty
        elif pattern == 2:
            r[:] = np.nan                                  # both empty
        elif pattern == 3:
            r[c1[1:]] = np.nan                             # one value left in group 1
        elif pattern == 4:
            r[c1[1:]] = np.nan
            r[c2[:-1]] = np.nan                            # one value left in each
        elif pattern == 5:
            r[np.concatenate([c1, c2])] = np.nan
            r[64:] = 0.3                                   # only unused columns defined
        elif pattern == 6:
            r[c1] = np.inf
            r[c2[:5]] = -np.inf                            # infinities are ordinary values
        rows.append(r)
    ps = np.array(rows)
    got, want = kernel_rows(ps, c1, c2), scipy_rows(ps, c1, c2)
    assert_rows_match(got, want)
    assert np.isnan(got[1][[0, 1, 2, 5], 2:]).all()
    np.testing.assert_array_equal(got[0][[0, 2, 3, 4]], [[0, 32], [0, 0], [1, 32], [1, 1]])


def test_padded_leading_dimension_and_row_range():
    from splicedice_b200 import ops
    rng = np.random.default_rng(4)
    J, S = 500, 70
    ps = tied_matrix(rng, J, S)
    perm = rng.permutation(S)
    c1, c2 = perm[:30], perm[30:60]
    buf = torch.full((J, S + 9), 7.0, dtype=torch.float64, device=_dev())
    buf[:, :S] = torch.from_numpy(ps).to(_dev())
    n_buf = torch.full((J, 5), -9, dtype=torch.int32, device=_dev())
    st_buf = torch.full((J, 6), -9.0, dtype=torch.float64, device=_dev())
    r0, r1 = 123, 401
    ops.ranksum_rows(buf[:, :S], c1, c2, row_begin=r0, row_end=r1, out=(n_buf[:, :2], st_buf[:, :4]))
    n, st = n_buf.cpu().numpy(), st_buf.cpu().numpy()
    assert (n[:r0] == -9).all() and (n[r1:] == -9).all() and (n[:, 2:] == -9).all()
    assert (st[:r0] == -9).all() and (st[r1:] == -9).all() and (st[:, 4:] == -9).all()
    want = scipy_rows(ps[r0:r1], c1, c2)
    assert_rows_match((n[r0:r1, :2], st[r0:r1, :4]), want)
    whole = kernel_rows(ps, c1, c2)
    assert np.array_equal(whole[1][r0:r1].view(np.uint64), st[r0:r1, :4].view(np.uint64))


def test_balanced_rank_sums_are_exact_at_large_n():
    rng = np.random.default_rng(5)
    n1 = n2 = 6000
    S = n1 + n2
    v = np.round(rng.random(n1), 4)
    ps = np.empty((3, S))
    ps[0, :n1], ps[0, n1:] = v, rng.permutation(v)        # the same multiset in both groups
    ps[1] = 0.25                                           # every value tied
    w = rng.random(n1 // 2)
    ps[2, :n1] = np.concatenate([w, 2 + w])                # mirrored: rank sums balance
    ps[2, n1:] = np.concatenate([1 + w, 1 + w])
    c1, c2 = np.arange(n1), np.arange(n1, S)
    for dtype in (np.float64, np.float32):
        n, st = kernel_rows(ps.astype(dtype), c1, c2)
        assert (st[:, 2] == 0.0).all() and (st[:, 3] == 1.0).all(), st
        assert (st[:, 2] == scipy_rows(ps.astype(dtype), c1, c2)[1][:, 2]).all()


def test_float32_rounding_of_a_float64_matrix():
    """Wherever rounding to float32 keeps a row's order (and its ties), the ranks and hence z are the same."""
    from scipy.stats import rankdata
    rng = np.random.default_rng(6)
    J, S = 400, 96
    ps = np.round(rng.random((J, S)), 3)
    close = np.arange(J) % 3 == 0
    ps[close, 1::4] = ps[close, 0::4] + 1e-12              # distinct in float64, merged in float32
    ps[rng.random((J, S)) < 0.1] = np.nan
    c1, c2 = np.arange(0, S, 2), np.arange(1, S, 2)
    f32 = ps.astype(np.float32)
    _, st64 = kernel_rows(ps, c1, c2)
    _, st32 = kernel_rows(f32, c1, c2)
    cols = np.concatenate([c1, c2])
    same = np.array([np.array_equal(rankdata(ps[j, cols], nan_policy="omit"),
                                    rankdata(f32[j, cols].astype(np.float64), nan_policy="omit"), equal_nan=True)
                     for j in range(J)])
    assert same.sum() > J // 2 and (~same).sum() > 50
    assert np.array_equal(st64[same, 2], st32[same, 2])
    assert not np.array_equal(st64[~same, 2], st32[~same, 2])


def test_too_many_samples_refused_by_the_library():
    from splicedice_b200 import native, ops
    ps = torch.zeros((2, 16385), dtype=torch.float32, device=_dev())
    with pytest.raises(native.NativeCallError) as e:
        ops.ranksum_rows(ps, np.arange(8192), np.arange(8192, 16385))
    assert e.value.code == native.SD_ERR_INVALID and "n1 + n2 = 16385 exceeds 16384" in str(e.value)
    r = ops.ranksum_rows(ps, np.arange(8192), np.arange(8192, 16384))     # the limit itself runs
    assert (r["z"].cpu().numpy() == 0).all()


def test_argument_errors():
    from splicedice_b200 import native, ops
    ps = torch.zeros((4, 10), dtype=torch.float64, device=_dev())
    for c1, c2 in (([0, 1], [1, 2]), ([0, 0], [1]), ([0], [10]), ([], [1]), ([-1], [2])):
        with pytest.raises(ValueError):
            ops.ranksum_rows(ps, c1, c2)
    with pytest.raises(TypeError):
        ops.ranksum_rows(ps.to(torch.int32), [0], [1])
    with pytest.raises(native.NativeCallError):
        ops.ranksum_rows(ps, [0], [1], row_begin=2, row_end=5)


def test_device_column_outside_the_matrix_is_never_read():
    from splicedice_b200 import ops
    ps = torch.rand((50, 10), dtype=torch.float64, device=_dev())
    c1 = torch.tensor([0, 1, 12], dtype=torch.int32, device=_dev())
    c2 = torch.tensor([2, 3], dtype=torch.int32, device=_dev())
    r = ops.ranksum_rows(ps, c1, c2)
    assert (r["n1"].cpu().numpy() == -1).all() and (r["n2"].cpu().numpy() == -1).all()
    assert torch.isnan(r["p"]).all() and torch.isnan(r["mean1"]).all()


# ---- the CLI -------------------------------------------------------------------------------------
def _args(module, argv):
    p = argparse.ArgumentParser()
    module.add_parser(p)
    return p.parse_args(argv)


def _groups(golden_dir, case, tmp_path):
    """Group files in two formats: the cond0 lines of the quant manifest, and a plain list."""
    lines = open(os.path.join(golden_dir, case, "input", "manifest.txt")).read().splitlines()
    g1, g2 = tmp_path / "g1.txt", tmp_path / "g2.txt"
    g1.write_text("\n".join(l for l in lines if l.endswith("cond0")) + "\n")
    g2.write_text("\n\n".join(l.split("\t")[0] for l in lines if l.endswith("cond1")) + "\n")
    return str(g1), str(g2)


def _expected_file(path, events, ps, cols1, cols2):
    from oracle import oracle_np
    from splicedice_b200 import compare_groups, textio
    _, st = scipy_rows(ps, cols1, cols2)
    p = st[:, 3]
    corrected = np.full_like(p, np.nan)
    fin = np.isfinite(p)
    corrected[fin] = oracle_np.bh_adjust(p[fin])
    res = np.column_stack([st[:, 0], st[:, 1], st[:, 0] - st[:, 1], st[:, 2], p, corrected])
    textio.write_matrix(path, compare_groups.HEADER, events, res, repr_floats=True)


def _assert_same_file(got_path, want_path):
    got, want = open(got_path, "rb").read().split(b"\n"), open(want_path, "rb").read().split(b"\n")
    assert got[0] == want[0] == b"event\tmean1\tmean2\tdelta\tz\tpvalue\tcorrected"
    assert [l.split(b"\t")[0] for l in got] == [l.split(b"\t")[0] for l in want]
    g = np.array([[float(x) for x in l.split(b"\t")[1:]] for l in got[1:-1]])
    w = np.array([[float(x) for x in l.split(b"\t")[1:]] for l in want[1:-1]])
    assert np.array_equal(np.isnan(g), np.isnan(w))
    ok = ~np.isnan(w)
    np.testing.assert_allclose(g[:, :3][ok[:, :3]], w[:, :3][ok[:, :3]], rtol=0, atol=1e-12)
    np.testing.assert_allclose(g[:, 3][ok[:, 3]], w[:, 3][ok[:, 3]], rtol=0, atol=1e-13)
    for k in (4, 5):
        big = ok[:, k] & (w[:, k] > 1e-300)
        np.testing.assert_allclose(g[big, k], w[big, k], rtol=1e-12, atol=0)
    return w


def _run(ps_path, g1, g2, out):
    from splicedice_b200 import compare_groups
    compare_groups.run_with(_args(compare_groups, ["-p", ps_path, "-g1", g1, "-g2", g2, "-o", str(out)]))


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_tsv_equals_a_scipy_loop(case, golden_dir, tmp_path):
    tsv = os.path.join(golden_dir, case, "expected", "ref_allPS.tsv")
    g1, g2 = _groups(golden_dir, case, tmp_path)
    _run(tsv, g1, g2, tmp_path / "cmp.tsv")
    lines = [l.rstrip("\n").split("\t") for l in open(tsv)]
    samples, events = lines[0][1:], [r[0] for r in lines[1:]]
    ps = np.array([[float(x) for x in r[1:]] for r in lines[1:]])
    c1 = [samples.index(s) for s in ("s0", "s2", "s4", "s6")]
    c2 = [samples.index(s) for s in ("s1", "s3", "s5", "s7")]
    _expected_file(tmp_path / "want.tsv", events, ps, c1, c2)
    w = _assert_same_file(tmp_path / "cmp.tsv", tmp_path / "want.tsv")
    assert np.isfinite(w[:, 4]).sum() > 100
    if case == "cli_8x_lownan":
        assert np.isnan(w[:, 4]).any()                    # some events are untested


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_npz_from_quant(case, golden_dir, tmp_path):
    from splicedice_b200 import quant
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
    g1, g2 = _groups(golden_dir, case, tmp_path)
    _run(npz, g1, g2, tmp_path / "cmp.tsv")
    z = np.load(npz)
    samples, events, ps = list(z["cols"]), list(z["rows"]), z["data"]
    assert ps.dtype == np.float32
    c1 = [samples.index(s) for s in ("s0", "s2", "s4", "s6")]
    c2 = [samples.index(s) for s in ("s1", "s3", "s5", "s7")]
    _expected_file(tmp_path / "want.tsv", [str(e) for e in events], ps, c1, c2)
    _assert_same_file(tmp_path / "cmp.tsv", tmp_path / "want.tsv")
    # the same events, in the same order, as the TSV quant wrote beside it
    tsv_events = [l.split("\t")[0] for l in open(tmp_path / "out_allPS.tsv")][1:]
    assert [l.split("\t")[0] for l in open(tmp_path / "cmp.tsv")][1:] == tsv_events


@pytest.mark.parametrize("g1,g2,needle", [("s0\ns9\n", "s1\n", "'s9'"), ("s0\ns1\n", "s1\ns2\n", "'s1'"),
                                          ("\n\n", "s1\n", "group 1"), ("s0\n", "", "group 2")])
def test_cli_errors_name_the_sample(g1, g2, needle, golden_dir, tmp_path):
    tsv = os.path.join(golden_dir, "cli_8x", "expected", "ref_allPS.tsv")
    f1, f2 = tmp_path / "a.txt", tmp_path / "b.txt"
    f1.write_text(g1)
    f2.write_text(g2)
    out = tmp_path / "cmp.tsv"
    with pytest.raises(ValueError) as e:
        _run(tsv, str(f1), str(f2), out)
    assert needle in str(e.value)
    assert not out.exists()
