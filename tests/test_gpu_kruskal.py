"""sd_kruskal_rows on the GPU (Kruskal-Wallis H test per event across sample groups) against
scipy.stats.kruskal(*groups, nan_policy='omit') and the exact fraction oracle row by row, and
`compare_conditions` end to end on the golden PS tables (TSV, and the NPZ `quant --npz` writes)
against a scipy loop + the numpy BH restatement."""
import argparse
import json
import os
import warnings

import numpy as np
import pytest
from scipy.special import chdtrc
from scipy.stats import kruskal

from tests import kruskal_cases as cases

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _dev():
    return torch.device("cuda", 0)


def scipy_h(ps_row, groups):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return float(kruskal(*[ps_row[g] for g in groups], nan_policy="omit")[0])
        except ValueError:
            return np.nan


def reference_rows(ps, groups):
    """Per row: counts, means, exact H (NaN where the kernel reports NaN), scipy's H and the bound
    1e-13 * 3 (n + 1) / (1 - T / (n^3 - n)) on |H - H_scipy|."""
    J, k = ps.shape[0], len(groups)
    cols = np.concatenate(groups)
    labels = np.repeat(np.arange(k), [len(g) for g in groups])
    n = np.zeros((J, k), dtype=np.int64)
    mean = np.full((J, k), np.nan)
    h_exact, h_scipy, bound = np.full(J, np.nan), np.full(J, np.nan), np.full(J, np.nan)
    for j in range(J):
        row = ps[j].astype(np.float64)
        for g, c in enumerate(groups):
            v = row[c][~np.isnan(row[c])]
            n[j, g] = len(v)
            if len(v):
                mean[j, g] = np.mean(v)
        d, n_g, m, t = cases.rank_terms(row[cols], labels, k)
        h = cases.exact_h(d, n_g, m, t)
        if h is not None:
            h_exact[j] = float(h)
            bound[j] = 1e-13 * 3 * (m + 1) / (1 - t / (m ** 3 - m))
            h_scipy[j] = scipy_h(row, groups)
    return n, mean, h_exact, h_scipy, bound


def kernel_rows(ps, groups, **kw):
    from splicedice_b200 import ops
    r = ops.kruskal_rows(torch.from_numpy(ps).to(_dev()), groups, **kw)
    return r["n"].cpu().numpy(), r["mean"].cpu().numpy(), r["H"].cpu().numpy(), r["p"].cpu().numpy()


def assert_rows_match(got, want, k):
    gn, gmean, gh, gp = got
    wn, wmean, wh, ws, bound = want
    np.testing.assert_array_equal(gn, wn)
    assert np.array_equal(np.isnan(gmean), np.isnan(wmean))
    ok = ~np.isnan(wmean)
    np.testing.assert_allclose(gmean[ok], wmean[ok], rtol=0, atol=1e-12)
    assert np.array_equal(np.isnan(gh), np.isnan(wh)) and np.array_equal(np.isnan(gp), np.isnan(wh))
    t = ~np.isnan(wh)
    assert (gh[t] >= 0).all()
    assert ((gh[t] == 0) == (wh[t] == 0)).all()
    np.testing.assert_allclose(gh[t], wh[t], rtol=1e-13, atol=0)
    fin = t & np.isfinite(ws) & (ws >= 0)
    assert (np.abs(gh[fin] - ws[fin]) <= bound[fin]).all(), np.max(np.abs(gh[fin] - ws[fin]) / bound[fin])
    assert (gp[t & (gh == 0)] == 1.0).all()
    want_p = chdtrc(k - 1, gh[t])
    big = want_p > 1e-300
    np.testing.assert_allclose(gp[t][big], want_p[big], rtol=1e-12, atol=0)
    assert ((gp[t] >= 0) & (gp[t] <= 1)).all()
    return t.sum()


def split_groups(rng, S, sizes, contiguous=False):
    cols = np.arange(S) if contiguous else rng.permutation(S)
    out, at = [], 0
    for s in sizes:
        out.append(cols[at:at + s])
        at += s
    return out


def tied_matrix(rng, J, S):
    """Heavy ties: mostly 0 or 1, the rest rounded to 2 decimals; -0.0 next to +0.0; +-inf; NaN."""
    ps = np.round(rng.random((J, S)), 2)
    u = rng.random((J, S))
    ps[u < 0.3] = 0.0
    ps[(u >= 0.3) & (u < 0.5)] = 1.0
    ps[rng.random((J, S)) < 0.15] = -0.0
    ps[rng.random((J, S)) < 0.02] = np.inf
    ps[rng.random((J, S)) < 0.02] = -np.inf
    ps[rng.random((J, S)) < 0.1] = np.nan
    return ps


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("k", [2, 3, 7, 64, 256])
def test_heavy_ties_signed_zero_and_infinities(k, dtype):
    rng = np.random.default_rng(k)
    J, S = (40, 5 * k + 9) if k >= 64 else (200, 12 * k + 7)
    ps = tied_matrix(rng, J, S)
    groups = split_groups(rng, S, [(S - 9) // k] * k)
    ps[::5, groups[0]] += 0.5                                # some rows far from balanced
    ps = ps.astype(dtype)
    tested = assert_rows_match(kernel_rows(ps, groups), reference_rows(ps, groups), k)
    assert tested > J // 2


def test_nan_patterns_balanced_and_all_tied_rows():
    rng = np.random.default_rng(3)
    S, k = 60, 3
    groups = [np.arange(0, 60, 3), np.arange(1, 60, 3), np.arange(2, 60, 3)]
    rows = []
    for pattern in range(8):
        r = rng.random(S)
        if pattern == 0:
            r[groups[1]] = np.nan                            # one group empty
        elif pattern == 1:
            r[:] = np.nan                                    # everything NaN
        elif pattern == 2:
            for g in groups:
                r[g[1:]] = np.nan                            # one cell per group
        elif pattern == 3:
            r[:] = 0.7                                       # all tied
        elif pattern == 4:
            r[:] = rng.choice([0.0, -0.0], S)                # all tied through the signed zeros
            r[groups[2][:4]] = np.nan
        elif pattern == 5:
            base = np.round(rng.random(20), 1)
            for g in groups:
                r[g] = rng.permutation(base)                 # balanced: the same multiset per group
        elif pattern == 6:
            r[groups[0]] = np.inf
            r[groups[1]] = -np.inf                           # infinities are ordinary values
        rows.append(r)
    ps = np.array(rows)
    got, want = kernel_rows(ps, groups), reference_rows(ps, groups)
    assert_rows_match(got, want, k)
    n, _, h, p = got
    assert np.isnan(h[[0, 1, 3, 4]]).all() and np.isnan(p[[0, 1, 3, 4]]).all()
    np.testing.assert_array_equal(n[[0, 1, 2]], [[20, 0, 20], [0, 0, 0], [1, 1, 1]])
    assert h[5] == 0.0 and p[5] == 1.0
    assert h[6] > 0 and np.isfinite(h[6])


@pytest.mark.parametrize("sizes", [[1, 3, 100, 8000, 8280], [8192, 8192], [64] * 256, [1] * 255 + [16129]])
def test_totals_up_to_the_limit_with_uneven_groups(sizes):
    rng = np.random.default_rng(len(sizes))
    S = sum(sizes) + 5
    J = 6
    ps = rng.random((J, S))
    ps[:, ::3] = np.round(ps[:, ::3], 2)
    ps[rng.random((J, S)) < 0.05] = np.nan
    ps[1] = 0.5                                              # all tied
    groups = split_groups(rng, S, sizes)
    for g in groups:
        ps[2:, g[0]] = rng.random(J - 2)                     # every group keeps a defined cell
    assert_rows_match(kernel_rows(ps, groups), reference_rows(ps, groups), len(sizes))


def test_deep_chi_square_tail_on_the_device():
    """256 groups of 64 with a growing shift per group: H from ~300 to ~2,200, so x = H / 2 passes 745
    (where a recurrence started at e^-x underflows) while p is still above 1e-300; the device's exp /
    log / lgamma against chdtrc and mpmath at 50 digits."""
    k, per = 256, 64
    rng = np.random.default_rng(7)
    labels = np.repeat(np.arange(k), per)
    shifts = np.linspace(0.0002, 0.0016, 16)
    ps = rng.random((len(shifts), k * per)) + shifts[:, None] * labels[None, :]
    groups = [np.arange(g * per, (g + 1) * per) for g in range(k)]
    got = kernel_rows(ps, groups)
    assert_rows_match(got, reference_rows(ps, groups), k)
    h, p = got[2], got[3]
    exact = np.array([cases.mpmath_sf(k - 1, x) for x in h])
    keep = exact >= 1e-300
    assert (keep & (h / 2 > 745)).sum() >= 2 and (exact[keep] < 1e-250).any()
    np.testing.assert_allclose(p[keep], exact[keep], rtol=1e-12, atol=0)


def test_balanced_rank_sums_are_exact_at_large_n():
    rng = np.random.default_rng(5)
    k, per = 4, 4000
    v = np.round(rng.random(per), 3)
    ps = np.empty((2, k * per))
    for g in range(k):
        ps[0, g * per:(g + 1) * per] = rng.permutation(v)   # the same multiset in every group
    # every group symmetric about 1/2 (values on a 1/1024 grid: exact in float32 too), so every mean
    # rank is (n + 1) / 2
    for lo, hi in ((0, 3000), (3000, 4000), (4000, 16000)):
        a = rng.integers(0, 1024, (hi - lo) // 2) / 1024
        ps[1, lo:hi] = np.concatenate([a, 1 - a])
    three = [np.arange(0, 3000), np.arange(3000, 4000), np.arange(4000, 16000)]
    for dtype in (np.float64, np.float32):
        x = ps.astype(dtype)
        _, _, h, p = kernel_rows(x, [np.arange(g * per, (g + 1) * per) for g in range(k)])
        assert h[0] == 0.0 and p[0] == 1.0
        _, _, h, p = kernel_rows(x, three)
        assert h[1] == 0.0 and p[1] == 1.0
        assert cases.exact_h(*cases.rank_terms(x[1, :16000], np.repeat([0, 1, 2], [3000, 1000, 12000]), 3)) == 0


def test_padded_leading_dimensions_and_row_range():
    from splicedice_b200 import ops
    rng = np.random.default_rng(4)
    J, S, k = 500, 70, 5
    ps = tied_matrix(rng, J, S)
    groups = split_groups(rng, S, [10, 20, 5, 15, 12])
    buf = torch.full((J, S + 9), 7.0, dtype=torch.float64, device=_dev())
    buf[:, :S] = torch.from_numpy(ps).to(_dev())
    n_buf = torch.full((J, k + 3), -9, dtype=torch.int32, device=_dev())
    m_buf = torch.full((J, k + 2), -9.0, dtype=torch.float64, device=_dev())
    st_buf = torch.full((J, 5), -9.0, dtype=torch.float64, device=_dev())
    r0, r1 = 123, 401
    ops.kruskal_rows(buf[:, :S], groups, row_begin=r0, row_end=r1, out=(n_buf, m_buf, st_buf))
    n, m, st = n_buf.cpu().numpy(), m_buf.cpu().numpy(), st_buf.cpu().numpy()
    for a, w in ((n, k), (m, k), (st, 2)):
        assert (a[:r0] == -9).all() and (a[r1:] == -9).all() and (a[:, w:] == -9).all()
    got = (n[r0:r1, :k], m[r0:r1, :k], st[r0:r1, 0], st[r0:r1, 1])
    assert_rows_match(got, reference_rows(ps[r0:r1], groups), k)
    whole = kernel_rows(ps, groups)
    for a, b in zip(whole, got):
        assert np.array_equal(np.ascontiguousarray(a[r0:r1]).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _native(ps, cols, labels, k, n_cols=None):
    """sd_kruskal_rows on device column / label lists as given (ops checks host lists first)"""
    from splicedice_b200 import native
    J, S = ps.shape
    c = torch.tensor(cols, dtype=torch.int32, device=_dev())
    g = torch.tensor(labels, dtype=torch.int32, device=_dev())
    n = torch.zeros((J, max(k, 1)), dtype=torch.int32, device=_dev())
    mean = torch.zeros((J, max(k, 1)), dtype=torch.float64, device=_dev())
    st = torch.zeros((J, 2), dtype=torch.float64, device=_dev())
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    native.call("sd_kruskal_rows", J, S, native.ptr(ps), ps.stride(0), kind, k, len(cols) if n_cols is None else n_cols,
                native.ptr(c), native.ptr(g), 0, J, native.ptr(n), n.stride(0), native.ptr(mean), mean.stride(0),
                native.ptr(st), st.stride(0), native.stream_ptr())
    return n.cpu().numpy(), mean.cpu().numpy(), st.cpu().numpy()


def test_column_or_label_outside_its_range_is_never_read():
    ps = torch.rand((50, 10), dtype=torch.float64, device=_dev())
    for cols, labels in (([0, 1, 12, 3], [0, 0, 1, 1]), ([0, 1, 2, 3], [0, 3, 1, 1]), ([0, 1, -1, 3], [0, 0, 1, 1]),
                         ([0, 1, 2, 3], [0, -1, 1, 1])):
        n, mean, st = _native(ps, cols, labels, 2)
        assert (n == -1).all() and np.isnan(mean).all() and np.isnan(st).all()
    n, mean, st = _native(ps, [0, 1, 2, 3], [0, 0, 1, 1], 2)               # the same call, in range
    assert (n == 2).all() and np.isfinite(st).all()


def test_sizes_outside_the_limits_are_refused():
    from splicedice_b200 import native, ops
    ps = torch.zeros((2, 16385), dtype=torch.float32, device=_dev())
    for cols, labels, k, needle in ((np.arange(16385), np.arange(16385) % 2, 2, "n_cols = 16385"),
                                    (np.arange(300), np.arange(300) % 257, 257, "n_groups = 257"),
                                    (np.arange(10), np.zeros(10), 1, "n_groups = 1")):
        with pytest.raises(native.NativeCallError) as e:
            _native(ps, cols, labels, k)
        assert e.value.code == native.SD_ERR_INVALID and needle in str(e.value)
    with pytest.raises(ValueError, match="16385 columns"):
        ops.kruskal_rows(ps, [np.arange(8192), np.arange(8192, 16385)])
    with pytest.raises(ValueError, match="257 groups"):
        ops.kruskal_rows(ps, [[i] for i in range(257)])
    with pytest.raises(ValueError, match="1 groups"):
        ops.kruskal_rows(ps, [np.arange(10)])
    r = ops.kruskal_rows(ps, [np.arange(8192), np.arange(8192, 16384)])     # the limit itself runs
    assert torch.isnan(r["H"]).all() and (r["n"] == 8192).all().item()    # all tied at 0.0
    r = ops.kruskal_rows(ps, [[i] for i in range(256)])
    assert (r["n"] == 1).all().item()


def test_argument_errors():
    from splicedice_b200 import native, ops
    ps = torch.zeros((4, 10), dtype=torch.float64, device=_dev())
    for groups in (([0, 1], [1, 2]), ([0, 0], [1]), ([0], [10]), ([], [1]), ([-1], [2])):
        with pytest.raises(ValueError):
            ops.kruskal_rows(ps, groups)
    with pytest.raises(TypeError):
        ops.kruskal_rows(ps.to(torch.int32), [[0], [1]])
    with pytest.raises(native.NativeCallError):
        ops.kruskal_rows(ps, [[0], [1]], row_begin=2, row_end=5)
    n, mean, st = (torch.empty((4, 3), dtype=torch.int32, device=_dev()),
                   torch.empty((4, 3), dtype=torch.float64, device=_dev()),
                   torch.empty((4, 2), dtype=torch.float64, device=_dev()))
    ops.kruskal_rows(ps, [[0], [1], [2]], out=(n, mean, st))
    for narrow in ((n[:, :2], mean, st), (n, mean[:, :2], st), (n, mean, st[:, :1])):
        with pytest.raises(TypeError):
            ops.kruskal_rows(ps, [[0], [1], [2]], out=narrow)


# ---- the CLI -------------------------------------------------------------------------------------
def _args(module, argv):
    p = argparse.ArgumentParser()
    module.add_parser(p)
    return p.parse_args(argv)


def _groups_files(golden_dir, tmp_path):
    """The case's own manifest (cond0 / cond1) and a three-group sample<TAB>group file."""
    manifest = os.path.join(golden_dir, "cli_8x", "input", "manifest.txt")
    three = tmp_path / "three.txt"
    three.write_text("s5\tC\ns0\tA\ns1\tA\r\n\ns2\tB\ns3\tA\ns4\tB\ns6\tC\n")
    return [(manifest, ["cond0", "cond1"], [["s0", "s2", "s4", "s6"], ["s1", "s3", "s5", "s7"]]),
            (str(three), ["C", "A", "B"], [["s5", "s6"], ["s0", "s1", "s3"], ["s2", "s4"]])]


def _check_file(path, events, samples, ps, names, members):
    from oracle import oracle_np
    groups = [np.array([samples.index(s) for s in m]) for m in members]
    k = len(groups)
    lines = open(path).read().split("\n")
    assert lines[0] == "\t".join(["event", "H", "pvalue", "corrected"] + [f"mean_{g}" for g in names])
    assert lines[-1] == "" and [l.split("\t")[0] for l in lines[1:-1]] == list(events)
    got = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines[1:-1]])
    n, mean, h_exact, h_scipy, bound = reference_rows(ps, groups)
    gh, gp, gc = got[:, 0], got[:, 1], got[:, 2]
    t = ~np.isnan(h_exact)
    assert np.array_equal(np.isnan(gh), ~t) and np.array_equal(np.isnan(gc), ~t)
    np.testing.assert_allclose(gh[t], h_exact[t], rtol=1e-13, atol=0)
    fin = t & np.isfinite(h_scipy) & (h_scipy >= 0)
    assert (np.abs(gh[fin] - h_scipy[fin]) <= bound[fin]).all()
    want_p = chdtrc(k - 1, gh[t])
    big = want_p > 1e-300
    np.testing.assert_allclose(gp[t][big], want_p[big], rtol=1e-12, atol=0)
    corrected = oracle_np.bh_adjust(gp[t])
    np.testing.assert_allclose(gc[t], corrected, rtol=1e-12, atol=0)
    assert np.array_equal(np.isnan(got[:, 3:]), np.isnan(mean))
    ok = ~np.isnan(mean)
    np.testing.assert_allclose(got[:, 3:][ok], mean[ok], rtol=0, atol=1e-12)
    return t.sum()


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_tsv_equals_a_scipy_loop(case, golden_dir, tmp_path):
    from splicedice_b200 import compare_conditions, compare_groups
    tsv = os.path.join(golden_dir, case, "expected", "ref_allPS.tsv")
    samples, events, ps = compare_groups.read_ps(tsv)
    for groups_file, names, members in _groups_files(golden_dir, tmp_path):
        out = tmp_path / "cmp.tsv"
        compare_conditions.run_with(_args(compare_conditions, ["-p", tsv, "-g", groups_file, "-o", str(out)]))
        assert _check_file(out, events, samples, ps, names, members) > 100


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_npz_from_quant(case, golden_dir, tmp_path):
    from splicedice_b200 import compare_conditions, quant
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
    for groups_file, names, members in _groups_files(golden_dir, tmp_path):
        out = tmp_path / "cmp.tsv"
        compare_conditions.run_with(_args(compare_conditions, ["-p", npz, "-g", groups_file, "-o", str(out)]))
        assert _check_file(out, events, samples, ps, names, members) > 100
