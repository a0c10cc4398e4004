"""sd_friedman_rows on the GPU (Friedman test per event across conditions measured on the same subjects)
against the exact fraction oracle and scipy.stats.friedmanchisquare(*conditions, nan_policy='omit') on the
float64-widened row, row by row, and `compare_repeated` end to end on the golden PS tables (TSV, and the
NPZ `quant --npz` writes) against a scipy loop + the numpy BH restatement."""
import argparse
import json
import os

import numpy as np
import pytest
from scipy.special import chdtrc

from tests import friedman_cases as cases

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _dev():
    return torch.device("cuda", 0)


def reference_rows(ps, blocks):
    """Per row: n, condition means over the complete blocks, exact Q (NaN where the kernel reports NaN),
    scipy's Q on the float64-widened cells, and the bound 1e-13 * 3 n (k + 1) / c on |Q - Q_scipy|."""
    J, k = ps.shape[0], blocks.shape[1]
    n = np.zeros(J, dtype=np.int64)
    mean = np.full((J, k), np.nan)
    q_exact, q_scipy, bound = np.full(J, np.nan), np.full(J, np.nan), np.full(J, np.nan)
    for j in range(J):
        cells = ps[j].astype(np.float64)[blocks]
        complete = cells[~np.isnan(cells).any(axis=1)]
        d, n[j], t = cases.block_terms(cells)
        if n[j]:
            mean[j] = complete.mean(axis=0)
        q = cases.exact_q(d, n[j], k, t)
        if q is not None:
            q_exact[j] = float(q)
            bound[j] = 1e-13 * 3 * n[j] * (k + 1) / cases.tie_factor(n[j], k, t)
            q_scipy[j] = cases.scipy_q(cells)
    return n, mean, q_exact, q_scipy, bound


def kernel_rows(ps, blocks, **kw):
    from splicedice_b200 import ops
    r = ops.friedman_rows(torch.from_numpy(ps).to(_dev()), blocks, **kw)
    return r["n"].cpu().numpy(), r["mean"].cpu().numpy(), r["Q"].cpu().numpy(), r["p"].cpu().numpy()


def assert_rows_match(got, want, k):
    gn, gmean, gq, gp = got
    wn, wmean, wq, ws, bound = want
    np.testing.assert_array_equal(gn, wn)
    assert np.array_equal(np.isnan(gmean), np.isnan(wmean))
    ok = ~np.isnan(wmean)
    np.testing.assert_allclose(gmean[ok], wmean[ok], rtol=0, atol=1e-12)
    assert np.array_equal(np.isnan(gq), np.isnan(wq)) and np.array_equal(np.isnan(gp), np.isnan(wq))
    t = ~np.isnan(wq)
    assert np.array_equal(gq[t].view(np.uint64), wq[t].view(np.uint64))      # the exact fraction, rounded once
    fin = t & np.isfinite(ws)
    assert (np.abs(gq[fin] - ws[fin]) <= bound[fin]).all(), np.max(np.abs(gq[fin] - ws[fin]) / bound[fin])
    assert (gp[t & (gq == 0)] == 1.0).all()
    want_p = chdtrc(k - 1, gq[t])
    big = want_p > 1e-300
    np.testing.assert_allclose(gp[t][big], want_p[big], rtol=1e-12, atol=0)
    assert ((gp[t] >= 0) & (gp[t] <= 1)).all()
    return t.sum()


def random_blocks(rng, S, n_blocks, k):
    return rng.permutation(S)[:n_blocks * k].reshape(n_blocks, k)


def tied_matrix(rng, J, S):
    """Heavy ties: mostly 0 or 1, the rest rounded to 2 decimals; -0.0 next to +0.0; +-inf; NaN."""
    ps = np.round(rng.random((J, S)), 2)
    u = rng.random((J, S))
    ps[u < 0.3] = 0.0
    ps[(u >= 0.3) & (u < 0.5)] = 1.0
    ps[rng.random((J, S)) < 0.15] = -0.0
    ps[rng.random((J, S)) < 0.02] = np.inf
    ps[rng.random((J, S)) < 0.02] = -np.inf
    ps[rng.random((J, S)) < 0.03] = np.nan
    return ps


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("k", [3, 4, 7, 64, 256])
def test_heavy_ties_signed_zero_and_infinities(k, dtype):
    rng = np.random.default_rng(k)
    n_blocks = {3: 40, 4: 33, 7: 20, 64: 9, 256: 5}[k]
    J, S = (60 if k >= 64 else 200), n_blocks * k + 11
    ps = tied_matrix(rng, J, S)
    blocks = random_blocks(rng, S, n_blocks, k)
    ps[::5, blocks[:, 0]] += 0.5                             # some rows far from balanced
    if k >= 64:                                              # NaN per block, not per cell: most blocks complete
        ps[np.isnan(ps)] = 0.25
        ps[rng.random((J, S)) < 0.2 / k] = np.nan
    ps = ps.astype(dtype)
    tested = assert_rows_match(kernel_rows(ps, blocks), reference_rows(ps, blocks), k)
    assert tested > J // 2


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_nan_patterns_balanced_all_tied_and_single_block_rows(dtype):
    rng = np.random.default_rng(3)
    k, n_blocks = 3, 10
    S = k * n_blocks
    blocks = np.arange(S).reshape(n_blocks, k)
    rows = []
    for pattern in range(9):
        r = rng.random(S)
        if pattern == 0:
            r[blocks[:, 1]] = np.nan                         # one condition empty: every block dropped
        elif pattern == 1:
            r[:] = np.nan
        elif pattern == 2:
            r[blocks[1:, 0]] = np.nan                        # one complete block left
        elif pattern == 3:
            r[:] = 0.7                                       # all tied
        elif pattern == 4:
            r[:] = rng.choice([0.0, -0.0], S)                # all tied through the signed zeros
            r[blocks[:4, 2]] = np.nan
        elif pattern == 5:
            for b in range(n_blocks):                        # balanced: each condition takes every rank equally
                r[blocks[b]] = np.roll([0.1, 0.2, 0.3], b % 3)
            r[blocks[9]] = np.nan
        elif pattern == 6:
            r[blocks[:, 0]] = -np.inf
            r[blocks[:, 2]] = np.inf                         # infinities are ordinary values
        elif pattern == 7:
            r[blocks[:5]] = 0.25                             # half the blocks tied throughout
            r[blocks[5:, 1]] = np.nan                        # and the others dropped
        rows.append(r)
    ps = np.array(rows).astype(dtype)
    got, want = kernel_rows(ps, blocks), reference_rows(ps, blocks)
    assert_rows_match(got, want, k)
    n, mean, q, p = got
    np.testing.assert_array_equal(n, [0, 0, 1, 10, 6, 9, 10, 5, 10])
    assert np.isnan(q[[0, 1, 3, 4, 7]]).all() and np.isnan(p[[0, 1, 3, 4, 7]]).all()
    assert np.isnan(mean[[0, 1]]).all() and not np.isnan(mean[2:]).any()
    assert q[2] >= 0 and np.isfinite(p[2])                   # n = 1 is a valid test
    assert q[5] == 0.0 and p[5] == 1.0
    assert q[6] == 2.0 * n_blocks and np.isfinite(p[6])      # every block ranked -inf < x < +inf


def test_one_block_of_three():
    ps = np.array([[0.1, 0.5, 0.3]])
    n, _, q, p = kernel_rows(ps, np.array([[0, 1, 2]]))
    assert n[0] == 1 and q[0] == 2.0 and abs(p[0] - np.exp(-1.0)) <= 1e-15
    assert abs(cases.scipy_q(ps[:, [0, 1, 2]]) - 2.0) < 1e-12


@pytest.mark.parametrize("n_blocks,k", [(5461, 3), (4096, 4), (64, 256), (128, 128)])
def test_cells_up_to_the_limit(n_blocks, k):
    rng = np.random.default_rng(n_blocks + k)
    J = 6
    S = n_blocks * k + 3
    ps = rng.random((J, S))
    ps[:, ::3] = np.round(ps[:, ::3], 1)
    ps[rng.random((J, S)) < 0.002] = np.nan
    ps[1] = 0.5                                              # all tied
    blocks = random_blocks(rng, S, n_blocks, k)
    ps[2, blocks] += np.arange(k)[None, :] * 1e-3            # a strong condition effect
    assert_rows_match(kernel_rows(ps, blocks), reference_rows(ps, blocks), k)


def test_deep_chi_square_tail_on_the_device():
    """64 subjects x 256 conditions with a growing shift per condition: Q past 1,490, so Q / 2 passes 745
    (where a recurrence started at e^-x underflows) while p is still above 1e-300."""
    k, n_blocks = 256, 64
    rng = np.random.default_rng(7)
    shifts = np.linspace(0.00125, 0.0019, 12)
    blocks = np.arange(n_blocks * k).reshape(n_blocks, k)
    ps = rng.random((len(shifts), n_blocks * k))
    ps += shifts[:, None] * np.tile(np.arange(k), n_blocks)[None, :]
    got = kernel_rows(ps, blocks)
    assert_rows_match(got, reference_rows(ps, blocks), k)
    q, p = got[2], got[3]
    want = chdtrc(k - 1, q)
    keep = want > 1e-300
    assert (keep & (q / 2 > 745)).sum() >= 2 and (want[keep] < 1e-200).any()


def test_padded_leading_dimensions_row_range_and_out_buffers():
    from splicedice_b200 import ops
    rng = np.random.default_rng(4)
    J, S, k = 500, 70, 5
    ps = tied_matrix(rng, J, S)
    blocks = random_blocks(rng, S, 12, k)
    buf = torch.full((J, S + 9), 7.0, dtype=torch.float64, device=_dev())
    buf[:, :S] = torch.from_numpy(ps).to(_dev())
    n_buf = torch.full((J,), -9, dtype=torch.int32, device=_dev())
    m_buf = torch.full((J, k + 2), -9.0, dtype=torch.float64, device=_dev())
    st_buf = torch.full((J, 5), -9.0, dtype=torch.float64, device=_dev())
    r0, r1 = 123, 401
    r = ops.friedman_rows(buf[:, :S], blocks, row_begin=r0, row_end=r1, out=(n_buf, m_buf, st_buf))
    assert r["n"].data_ptr() == n_buf.data_ptr() and r["mean"].data_ptr() == m_buf.data_ptr()
    n, m, st = n_buf.cpu().numpy(), m_buf.cpu().numpy(), st_buf.cpu().numpy()
    assert (n[:r0] == -9).all() and (n[r1:] == -9).all()
    for a, w in ((m, k), (st, 2)):
        assert (a[:r0] == -9).all() and (a[r1:] == -9).all() and (a[:, w:] == -9).all()
    got = (n[r0:r1], m[r0:r1, :k], st[r0:r1, 0], st[r0:r1, 1])
    assert_rows_match(got, reference_rows(ps[r0:r1], blocks), k)
    whole = kernel_rows(ps, blocks)
    for a, b in zip(whole, got):
        assert np.array_equal(np.ascontiguousarray(a[r0:r1]).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def resident_bound(n_blocks, k, itemsize):
    """An upper bound on the kernel's resident grid: 148-ish SMs times the CTAs of its thread count and
    dynamic shared memory that fit on one (228 KB, 1 KB reserved per CTA), at most 32"""
    cells = n_blocks * k
    threads = min(256, (cells + 31) // 32 * 32)
    smem = 8 * k + (itemsize + 4) * cells + 4 * n_blocks + 48
    per_sm = min(32, 2048 // threads, (228 * 1024) // (smem + 1024))
    return torch.cuda.get_device_properties(0).multi_processor_count * per_sm


def varying_rows(rng, J, S, blocks):
    """Rows that differ from one to the next: ties on a 2-decimal grid, a different random set of dropped
    blocks in every row (one NaN cell each, 0 to ~50 % of the blocks), a condition effect in some rows, and
    all-tied, balanced and all-NaN rows at random row indices."""
    nb, k = blocks.shape
    ps = np.round(rng.random((J, S)), 2)
    effect = rng.random(J) < 0.3
    ps[np.ix_(effect, blocks.T.reshape(-1))] += np.repeat(np.arange(k) * 0.05, nb)[None, :]
    drop = rng.random((J, nb)) < rng.random(J)[:, None] * 0.5
    rows, bs = np.nonzero(drop)
    ps[rows, blocks[bs, rng.integers(0, k, bs.size)]] = np.nan
    special = rng.permutation(J)[:3 * max(1, J // 40)].reshape(3, -1)
    ps[special[0]] = 0.5                                             # all tied
    ps[special[2]] = np.nan                                          # no complete block
    full = nb - nb % k                                               # balanced: every condition takes each rank
    for j in special[1]:                                             # equally often; the rest dropped
        for b in range(nb):
            ps[j, blocks[b]] = np.roll(np.arange(k) / k, b % k) if b < full else np.nan
    return ps, special


@pytest.mark.parametrize("n_blocks,k,dtype,rows_per_cta", [
    (250, 4, np.float32, 8),          # 1,000 cells: every cell loaded a row ahead
    (250, 4, np.float64, 8),
    (16, 4, np.float32, 4),           # 64 cells, 64-thread CTAs
    (5461, 3, np.float64, 4),         # 16,383 cells, 213 KB of shared memory: one CTA per SM, most cells
])                                    # loaded in the row itself
def test_many_rows_per_cta(n_blocks, k, dtype, rows_per_cta):
    """J several times the resident grid, so every CTA stages, prefetches, stamps dropped blocks and
    overlaps warp 0's tail over several rows, and its p epilogue covers several rows; every row against
    the oracles, then a row range that starts off a multiple of the grid, bit for bit against the whole."""
    from splicedice_b200 import ops
    rng = np.random.default_rng(n_blocks * k)
    bound = resident_bound(n_blocks, k, np.dtype(dtype).itemsize)
    J = rows_per_cta * bound
    S = n_blocks * k + 5
    blocks = random_blocks(rng, S, n_blocks, k)
    ps, special = varying_rows(rng, J, S, blocks)
    ps = ps.astype(dtype)
    got = kernel_rows(ps, blocks)
    want = reference_rows(ps, blocks)
    assert assert_rows_match(got, want, k) > J // 2
    n, _, q, p = got
    assert np.isnan(q[special[0]]).all() and (n[special[0]] == n_blocks).all()
    assert (q[special[1]] == 0).all() and (p[special[1]] == 1).all()
    assert (n[special[2]] == 0).all() and np.isnan(q[special[2]]).all()
    assert len(np.unique(n)) > 10                                    # the dropped blocks differ row to row
    r0, r1 = bound + 37, J - 101
    dev = _dev()
    out = (torch.full((J,), -9, dtype=torch.int32, device=dev), torch.full((J, k), -9.0, dtype=torch.float64, device=dev),
           torch.full((J, 2), -9.0, dtype=torch.float64, device=dev))
    ops.friedman_rows(torch.from_numpy(ps).to(dev), blocks, row_begin=r0, row_end=r1, out=out)
    part = [t.cpu().numpy() for t in out]
    for a in part:
        assert (a[:r0] == -9).all() and (a[r1:] == -9).all()
    for a, b in zip((n, got[1], np.stack([q, p], axis=1)), part):
        assert np.array_equal(np.ascontiguousarray(a[r0:r1]).view(np.uint8), np.ascontiguousarray(b[r0:r1]).view(np.uint8))


def _native(ps, cols, k, n_blocks):
    """sd_friedman_rows on a device column list as given (ops checks host lists first)"""
    from splicedice_b200 import native
    J, S = ps.shape
    c = torch.tensor(cols, dtype=torch.int32, device=_dev())
    n = torch.zeros(J, dtype=torch.int32, device=_dev())
    mean = torch.zeros((J, k), dtype=torch.float64, device=_dev())
    st = torch.zeros((J, 2), dtype=torch.float64, device=_dev())
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    native.call("sd_friedman_rows", J, S, native.ptr(ps), ps.stride(0), kind, k, n_blocks, native.ptr(c), 0, J,
                native.ptr(n), native.ptr(mean), mean.stride(0), native.ptr(st), st.stride(0), native.stream_ptr())
    return n.cpu().numpy(), mean.cpu().numpy(), st.cpu().numpy()


def test_column_outside_its_range_is_never_read():
    ps = torch.rand((50, 10), dtype=torch.float64, device=_dev())
    for cols in ([0, 1, 2, 3, 4, 12], [0, 1, -1, 3, 4, 5], [0, 1, 2, 3, 4, 10]):
        n, mean, st = _native(ps, cols, 3, 2)
        assert (n == -1).all() and np.isnan(mean).all() and np.isnan(st).all()
    n, mean, st = _native(ps, [0, 1, 2, 3, 4, 5], 3, 2)               # the same call, in range
    assert (n == 2).all() and np.isfinite(st).all()


def test_sizes_outside_the_limits_are_refused():
    from splicedice_b200 import native, ops
    ps = torch.zeros((2, 16385), dtype=torch.float32, device=_dev())
    for cols, k, nb, needle in ((np.arange(16385), 5, 3277, "n_blocks = 3277"),
                                (np.arange(257 * 2), 257, 2, "n_conditions = 257"),
                                (np.arange(10), 2, 5, "n_conditions = 2")):
        with pytest.raises(native.NativeCallError) as e:
            _native(ps, cols, k, nb)
        assert e.value.code == native.SD_ERR_INVALID and needle in str(e.value)
    with pytest.raises(ValueError, match="16385 cells"):
        ops.friedman_rows(ps, np.arange(16385).reshape(3277, 5))
    with pytest.raises(ValueError, match="257 conditions"):
        ops.friedman_rows(ps, np.arange(514).reshape(2, 257))
    with pytest.raises(ValueError, match="2 conditions"):
        ops.friedman_rows(ps, np.arange(10).reshape(5, 2))
    r = ops.friedman_rows(ps, np.arange(16384).reshape(4096, 4))     # the limit itself runs
    assert torch.isnan(r["Q"]).all() and (r["n"] == 4096).all().item()  # all tied at 0.0
    r = ops.friedman_rows(ps, np.arange(16384).reshape(64, 256))
    assert (r["n"] == 64).all().item()


def test_argument_errors():
    from splicedice_b200 import native, ops
    ps = torch.zeros((4, 10), dtype=torch.float64, device=_dev())
    for blocks in (np.array([[0, 1, 1]]), np.array([[0, 1, 10]]), np.array([[-1, 1, 2]]), np.array([0, 1, 2]),
                   np.array([[0.0, 1.0, 2.0]]), np.zeros((0, 3), dtype=np.int64), np.array([[0, 1, 2], [3, 4, 0]])):
        with pytest.raises(ValueError):
            ops.friedman_rows(ps, blocks)
    with pytest.raises(TypeError):
        ops.friedman_rows(ps.to(torch.int32), [[0, 1, 2]])
    with pytest.raises(native.NativeCallError):
        ops.friedman_rows(ps, [[0, 1, 2]], row_begin=2, row_end=5)
    n, mean, st = (torch.empty(4, dtype=torch.int32, device=_dev()),
                   torch.empty((4, 3), dtype=torch.float64, device=_dev()),
                   torch.empty((4, 2), dtype=torch.float64, device=_dev()))
    ops.friedman_rows(ps, [[0, 1, 2]], out=(n, mean, st))
    for bad in ((n[:3], mean, st), (n, mean[:, :2], st), (n, mean, st[:, :1]), (n.view(4, 1), mean, st),
                (n.to(torch.int64), mean, st)):
        with pytest.raises(TypeError):
            ops.friedman_rows(ps, [[0, 1, 2]], out=bad)


# ---- the CLI -------------------------------------------------------------------------------------
def _args(module, argv):
    p = argparse.ArgumentParser()
    module.add_parser(p)
    return p.parse_args(argv)


def _blocks_files(tmp_path):
    """2 subjects x 4 conditions (s0-s3 / s4-s7), and 3 conditions with one subject skipped (an empty field)."""
    four = tmp_path / "four.txt"
    four.write_text("c0\tc1\tc2\tc3\ns0\ts1\ts2\ts3\ns4\ts5\ts6\ts7\n")
    three = tmp_path / "three.txt"
    three.write_text("wk12\tbase\twk4\r\n\ns5\ts0\ts2\r\ns7\t\ts1\ns3\ts6\ts4\n")
    return [(str(four), ["c0", "c1", "c2", "c3"], [["s0", "s1", "s2", "s3"], ["s4", "s5", "s6", "s7"]]),
            (str(three), ["wk12", "base", "wk4"], [["s5", "s0", "s2"], ["s3", "s6", "s4"]])]


def _check_file(path, events, samples, ps, names, subjects):
    from oracle import oracle_np
    blocks = np.array([[samples.index(s) for s in subject] for subject in subjects])
    k = len(names)
    lines = open(path).read().split("\n")
    assert lines[0] == "\t".join(["event", "n", "Q", "pvalue", "corrected"] + [f"mean_{c}" for c in names])
    assert lines[-1] == "" and [l.split("\t")[0] for l in lines[1:-1]] == list(events)
    got = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines[1:-1]])
    n, mean, q_exact, q_scipy, bound = reference_rows(ps, blocks)
    gn, gq, gp, gc = got[:, 0], got[:, 1], got[:, 2], got[:, 3]
    np.testing.assert_array_equal(gn, n)
    t = ~np.isnan(q_exact)
    assert np.array_equal(np.isnan(gq), ~t) and np.array_equal(np.isnan(gc), ~t)
    assert np.array_equal(gq[t], q_exact[t])
    fin = t & np.isfinite(q_scipy)
    assert (np.abs(gq[fin] - q_scipy[fin]) <= bound[fin]).all()
    want_p = chdtrc(k - 1, gq[t])
    big = want_p > 1e-300
    np.testing.assert_allclose(gp[t][big], want_p[big], rtol=1e-12, atol=0)
    np.testing.assert_allclose(gc[t], oracle_np.bh_adjust(gp[t]), rtol=1e-12, atol=0)
    assert np.array_equal(np.isnan(got[:, 4:]), np.isnan(mean))
    ok = ~np.isnan(mean)
    np.testing.assert_allclose(got[:, 4:][ok], mean[ok], rtol=0, atol=1e-12)
    return t.sum()


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_tsv_equals_a_scipy_loop(case, golden_dir, tmp_path, capsys):
    from splicedice_b200 import compare_groups, compare_repeated
    tsv = os.path.join(golden_dir, case, "expected", "ref_allPS.tsv")
    samples, events, ps = compare_groups.read_ps(tsv)
    for blocks_file, names, subjects in _blocks_files(tmp_path):
        out = tmp_path / "cmp.tsv"
        compare_repeated.run_with(_args(compare_repeated, ["-p", tsv, "--blocks", blocks_file, "-o", str(out)]))
        tested = _check_file(out, events, samples, ps, names, subjects)
        assert tested > 100
        text = capsys.readouterr().out
        assert f"{tested} / {len(events)} events tested" in text
        assert ("1 subject(s) without a sample for every condition skipped" in text) == (len(names) == 3)


@pytest.mark.parametrize("case", ["cli_8x", "cli_8x_lownan"])
def test_cli_npz_from_quant(case, golden_dir, tmp_path):
    from splicedice_b200 import compare_repeated, quant
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
    for blocks_file, names, subjects in _blocks_files(tmp_path):
        out = tmp_path / "cmp.tsv"
        compare_repeated.run_with(_args(compare_repeated, ["-p", npz, "--blocks", blocks_file, "-o", str(out)]))
        assert _check_file(out, events, samples, ps, names, subjects) > 100
