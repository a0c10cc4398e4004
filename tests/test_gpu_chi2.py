"""sd_chi2_pairwise on the GPU (Yates-corrected chi-squared per (event, sample pair)) and `pairwise
--chi2` end to end: the twin's vectors through the kernel against scipy / mpmath / the CPU twin, the
matrix layout (row ranges, padded leading dimensions, pair subsets), the first-refused index, and
the CLI on the golden inputs (refusal) and on filtered inputs (files equal to a chi2_contingency loop)."""
import argparse
import os

import numpy as np
import pytest

from tests import chi2_cases as cases
from tests.test_chi2_twin import twin  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NONE = -1


def _dev():
    return torch.device("cuda", 0)


def _tables_as_rows(t):
    """Table i as row i of a two-sample problem: inc[i] = (a, b), exc[i] = (c, d), one pair (0, 1)."""
    inc = torch.from_numpy(np.ascontiguousarray(t[:, :2], dtype=np.int32)).to(_dev())
    exc = torch.from_numpy(np.ascontiguousarray(t[:, 2:], dtype=np.int64)).to(_dev())
    return inc, exc


def _kernel_tables(t, refused=None):
    from splicedice_b200 import ops
    inc, exc = _tables_as_rows(t)
    return ops.chi2_pairwise(inc, exc, [0], [1], refused=refused)[:, 0].cpu().numpy()


def test_vectors_through_the_kernel(twin):  # noqa: F811
    domain = np.array([[1, 2, 1 << 61, 4], [1, 2, 3, (1 << 61) + 5], [(1 << 31) - 1, 2, (1 << 61) - 1, 4]])
    t = np.concatenate([cases.random_tables(seed=1), cases.small_tables(8), domain])
    got = _kernel_tables(t)
    want, status = twin(t)
    val = status == cases.VALUE
    assert np.isnan(got[~val]).all()
    np.testing.assert_allclose(got[val], want[val], rtol=2e-15 * 64, atol=1e-300)      # device vs glibc erfc
    assert np.array_equal(got[val] == 1.0, want[val] == 1.0)
    rnd = cases.random_tables(seed=1)
    assert cases.max_rel(got[: len(rnd)], cases.mpmath_p(rnd)) < 1e-12
    cases.assert_scipy_parity(rnd, got[: len(rnd)])
    small = cases.small_tables(8)
    sv = cases.expected_status(small) == cases.VALUE
    np.testing.assert_allclose(got[len(rnd):-len(domain)][sv], cases.scipy_p(small)[sv], rtol=1e-9, atol=0)
    np.testing.assert_array_equal(status[-len(domain):], [cases.REFUSED_ENTRY] * 2 + [cases.VALUE])


def _random_problem(J, S, seed, zero_frac=0.3):
    rng = np.random.default_rng(seed)
    inc = rng.integers(0, 50, size=(J, S)).astype(np.int64)
    inc[rng.random((J, S)) < zero_frac] = 0
    exc = rng.integers(0, 400, size=(J, S)).astype(np.int64)
    exc[rng.random((J, S)) < zero_frac] = 0
    return inc, exc


def _host_reference(twin_fn, inc, exc, pa, pb):  # noqa: F811
    t = np.stack([inc[:, pa], inc[:, pb], exc[:, pa], exc[:, pb]], axis=-1).reshape(-1, 4)
    p, status = twin_fn(t)
    return p.reshape(len(inc), len(pa)), status.reshape(len(inc), len(pa))


def test_layout_row_ranges_padding_and_pair_subsets(twin):  # noqa: F811
    from splicedice_b200 import ops
    J, S = 3000, 20
    inc_h, exc_h = _random_problem(J, S, seed=4)
    rng = np.random.default_rng(5)
    pa_all, pb_all = ops.all_pairs(S)
    pick = rng.permutation(len(pa_all))[:77]
    pa, pb = pa_all[pick], pb_all[pick]
    inc_buf = torch.zeros((J, S + 5), dtype=torch.int32, device=_dev())
    exc_buf = torch.zeros((J, S + 3), dtype=torch.int64, device=_dev())
    inc_buf[:, :S] = torch.from_numpy(inc_h.astype(np.int32)).to(_dev())
    exc_buf[:, :S] = torch.from_numpy(exc_h).to(_dev())
    inc, exc = inc_buf[:, :S], exc_buf[:, :S]
    P = len(pa)
    out_buf = torch.full((J, P + 3), -7.0, dtype=torch.float64, device=_dev())
    out = out_buf[:, :P]
    r0, r1 = 700, 2100
    ops.chi2_pairwise(inc, exc, pa, pb, row_begin=r0, row_end=r1, out=out)
    got = out_buf.cpu().numpy()
    want, _ = _host_reference(twin, inc_h, exc_h, pa, pb)
    assert (got[:r0] == -7.0).all() and (got[r1:] == -7.0).all() and (got[:, P:] == -7.0).all()
    np.testing.assert_allclose(got[r0:r1, :P], want[r0:r1], rtol=2e-15 * 64, atol=1e-300)
    assert np.array_equal(np.isnan(got[r0:r1, :P]), np.isnan(want[r0:r1]))
    # bit-identical whatever the row ranges the rows are computed in
    whole = ops.chi2_pairwise(inc, exc, pa, pb).cpu().numpy()
    parts = torch.empty((J, P), dtype=torch.float64, device=_dev())
    for a, b in ((0, 1), (1, 999), (999, 2500), (2500, J)):
        ops.chi2_pairwise(inc, exc, pa, pb, row_begin=a, row_end=b, out=parts)
    assert np.array_equal(whole.view(np.uint64), parts.cpu().numpy().view(np.uint64))
    assert np.array_equal(whole[r0:r1].view(np.uint64), got[r0:r1, :P].view(np.uint64))


def _refused_value(ref):
    return int(ref.item())


def test_first_refused_among_many_scattered_refusals(twin):  # noqa: F811
    """~2,000 refused tables spread over hundreds of CTAs, none in the first 20,000 rows: the index is
    numpy's first refused (row, pair) in row-major order; NULL tracking gives the same matrix."""
    from splicedice_b200 import ops
    J, S = 60000, 16
    rng = np.random.default_rng(8)
    inc_h = rng.integers(1, 60, size=(J, S)).astype(np.int64)
    exc_h = rng.integers(1, 300, size=(J, S)).astype(np.int64)
    rows = rng.choice(np.arange(20000, J), size=300, replace=False)
    cols = rng.integers(0, S, size=300)
    inc_h[rows, cols] = 0
    exc_h[rows, cols] = 0                                   # sample column all zero: c1 or c2 == 0
    pa, pb = ops.all_pairs(S)
    want_p, status = _host_reference(twin, inc_h, exc_h, pa, pb)
    bad = np.flatnonzero(cases.refused_mask(status.reshape(-1)))
    assert len(bad) > 1000
    inc = torch.from_numpy(inc_h.astype(np.int32)).to(_dev())
    exc = torch.from_numpy(exc_h).to(_dev())
    ref = torch.full((1,), NONE, dtype=torch.int64, device=_dev())
    p = ops.chi2_pairwise(inc, exc, pa, pb, refused=ref).cpu().numpy()
    assert _refused_value(ref) == bad[0]
    assert np.array_equal(np.isnan(p).reshape(-1)[bad], np.ones(len(bad), bool))
    # a row range past the first refusal: the first refusal inside it, in absolute rows
    r0 = int(bad[0] // len(pa)) + 1
    ref.fill_(NONE)
    ops.chi2_pairwise(inc, exc, pa, pb, row_begin=r0, refused=ref)
    assert _refused_value(ref) == bad[bad >= r0 * len(pa)][0]
    # only ever lowered: a smaller initial value stays
    ref.fill_(5)
    ops.chi2_pairwise(inc, exc, pa, pb, refused=ref)
    assert _refused_value(ref) == 5
    # untouched without refusals
    ref.fill_(NONE)
    ops.chi2_pairwise(inc[:20000], exc[:20000], pa, pb, refused=ref)
    assert _refused_value(ref) == NONE
    q = ops.chi2_pairwise(inc, exc, pa, pb).cpu().numpy()
    assert np.array_equal(p.view(np.uint64), q.view(np.uint64))
    np.testing.assert_allclose(p[~np.isnan(p)], want_p[~np.isnan(want_p)], rtol=2e-15 * 64, atol=1e-300)


def test_argument_errors():
    from splicedice_b200 import native, ops
    inc, exc = _tables_as_rows(np.array([[1, 2, 3, 4]]))
    with pytest.raises(ValueError):
        ops.chi2_pairwise(inc, exc, [0], [2])
    with pytest.raises(native.NativeCallError):
        ops.chi2_pairwise(inc, exc, [0], [1], row_begin=0, row_end=2)
    with pytest.raises(TypeError):
        ops.chi2_pairwise(inc, exc, [0], [1], refused=torch.full((1,), -1, dtype=torch.int32, device=_dev()))


# ---- the CLI -------------------------------------------------------------------------------------
def _args(module, argv):
    p = argparse.ArgumentParser()
    module.add_parser(p)
    return p.parse_args(argv)


def _golden(golden_dir, case):
    exp = os.path.join(golden_dir, case, "expected")
    counts_tsv, clusters_tsv = os.path.join(exp, "ref_inclusionCounts.tsv"), os.path.join(exp, "ref_allClusters.tsv")
    lines = [l.rstrip("\n").split("\t") for l in open(counts_tsv)]
    samples, names = lines[0][1:], [r[0] for r in lines[1:]]
    counts = np.array([[int(x) for x in r[1:]] for r in lines[1:]], dtype=np.int64)
    adj = {}
    for l in open(clusters_tsv):
        f = l.split()
        adj[f[0]] = f[1].split(",") if len(f) > 1 else []
    return counts_tsv, clusters_tsv, samples, names, counts, adj


def _exclusions(names, counts, adj, keep):
    idx = {n: i for i, n in enumerate(names)}
    return np.array([sum((counts[idx[o]] for o in adj[n] if o in keep), np.zeros(counts.shape[1], np.int64))
                     for n in names])


def _chi2_loop(names, counts, adj, keep):
    """ref_port.pairwise_loop's shape with scipy.stats.chi2_contingency: per listed event, exclusions
    over listed partners, one test per sample pair in pair order; the first refusal raises."""
    from scipy.stats import chi2_contingency
    rows = [i for i, n in enumerate(names) if n in keep]
    exc = _exclusions(names, counts, adj, keep)
    S = counts.shape[1]
    pairs = [(a, b) for a in range(S - 1) for b in range(a + 1, S)]
    out = []
    for r in rows:
        out.append([chi2_contingency([[float(counts[r, a]), float(counts[r, b])],
                                      [float(exc[r, a]), float(exc[r, b])]])[1] for a, b in pairs])
    return [names[r] for r in rows], np.array(out).reshape(len(rows), len(pairs))


def _first_refusal(names, counts, adj, samples):
    """(event, column, position) of the first table the reference's loop stops at (unfiltered input)."""
    exc = _exclusions(names, counts, adj, set(names))
    S = counts.shape[1]
    for r, n in enumerate(names):
        for a in range(S - 1):
            for b in range(a + 1, S):
                pos = cases.scipy_refusal_position([counts[r, a], counts[r, b], exc[r, a], exc[r, b]])
                if pos is not None:
                    return n, f"{samples[a]}_{samples[b]}", pos
    return None


def _nonzero_margin_filter(names, counts, adj):
    """Largest event set, by repeated removal, in which every table (exclusions over listed partners
    only, as with -f) has four non-zero margins."""
    keep = set(names)
    while True:
        exc = _exclusions(names, counts, adj, keep)
        bad = set()
        for r, n in enumerate(names):
            if n not in keep:
                continue
            i, e = counts[r], exc[r]
            for a in range(len(i) - 1):
                for b in range(a + 1, len(i)):
                    if min(i[a] + i[b], e[a] + e[b], i[a] + e[a], i[b] + e[b]) == 0:
                        bad.add(n)
        if not bad:
            return keep
        keep -= bad


def _run(counts_tsv, clusters_tsv, out, mode, extra=()):
    from splicedice_b200 import pairwise_fisher
    pairwise_fisher.run_with(_args(pairwise_fisher, ["--inclusionSPLICEDICE", counts_tsv, "-c", clusters_tsv, "--chi2",
                                                     "--multiple_test_correction", mode, "-o", str(out), *extra]))


@pytest.mark.parametrize("case", ["survey_vector", "cli_5x_pairwise"])
def test_cli_refuses_like_scipy_and_writes_nothing(case, golden_dir, tmp_path):
    counts_tsv, clusters_tsv, samples, names, counts, adj = _golden(golden_dir, case)
    event, column, pos = _first_refusal(names, counts, adj, samples)
    out = tmp_path / "pw.tsv"
    with pytest.raises(ValueError) as e:
        _run(counts_tsv, clusters_tsv, out, "pairwise")
    msg = str(e.value)
    assert f"zero element at ({pos[0]}, {pos[1]})" in msg
    assert f"event {event}," in msg and f"column {column}," in msg
    assert not out.exists()


@pytest.mark.parametrize("case", ["survey_vector", "cli_5x_pairwise"])
@pytest.mark.parametrize("mode", ["none", "pairwise", "all"])
def test_cli_filtered_file_equals_a_chi2_contingency_loop(case, mode, golden_dir, tmp_path):
    from oracle import oracle_np
    counts_tsv, clusters_tsv, samples, names, counts, adj = _golden(golden_dir, case)
    keep = _nonzero_margin_filter(names, counts, adj)
    assert len(keep) >= 6
    flt = tmp_path / "filter.txt"
    flt.write_text("\n".join(sorted(keep)) + "\n")
    out = tmp_path / "pw.tsv"
    _run(counts_tsv, clusters_tsv, out, mode, ["-f", str(flt)])
    got = [l.rstrip("\n").split("\t") for l in open(out)]
    events, want = _chi2_loop(names, counts, adj, keep)
    if mode == "pairwise":
        want = np.stack([oracle_np.bh_adjust(want[:, k]) for k in range(want.shape[1])], axis=1)
    elif mode == "all":
        want = oracle_np.bh_adjust(want.reshape(-1)).reshape(want.shape)
    S = len(samples)
    assert got[0] == ["clusterID"] + [f"{samples[a]}_{samples[b]}" for a in range(S - 1) for b in range(a + 1, S)]
    assert [r[0] for r in got[1:]] == events
    g = np.array([[float(x) for x in r[1:]] for r in got[1:]])
    np.testing.assert_allclose(g, want, rtol=1e-9, atol=0)
    assert np.array_equal(g == 1.0, want == 1.0)


# ---- two GPUs ------------------------------------------------------------------------------------
two_gpus = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2,
                              reason="needs two CUDA devices")


@two_gpus
def test_two_gpu_chi2_matrices_are_bit_identical():
    from splicedice_b200 import pairwise_fisher
    J, S = 20000, 10
    rng = np.random.default_rng(6)
    counts = rng.integers(1, 200, size=(J, S)).astype(np.float64)
    names = [f"chr1:{i}-{i + 1}:+" for i in range(J)]
    clusters = {names[i]: [names[i ^ 1]] + ([names[i - 2]] if i >= 2 and i % 2 else []) for i in range(J)}
    for mode in ("none", "pairwise", "all"):
        a = pairwise_fisher.pairwise_pvalues(names, counts, clusters, correction=mode, gpus=1, test="chi2")
        b = pairwise_fisher.pairwise_pvalues(names, counts, clusters, correction=mode, gpus=2, test="chi2")
        assert np.isfinite(a).all()
        np.testing.assert_array_equal(a.view(np.uint64), b.view(np.uint64))


@two_gpus
def test_two_gpu_refusal_names_the_same_table(golden_dir, tmp_path):
    counts_tsv, clusters_tsv, *_ = _golden(golden_dir, "cli_5x_pairwise")
    msgs = []
    for gpus in ("1", "2"):
        out = tmp_path / f"pw{gpus}.tsv"
        with pytest.raises(ValueError) as e:
            _run(counts_tsv, clusters_tsv, out, "pairwise", ["--gpus", gpus])
        assert not out.exists()
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1]


# ---- the unmodified reference, live ---------------------------------------------------------------
@pytest.mark.needs_reference
def test_reference_chi2_matches_on_filtered_input_and_raises_on_unfiltered(golden_dir, tmp_path):
    import contextlib
    import io
    from oracle import ref_harness
    counts_tsv, clusters_tsv, samples, names, counts, adj = _golden(golden_dir, "cli_5x_pairwise")
    keep = _nonzero_margin_filter(names, counts, adj)
    flt = tmp_path / "filter.txt"
    flt.write_text("\n".join(sorted(keep)) + "\n")
    mod = ref_harness.load("pairwise_fisher")
    ref_out, ours = tmp_path / "ref.tsv", tmp_path / "ours.tsv"
    args = ref_harness._Args(inclusionSPLICEDICE=counts_tsv, clusters=clusters_tsv, chi2=True,
                             multiple_test_correction="none", filter_list=str(flt), output=str(ref_out))
    with contextlib.redirect_stdout(io.StringIO()):
        mod.run_with(args)
    _run(counts_tsv, clusters_tsv, ours, "none", ["-f", str(flt)])
    want = [l.rstrip("\n").split("\t") for l in open(ref_out)]
    got = [l.rstrip("\n").split("\t") for l in open(ours)]
    assert got[0] == want[0] and [r[0] for r in got] == [r[0] for r in want]
    np.testing.assert_allclose(np.array([[float(x) for x in r[1:]] for r in got[1:]]),
                               np.array([[float(x) for x in r[1:]] for r in want[1:]]), rtol=1e-9, atol=0)
    args.filter_list, args.output = None, str(tmp_path / "ref_unfiltered.tsv")
    with pytest.raises(ValueError), contextlib.redirect_stdout(io.StringIO()):
        mod.run_with(args)
