"""K3 parity on the GPU: two-sided Fisher p-values vs scipy goldens and the binary128 oracle."""
import numpy as np
import pytest

from oracle import fisher_c, oracle_np
from tests import util

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RTOL = 1e-9          # BASELINE.json north_star: 1e-9 relative for p > 1e-300


def _ops():
    from splicedice_b200 import native, ops
    ops.require_cuda()
    return native, ops


def _check(got, want, rtol=RTOL):
    ok = want > 1e-300
    rel = np.abs(got[ok] - want[ok]) / want[ok]
    assert rel.max(initial=0.0) <= rtol, f"max rel err {rel.max()}"
    assert np.all(got[~ok] <= 1e-299)


def test_scipy_golden_tables():
    _, ops = _ops()
    g = util.load_npz("fisher_tables.npz")
    t, p = g["tables"], g["p"]
    got = ops.fisher_tables(t[:, 0], t[:, 1], t[:, 2], t[:, 3]).cpu().numpy()
    _check(got, p)
    assert np.array_equal(got[p == 1.0], p[p == 1.0])      # ties / zero margins are exactly 1


def test_exact_rational_small_tables():
    _, ops = _ops()
    g = util.load_npz("fisher_exact_small.npz")
    t, p = g["tables"], g["p"]
    got = ops.fisher_tables(t[:, 0], t[:, 1], t[:, 2], t[:, 3]).cpu().numpy()
    np.testing.assert_allclose(got, p, rtol=1e-12, atol=0)


@pytest.mark.parametrize("scale,n", [(4, 100000), (40, 200000), (400, 200000), (5000, 50000), (200000, 3000)])
def test_random_tables_vs_binary128_oracle(scale, n):
    _, ops = _ops()
    rng = np.random.default_rng(scale)
    t = rng.integers(0, scale, size=(n, 4))
    t[::3, 1] *= rng.integers(1, 20)
    t[::5, 2] //= 3
    got = ops.fisher_tables(t[:, 0], t[:, 1], t[:, 2], t[:, 3]).cpu().numpy()
    want = fisher_c.fisher_two_sided(t[:, 0], t[:, 1], t[:, 2], t[:, 3])
    _check(got, want, rtol=1e-11)


def test_pairwise_layout_and_exclusions():
    """inc/exc matrices -> [J, P] with the reference's pair order (pairwise_fisher.py:142-145)."""
    _, ops = _ops()
    J, S = 3000, 12
    _, csr, counts = util.synthetic_problem(J, S, seed=11, zero_frac=0.1)
    exc = oracle_np.exclusion_sums(counts, csr["row_ptr"], csr["col_idx"])
    pa, pb = oracle_np.all_pairs(S)
    dev = torch.device("cuda", 0)
    got = ops.fisher_pairwise(torch.from_numpy(counts).to(dev), torch.from_numpy(exc).to(dev), pa, pb).cpu().numpy()
    want = fisher_c.pairwise(counts, exc, pa, pb)
    assert got.shape == (J, S * (S - 1) // 2)
    _check(got.ravel(), want.ravel(), rtol=1e-11)
    # rows with an empty adjacency list have a zero margin: p = 1 everywhere
    empty = np.diff(csr["row_ptr"]) == 0
    assert empty.any() and np.all(got[empty] == 1.0)
    # host-buffer entry point, ragged row range
    got_h = ops.fisher_pairwise_host(counts, exc, pa, pb).numpy()
    np.testing.assert_array_equal(got_h, got)
    # the whole hot loop for host buffers: exclusion counts summed on the device from the CSR
    got_w = ops.pairwise_host(counts, csr["row_ptr"], csr["col_idx"], pa, pb).numpy()
    np.testing.assert_array_equal(got_w, got)
    wide = np.zeros((J, S + 5), dtype=np.int32)                   # strided host input, odd sample count
    wide[:, :S] = counts
    sub = torch.from_numpy(wide)[:, :S - 1]
    pa2, pb2 = oracle_np.all_pairs(S - 1)
    exc2 = oracle_np.exclusion_sums(counts[:, :S - 1], csr["row_ptr"], csr["col_idx"])
    got_s = ops.pairwise_host(sub, csr["row_ptr"], csr["col_idx"], pa2, pb2).numpy()
    _check(got_s.ravel(), fisher_c.pairwise(counts[:, :S - 1], exc2, pa2, pb2).ravel(), rtol=1e-11)


def test_negative_entries_are_rejected():
    native, ops = _ops()
    with pytest.raises(native.NativeCallError):
        ops.fisher_tables([1, 2], [3, -1], [4, 4], [5, 5])


def test_survey_vector_pairwise_file(golden_dir):
    """SURVEY.md section 4 known-answer vector, values taken from the reference's own output file."""
    import os
    _, ops = _ops()
    path = os.path.join(golden_dir, "survey_vector", "expected", "pairwise_none.tsv")
    rows = [l.rstrip("\n").split("\t") for l in open(path)]
    want = np.array([[float(x) for x in r[1:]] for r in rows[1:]])
    cpath = os.path.join(golden_dir, "survey_vector", "expected", "ref_inclusionCounts.tsv")
    crow = [l.rstrip("\n").split("\t") for l in open(cpath)][1:]
    names = [r[0] for r in crow]
    counts = np.array([[int(x) for x in r[1:]] for r in crow], dtype=np.int32)
    adj = {}
    for l in open(os.path.join(golden_dir, "survey_vector", "expected", "ref_allClusters.tsv")):
        f = l.rstrip("\n").split("\t")
        adj[f[0]] = [x for x in f[1].split(",") if x] if len(f) > 1 else []
    idx = {n: i for i, n in enumerate(names)}
    exc = np.array([counts[[idx[o] for o in adj[n]]].sum(axis=0) if adj[n] else np.zeros(3, int) for n in names],
                   dtype=np.int64)
    pa, pb = oracle_np.all_pairs(3)
    dev = torch.device("cuda", 0)
    got = ops.fisher_pairwise(torch.from_numpy(counts).to(dev), torch.from_numpy(exc).to(dev), pa, pb).cpu().numpy()
    by_name = {r[0]: i for i, r in enumerate(rows[1:])}
    order = [by_name[n] for n in names]
    np.testing.assert_allclose(got, want[order], rtol=RTOL, atol=0)


def test_bounded_entry_point_matches_and_guards():
    """sd_fisher_pairwise_bounded: same p-values without the device-side reduction; a cell outside
    the promised bound yields NaN for the tables that use it, never a wrong number."""
    _, ops = _ops()
    J, S = 1500, 10
    _, csr, counts = util.synthetic_problem(J, S, seed=21, zero_frac=0.1)
    exc = oracle_np.exclusion_sums(counts, csr["row_ptr"], csr["col_idx"])
    pa, pb = oracle_np.all_pairs(S)
    dev = torch.device("cuda", 0)
    inc_d, exc_d = torch.from_numpy(counts).to(dev), torch.from_numpy(exc).to(dev)
    ref = ops.fisher_pairwise(inc_d, exc_d, pa, pb).cpu().numpy()
    bound = int((counts + exc).max())
    got = ops.fisher_pairwise(inc_d, exc_d, pa, pb, max_cell_bound=bound).cpu().numpy()
    np.testing.assert_array_equal(got, ref)
    loose = ops.fisher_pairwise(inc_d, exc_d, pa, pb, max_cell_bound=bound * 50).cpu().numpy()   # other instantiation
    _check(loose.ravel(), ref.ravel(), rtol=1e-12)
    tight = ops.fisher_pairwise(inc_d, exc_d, pa, pb, max_cell_bound=bound // 2).cpu().numpy()
    over = (counts + exc) > bound // 2
    bad = over[:, pa] | over[:, pb]
    assert bad.any() and np.isnan(tight[bad]).all()
    np.testing.assert_array_equal(tight[~bad], ref[~bad])


def test_kernel_instantiations_agree():
    """Every instantiation of the pairwise kernel on the same tables: staged table (mode 0), table
    partly / wholly in global memory (modes 1, 2 with the Stirling fallback, chosen through the
    promised bound), 64-bit totals (the pair-order kernel, bound 2^31) -- and more than 512
    samples, where the junction row is not staged in shared memory."""
    import os
    _, ops = _ops()
    J, S = 700, 10
    _, csr, counts = util.synthetic_problem(J, S, seed=33, zero_frac=0.1)
    exc = oracle_np.exclusion_sums(counts, csr["row_ptr"], csr["col_idx"])
    pa, pb = oracle_np.all_pairs(S)
    dev = torch.device("cuda", 0)
    inc_d, exc_d = torch.from_numpy(counts).to(dev), torch.from_numpy(exc).to(dev)
    want = fisher_c.pairwise(counts, exc, pa, pb)
    for bound in (int((counts + exc).max()), 20_000, 3_000_000, 2 ** 31):
        got = ops.fisher_pairwise(inc_d, exc_d, pa, pb, max_cell_bound=bound).cpu().numpy()
        _check(got.ravel(), want.ravel(), rtol=1e-11)
    # per-sample log-factorial terms staged once per junction (the default whenever they fit next
    # to the table) against the same arithmetic evaluated per pair: identical bits; a table that
    # fills shared memory (bound 5,000 -> 10,001 entries) leaves no room for 400 samples' terms
    staged = ops.fisher_pairwise(inc_d, exc_d, pa, pb).cpu().numpy()
    os.environ["SD_FISHER_NO_PRE"] = "1"
    try:
        per_pair = ops.fisher_pairwise(inc_d, exc_d, pa, pb).cpu().numpy()
    finally:
        del os.environ["SD_FISHER_NO_PRE"]
    np.testing.assert_array_equal(staged.view(np.uint64), per_pair.view(np.uint64))
    J3, S3 = 30, 400
    _, csr3, counts3 = util.synthetic_problem(J3, S3, seed=35, zero_frac=0.05)
    exc3 = oracle_np.exclusion_sums(counts3, csr3["row_ptr"], csr3["col_idx"])
    qa3, qb3 = oracle_np.all_pairs(S3)
    qa3, qb3 = qa3[::37], qb3[::37]
    want3 = fisher_c.pairwise(counts3, exc3, qa3, qb3)
    for bound in (int((counts3 + exc3).max()), 5_000):
        got3 = ops.fisher_pairwise(torch.from_numpy(counts3).to(dev), torch.from_numpy(exc3).to(dev), qa3, qb3,
                                   max_cell_bound=bound).cpu().numpy()
        _check(got3.ravel(), want3.ravel(), rtol=1e-11)

    # 600 samples (> 512: unstaged row), an arbitrary pair list with repeats and a == b
    J2, S2 = 40, 600
    _, csr2, counts2 = util.synthetic_problem(J2, S2, seed=34, zero_frac=0.05)
    exc2 = oracle_np.exclusion_sums(counts2, csr2["row_ptr"], csr2["col_idx"])
    rng = np.random.default_rng(0)
    qa = rng.integers(0, S2, size=3001).astype(np.int32)
    qb = rng.integers(0, S2, size=3001).astype(np.int32)
    got2 = ops.fisher_pairwise(torch.from_numpy(counts2).to(dev), torch.from_numpy(exc2).to(dev), qa, qb).cpu().numpy()
    want2 = fisher_c.pairwise(counts2, exc2, qa, qb)
    _check(got2.ravel(), want2.ravel(), rtol=1e-11)


def test_totals_straddling_the_table_cap():
    """Table totals either side of 2^22 (the log-factorial table's cap): beyond it the kernel uses
    the double-double Stirling series (fisher::lgfact_stirling), which keeps the 1e-9 contract where
    a binary64 lgamma() (7e-9 of rounding at log 4e6!) would not.  Element-wise kernel and the
    pairwise kernels (cells of 1-3 million), against the binary128 oracle."""
    _, ops = _ops()
    rng = np.random.default_rng(12)
    rows = []
    for total in (3_900_000, 4_194_303, 4_194_304, 4_194_305, 4_500_000, 6_000_000, 8_000_000):
        for skew in (0.0, 0.001, 0.004):
            n1 = int(total * rng.uniform(0.3, 0.7)); n = int(total * rng.uniform(0.3, 0.7))
            a = int(n1 * n / total * (1.0 + skew))
            rows.append([a, n1 - a, n - a, total - n1 - n + a])
    t = np.array(rows)
    want = fisher_c.fisher_two_sided(t[:, 0], t[:, 1], t[:, 2], t[:, 3])
    got = ops.fisher_tables(t[:, 0], t[:, 1], t[:, 2], t[:, 3]).cpu().numpy()
    _check(got, want)
    # pairwise form: 4 samples whose (inc, exc) columns are the table columns above
    dev = torch.device("cuda", 0)
    inc = np.stack([t[:, 0], t[:, 1], t[:, 1], t[:, 0]], axis=1).astype(np.int32)
    exc = np.stack([t[:, 2], t[:, 3], t[:, 3] // 2, t[:, 2] + 7], axis=1).astype(np.int64)
    pa, pb = oracle_np.all_pairs(4)
    wantp = fisher_c.pairwise(inc, exc, pa, pb)
    gotp = ops.fisher_pairwise(torch.from_numpy(inc).to(dev), torch.from_numpy(exc).to(dev), pa, pb).cpu().numpy()
    _check(gotp.ravel(), wantp.ravel())
    np.testing.assert_array_equal(gotp[:, 0], got)


def test_tie_rule_is_the_modern_scipy_one():
    """See tests/test_fisher_twin.py: tables where scipy 1.4.1's 1e-4 tie window would return exactly 1
    and scipy >= 1.9 does not; the kernel follows the latter."""
    from scipy.stats import fisher_exact
    from tests.test_fisher_twin import TIE_RULE_TABLES
    _, ops = _ops()
    t = np.array(TIE_RULE_TABLES)
    want = np.array([fisher_exact([[a, b], [c, d]])[1] for a, b, c, d in t.tolist()])
    got = ops.fisher_tables(t[:, 0], t[:, 1], t[:, 2], t[:, 3]).cpu().numpy()
    assert (got < 0.999).all()
    _check(got, want)
