"""K1 (sd_cluster_build / sd_cluster_fill) at the edges of its documented input domain, bit-exact
against oracle_np.cluster_csr (int64, no key packing).

The cluster key packs chrom into bits 39..63, strand into 31..38 and the coordinate into 0..30, so
chrom_rank 2^25 - 1, strand_rank 255 and coordinates near 2^31 - 1 are where a probe built from
that key can carry into the next field or wrap.  Input outside the domain must be refused with
SD_ERR_INVALID rather than aliased onto another key.

Every set is compared in two steps: the build alone first (row order, components, row pointer,
nnz), and the adjacency fill only once those match, because the fill sizes its scratch from nnz and
writes every edge the build found.  Strand-255 segments on odd chromosome ranks are kept to at most
8 junctions: a rank computed with a carried strand probe is then off by at most 28 rows.
"""
import ctypes

import numpy as np
import pytest

from oracle import oracle_np

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOP = 2**31 - 1                       # largest start / end
CHROM_MAX = 2**25 - 1                 # largest chrom_rank
EDGE_CHROMS = [0, 1, 2, 3, 2**24, 2**25 - 2, CHROM_MAX]
EDGE_STRANDS = [0, 1, 127, 128, 254, 255]
SD_ERR_INVALID = 1


def _ops():
    from splicedice_b200 import ops
    ops.require_cuda()
    return ops


def _arrays(rows):
    a = np.asarray(rows, dtype=np.int64).reshape(-1, 4)
    return tuple(np.ascontiguousarray(a[:, k]).astype(np.int32) for k in range(4))


def _shuffled_unique(rows, rng):
    a = np.unique(np.asarray(rows, dtype=np.int64).reshape(-1, 4), axis=0)
    return _arrays(a[rng.permutation(len(a))])


def _brute_adjacency(arrays, got):
    """Every pair on the same (chrom, strand) whose closed intervals overlap, and nothing else."""
    c, s, st, en = (np.asarray(x, dtype=np.int64) for x in arrays)
    adj = ((c[:, None] == c[None, :]) & (s[:, None] == s[None, :]) & (st[:, None] <= en[None, :])
           & (st[None, :] <= en[:, None]))
    np.fill_diagonal(adj, False)
    out_row = got["out_row"].cpu().numpy()
    rp, ci = got["row_ptr"].cpu().numpy(), got["col_idx"].cpu().numpy()
    for i in range(len(c)):
        r = out_row[i]
        lst = ci[rp[r]:rp[r + 1]]
        assert len(lst) == len(set(lst.tolist())), f"junction {i}: repeated neighbour"
        assert sorted(lst.tolist()) == sorted(out_row[np.nonzero(adj[i])[0]].tolist()), f"junction {i}"


def _compare(arrays):
    ops = _ops()
    want = oracle_np.cluster_csr(*arrays)
    got = ops.cluster_build(*arrays, with_adjacency=False)
    for k in ("cluster_order", "out_row", "row_of_pos", "comp_id", "row_ptr"):
        np.testing.assert_array_equal(got[k].cpu().numpy(), want[k], err_msg=k)
    assert got["nnz"] == int(want["row_ptr"][-1])
    assert got["n_comp"] == want["n_comp"]
    got = ops.cluster_build(*arrays)
    for k in ("cluster_order", "out_row", "row_of_pos", "comp_id", "row_ptr", "col_idx"):
        np.testing.assert_array_equal(got[k].cpu().numpy(), want[k], err_msg=k)
    assert got["nnz"] == int(want["row_ptr"][-1]) and got["n_comp"] == want["n_comp"]
    if len(arrays[0]) <= 2000:
        _brute_adjacency(arrays, got)
    return got, want


def _segment(rng, chrom, strand, base, k):
    """k junctions around `base`: touching, nested and shared-start intervals, plus (base + 10,
    base + 20), which every strand of the chromosome holds (a tie that only the strand rank breaks)."""
    rows = {(chrom, strand, base + 10, base + 20)}
    while len(rows) < k:
        a = base + int(rng.integers(0, 30))
        rows.add((chrom, strand, a, a + int(rng.integers(0, 12))))
    return sorted(rows)


def _segments(rng, chroms, base):
    rows = []
    for c in chroms:
        for s in EDGE_STRANDS:
            rows += _segment(rng, c, s, base, int(rng.integers(1, 9)))
    return rows


@pytest.mark.parametrize("chrom", EDGE_CHROMS)
@pytest.mark.parametrize("base", [0, TOP - 40])
def test_rank_edges_one_chromosome(chrom, base):
    """Six strand segments (ranks 0, 1, 127, 128, 254, 255) on one chromosome rank."""
    rng = np.random.default_rng(chrom % 1000 + base % 7)
    _compare(_shuffled_unique(_segments(rng, [chrom], base), rng))


@pytest.mark.parametrize("seed", range(3))
def test_rank_edges_all_chromosomes(seed):
    """Every edge chromosome rank with every edge strand rank in one set, so that the chromosome
    bounds are searched across neighbours (2^25 - 2 next to 2^25 - 1 included)."""
    rng = np.random.default_rng(10 + seed)
    _compare(_shuffled_unique(_segments(rng, EDGE_CHROMS, [0, 2**30, TOP - 40][seed]), rng))


@pytest.mark.parametrize("chrom,strands", [(1, (0, 1)), (2, (0, 255)), (3, (0, 255)), (CHROM_MAX, (0, 1)),
                                           (CHROM_MAX, (0, 255))])
def test_four_junctions_on_two_strands(chrom, strands):
    """(10, 20), (10, 40), (30, 50), (5, 60) on alternating strands: a probe for the end of a
    strand-255 segment that carries into an odd chromosome rank, or a probe for the next chromosome
    that wraps past 2^25 - 1, gives out_row [1, 2, 3, -1] or [0, 2, 1, 0] instead of [1, 2, 3, 0]."""
    rows = [(chrom, strands[k % 2], a, b) for k, (a, b) in enumerate([(10, 20), (10, 40), (30, 50), (5, 60)])]
    got, _ = _compare(_arrays(rows))
    assert got["out_row"].cpu().numpy().tolist() == [1, 2, 3, 0]


COORDS = [0, 1, 2**30, TOP - 1, TOP]


def _coordinate_segment(chrom, strand):
    # every (start <= end) pair of edge coordinates: [0, 2^31 - 1] spanning the chromosome, intervals
    # touching at 2^30 and 2^31 - 2, several junctions sharing the start 2^31 - 2, zero-length ones
    rows = [(chrom, strand, a, b) for a in COORDS for b in COORDS if a <= b]
    rows += [(chrom, strand, TOP - 2, TOP - 1), (chrom, strand, TOP - 3, TOP - 2), (chrom, strand, 1, 2**30)]
    if chrom % 2 and strand == 255:
        keep = [(0, TOP), (2**30, TOP - 1), (TOP - 1, TOP - 1), (TOP - 1, TOP), (TOP, TOP), (TOP - 2, TOP - 1),
                (TOP - 3, TOP - 2), (1, 2**30)]
        rows = [r for r in rows if (r[2], r[3]) in keep]
    return rows


@pytest.mark.parametrize("chroms", [[0], [2**25 - 2], [CHROM_MAX], [1, 2, 3, 2**24, 2**25 - 2, CHROM_MAX]])
def test_coordinate_edges(chroms):
    """start / end in {0, 1, 2^30, 2^31 - 2, 2^31 - 1} on strands 0, 1, 254 and 255."""
    rows = [r for c in chroms for s in (0, 1, 254, 255) for r in _coordinate_segment(c, s)]
    _compare(_shuffled_unique(rows, np.random.default_rng(len(rows))))


@pytest.mark.parametrize("run", [2, 64, 65, 300])
def test_runs_sharing_a_start_at_the_key_limits(run):
    """A run of junctions sharing (chrom, strand, start) is sorted in place up to 64 long; a longer
    one repeats the build with the two-pass sort.  Runs at the top of the coordinate range on
    (2^25 - 2, strand 255) and (2^25 - 1, strand 254), with clutter and a short strand-255 segment
    on the last chromosome."""
    rng = np.random.default_rng(run)
    start = TOP - 1 - 3 * run
    rows = []
    for chrom, strand in [(2**25 - 2, 255), (CHROM_MAX, 254)]:
        ends = rng.choice(np.arange(start, TOP + 1), size=run, replace=False)
        rows += [(chrom, strand, start, int(e)) for e in ends]
        for _ in range(40):
            a = int(rng.integers(start - 400, TOP))
            rows.append((chrom, strand, a, min(TOP, a + int(rng.integers(0, 400)))))
    rows += [(CHROM_MAX, 255, start - k, start + k) for k in range(8)]          # nested, up to 2^31 - 1
    _compare(_shuffled_unique(rows, rng))


def test_many_contigs():
    """About 50,000 scaffolds whose string order differs from their numeric order, 1-4 junctions
    each on both strands, ranked by name as quant ranks them."""
    rng = np.random.default_rng(5)
    js = set()
    for k in range(50_000):
        name = f"scaffold_{k}"
        for _ in range(int(rng.integers(1, 5))):
            a = int(rng.integers(0, 2_000))
            js.add((name, a, a + int(rng.integers(1, 300)), "+-"[int(rng.integers(0, 2))]))
    js = sorted(js)
    rng.shuffle(js)
    c, s, st, en, names, _ = oracle_np.junctions_to_arrays(js)
    assert len(names) == 50_000 and names[:3] == ["scaffold_0", "scaffold_1", "scaffold_10"]
    _compare((c, s, st, en))


@pytest.mark.parametrize("seed", range(3))
def test_random_sets_at_the_limits(seed):
    """About 200,000 junctions: sparse chromosome ranks up to 2^25 - 2 with the edge ranks among
    them, strand ranks 0, 1, 127, 128, 254, coordinates anywhere in [0, 2^31 - 1] with clusters at
    0, 2^30 and the top, and runs sharing a start (longer than 64 in odd seeds)."""
    rng = np.random.default_rng(1000 + seed)
    n = 200_000
    chroms = np.unique(np.concatenate([[0, 1, 2, 3, 2**24, 2**25 - 2], rng.integers(0, 2**25 - 1, 300)]))
    strands = np.array([0, 1, 127, 128, 254])
    c = chroms[rng.integers(0, len(chroms), n)]
    s = strands[rng.integers(0, len(strands), n)]
    where = rng.integers(0, 4, n)
    st = np.where(where == 0, rng.integers(0, TOP, n),
                  np.where(where == 1, rng.integers(0, 20_000, n),
                           np.where(where == 2, rng.integers(2**30 - 10_000, 2**30 + 10_000, n),
                                    rng.integers(TOP - 20_000, TOP + 1, n))))
    length = np.where(rng.random(n) < 0.9, rng.integers(0, 3_000, n), rng.integers(0, 2**31, n))
    en = np.minimum(st + length, TOP)
    rows = [np.stack([c, s, st, en], axis=1)]
    max_run = 100 if seed % 2 else 64
    for _ in range(30):
        r = int(rng.integers(2, max_run + 1))
        a = int(rng.integers(0, TOP - 2 * max_run)) if rng.random() < 0.5 else TOP - 2 * max_run
        cc, ss = int(chroms[rng.integers(0, len(chroms))]), int(strands[rng.integers(0, len(strands))])
        ends = a + rng.choice(np.arange(2 * max_run), size=r, replace=False)
        rows.append(np.stack([np.full(r, cc), np.full(r, ss), np.full(r, a), ends], axis=1))
    arrays = _shuffled_unique(np.concatenate(rows), rng)
    longest = np.unique(np.stack(arrays[:3], axis=1), axis=0, return_counts=True)[1].max()
    assert (longest > 64) == bool(seed % 2)
    _compare(arrays)


# ---- refusals --------------------------------------------------------------------------------
GUARD = 64                             # int32 / 256 bytes of canary on each side of every buffer
CANARY = 0x5A5A5A5A


class _Guarded:
    """A device buffer of `count` int32 between two canary bands."""

    def __init__(self, count):
        self.buf = torch.full((count + 2 * GUARD,), CANARY, dtype=torch.int32, device="cuda")
        self.view = self.buf[GUARD:GUARD + count]

    def guards_intact(self):
        b = self.buf.cpu().numpy()
        return bool((b[:GUARD] == CANARY).all() and (b[-GUARD:] == CANARY).all())


def _native_build(arrays, ws, ws_bytes):
    """sd_cluster_build through the C ABI on caller-chosen buffers: every output between canaries."""
    from splicedice_b200 import native
    n = len(arrays[0])
    ins = [torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).cuda() for x in arrays]
    outs = {k: _Guarded(n) for k in ("cluster_order", "out_row", "row_of_pos", "comp_id")}
    outs["row_ptr"] = _Guarded(n + 1)
    nnz, ncomp = ctypes.c_int64(-7), ctypes.c_int64(-7)
    rc = native.load().sd_cluster_build(n, *(native.ptr(x) for x in ins),
                                        *(native.ptr(outs[k].view) for k in ("cluster_order", "out_row", "row_of_pos",
                                                                             "comp_id", "row_ptr")),
                                        ctypes.byref(nnz), ctypes.byref(ncomp), native.ptr(ws.view), ws_bytes,
                                        native.stream_ptr())
    torch.cuda.synchronize()
    return rc, outs, nnz.value, ncomp.value


VALID = [(1, 0, 10, 20), (1, 1, 10, 40), (1, 0, 30, 50), (1, 1, 5, 60), (2, 0, 10, 20), (CHROM_MAX, 0, 7, 9)]
BAD = [("chrom", 0, -1), ("chrom", 0, 2**25), ("chrom", 0, -(2**31)), ("strand", 1, -1), ("strand", 1, 256),
       ("start", 2, -1), ("end", 3, -1), ("start", 2, -(2**31))]


def _run_of_66():
    return [(0, 0, 100, 101 + k) for k in range(66)]


@pytest.mark.parametrize("with_long_run", [False, True])
@pytest.mark.parametrize("field,column,value", BAD)
def test_out_of_range_input_is_refused(field, column, value, with_long_run):
    """One junction with one field outside the domain: SD_ERR_INVALID, nothing written outside the
    caller's arrays and the workspace, the result pointers untouched.  With a run longer than 64
    in the same set, the refusal is not lost to the repeated build.  A valid call on the same
    workspace afterwards matches the oracle."""
    from splicedice_b200 import native
    _ops()
    rows = [list(r) for r in VALID] + ([list(r) for r in _run_of_66()] if with_long_run else [])
    rows[len(VALID) // 2][column] = value
    arrays = _arrays(rows)
    n = len(rows)
    ws_bytes = native.load().sd_cluster_workspace_bytes(n)
    ws = _Guarded((ws_bytes + 3) // 4)
    rc, outs, nnz, ncomp = _native_build(arrays, ws, ws_bytes)
    assert rc == SD_ERR_INVALID, f"{field} = {value} was not refused (rc {rc})"
    assert native.last_error().startswith("sd_cluster_build:")
    assert (nnz, ncomp) == (-7, -7)
    assert ws.guards_intact() and all(o.guards_intact() for o in outs.values())

    # the same workspace, now with valid input (the bad junction removed): build and fill
    good = _arrays([r for k, r in enumerate(rows) if k != len(VALID) // 2])
    m = len(good[0])
    rc, outs, nnz, ncomp = _native_build(good, ws, ws_bytes)
    assert rc == 0, native.last_error()
    want = oracle_np.cluster_csr(*good)
    for k in ("cluster_order", "out_row", "row_of_pos", "comp_id", "row_ptr"):
        np.testing.assert_array_equal(outs[k].view.cpu().numpy(), want[k], err_msg=k)
    assert nnz == int(want["row_ptr"][-1]) and ncomp == want["n_comp"]
    col = _Guarded(max(nnz, 1))
    fw_bytes = native.load().sd_cluster_fill_workspace_bytes(m, nnz)
    fw = torch.empty(fw_bytes, dtype=torch.uint8, device="cuda")
    native.call("sd_cluster_fill", m, nnz, native.ptr(outs["row_of_pos"].view), native.ptr(outs["row_ptr"].view),
                native.ptr(col.view), native.ptr(ws.view), ws_bytes, native.ptr(fw), fw_bytes, native.stream_ptr())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(col.view[:nnz].cpu().numpy(), want["col_idx"])
    assert ws.guards_intact() and col.guards_intact() and all(o.guards_intact() for o in outs.values())


def test_refusal_through_ops():
    """ops.cluster_build raises NativeCallError with code SD_ERR_INVALID (it has no check of its own)."""
    from splicedice_b200 import native
    ops = _ops()
    c, s, st, en = _arrays(VALID)
    s[0] = 256
    with pytest.raises(native.NativeCallError) as e:
        ops.cluster_build(c, s, st, en, with_adjacency=False)
    assert e.value.code == SD_ERR_INVALID
    s[0] = 0
    _compare((c, s, st, en))
