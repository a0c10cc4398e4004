"""Host-side logic that needs no GPU: name <-> tuple, CSR construction from the cluster files
with the reference's two lookup semantics, Benjamini-Hochberg, file parsers on the goldens."""
import os

import numpy as np
import pytest

from oracle import oracle_np
from splicedice_b200 import counts_to_ps, ir_table, junctions as jn, ops, pairwise_fisher


def test_names_round_trip():
    j = ("chr10", 50, 250, "-")
    assert jn.junction_name(j) == "chr10:50-250:-" and jn.parse_name("chr10:50-250:-") == j
    with pytest.raises(ValueError):
        jn.parse_name("chr1:100:+")


def test_string_ranks_follow_python_order():
    ranks, names = jn.dense_ranks(["chr2", "chr10", "chr1", "chr10"])
    assert names == ["chr1", "chr10", "chr2"] and ranks.tolist() == [2, 1, 0, 1]
    t = jn.JunctionTable([("chr2", 5, 9, "-"), ("chr10", 1, 4, "+")])
    assert t.chrom_rank.tolist() == [1, 0] and t.strand_rank.tolist() == [1, 0]      # '+' < '-'
    with pytest.raises(ValueError):
        jn.JunctionTable([("chr1", -1, 5, "+")])


def test_csr_sum_semantics():
    names = ["a", "b", "c"]
    clusters = {"a": ["b", "b", ""], "b": [""], "c": ["a"]}
    rp, ci = jn.csr_from_named_lists(names, clusters, "sum")
    assert rp.tolist() == [0, 2, 2, 3] and ci.tolist() == [1, 1, 0]        # duplicates count twice
    with pytest.raises(KeyError):
        jn.csr_from_named_lists(names, {"a": ["zz"], "b": [], "c": []}, "sum")


def test_csr_isin_semantics():
    names = ["a", "b", "a", "c"]                                             # a repeated row name
    clusters = {"a": ["b", "b", "missing"], "b": ["a"], "c": []}
    rp, ci = jn.csr_from_named_lists(names, clusters, "isin")
    assert rp.tolist() == [0, 1, 3, 4, 4] and ci.tolist() == [1, 0, 2, 1]    # sets; both 'a' rows selected
    with pytest.raises(KeyError):
        jn.csr_from_named_lists(["a", "d"], clusters, "isin")


def test_bh_oracle_known_values():
    """The BH restatement on textbook values (the device version is checked against it in
    tests/test_gpu_bh.py)."""
    np.testing.assert_allclose(oracle_np.bh_adjust([0.01, 0.04, 0.03, 0.005]), [0.02, 0.04, 0.04, 0.02])
    np.testing.assert_allclose(oracle_np.bh_adjust([0.5, 0.9, 1.0]), [1.0, 1.0, 1.0])
    assert oracle_np.bh_adjust([]).size == 0
    assert pairwise_fisher.fdr_bh([]).size == 0                              # empty input never reaches the device


def test_pair_order():
    assert pairwise_fisher.sample_pairs(4) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    for n in (0, 1, 2, 5, 13):              # the column header and the device pair arrays agree
        assert pairwise_fisher.sample_pairs(n) == list(zip(*ops.all_pairs(n)))


def test_parsers_on_reference_files(golden_dir):
    exp = os.path.join(golden_dir, "survey_vector", "expected")
    cl = counts_to_ps.get_clusters(os.path.join(exp, "ref_allClusters.tsv"))
    assert cl["chr1:100-300:-"] == [""] and cl["chr2:50-250:+"] == ["chr2:60-200:+"]
    header, counts = counts_to_ps.get_counts(os.path.join(exp, "ref_inclusionCounts.tsv"))
    assert header == "cluster\ts0\ts1\ts2\n" and counts["chr1:100-300:+"].tolist() == [34.0, 32.0, 22.0]
    pc = pairwise_fisher.getClusters(os.path.join(exp, "ref_allClusters.tsv"))
    assert pc["chr1:100-300:-"] == [] and pc["chr1:301-600:+"] == ["chr1:300-500:+", "chr1:100-400:+"]
    samples, events, mat = pairwise_fisher.getEventCounts(os.path.join(exp, "ref_inclusionCounts.tsv"))
    assert samples == ["s0", "s1", "s2"] and len(events) == 9 and mat.shape == (9, 3)
    _, ev2, m2 = pairwise_fisher.getEventCounts(os.path.join(exp, "ref_inclusionCounts.tsv"), {"chr2:60-200:+"})
    assert ev2 == ["chr2:60-200:+"] and m2.tolist() == [[7.0, 21.0, 22.0]]
    ic = ir_table.getClusters(os.path.join(exp, "ref_allClusters.tsv"))
    assert ic["chr1:700-900:+"] == []


def test_gtf_introns(tmp_path):
    gtf = tmp_path / "a.gtf"
    gtf.write_text(
        "#comment\n"
        'chr1\tx\ttranscript\t100\t900\t.\t+\t.\tgene_id "g1"; transcript_id "t1"; gene_name "G";\n'
        'chr1\tx\texon\t100\t200\t.\t+\t.\tgene_id "g1"; transcript_id "t1";\n'
        'chr1\tx\texon\t400\t500\t.\t+\t.\tgene_id "g1"; transcript_id "t1";\n'
        'chr1\tx\texon\t800\t900\t.\t+\t.\tgene_id "g1"; transcript_id "t1";\n')
    assert ir_table.getAnnotated(str(gtf)) == {"chr1:200-399:+", "chr1:500-799:+"}


def test_sample_type_sniffing(tmp_path):
    from splicedice_b200 import quant
    plain = tmp_path / "a.junc.bed"
    plain.write_text("chr1\t1\t100\tj0\t7\t+\n")
    tagged = tmp_path / "b.bed"
    tagged.write_text("chr1\t1\t100\te:1.20:1.30;o:9;m:GT_AG;a:?\t7\t+\n")
    assert quant.Sample(["a", str(plain), "m", "c"]).type == "bed"
    assert quant.Sample(["b", str(tagged), "m", "c"]).type == "splicedicebed"
    assert quant.Sample(["c", "x.SJ.out.tab", "m", "c"]).type == "SJ"
    assert quant.Sample(["d", "x.bam", "m", "c"]).type == "bam"
    assert quant.Sample(["e", "x.leafcutter.junc", "m", "c"]).type == "leafcutter"
    assert quant.Sample(["f", "x.junc", "m", "c"]).type == "unknown"


def test_junction_filters(tmp_path):
    """SJ.out.tab uses strict length bounds, BED inclusive ones; tagged BED filters only unannotated."""
    import argparse
    from splicedice_b200 import quant
    sj = tmp_path / "s.SJ.out.tab"
    sj.write_text("chr1\t101\t150\t1\t1\t0\t9\t0\t20\n"        # length 50: not > minLength -> out
                  "chr1\t101\t151\t1\t1\t0\t3\t2\t20\n"        # length 51, score 3+2 -> in
                  "chr1\t101\t400\t0\t1\t0\t9\t0\t20\n"        # undefined strand -> out
                  "chr1\t101\t500\t2\t3\t0\t9\t0\t20\n")       # motif 3 not in gtag_only -> out
    bed = tmp_path / "p.bed"
    bed.write_text("chr2\t100\t150\tj\t5\t+\n"                 # length 50 inclusive -> in
                   "chr2\t100\t149\tj\t9\t+\n"                 # too short
                   "chr2\t100\t900\tj\t4\t-\n"                 # score < minUnique
                   "chr2\t100\t800\tj\t9\t.\n")                # no strand
    tag = tmp_path / "t.bed"
    tag.write_text("chr3\t100\t900\te:0.10:0.20;o:1;m:GT_AG;a:GENE\t1\t+\n"   # annotated: no filter at all
                   "chr3\t100\t800\te:0.10:2.00;o:9;m:GT_AG;a:?\t9\t+\n"      # low entropy
                   "chr3\t100\t700\te:1.10:2.00;o:9;m:GT_AG;a:?\t9\t-\n")     # passes
    man = tmp_path / "m.txt"
    man.write_text(f"a\t{sj}\tx\ty\nb\t{bed}\tx\ty\nc\t{tag}\tx\ty\n")
    p = argparse.ArgumentParser()
    quant.add_parser(p)
    args = p.parse_args(["-m", str(man), "-o", str(tmp_path / "o")])
    job = quant.SPLICEDICE(args.manifest, args.output_prefix, args, run=False)
    job.manifest = job.parseManifest()
    assert job.getAllJunctions() == {("chr1", 100, 151, "+"), ("chr2", 100, 150, "+"),
                                     ("chr3", 100, 900, "+"), ("chr3", 100, 700, "-")}


def test_native_row_formatter_is_byte_identical_to_python():
    """sd_host_format_rows against the reference's per-cell f-strings (SPLICEDICE.py:340,353;
    counts_to_ps.py:69): exact round-half-even on the binary value, 'nan' for any NaN."""
    from splicedice_b200 import textio
    rng = np.random.default_rng(0)
    x = rng.random((700, 130)).astype(np.float32)
    x[rng.random(x.shape) < 0.05] = np.nan
    x[0, :9] = [0.0625, 0.1875, 0.0005, 0.0015, 0.9995, 1.0, 0.0, -0.0, np.float32(-np.nan)]
    names = [f"chr{i % 22 + 1}:{i}-{i + 100}:{'+-'[i % 2]}" for i in range(700)]
    want = "".join(n + "\t" + "\t".join(f"{v:.3f}" for v in row) + "\n" for n, row in zip(names, x.tolist()))
    assert textio.format_rows(x, names) == want.encode()
    assert textio.format_rows(x, names, threads=1) == want.encode()
    y = np.concatenate([rng.random(60000), rng.integers(0, 10 ** 7, 60000) / 8000.0,
                        np.array([0.0005, 0.0015, 0.0025, 1e15, 1e17, -3.14159, np.inf, -np.inf, np.nan, 5e-324, 4.0e12]),
                        rng.standard_normal(30000) * 1e6])
    y = np.concatenate([y, np.zeros((-len(y)) % 40)]).reshape(-1, 40)
    want = "".join("\t".join(f"{v:0.3f}" for v in row) + "\n" for row in y.tolist())
    assert textio.format_rows(y) == want.encode()
    z = rng.integers(0, 2 ** 31 - 1, size=(300, 17)).astype(np.int32)
    z[0, :2] = [0, 2 ** 31 - 1]
    want = "".join("\t".join(f"{float(v):.0f}" for v in row) + "\n" for row in z.tolist())
    assert textio.format_rows(z) == want.encode()
    assert textio.format_rows(np.zeros((0, 5), dtype=np.float32), []) == b""


def test_pairwise_value_formatter_matches_str():
    from splicedice_b200 import textio
    rng = np.random.default_rng(1)
    y = np.concatenate([rng.random(50000), 10.0 ** rng.uniform(-320, 300, 50000),
                        np.array([1.0, 0.5, 1e-5, 1e-4, 1e16, 1e15, 9999999999999998.0, 1e22, 5e-324, 0.1, 1 / 3,
                                  np.inf, -np.inf, np.nan, 0.0, -0.0, -1.5e-10, 100.0, 12345.678])])
    y = np.concatenate([y, np.ones((-len(y)) % 30)]).reshape(-1, 30)
    want = "".join("\t".join(str(np.float64(v)) for v in row) + "\n" for row in y)
    assert textio.format_rows(y, repr_floats=True) == want.encode()


def test_write_matrix_streams_segments_byte_identically(tmp_path):
    """write_matrix (sd_host_format_rows_segments: per-thread slices written in order, no
    compaction) produces the same file as the one-shot formatter, for every chunking / thread
    count, including a buffer that starts too small and rows of very uneven text length."""
    import ctypes
    from splicedice_b200 import native, textio
    rng = np.random.default_rng(5)
    x = rng.random((3000, 37))
    x[:1500] *= 1e11                                  # first half ~15 bytes per cell, second half 5
    names = [f"chrX:{i}-{i * 3 + 7}:-" for i in range(3000)]
    want = b"h\tcols\n" + textio.format_rows(x, names)
    for chunk, threads in ((None, 0), (7, 3), (1000, 1), (2999, 8)):
        path = tmp_path / f"m_{chunk}_{threads}.tsv"
        textio.write_matrix(str(path), "h\tcols\n", names, x, chunk_rows=chunk, threads=threads)
        assert path.read_bytes() == want
    p = rng.random((500, 20)) * 10.0 ** rng.integers(-300, 0, (500, 20))
    path = tmp_path / "p.tsv"
    textio.write_matrix(str(path), "", None, p, repr_floats=True, chunk_rows=128)
    assert path.read_bytes() == textio.format_rows(p, repr_floats=True)
    textio.write_matrix(str(path), "only header\n", [], np.zeros((0, 4), dtype=np.float32))
    assert path.read_bytes() == b"only header\n"
    # too-small buffer: SD_ERR_WORKSPACE and a sufficient size, never an overrun
    lib = native.load()
    m, blob, off = textio._prepare(x, names, False)
    buf = np.full(4096 + 64, 0x55, dtype=np.uint8)
    so, sl = np.empty(8, dtype=np.int64), np.empty(8, dtype=np.int64)
    ns, need = ctypes.c_int32(), ctypes.c_size_t()
    rc = lib.sd_host_format_rows_segments(1, native.ptr(m), 3000, 37, 37, blob, native.ptr(off), native.ptr(buf), 4096,
                                          native.ptr(so), native.ptr(sl), 8, ctypes.byref(ns), ctypes.byref(need), 4)
    assert rc == native.SD_ERR_WORKSPACE and need.value >= len(want) - 7 and (buf[4096:] == 0x55).all()
    buf, segs = textio._format_segments(m, blob, off, 4, False, np.empty(4096, dtype=np.uint8))
    assert b"".join(bytes(buf[o:o + n]) for o, n in segs) == want[7:]


def _quant_job(manifest, out, extra=(), native_io=True):
    import argparse
    from splicedice_b200 import quant
    p = argparse.ArgumentParser()
    quant.add_parser(p)
    args = p.parse_args(["-m", str(manifest), "-o", str(out), *extra])
    job = quant.SPLICEDICE(args.manifest, args.output_prefix, args, run=False, native_io=native_io)
    job.manifest = job.parseManifest()
    return job


def test_native_ingest_equals_python_parsers(tmp_path, golden_dir):
    """sd_ingest_collect / sd_ingest_counts against the per-line python readers on every sample
    type, with duplicates, filters at their boundaries and low-coverage cells."""
    rng = np.random.default_rng(5)
    sj = tmp_path / "a.SJ.out.tab"
    lines = []
    for i in range(3000):
        start = int(rng.integers(1, 5000)); length = int(rng.integers(40, 70)) if i % 3 else int(rng.integers(49000, 50010))
        lines.append(f"chr{rng.integers(1, 4)}\t{start}\t{start + length - 1}\t{rng.integers(0, 3)}\t{rng.integers(0, 7)}\t0\t"
                     f"{rng.integers(0, 9)}\t{rng.integers(0, 4)}\t{rng.integers(1, 30)}\n")
    sj.write_text("".join(lines))
    bed = tmp_path / "b.junc.bed"
    lines = []
    for i in range(3000):
        left = int(rng.integers(0, 5000)); length = int(rng.integers(45, 60))
        lines.append(f"chr{rng.integers(1, 4)}\t{left}\t{left + length}\tj{i}\t{rng.integers(0, 12)}\t{'+-.'[int(rng.integers(0, 3))]}\n")
    lines += lines[:200]                                       # duplicates: last line wins
    bed.write_text("".join(lines))
    tag = tmp_path / "c.bed"
    lines = []
    for i in range(3000):
        left = int(rng.integers(0, 5000)); length = int(rng.integers(45, 60))
        ann = "?" if i % 2 else "GENE1"
        lines.append(f"chr{rng.integers(1, 4)}\t{left}\t{left + length}\te:{rng.random() * 2:.2f}:{rng.random() * 2:.2f};"
                     f"o:{rng.integers(0, 12)};m:GT_AG;a:{ann}\t{rng.integers(0, 12)}\t{'+-'[int(rng.integers(0, 2))]}\n")
    tag.write_text("".join(lines))
    leaf = tmp_path / "d.leafcutter.junc"
    leaf.write_text("".join(f"chrX\t{100 * i}\t{100 * i + 55 + i % 3}\t.\t{i % 9}\t+\n" for i in range(500)))
    ignored = tmp_path / "e.junc"
    ignored.write_text("not a junction file\n")
    man = tmp_path / "m.txt"
    man.write_text("".join(f"s{i}\t{p}\tmeta\tcond\n" for i, p in enumerate([sj, bed, tag, leaf, ignored])))
    for extra in ((), ("--lowCoverageNan", "--minUnique", "7"), ("--noMultimap", "--minLength", "48", "--maxLength", "56"),
                  ("--minEntropy", "0.5", "--minOverhang", "8")):
        fast = _quant_job(man, tmp_path / "o", extra, native_io=True)
        slow = _quant_job(man, tmp_path / "o", extra, native_io=False)
        fast.junctions = fast.getAllJunctions()
        slow.junctions = slow.getAllJunctions()
        assert fast.junctions == slow.junctions and len(fast.junctions) > 500
        rows = sorted(fast.junctions)
        for job in (fast, slow):
            job._rows = rows
            job.junctionIndex = {j: r for r, j in enumerate(rows)}
        c_fast, low_fast = fast.getJunctionCounts()
        c_slow, low_slow = slow.getJunctionCounts()
        np.testing.assert_array_equal(c_fast, c_slow)
        assert sorted(set(low_fast)) == sorted(set(low_slow))
        assert (c_fast[:, 4] == 0).all()                       # the unknown-suffix sample stays a zero column


def test_native_ingest_reports_malformed_lines(tmp_path):
    bad = tmp_path / "bad.junc.bed"
    bad.write_text("chr1\t10\t90\tj\t5\t+\nchr1\tten\t90\tj\t5\t+\n")
    man = tmp_path / "m.txt"
    man.write_text(f"s0\t{bad}\tm\tc\n")
    job = _quant_job(man, tmp_path / "o")
    with pytest.raises(ValueError) as e:
        job.getAllJunctions()
    assert "bad.junc.bed:2" in str(e.value)


def test_native_table_reader(tmp_path, golden_dir):
    from splicedice_b200 import textio
    exp = os.path.join(golden_dir, "cli_8x", "expected", "ref_inclusionCounts.tsv")
    header, names, values = textio.read_table(exp)
    lines = open(exp).read().split("\n")
    assert header == lines[0] + "\n" and names == [l.split("\t")[0] for l in lines[1:] if l]
    want = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines[1:] if l])
    np.testing.assert_array_equal(values, want)
    odd = tmp_path / "odd.tsv"
    odd.write_text("h\ta\tb\nx\t1.5\t2e3\ny\tnan\t-0.0\nz\t007\t1e-3")           # no trailing newline
    h, n, v = textio.read_table(str(odd))
    assert n == ["x", "y", "z"] and v[0].tolist() == [1.5, 2000.0] and np.isnan(v[1, 0]) and v[2].tolist() == [7.0, 0.001]
    ragged = tmp_path / "ragged.tsv"
    ragged.write_text("h\ta\tb\nx\t1\t2\ny\t1\n")
    with pytest.raises(ValueError):
        textio.read_table(str(ragged))
    with pytest.raises(FileNotFoundError):
        textio.read_table(str(tmp_path / "missing.tsv"))
    empty = tmp_path / "empty.tsv"
    empty.write_text("cluster\ts0\n")
    h, n, v = textio.read_table(str(empty))
    assert h == "cluster\ts0\n" and n == [] and v.shape[0] == 0


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to the GPU arm): exactly one
    line on stdout, valid JSON with the contract's keys, the same `config` the GPU arm prints; ranks
    other than 0 print nothing.  The timed code is the unmodified reference when oracle/_ref (or
    /root/reference) is present, the port otherwise -- the line says which."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--junctions", "3000", "--samples", "16", "--cpu-workers", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "quant_ps_cells_per_s" and line["unit"] == "cells/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["gpu_launches"] == 0
    from oracle import ref_harness
    kind = "reference" if ref_harness.available() else "port"
    assert line["cpu_baseline"]["kind"] == kind
    # the reference fans out over --cpu-workers processes; the port runs in one
    assert line["cpu_baseline"]["cores"] == (2 if kind == "reference" else 1)
    assert line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    import argparse
    import bench
    assert line["config"] == bench.base_config(argparse.Namespace(samples=16, junctions=3000))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root, env=env)
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_reference_fan_out_equals_one_process():
    """oracle/ref_harness.ref_quant_seconds: the closed-row-slab fan-out of the reference's own
    getClusters / calculatePsi gives the same PS matrix (checksum, NaN count) as one process on the
    whole problem, and the slabs are closed under overlap."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip("no reference tree (neither /root/reference nor oracle/_ref)")
    from splicedice_b200 import synth
    rows = sorted(set(synth.junction_tuples(5000, 3)) | set(synth.adversarial_tuples(4)))
    counts = synth.counts_host(7, 0, len(rows), 12).astype(np.float32)
    counts[::7] = 0
    keep = np.zeros(counts.shape, dtype=np.float32)
    with ref_harness.warnings_off():
        _, sum1, nan1 = ref_harness.ref_quant_seconds(rows, counts, 1, keep=keep)
        _, sum3, nan3 = ref_harness.ref_quant_seconds(rows, counts, 3)
    assert nan1 == nan3 and nan1 == int(np.isnan(keep).sum()) and abs(sum1 - sum3) <= 1e-9 * abs(sum1)
    slabs = ref_harness.closed_row_slabs(rows, 18)
    assert slabs[0][0] == 0 and slabs[-1][1] == len(rows) and all(a[1] == b[0] for a, b in zip(slabs, slabs[1:]))
    clusters = ref_harness.ref_get_clusters(rows)
    index = {j: i for i, j in enumerate(rows)}
    for a, b in slabs:
        for j in rows[a:b]:
            assert all(a <= index[o] < b for o in clusters[j])


def test_npz_writer_layout(tmp_path):
    """--npz: cols / rows / data exactly as findOutliers.py:117-118 unpacks them, data identical
    to the matrix the TSV writer prints, NaN cells kept."""
    import argparse
    from splicedice_b200 import quant
    p = argparse.ArgumentParser()
    quant.add_parser(p)
    man = tmp_path / "m.txt"
    man.write_text("")
    args = p.parse_args(["-m", str(man), "-o", str(tmp_path / "o"), "--npz"])
    assert args.npz is True
    job = quant.SPLICEDICE(args.manifest, args.output_prefix, args, run=False)

    class S:
        def __init__(self, name):
            self.name = name
    job.manifest = [S("a"), S("b"), S("c")]
    job._rows = [("chr1", 5, 90, "+"), ("chr1", 7, 80, "-")]
    job.psi = np.array([[0.25, np.nan, 1.0], [0.0, 0.5, 0.125]], dtype=np.float32)
    job.writeNpz()
    z = np.load(str(tmp_path / "o_allPS.npz"))
    assert sorted(z.files) == ["cols", "data", "rows"]
    assert z["cols"].tolist() == ["a", "b", "c"] and z["rows"].tolist() == ["chr1:5-90:+", "chr1:7-80:-"]
    assert z["data"].dtype == np.float32 and np.array_equal(z["data"], job.psi, equal_nan=True)


def test_fractional_counts_are_refused_not_truncated():
    """The reference would sum fractional rows in float and let scipy truncate the summed table
    (pairwise_fisher.py:158-165); the integer device matrix cannot reproduce that, so such input is
    refused loudly instead of being truncated cell by cell (no GPU is touched before the check)."""
    from splicedice_b200 import pairwise_fisher
    events = ["chr1:1-100:+", "chr1:50-200:+"]
    clusters = {events[0]: [events[1]], events[1]: [events[0]]}
    with pytest.raises(ValueError, match="integers"):
        pairwise_fisher.pairwise_pvalues(events, np.array([[3.0, 4.6], [2.0, 5.0]]), clusters)
    with pytest.raises(ValueError, match="nonnegative"):
        pairwise_fisher.pairwise_pvalues(events, np.array([[3.0, -4.0], [2.0, 5.0]]), clusters)


def test_bench_rejects_bad_arguments():
    """--steps below 1, a negative --warmup, and --dump-outputs on the reference arm stop at parsing."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *argv], capture_output=True, text=True,
                             timeout=120, cwd=root)
        assert out.returncode == 2 and out.stdout == "" and "error:" in out.stderr, argv
