"""``splicedice ir_table`` on a B200: intron-retention ratios from per-sample intron coverage.

Host mirror of /root/reference/splicedice/ir_table.py (same flags, inputs and output files).
The per-(junction, sample) arithmetic of calculateIR (ir_table.py:118-132) runs on the GPU:
    IR  = median / (median + inc + sum of inc over the junction's cluster)   (sd_ir_ratio)
    RSD = std(cov) / mean(cov) over the 5 coverage points                    (sd_rsd5)
Reading the coverage files, the GTF and the RSD filter / writers stay on the host.

Departures from the reference, both places where it cannot run as written: ``np.float``
(ir_table.py:118, removed from numpy 1.24) is plain float64 here, and ``--RSDthreshold`` is
parsed as a float (the reference leaves it a string, which fails at the comparison :140).
"""
from __future__ import annotations

import os

import numpy as np


def add_parser(parser):
    parser.add_argument("-i", "--inclusionCounts", help="inclusionCounts.tsv written by quant")
    parser.add_argument("-c", "--clusters", help="allClusters.tsv written by quant")
    parser.add_argument("-d", "--coverageDirectory", help="directory of {sample}_intron_coverage.txt files")
    parser.add_argument("-o", "--outputPrefix", help="prefix of the output files")
    parser.add_argument("-r", "--makeRSDtable", action="store_true", help="also write the RSD table")
    parser.add_argument("-s", "--singleJunctionCalculation", action="store_true",
                        help="use the junction's own count only, not its cluster")
    parser.add_argument("-a", "--annotation", help="GTF with the gene annotation")
    parser.add_argument("-j", "--allJunctions", action="store_true",
                        help="keep every junction under the RSD threshold, not only annotated introns")
    parser.add_argument("-t", "--RSDthreshold", default=1.0, type=float, help="RSD cutoff (default 1.0)")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def _attr(field, key):
    for part in field.split(";"):
        if key in part.split('"')[0]:
            return part.split('"')[1]
    raise IndexError(key)


def getAnnotated(annotation):
    """Names ``chrom:exon_end-next_exon_start-1:strand`` of every annotated intron (ir_table.py:39-68)."""
    exons = {}
    with open(annotation) as gtf:
        for line in gtf:
            if line.startswith("#"):
                continue
            row = line.rstrip().split("\t")
            if row[2] == "transcript":
                exons[(_attr(row[8], "transcript_id"), row[0], row[6])] = []
            elif row[2] == "exon":
                exons[(_attr(row[8], "transcript_id"), row[0], row[6])].append((int(row[3]), int(row[4])))
    annotated = set()
    for (_, chrom, strand), spans in exons.items():
        for left, right in zip(spans, spans[1:]):
            annotated.add(f"{chrom}:{left[1]}-{right[0] - 1}:{strand}")
    return annotated


class _SampleCounts:
    """junction name -> float count of one sample: a column of the parsed table."""

    def __init__(self, rows, values, col):
        self._rows, self._values, self._col = rows, values, col

    def __contains__(self, name):
        return name in self._rows

    def __getitem__(self, name):
        return float(self._values[self._rows[name], self._col])


def getInclusionCounts(filename):
    """sample -> {junction name -> float count} (ir_table.py:72-80), as column views over the
    natively parsed table (sd_host_table_read)."""
    from . import textio
    header, names, values = textio.read_table(filename)
    rows = {n: i for i, n in enumerate(names)}
    return {s: _SampleCounts(rows, values, c) for c, s in enumerate(header.strip().split("\t")[1:])}


def getClusters(filename):
    clusters = {}
    with open(filename) as handle:
        for line in handle:
            row = line.strip().split("\t")
            clusters[row[0]] = row[1].split(",") if len(row) > 1 else []
    return clusters


class _Table:
    """sample -> junction -> value view over a dense [junction, sample] array."""

    def __init__(self, samples, names, values):
        self._col = {s: i for i, s in enumerate(samples)}
        self._row = {n: i for i, n in enumerate(names)}
        self.values = values

    def __getitem__(self, sample):
        col = self._col[sample]
        return _Column(self, col)


class _Column:
    def __init__(self, table, col):
        self._t, self._c = table, col

    def __getitem__(self, name):
        return float(self._t.values[self._t._row[name], self._c])


def calculateIR(samples, coverageDirectory, counts, clusters, annotated, args, device=0):
    """(junction names passing the RSD filter, IR view, RSD view) -- the reference's return
    shape; ``.values`` of the views are the dense float64 [junction, sample] arrays."""
    from . import ops
    import torch
    names, index = [], {}
    cells = []                                   # (row, sample, median, cov5)
    for s, sample in enumerate(samples):
        with open(os.path.join(coverageDirectory, f"{sample}_intron_coverage.txt")) as handle:
            for line in handle:
                row = line.strip().split("\t")
                name = f"{row[0]}:{row[1]}-{row[2]}:{row[5]}"
                if not args.allJunctions and name not in annotated:
                    continue
                r = index.get(name)
                if r is None:
                    r = index[name] = len(names)
                    names.append(name)
                cells.append((r, s, float(row[4]), [float(x) for x in row[-1].split(",")]))
    J, S = len(names), len(samples)
    if J == 0:
        empty = np.zeros((0, S))
        return [], _Table(samples, names, empty), _Table(samples, names, empty)
    median = np.full((J, S), np.nan)
    cov = np.full((J, S, 5), np.nan)
    for r, s, m, c in cells:
        median[r, s] = m
        cov[r, s, :] = c
    if np.isnan(median).any():
        r, s = np.argwhere(np.isnan(median))[0]
        raise KeyError(names[r])                 # the reference fails on IR[sample][junction] at write time
    # rows of the count matrix: the coverage junctions, then cluster members that only appear as partners
    all_names, all_index = list(names), dict(index)
    if clusters is not None:
        for n in names:
            for o in clusters[n]:
                if o not in all_index:
                    all_index[o] = len(all_names)
                    all_names.append(o)
    inc = np.zeros((len(all_names), S), dtype=np.int64)
    for s, sample in enumerate(samples):
        have = counts[sample]
        for r, n in enumerate(all_names):
            if n in have:
                value = have[n]
                if value != int(value):
                    # the count matrix is integer on the device; the reference would carry the fraction
                    # through its float arithmetic (ir_table.py:122-130) -- refuse rather than truncate
                    raise ValueError(f"inclusion count {value!r} of {n} in {sample} is not an integer: the B200 path "
                                     "takes the integer counts `quant` writes")
                inc[r, s] = int(value)
            elif r < J:
                raise KeyError(n)                # reference: prints and abandons the sample's file (:133-135)
    if (inc < 0).any() or (inc >= 2 ** 31).any():
        raise ValueError("inclusion counts must be non-negative integers below 2^31")
    dev = torch.device("cuda", device)
    inc_d = ops.upload_counts(inc, dev)
    med = torch.zeros((len(all_names), S), dtype=torch.float64, device=dev)
    med[:J] = torch.from_numpy(median).to(dev)
    if clusters is None or args.singleJunctionCalculation:
        ir = ops.ir_ratio(med, inc_d, row_end=J)
    else:
        row_ptr = np.zeros(len(all_names) + 1, dtype=np.int64)
        cols = []
        for r, n in enumerate(names):
            cols.extend(all_index[o] for o in clusters[n])
            row_ptr[r + 1] = len(cols)
        row_ptr[J + 1:] = len(cols)
        ir = ops.ir_ratio(med, inc_d, row_ptr.astype(np.int32), np.asarray(cols, dtype=np.int32), row_end=J)
    ir = ir[:J].cpu().numpy()
    rsd = ops.rsd5(torch.from_numpy(cov).to(dev)).cpu().numpy()
    keep = np.flatnonzero((rsd < args.RSDthreshold).any(axis=1))
    return [names[r] for r in keep], _Table(samples, names, ir), _Table(samples, names, rsd)


def _write(path, header, samples, junctions, table):
    from . import textio
    ordered = sorted(junctions)
    rows = [table._row[name] for name in ordered]
    cols = [table._col[s] for s in samples]
    block = np.ascontiguousarray(table.values[np.ix_(rows, cols)], dtype=np.float64) if rows else np.zeros((0, len(cols)))
    textio.write_matrix(path, header, ordered, block)


def writeIRtable(samples, outputPrefix, junctions, IR):
    _write(f"{outputPrefix}_intron_retention.tsv", "Junction\t" + "\t".join(samples) + "\n", samples, junctions, IR)


def writeRSDtable(samples, outputPrefix, junctions, RSD):
    _write(f"{outputPrefix}_intron_retention_RSD.tsv",
           "Junction\t" + "\t".join(f"{s}_RSD" for s in samples) + "\n", samples, junctions, RSD)


def run_with(args):
    import time
    start = time.time()
    suffix = "_intron_coverage.txt"
    samples = [f.replace(suffix, "") for f in os.listdir(args.coverageDirectory) if f.endswith("intron_coverage.txt")]
    print("Gathering inclusion counts and clusters...")
    counts = getInclusionCounts(args.inclusionCounts)
    annotated = None if args.allJunctions else getAnnotated(args.annotation)
    clusters = None if args.singleJunctionCalculation else getClusters(args.clusters)
    print("Calculating IR values...")
    junctions, IR, RSD = calculateIR(samples, args.coverageDirectory, counts, clusters, annotated, args,
                                     getattr(args, "device", 0))
    print("Done", time.time() - start)
    print("Writing output...")
    writeIRtable(samples, args.outputPrefix, junctions, IR)
    if args.makeRSDtable:
        writeRSDtable(samples, args.outputPrefix, junctions, RSD)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="intron-retention table (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
