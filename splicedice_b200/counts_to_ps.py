"""``splicedice counts_to_ps`` on a B200: PS from an inclusion-count table and a cluster table.

Host mirror of /root/reference/splicedice/counts_to_ps.py (same functions, flags and files).
The arithmetic of writePsValues (counts_to_ps.py:58-70: exclusion = inc + sum over the listed
overlaps, ps = inc / exclusion in float64) runs in sd_quant_ps (float64 PS output); with
--recluster the adjacency is rebuilt on the device by sd_cluster_build (determine_clusters,
counts_to_ps.py:16-41).
"""
from __future__ import annotations

import numpy as np

from . import junctions as jn


def get_clusters(cluster_file):
    """name -> list of overlap names; an empty list is [''] exactly as the reference parses it."""
    clusters = {}
    with open(cluster_file) as handle:
        for line in handle:
            name, overlaps = line.rstrip("\n").split("\t")
            clusters[name] = overlaps.split(",")
    return clusters


def _names_in_counts_file(counts_file):
    with open(counts_file) as handle:
        handle.readline()
        return [line.split("\t", 1)[0] for line in handle]


def determine_clusters(counts_file, device=0):
    """Adjacency from the junction names of a counts file (sd_cluster_build), keyed and listed by
    name in the reference's list order."""
    from . import ops
    tuples = [jn.parse_name(n) for n in _names_in_counts_file(counts_file)]
    table = jn.JunctionTable(tuples)
    built = ops.cluster_build(*table.arrays(), device=device)
    rows = jn.rows_in_output_order(table.tuples, built["out_row"].cpu().numpy())
    names = [jn.junction_name(j) for j in rows]
    rp = built["row_ptr"].cpu().numpy().tolist()
    ci = built["col_idx"].cpu().numpy().tolist()
    # insertion order follows cluster order in the reference; only membership and list order matter
    order = built["row_of_pos"].cpu().numpy().tolist()
    return {names[r]: [names[c] for c in ci[rp[r]:rp[r + 1]]] for r in order}


def get_counts(count_file):
    """(header line, name -> float64 row); a repeated name keeps its last row.  Parsed natively
    (sd_host_table_read)."""
    from . import textio
    header, names, values = textio.read_table(count_file)
    return header, {n: values[i] for i, n in enumerate(names)}


def junctionStringToTuple(string):
    return jn.parse_name(string)


def ps_matrix(clusters, counts, device=0):
    """(row names sorted as the reference writes them, float64 PS matrix)."""
    from . import ops
    import torch
    names = sorted(clusters.keys(), key=junctionStringToTuple)
    if not names:
        return names, np.zeros((0, 0))
    # rows of the device matrix: every cluster key first, then any counted name only reachable as an overlap
    index = {n: i for i, n in enumerate(names)}
    extra = []
    for n in names:
        for o in clusters[n]:
            if o != "" and o not in index:
                if o not in counts:
                    raise KeyError(o)
                index[o] = len(names) + len(extra)
                extra.append(o)
    all_names = names + extra
    dense = np.stack([counts[n] for n in all_names])           # KeyError if a cluster key has no counts
    as_int = dense.astype(np.int64)
    if not np.array_equal(as_int, dense) or (as_int < 0).any() or (as_int >= 2 ** 31).any():
        raise ValueError("inclusion counts must be non-negative integers below 2^31")
    listing = {n: clusters.get(n, [""]) for n in all_names}
    row_ptr, col_idx = jn.csr_from_named_lists(all_names, listing, "sum")
    inc = ops.upload_counts(as_int, torch.device("cuda", device))
    ps = ops.quant_ps(inc, row_ptr, col_idx, want_f32=False, want_f64=True, row_end=len(names))["ps_f64"]
    return names, ps[:len(names)].cpu().numpy()


def writePsValues(clusters, header, counts, output_prefix, device=0):
    from . import textio
    names, ps = ps_matrix(clusters, counts, device)
    textio.write_matrix(f"{output_prefix}_allPS.tsv", header, names, np.ascontiguousarray(ps, dtype=np.float64))


def writeClusters(clusters, output_prefix):
    with open(f"{output_prefix}_allClusters.tsv", "w") as out:
        for name in sorted(clusters):                      # plain string order here (counts_to_ps.py:76)
            out.write(f"{name}\t{','.join(clusters[name])}\n")


def add_parser(parser):
    parser.add_argument("--clusters", "-c", default=None, help="allClusters.tsv written by quant")
    parser.add_argument("--recluster", "-r", action="store_true",
                        help="rebuild the clusters from the junction names of the counts file")
    parser.add_argument("--inclusion_counts", "-i", required=True, help="inclusionCounts.tsv written by quant")
    parser.add_argument("--output_prefix", "-o", required=True, help="prefix of the output files")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def run_with(args):
    device = getattr(args, "device", 0)
    if args.clusters:
        print("Gathering clusters...")
        clusters = get_clusters(args.clusters)
    elif args.recluster:
        print("Determining clusters from counts file...")
        clusters = determine_clusters(args.inclusion_counts, device)
        writeClusters(clusters, args.output_prefix)
    else:
        raise UnboundLocalError("cannot access local variable 'clusters': give --clusters or --recluster")
    print("Gathering counts...")
    header, counts = get_counts(args.inclusion_counts)
    print("Calculating PS values...")
    writePsValues(clusters, header, counts, args.output_prefix, device)
    print("Done.")


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="PS values from an inclusion-count table (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
