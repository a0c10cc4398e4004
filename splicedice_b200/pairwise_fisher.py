"""``splicedice pairwise`` on a B200: per-event Fisher exact (or ``--chi2``) test for every sample pair.

Host mirror of /root/reference/splicedice/pairwise_fisher.py (same flags, inputs and output
file).  The hot loop (pairwise_fisher.py:154-180) runs on the GPU: exclusion counts with
sd_quant_ps over the cluster CSR, then sd_fisher_pairwise (or sd_chi2_pairwise) for the
[events x pairs] p-values.  Benjamini-Hochberg runs on the device too (sd_bh_adjust); the writer
is the native host formatter.  With ``--chi2`` a table scipy's chi2_contingency refuses (a zero
margin) raises the same ValueError the reference's loop stops on, and no file is written.
"""
from __future__ import annotations

import numpy as np

from . import junctions as jn


def getClusters(filename, filter_list=None):
    """event -> list of mutually exclusive events.  Whitespace split; a line that is not exactly
    two fields is an event with no partners (pairwise_fisher.py:26-43)."""
    clusters = {}
    with open(filename) as handle:
        for line in handle:
            fields = line.rstrip().split()
            if len(fields) == 2:
                clusters[fields[0]] = fields[1].split(",")
            else:
                clusters[line.strip()] = []
    return clusters


def getEventCounts(filename, filter_list=None):
    """(sample names, event names, float64 counts); with a filter only listed events are kept.
    Parsed natively (sd_host_table_read); same results as the reference's per-line reader."""
    from . import textio
    header, events, counts = textio.read_table(filename)
    samples = header.rstrip().split("\t")[1:]
    if filter_list is not None:
        keep = [i for i, e in enumerate(events) if e in filter_list]
        events = [events[i] for i in keep]
        counts = counts[keep]
    return samples, events, counts


def fdr_bh(p, device=0):
    """Benjamini-Hochberg adjusted p-values of a 1-D array, as statsmodels
    multipletests(method='fdr_bh')[1] (pairwise_fisher.py:185,190), computed on the GPU
    (sd_bh_adjust: radix sort, p / (rank / n), running minimum from the right, clip at 1)."""
    from . import ops
    import torch
    p = np.ascontiguousarray(p, dtype=np.float64).reshape(-1)
    if p.size == 0:
        return p.copy()
    d = torch.from_numpy(p).to(torch.device("cuda", device)).reshape(-1, 1)
    return ops.bh_adjust(d, "all", out=d).reshape(-1).cpu().numpy()


def sample_pairs(n_samples):
    return [(i, j) for i in range(n_samples - 1) for j in range(i + 1, n_samples)]


def checked_counts(counts):
    """int64 copy of a host inclusion-count matrix; ValueError on counts the device path cannot take."""
    counts = np.asarray(counts)
    as_int = counts.astype(np.int64)
    if not np.array_equal(as_int, counts):
        # the reference sums the float rows first and lets scipy truncate the summed table
        # (pairwise_fisher.py:158-165), so fractions would add up differently: refuse rather than guess
        raise ValueError("inclusion counts must be integers (the table `quant` writes); fractional counts are "
                         "not supported on the B200 path")
    if (as_int < 0).any():
        raise ValueError("All values in `table` must be nonnegative.")
    if (as_int >= 2 ** 31).any():
        raise ValueError("counts of 2^31 and above are not supported")
    return as_int


def fisher_inputs(counts_int, row_ptr, col_idx, device):
    """Upload a checked count matrix (or row slab with its local CSR) and sum its exclusion counts on
    ``device``: (inc, exc, pair_a, pair_b, bound) for ops.fisher_pairwise over every sample pair."""
    from . import ops
    inc = ops.upload_counts(counts_int, device)
    exc = ops.quant_ps(inc, row_ptr, col_idx, want_f32=False, want_exc=True)["exc"]
    pa, pb = ops.all_pairs(counts_int.shape[1])
    # the host filled the matrix, so it can vouch for a bound on inc + exc: no reduction / sync on the device
    bound = int(counts_int.max(initial=0)) * (1 + int(np.diff(row_ptr).max(initial=0)))
    return inc, exc, pa, pb, bound


def chi2_refusal(first, counts_int, row_ptr, col_idx, events, samples=None):
    """ValueError for the first table scipy.stats.chi2_contingency refuses, ``first`` = row * n_pairs +
    pair (sd_chi2_pairwise's index): scipy's message with the (i, j) of the first zero expected frequency,
    then the event, the ``a_b`` column and the table.  The table is rebuilt on the host from the CSR."""
    pa, pb = np.triu_indices(counts_int.shape[1], k=1)          # the pair order of ops.all_pairs
    j, k = divmod(int(first), len(pa))
    sa, sb = int(pa[k]), int(pb[k])
    members = col_idx[row_ptr[j]:row_ptr[j + 1]]
    a, b = int(counts_int[j, sa]), int(counts_int[j, sb])
    c, d = int(counts_int[members, sa].sum()), int(counts_int[members, sb].sum())
    column = f"{samples[sa]}_{samples[sb]}" if samples is not None else f"{sa}_{sb}"
    where = f"event {events[j]}, column {column}, table [[{a}, {b}], [{c}, {d}]]"
    if a + b == 0 or a + c == 0:
        pos = "(0, 0)"
    elif b + d == 0:
        pos = "(0, 1)"
    elif c + d == 0:
        pos = "(1, 0)"
    else:
        return ValueError(f"chi-squared test: table outside the supported range ({where})")
    return ValueError(f"The internally computed table of expected frequencies has a zero element at {pos}. ({where})")


def pairwise_pvalues(events, counts, clusters, device=0, correction="none", gpus=1, test="fisher", samples=None):
    """float64[len(events), n_pairs] p-values, pair order as ``sample_pairs``: two-sided Fisher
    (``test='fisher'``) or Yates-corrected chi-squared (``test='chi2'``, scipy's chi2_contingency; a
    refused table raises ValueError naming the event and the column, from ``samples`` when given);
    ``correction`` = 'none' | 'pairwise' | 'all' applies Benjamini-Hochberg on the device before the
    matrix comes back (pairwise_fisher.py:182-191)."""
    from . import ops
    import torch
    if test not in ("fisher", "chi2"):
        raise ValueError("test must be 'fisher' or 'chi2'")
    n_events, n_samples = counts.shape if counts.ndim == 2 else (0, 0)
    n_pairs = n_samples * (n_samples - 1) // 2
    if n_events == 0 or not n_pairs:
        return np.zeros((n_events, n_pairs))
    as_int = checked_counts(counts)
    row_ptr, col_idx = jn.csr_from_named_lists(events, clusters, "isin")
    if gpus > 1:                                    # one worker process per GPU (row slabs; NCCL for the correction)
        from . import multigpu
        p, first = multigpu.pairwise(as_int, row_ptr, col_idx, n_pairs, correction=correction, n_gpus=gpus, test=test)
        if first is not None:
            raise chi2_refusal(first, as_int, row_ptr, col_idx, events, samples)
        return p
    inc, exc, pa, pb, bound = fisher_inputs(as_int, row_ptr, col_idx, torch.device("cuda", device))
    if test == "chi2":
        refused = torch.full((1,), -1, dtype=torch.int64, device=inc.device)
        p = ops.chi2_pairwise(inc, exc, pa, pb, refused=refused)
        first = int(refused.item())
        if first != -1:                             # the reference's loop stops at this table
            raise chi2_refusal(first, as_int, row_ptr, col_idx, events, samples)
    else:
        p = ops.fisher_pairwise(inc, exc, pa, pb, max_cell_bound=bound)
    if correction != "none":
        ops.bh_adjust(p, correction, out=p)
    return p.cpu().numpy()


def add_parser(parser):
    parser.add_argument("--inclusionSPLICEDICE", type=str, required=True,
                        help="inclusionCounts.tsv written by quant")
    parser.add_argument("-c", "--clusters", type=str, required=True, help="allClusters.tsv written by quant")
    parser.add_argument("--chi2", action="store_true", default=False,
                        help="Yates-corrected chi-squared test (scipy's chi2_contingency) instead of Fisher")
    parser.add_argument("--multiple_test_correction", default="pairwise", choices=["pairwise", "all", "none"],
                        help="Benjamini-Hochberg per sample pair (default), over all p-values, or none")
    parser.add_argument("-f", "--filter_list", help="text file of events to analyse, one per line")
    parser.add_argument("-o", "--output", default="pairwise.tsv", help="output TSV")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")
    parser.add_argument("--gpus", type=int, default=1,
                        help="GPUs: one worker process per GPU on devices 0..N-1, events cut into row slabs")


def run_with(args):
    filter_list = None
    if args.filter_list is not None:
        with open(args.filter_list) as handle:
            filter_list = {line.rstrip() for line in handle}
    samples, events, counts = getEventCounts(args.inclusionSPLICEDICE, filter_list)
    print("Counts loaded from", args.inclusionSPLICEDICE, "...")
    clusters = getClusters(args.clusters, filter_list)
    print("Clusters loaded from", args.clusters, "...")
    pairs = sample_pairs(len(samples))
    columns = [f"{samples[a]}_{samples[b]}" for a, b in pairs]
    print("Analyzing pairs:")
    print(",".join(columns))
    parray = pairwise_pvalues(events, counts, clusters, getattr(args, "device", 0),
                              correction=args.multiple_test_correction, gpus=getattr(args, "gpus", 1),
                              test="chi2" if args.chi2 else "fisher", samples=samples)
    print(f"[{len(events)} / {len(events)}] events analyzed...")
    from . import textio
    textio.write_matrix(args.output, "clusterID\t" + "\t".join(columns) + "\n", events,
                        np.ascontiguousarray(parray, dtype=np.float64), repr_floats=True)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="pairwise Fisher exact / chi-squared tests (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
