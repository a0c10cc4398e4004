"""``splicedice_b200 compare_groups``: per-event Wilcoxon rank-sum test between two sample groups.

Reads a PS matrix (``{prefix}_allPS.tsv`` from ``quant`` / ``counts_to_ps``, or ``{prefix}_allPS.npz``
from ``quant --npz``) and two sample lists, runs ``scipy.stats.ranksums(x, y, nan_policy='omit')`` per
event on the GPU (sd_ranksum_rows) and Benjamini-Hochberg over the tested events (sd_bh_adjust), and
writes one row per input event, in input order:

    event  mean1  mean2  delta  z  pvalue  corrected

An event with no defined cell in one group is untested: z, pvalue and corrected are ``nan``, and so is
that group's mean.  The file layout is this project's own; the reference's ``compare_sample_sets``
(whose source is not part of this project) may lay its output out differently.
"""
from __future__ import annotations

import numpy as np

HEADER = "event\tmean1\tmean2\tdelta\tz\tpvalue\tcorrected\n"


def read_samples(path):
    """The first tab-separated field of every non-blank line: a ``quant`` manifest or a plain list of
    sample names."""
    names = []
    with open(path, newline="") as handle:
        for line in handle:
            line = line.rstrip("\r\n")
            if line.strip():
                names.append(line.split("\t")[0])
    return names


def read_ps(path):
    """(sample names, event names, PS matrix): float32 from an ``_allPS.npz`` (``cols`` / ``rows`` /
    ``data``), float64 from a TSV table."""
    if path.endswith(".npz"):
        with np.load(path, allow_pickle=False) as z:
            return ([str(s) for s in z["cols"]], [str(r) for r in z["rows"]],
                    np.ascontiguousarray(z["data"], dtype=np.float32))
    from . import textio
    header, events, values = textio.read_table(path)
    return header.rstrip("\r\n").split("\t")[1:], events, values


def group_columns(samples, group1, group2):
    """Column indices of the two groups in ``samples``; ValueError naming the sample for an empty
    group, a sample listed twice or in both groups, or a sample missing from the header."""
    for k, group in ((1, group1), (2, group2)):
        if not group:
            raise ValueError(f"group {k} lists no samples")
        seen = set()
        for s in group:
            if s in seen:
                raise ValueError(f"sample {s!r} is listed twice in group {k}")
            seen.add(s)
    both = set(group1) & set(group2)
    if both:
        s = next(s for s in group1 if s in both)
        raise ValueError(f"sample {s!r} is in both groups")
    index = {s: i for i, s in enumerate(samples)}
    cols = []
    for group in (group1, group2):
        for s in group:
            if s not in index:
                raise ValueError(f"sample {s!r} is not a column of the PS table")
        cols.append(np.array([index[s] for s in group], dtype=np.int32))
    return cols[0], cols[1]


def bh_over_tested(p):
    """Benjamini-Hochberg ("all" mode, sd_bh_adjust) over the tested events of a CUDA p-value vector:
    the events with a p-value; NaN where p is NaN."""
    import torch

    from . import ops
    tested = torch.nonzero(~torch.isnan(p)).reshape(-1)
    corrected = torch.full_like(p, float("nan"))
    if tested.numel():
        corrected[tested] = ops.bh_adjust(p[tested].reshape(-1, 1).contiguous(), "all").reshape(-1)
    return corrected


def compare(ps, cols1, cols2, device=0):
    """float64 [J, 6] = mean1, mean2, delta, z, pvalue, corrected for a host PS matrix (float32 or
    float64), BH over the events with a finite p only."""
    import torch

    from . import ops
    J = ps.shape[0]
    out = np.full((J, 6), np.nan)
    if J == 0:
        return out
    dev = torch.device("cuda", device)
    r = ops.ranksum_rows(torch.from_numpy(ps).to(dev), cols1, cols2)
    p = r["p"]
    corrected = bh_over_tested(p)
    out[:, 0] = r["mean1"].cpu().numpy()
    out[:, 1] = r["mean2"].cpu().numpy()
    out[:, 2] = out[:, 0] - out[:, 1]
    out[:, 3] = r["z"].cpu().numpy()
    out[:, 4] = p.cpu().numpy()
    out[:, 5] = corrected.cpu().numpy()
    return out


def add_parser(parser):
    parser.add_argument("-p", "--ps", required=True,
                        help="PS table: {prefix}_allPS.tsv (quant / counts_to_ps) or {prefix}_allPS.npz (quant --npz)")
    parser.add_argument("-g1", "--group1", required=True,
                        help="samples of group 1: first tab-separated field of each line (a quant manifest works)")
    parser.add_argument("-g2", "--group2", required=True, help="samples of group 2, same format")
    parser.add_argument("-o", "--output", default="compare_groups.tsv", help="output TSV")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def run_with(args):
    group1, group2 = read_samples(args.group1), read_samples(args.group2)
    samples, events, ps = read_ps(args.ps)
    cols1, cols2 = group_columns(samples, group1, group2)
    print(f"PS loaded from {args.ps}: {len(events)} events x {len(samples)} samples; "
          f"group 1: {len(cols1)} samples, group 2: {len(cols2)}")
    res = compare(ps, cols1, cols2, getattr(args, "device", 0))
    print(f"{int(np.isfinite(res[:, 4]).sum())} / {len(events)} events tested")
    from . import textio
    textio.write_matrix(args.output, HEADER, events, res, repr_floats=True)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="Wilcoxon rank-sum test per event between two sample groups (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
