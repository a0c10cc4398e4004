"""``splicedice_b200 compare_paired``: per-event Wilcoxon signed-rank test between matched sample pairs.

Reads a PS matrix (``{prefix}_allPS.tsv`` from ``quant`` / ``counts_to_ps``, or ``{prefix}_allPS.npz``
from ``quant --npz``) and a pairs file, runs ``scipy.stats.wilcoxon(x, y, nan_policy='omit')`` per event
on the GPU (sd_signedrank_rows; x = the side-1 samples, y = their partners) and Benjamini-Hochberg over
the tested events (sd_bh_adjust), and writes one row per input event, in input order:

    event  n  mean1  mean2  delta  W  pvalue  corrected

Pairs file: per non-blank line, the first two tab-separated fields are a side-1 sample and its side-2
partner (tumour and adjacent normal of one patient, before and after treatment, ...); further fields
are ignored.  n is the number of pairs with both cells defined; mean1 / mean2 are over those pairs.
Differences are taken in the PS matrix's precision (float32 for an ``.npz``).  An event with no
complete pair, with one complete pair whose difference is zero, or with more than 13 complete pairs
and no nonzero difference (scipy's p is ``nan`` there) is untested: W, pvalue and corrected are ``nan``.
"""
from __future__ import annotations

import numpy as np

from .compare_groups import bh_over_tested, read_ps

HEADER = "event\tn\tmean1\tmean2\tdelta\tW\tpvalue\tcorrected\n"


def read_pairs(path):
    """(side-1 sample, side-2 sample) of every non-blank line, in file order; ValueError naming
    ``path:line`` for a line without two non-empty tab-separated fields."""
    pairs = []
    with open(path, newline="") as handle:
        for number, line in enumerate(handle, 1):
            line = line.rstrip("\r\n")
            if not line.strip():
                continue
            fields = line.split("\t")
            if len(fields) < 2 or not fields[0] or not fields[1]:
                raise ValueError(f"{path}:{number}: expected two samples separated by a tab")
            pairs.append((fields[0], fields[1]))
    return pairs


def pair_columns(samples, pairs):
    """Column indices of the side-1 and side-2 samples in ``samples``; ValueError naming the sample for
    a sample listed twice (on either side) or missing from the header, and for no pairs at all."""
    if not pairs:
        raise ValueError("the pairs file lists no pairs")
    seen = set()
    for pair in pairs:
        for s in pair:
            if s in seen:
                raise ValueError(f"sample {s!r} is listed twice")
            seen.add(s)
    index = {s: i for i, s in enumerate(samples)}
    for pair in pairs:
        for s in pair:
            if s not in index:
                raise ValueError(f"sample {s!r} is not a column of the PS table")
    return (np.array([index[a] for a, _ in pairs], dtype=np.int32),
            np.array([index[b] for _, b in pairs], dtype=np.int32))


def compare(ps, cols1, cols2, device=0):
    """float64 [J, 7] = n, mean1, mean2, delta, W, pvalue, corrected for a host PS matrix (float32 or
    float64), BH over the tested events only."""
    import torch

    from . import ops
    J = ps.shape[0]
    out = np.full((J, 7), np.nan)
    if J == 0:
        return out
    dev = torch.device("cuda", device)
    r = ops.signedrank_rows(torch.from_numpy(ps).to(dev), cols1, cols2)
    corrected = bh_over_tested(r["p"])
    out[:, 0] = r["n"].cpu().numpy()
    out[:, 1] = r["mean1"].cpu().numpy()
    out[:, 2] = r["mean2"].cpu().numpy()
    out[:, 3] = out[:, 1] - out[:, 2]
    out[:, 4] = r["W"].cpu().numpy()
    out[:, 5] = r["p"].cpu().numpy()
    out[:, 6] = corrected.cpu().numpy()
    return out


def add_parser(parser):
    parser.add_argument("-p", "--ps", required=True,
                        help="PS table: {prefix}_allPS.tsv (quant / counts_to_ps) or {prefix}_allPS.npz (quant --npz)")
    parser.add_argument("--pairs", required=True,
                        help="one pair per line: a side-1 sample and its side-2 partner, tab-separated")
    parser.add_argument("-o", "--output", default="compare_paired.tsv", help="output TSV")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def run_with(args):
    pairs = read_pairs(args.pairs)
    samples, events, ps = read_ps(args.ps)
    cols1, cols2 = pair_columns(samples, pairs)
    print(f"PS loaded from {args.ps}: {len(events)} events x {len(samples)} samples; {len(pairs)} pairs")
    res = compare(ps, cols1, cols2, getattr(args, "device", 0))
    print(f"{int(np.isfinite(res[:, 5]).sum())} / {len(events)} events tested")
    from . import textio
    textio.write_matrix(args.output, HEADER, events, res, repr_floats=True)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="Wilcoxon signed-rank test per event between matched sample pairs (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
