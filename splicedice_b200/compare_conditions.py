"""``splicedice_b200 compare_conditions``: per-event Kruskal-Wallis H test across any number of sample
groups.

Reads a PS matrix (``{prefix}_allPS.tsv`` from ``quant`` / ``counts_to_ps``, or ``{prefix}_allPS.npz``
from ``quant --npz``) and a groups file, runs ``scipy.stats.kruskal(*groups, nan_policy='omit')`` per
event on the GPU (sd_kruskal_rows) and Benjamini-Hochberg over the tested events (sd_bh_adjust), and
writes one row per input event, in input order:

    event  H  pvalue  corrected  mean_<group 1>  ...  mean_<group k>

Groups file: per non-blank line, the sample is the first tab-separated field and its group the last,
so a ``quant`` manifest (``name path metadata condition``) groups by condition and a two-column
``sample<TAB>group`` file works as well.  Groups are numbered in the order they first appear; samples
of the PS table the file does not list are unused.  An event with no defined cell in some group, or
with every defined cell tied, is untested: H, pvalue and corrected are ``nan``.
"""
from __future__ import annotations

import numpy as np

from .compare_groups import bh_over_tested, read_ps


def read_groups(path):
    """(group names in order of first appearance, the samples of each group in file order); ValueError
    naming ``path:line`` for a line with one field or an empty group label."""
    names, members = [], {}
    with open(path, newline="") as handle:
        for number, line in enumerate(handle, 1):
            line = line.rstrip("\r\n")
            if not line.strip():
                continue
            fields = line.split("\t")
            if len(fields) < 2:
                raise ValueError(f"{path}:{number}: expected a sample and a group separated by a tab")
            if not fields[-1].strip():
                raise ValueError(f"{path}:{number}: empty group label")
            if fields[-1] not in members:
                names.append(fields[-1])
                members[fields[-1]] = []
            members[fields[-1]].append(fields[0])
    return names, [members[g] for g in names]


def group_columns(samples, names, members):
    """Column indices of every group in ``samples``; ValueError naming the sample for a sample listed
    twice or missing from the header, and for fewer than two groups."""
    if len(names) < 2:
        raise ValueError(f"the groups file names {len(names)} group(s); at least two are needed")
    seen = set()
    for group in members:
        for s in group:
            if s in seen:
                raise ValueError(f"sample {s!r} is listed twice")
            seen.add(s)
    index = {s: i for i, s in enumerate(samples)}
    for group in members:
        for s in group:
            if s not in index:
                raise ValueError(f"sample {s!r} is not a column of the PS table")
    return [np.array([index[s] for s in group], dtype=np.int32) for group in members]


def header(names):
    return "\t".join(["event", "H", "pvalue", "corrected"] + [f"mean_{g}" for g in names]) + "\n"


def compare(ps, cols, device=0):
    """float64 [J, 3 + k] = H, pvalue, corrected, mean per group for a host PS matrix (float32 or
    float64), BH over the tested events only."""
    import torch

    from . import ops
    J, k = ps.shape[0], len(cols)
    out = np.full((J, 3 + k), np.nan)
    if J == 0:
        return out
    dev = torch.device("cuda", device)
    r = ops.kruskal_rows(torch.from_numpy(ps).to(dev), cols)
    corrected = bh_over_tested(r["p"])
    out[:, 0] = r["H"].cpu().numpy()
    out[:, 1] = r["p"].cpu().numpy()
    out[:, 2] = corrected.cpu().numpy()
    out[:, 3:] = r["mean"].cpu().numpy()
    return out


def add_parser(parser):
    parser.add_argument("-p", "--ps", required=True,
                        help="PS table: {prefix}_allPS.tsv (quant / counts_to_ps) or {prefix}_allPS.npz (quant --npz)")
    parser.add_argument("-g", "--groups", required=True,
                        help="sample in the first tab-separated field, its group in the last (a quant manifest "
                             "groups by condition)")
    parser.add_argument("-o", "--output", default="compare_conditions.tsv", help="output TSV")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def run_with(args):
    names, members = read_groups(args.groups)
    samples, events, ps = read_ps(args.ps)
    cols = group_columns(samples, names, members)
    print(f"PS loaded from {args.ps}: {len(events)} events x {len(samples)} samples; "
          f"{len(names)} groups: " + ", ".join(f"{g} ({len(c)})" for g, c in zip(names, cols)))
    res = compare(ps, cols, getattr(args, "device", 0))
    print(f"{int(np.isfinite(res[:, 1]).sum())} / {len(events)} events tested")
    from . import textio
    textio.write_matrix(args.output, header(names), events, res, repr_floats=True)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="Kruskal-Wallis H test per event across sample groups (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
