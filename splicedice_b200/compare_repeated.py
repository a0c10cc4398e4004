"""``splicedice_b200 compare_repeated``: per-event Friedman test across conditions measured on the same
subjects.

Reads a PS matrix (``{prefix}_allPS.tsv`` from ``quant`` / ``counts_to_ps``, or ``{prefix}_allPS.npz``
from ``quant --npz``) and a blocks file, runs ``scipy.stats.friedmanchisquare(*conditions,
nan_policy='omit')`` per event on the GPU (sd_friedman_rows; the cells of each subject are ranked within
the subject) and Benjamini-Hochberg over the tested events (sd_bh_adjust), and writes one row per input
event, in input order:

    event  n  Q  pvalue  corrected  mean_<condition 1>  ...  mean_<condition k>

Blocks file: the first non-blank line names the k >= 3 conditions, tab-separated; every further non-blank
line is one subject (a patient of a time course, a cell line under several treatments, a donor's
tissues): its k samples, tab-separated, in the header's order.  A subject with an empty field (no sample
for some condition) can never be complete and is skipped; the samples it does name are still checked
(listed once, present in the PS table).  n is the number of subjects with every cell of
the event defined; the means are over those subjects.  An event with no complete subject, or whose
complete subjects are tied throughout, is untested: Q, pvalue and corrected are ``nan``.
"""
from __future__ import annotations

import numpy as np

from .compare_groups import bh_over_tested, read_ps


def read_blocks(path):
    """(condition names, the complete subjects' sample lists, the skipped subjects' field lists);
    ValueError naming ``path:line`` for a header with fewer than three, repeated or empty condition names
    and for a subject line with the wrong number of fields, and ValueError for a file with no usable
    subject.  A skipped subject (one with an empty field) is still a list of samples: block_columns checks
    its named samples like any other."""
    names, subjects, skipped, header_line = None, [], [], 0
    with open(path, newline="") as handle:
        for number, line in enumerate(handle, 1):
            line = line.rstrip("\r\n")
            if not line.strip():
                continue
            fields = line.split("\t")
            if names is None:
                if any(not f.strip() for f in fields):
                    raise ValueError(f"{path}:{number}: empty condition name in the header")
                if len(set(fields)) != len(fields):
                    raise ValueError(f"{path}:{number}: a condition is named twice in the header")
                if len(fields) < 3:
                    raise ValueError(f"{path}:{number}: the header names {len(fields)} condition(s); the Friedman "
                                     "test needs at least three (compare_paired tests two matched conditions)")
                names, header_line = fields, number
                continue
            if len(fields) != len(names):
                raise ValueError(f"{path}:{number}: expected {len(names)} tab-separated samples, found {len(fields)}")
            if any(not f for f in fields):
                skipped.append(fields)
                continue
            subjects.append(fields)
    if names is None:
        raise ValueError(f"{path}: no header line naming the conditions")
    if not subjects:
        raise ValueError(f"{path}: no subject with a sample for every condition after the header "
                         f"(line {header_line})")
    return names, subjects, skipped


def block_columns(samples, subjects, skipped=()):
    """int32 [n_blocks, k] column indices of the subjects' samples in ``samples``; ValueError naming the
    sample for a sample listed twice or missing from the header.  The samples named on skipped subject
    lines are checked too (a typo or a reused sample there is as wrong as anywhere else), though they get
    no columns."""
    named = [s for subject in list(subjects) + list(skipped) for s in subject if s]
    seen = set()
    for s in named:
        if s in seen:
            raise ValueError(f"sample {s!r} is listed twice")
        seen.add(s)
    index = {s: i for i, s in enumerate(samples)}
    for s in named:
        if s not in index:
                raise ValueError(f"sample {s!r} is not a column of the PS table")
    return np.array([[index[s] for s in subject] for subject in subjects], dtype=np.int32)


def header(names):
    return "\t".join(["event", "n", "Q", "pvalue", "corrected"] + [f"mean_{c}" for c in names]) + "\n"


def compare(ps, blocks, device=0):
    """float64 [J, 4 + k] = n, Q, pvalue, corrected, mean per condition for a host PS matrix (float32 or
    float64) and int [n_blocks, k] columns, BH over the tested events only."""
    import torch

    from . import ops
    J, k = ps.shape[0], blocks.shape[1]
    out = np.full((J, 4 + k), np.nan)
    if J == 0:
        return out
    dev = torch.device("cuda", device)
    r = ops.friedman_rows(torch.from_numpy(ps).to(dev), blocks)
    corrected = bh_over_tested(r["p"])
    out[:, 0] = r["n"].cpu().numpy()
    out[:, 1] = r["Q"].cpu().numpy()
    out[:, 2] = r["p"].cpu().numpy()
    out[:, 3] = corrected.cpu().numpy()
    out[:, 4:] = r["mean"].cpu().numpy()
    return out


def add_parser(parser):
    parser.add_argument("-p", "--ps", required=True,
                        help="PS table: {prefix}_allPS.tsv (quant / counts_to_ps) or {prefix}_allPS.npz (quant --npz)")
    parser.add_argument("--blocks", required=True,
                        help="header: the k >= 3 condition names; then one subject per line: its k samples in "
                             "header order, tab-separated")
    parser.add_argument("-o", "--output", default="compare_repeated.tsv", help="output TSV")
    parser.add_argument("--device", type=int, default=0, help="CUDA device ordinal")


def run_with(args):
    names, subjects, skipped = read_blocks(args.blocks)
    samples, events, ps = read_ps(args.ps)
    blocks = block_columns(samples, subjects, skipped)
    print(f"PS loaded from {args.ps}: {len(events)} events x {len(samples)} samples; {len(subjects)} subjects x "
          f"{len(names)} conditions ({', '.join(names)})"
          + (f"; {len(skipped)} subject(s) without a sample for every condition skipped" if skipped else ""))
    res = compare(ps, blocks, getattr(args, "device", 0))
    print(f"{int(np.isfinite(res[:, 2]).sum())} / {len(events)} events tested")
    from . import textio
    textio.write_matrix(args.output, header(names), events, res, repr_floats=True)


if __name__ == "__main__":
    import argparse
    cli = argparse.ArgumentParser(description="Friedman test per event across conditions measured on the same "
                                              "subjects (B200)")
    add_parser(cli)
    run_with(cli.parse_args())
