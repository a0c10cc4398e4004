"""Time sd_kruskal_rows (compare_conditions) on two shapes, with sd_ranksum_rows (compare_groups) on the
same matrices, and print one JSON line:

  * 400,000 events x 1,000 samples: float32 PS of bench.py's configs[1] (synth counts -> quant_ps, seed
    SEED / SEED + 1), 4 groups of 250 columns (column c in group c % 4; listed group by group); the
    rank-sum arm splits the same columns 500 / 500 (even / odd).  1.6 GB of PS, far beyond the 126 MB
    L2, so every pass reads it from HBM;
  * 200,000 x 64, 4 groups of 16, rank sum 32 / 32 (the pairwise width; junctions SEED + 7, counts
    SEED + 8).

These are tools/ranksum_bench.py's matrices, so K7 reads against K6 on identical data.  Per shape: the
median CUDA-event time of each library call after two warm-up calls (the two alternate call by call;
device column lists built once),
events/s, the HBM floor (bytes read + written over sd_probe_copy's rate from the same run), and the
scipy.stats.kruskal loop on the first ~2,000 events timed on this host in the same run (one core: the
loop is serial), with the kernel's H / p on those events checked against it and H against the exact
fraction oracle.  ``--out FILE`` also writes the line."""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np
import torch
from scipy.special import chdtrc
from scipy.stats import kruskal

sys.path.insert(0, ".")
from splicedice_b200 import native, ops                       # noqa: E402
from tests import kruskal_cases as cases                      # noqa: E402
from tools.ranksum_bench import SEED, card, ps_matrix          # noqa: E402


def timed_pair(fa, fb, n):
    """medians (ms) of n per-call CUDA-event times of fa and fb, called alternately"""
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(2 * n)]
    torch.cuda.synchronize()
    for i in range(n):
        for f, (e0, e1) in ((fa, ev[2 * i]), (fb, ev[2 * i + 1])):
            e0.record()
            f()
            e1.record()
    torch.cuda.synchronize()
    t = [e0.elapsed_time(e1) for e0, e1 in ev]
    return float(np.median(t[0::2])), float(np.median(t[1::2]))


def scipy_loop(ps_host, groups):
    """(seconds per event, H) of scipy.stats.kruskal(..., nan_policy='omit') over the rows of ps_host"""
    h = np.full(len(ps_host), np.nan)
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for j, row in enumerate(ps_host):
            parts = [row[g] for g in groups]
            if all((~np.isnan(x)).any() for x in parts):
                try:
                    h[j] = kruskal(*parts, nan_policy="omit")[0]
                except ValueError:
                    pass
    return (time.perf_counter() - t0) / len(ps_host), h


def shape(label, J, S, k, junction_seed, count_seed, calls, copy_gbs, slice_rows, dev):
    ps = ps_matrix(J, S, junction_seed, count_seed, dev)
    groups = [np.arange(g, S, k, dtype=np.int32) for g in range(k)]
    c1, c2 = np.arange(0, S, 2, dtype=np.int32), np.arange(1, S, 2, dtype=np.int32)
    d1, d2 = torch.from_numpy(c1).to(dev), torch.from_numpy(c2).to(dev)
    d_cols = torch.from_numpy(np.concatenate(groups)).to(dev)
    d_group = torch.from_numpy(np.repeat(np.arange(k, dtype=np.int32), [len(g) for g in groups])).to(dev)
    n_kw, mean_kw, st_kw = (torch.empty((J, k), dtype=torch.int32, device=dev),
                            torch.empty((J, k), dtype=torch.float64, device=dev),
                            torch.empty((J, 2), dtype=torch.float64, device=dev))
    n_rs, st_rs = torch.empty((J, 2), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev)
    sp = native.stream_ptr()
    # both arms are the bare library call on device lists built once, so neither times host-side checks
    # or copies (ops.kruskal_rows adds those for host lists: the order ops lists the columns in is the
    # one used here, group by group)
    run_kw = lambda: native.call(                                       # noqa: E731
        "sd_kruskal_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, k, d_cols.numel(),
        native.ptr(d_cols), native.ptr(d_group), 0, J, native.ptr(n_kw), k, native.ptr(mean_kw), k,
        native.ptr(st_kw), 2, sp)
    run_rs = lambda: native.call(                                       # noqa: E731
        "sd_ranksum_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, len(c1), native.ptr(d1),
        len(c2), native.ptr(d2), 0, J, native.ptr(n_rs), 2, native.ptr(st_rs), 4, sp)
    for _ in range(2):
        run_kw()
        run_rs()
    ms_kw, ms_rs = timed_pair(run_kw, run_rs, calls)
    res = ops.kruskal_rows(ps, groups)
    torch.cuda.synchronize()
    if not (torch.equal(res["n"], n_kw) and torch.equal(res["H"].view(torch.int64), st_kw[:, 0].view(torch.int64))):
        raise SystemExit(f"{label}: ops.kruskal_rows differs from the timed call")
    read = J * S * ps.element_size()
    written = J * k * (4 + 8) + J * 2 * 8
    floor_ms = (read + written) / (copy_gbs * 1e9) * 1e3
    valid = (~torch.isnan(ps[:, :S])).sum(1).cpu().numpy()
    rows = min(slice_rows, J)
    # scipy 1.18.1 computes kruskal in float32 for float32 input; the kernel widens cells to double
    # exactly, so the reference is scipy on the same values as float64
    host = ps[:rows].cpu().numpy().astype(np.float64)
    per_event_s, h_ref = scipy_loop(host, groups)
    h = res["H"][:rows].cpu().numpy()
    p = res["p"][:rows].cpu().numpy()
    labels = np.repeat(np.arange(k), [len(g) for g in groups])
    cols = np.concatenate(groups)
    h_exact = np.full(rows, np.nan)
    scale = np.full(rows, np.nan)                      # 3 (n + 1) / (1 - T / (n^3 - n)): scipy's H cancels at this size
    for j in range(rows):
        d, n_g, m, t = cases.rank_terms(host[j, cols], labels, k)
        e = cases.exact_h(d, n_g, m, t)
        if e is not None:
            h_exact[j] = float(e)
            scale[j] = 3 * (m + 1) / (1 - t / (m ** 3 - m))
    if not np.array_equal(np.isnan(h), np.isnan(h_exact)):
        raise SystemExit(f"{label}: NaN pattern differs from the exact oracle")
    ok = ~np.isnan(h_exact)
    h_rel = float((np.abs(h[ok] - h_exact[ok]) / np.maximum(h_exact[ok], 1e-300)).max(initial=0))
    fin = ok & np.isfinite(h_ref) & (h_ref >= 0)
    h_scipy = float((np.abs(h[fin] - h_ref[fin]) / scale[fin]).max(initial=0))
    want_p = chdtrc(k - 1, h[ok])
    big = want_p > 1e-300
    p_err = float((np.abs(p[ok][big] - want_p[big]) / want_p[big]).max(initial=0))
    if h_rel > 1e-13 or h_scipy > 1e-13 or p_err > 1e-12:
        raise SystemExit(f"{label}: kernel differs (H rel {h_rel}, vs scipy {h_scipy} of its scale, p rel {p_err})")
    return {"shape": label, "events": J, "samples": S, "groups": k, "group_sizes": [len(g) for g in groups],
            "nan_fraction_of_group_cells": float(1 - valid.sum() / (J * S)),
            "kernel_ms": ms_kw, "events_per_s": J / (ms_kw * 1e-3),
            "ranksum_split": [len(c1), len(c2)], "ranksum_kernel_ms": ms_rs, "kruskal_over_ranksum": ms_kw / ms_rs,
            "bytes_read": read, "bytes_written": written, "hbm_floor_ms": floor_ms,
            "kernel_over_floor": ms_kw / floor_ms,
            "scipy_slice_events": rows, "scipy_tested_events": int(ok.sum()), "scipy_s_per_event": per_event_s,
            "scipy_loop_s_extrapolated_to_all_events": per_event_s * J,
            "speedup_over_scipy_loop": per_event_s * J / (ms_kw * 1e-3),
            "max_rel_h_err_vs_exact": h_rel, "max_abs_h_err_vs_scipy_over_its_scale": h_scipy,
            "max_rel_p_err_vs_chdtrc": p_err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=9)
    ap.add_argument("--slice", type=int, default=2000, help="events in the timed scipy loop")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.calls < 5:
        raise SystemExit("--calls must be at least 5")
    ops.require_cuda()
    dev = torch.device("cuda", 0)
    info = card()
    copy_gbs = ops.probe_copy(1 << 30, dev)
    shapes = [shape("400k x 1,000 (configs[1]), 4 x 250; rank sum 500 / 500", 400_000, 1000, 4, SEED, SEED + 1,
                    args.calls, copy_gbs, args.slice, dev),
              shape("200k x 64 (pairwise width), 4 x 16; rank sum 32 / 32", 200_000, 64, 4, SEED + 7, SEED + 8,
                    args.calls, copy_gbs, args.slice, dev)]
    res = {"tool": "tools/kruskal_bench.py", **info,
           "timing": f"median of {args.calls} per-call CUDA-event times after two warm-up calls, the two kernels "
                     "called alternately; scipy loop: host wall clock, one process on one core",
           "host_cpu_count": os.cpu_count(), "host_cpus_usable": len(os.sched_getaffinity(0)),
           "copy_probe_gbs": copy_gbs, "copy_probe_note": "sd_probe_copy: device-to-device copy, read + write bytes",
           "shapes": shapes}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
