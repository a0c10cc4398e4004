"""Time sd_ranksum_rows (compare_groups) on two shapes and print one JSON line:

  * 400,000 events x 1,000 samples: float32 PS of bench.py's configs[1] (synth counts -> quant_ps, seed
    SEED / SEED + 1), groups of 500 / 500 in interleaved columns (even / odd); 1.6 GB of PS, far beyond the
    126 MB L2, so every pass reads it from HBM;
  * 200,000 x 64, split 32 / 32 (the pairwise width; junctions SEED + 7, counts SEED + 8).

Per shape: the median CUDA-event kernel time after a warm-up, events/s, the HBM floor (bytes read + written
over sd_probe_copy's rate from the same run), the bitonic network's compare-exchange rate, and the
scipy.stats.ranksums loop on the first ~2,000 events timed on this host in the same run (one core: the loop
is serial), with the kernel's z / p on those events checked against it.  ``--out FILE`` also writes the line."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.stats import ranksums

sys.path.insert(0, ".")
from splicedice_b200 import ops, synth            # noqa: E402

SEED = 20261018                                   # bench.py's seed


def timed(fn, n):
    """median of n per-call CUDA-event times (ms)"""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
    torch.cuda.synchronize()
    ev[0].record()
    for i in range(n):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(n)]))


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = (x.strip() for x in r.stdout.strip().split(","))
        return {"device": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}
    except (OSError, ValueError, subprocess.SubprocessError):
        return {"device": torch.cuda.get_device_name(0), "power_limit_w": None, "max_sm_clock_mhz": None}


def ps_matrix(J, S, junction_seed, count_seed, dev):
    cl = ops.cluster_build(*synth.junction_arrays(J, junction_seed)[:4], device=dev)
    counts = ops.synth_counts(count_seed, 0, J, S, logical_cols=S, device=dev)
    return ops.quant_ps(counts, cl["row_ptr"], cl["col_idx"], want_f32=True)["ps_f32"]


def scipy_loop(ps_host, c1, c2):
    """(seconds per event, z, p) of scipy.stats.ranksums(..., nan_policy='omit') over the rows of ps_host"""
    z = np.full(len(ps_host), np.nan)
    p = np.full(len(ps_host), np.nan)
    t0 = time.perf_counter()
    for j, row in enumerate(ps_host):
        x, y = row[c1], row[c2]
        if (~np.isnan(x)).any() and (~np.isnan(y)).any():
            z[j], p[j] = ranksums(x, y, nan_policy="omit")
    return (time.perf_counter() - t0) / len(ps_host), z, p


def shape(label, J, S, junction_seed, count_seed, calls, copy_gbs, slice_rows, dev):
    ps = ps_matrix(J, S, junction_seed, count_seed, dev)
    c1, c2 = np.arange(0, S, 2, dtype=np.int32), np.arange(1, S, 2, dtype=np.int32)
    d1, d2 = torch.from_numpy(c1).to(dev), torch.from_numpy(c2).to(dev)
    out = (torch.empty((J, 2), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev))
    run = lambda: ops.ranksum_rows(ps, d1, d2, out=out)             # noqa: E731
    run()
    run()
    ms = timed(run, calls)
    res = run()
    torch.cuda.synchronize()
    n = len(c1) + len(c2)
    read = J * n * ps.element_size()
    written = J * (2 * 4 + 4 * 8)
    floor_ms = (read + written) / (copy_gbs * 1e9) * 1e3
    # the bitonic network on the next power of two above each row's valid count
    valid = (~torch.isnan(ps[:, :n])).sum(1).cpu().numpy()
    npad = np.where(valid > 1, 2 ** np.ceil(np.log2(np.maximum(valid, 1))), 1).astype(np.int64)
    lg = np.log2(npad).astype(np.int64)
    cx = int((npad // 2 * lg * (lg + 1) // 2).sum())
    rows = min(slice_rows, J)
    host = ps[:rows].cpu().numpy()
    per_event_s, z_ref, p_ref = scipy_loop(host, c1, c2)
    z = res["z"][:rows].cpu().numpy()
    p = res["p"][:rows].cpu().numpy()
    if not np.array_equal(np.isnan(z), np.isnan(z_ref)):
        raise SystemExit(f"{label}: NaN pattern differs from scipy")
    ok = ~np.isnan(z_ref)
    z_err = float(np.abs(z[ok] - z_ref[ok]).max(initial=0))
    big = ok & (p_ref > 1e-300)
    p_err = float((np.abs(p[big] - p_ref[big]) / p_ref[big]).max(initial=0))
    if z_err > 1e-13 or p_err > 1e-12:
        raise SystemExit(f"{label}: kernel differs from scipy (z {z_err}, p rel {p_err})")
    return {"shape": label, "events": J, "samples": S, "group_sizes": [len(c1), len(c2)],
            "nan_fraction_of_group_cells": float(1 - valid.sum() / (J * n)),
            "kernel_ms": ms, "events_per_s": J / (ms * 1e-3),
            "bytes_read": read, "bytes_written": written, "hbm_floor_ms": floor_ms,
            "kernel_over_floor": ms / floor_ms,
            "bitonic_compare_exchanges": cx, "compare_exchanges_per_s": cx / (ms * 1e-3),
            "scipy_slice_events": rows, "scipy_s_per_event": per_event_s,
            "scipy_loop_s_extrapolated_to_all_events": per_event_s * J,
            "speedup_over_scipy_loop": per_event_s * J / (ms * 1e-3),
            "max_abs_z_err_vs_scipy": z_err, "max_rel_p_err_vs_scipy": p_err}


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
    shapes = [shape("400k x 1,000 (configs[1]), 500 / 500", 400_000, 1000, SEED, SEED + 1, args.calls, copy_gbs,
                    args.slice, dev),
              shape("200k x 64 (pairwise width), 32 / 32", 200_000, 64, SEED + 7, SEED + 8, args.calls, copy_gbs,
                    args.slice, dev)]
    res = {"tool": "tools/ranksum_bench.py", **info,
           "timing": f"median of {args.calls} per-call CUDA-event times after two warm-up calls; "
                     "scipy loop: host wall clock, one process on one core",
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
