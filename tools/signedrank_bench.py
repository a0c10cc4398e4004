"""Time sd_signedrank_rows (compare_paired) on four shapes, one per method path, and print one JSON line:

  * 400,000 events x 1,000 samples as 500 pairs (column 2i with 2i + 1): float32 PS of bench.py's
    configs[1] (synth counts -> quant_ps, seed SEED / SEED + 1, tools/ranksum_bench.py's matrix) rounded
    to 3 decimals, so |d| ties heavily: the normal approximation.  sd_ranksum_rows (K6) runs on the same
    matrix with the same columns as 500 / 500, the two calls alternating;
  * 400,000 x 100 as 50 pairs, uniform float32 (seed SEED + 20), untied: the exact null distribution;
  * 400,000 x 24 as 12 pairs, uniform rounded to 2 decimals (seed SEED + 21), tied, with zeros: the
    sign-flip enumeration;
  * 200,000 x 64 as 32 pairs: tools/ranksum_bench.py's pairwise-width PS (junctions SEED + 7, counts
    SEED + 8), whose NaNs put rows on all three paths.

The first matrix is 1.6 GB, far beyond the 126 MB L2, so every pass reads it from HBM.  Per shape: the
median CUDA-event time of the bare library call on device column lists built once, after two warm-up
calls; events/s; the rows per method; the HBM floor (bytes read + written over sd_probe_copy's rate from
the same run); and the scipy.stats.wilcoxon(x, y, nan_policy='omit') loop on the first events timed on
this host in the same run (one core: the loop is serial), with the kernel's n, method, W and p on those
events checked against scipy and the row rule of tests/signedrank_cases.py.  ``--out FILE`` also writes
the line."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from splicedice_b200 import native, ops                       # noqa: E402
from tests import signedrank_cases as cases                   # noqa: E402
from tools.kruskal_bench import timed_pair                    # noqa: E402
from tools.ranksum_bench import SEED, card, ps_matrix, timed  # noqa: E402


def uniform(J, S, seed, decimals, dev):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    ps = torch.rand((J, S), generator=g, device=dev, dtype=torch.float32)
    return ps if decimals is None else torch.round(ps, decimals=decimals)


def scipy_loop(host, c1, c2):
    """(seconds per event, W, p) of scipy.stats.wilcoxon over the rows of host: on the float32 differences
    widened (cases.scipy_row), as the kernel subtracts; NaN where scipy raises"""
    w, p = np.full(len(host), np.nan), np.full(len(host), np.nan)
    t0 = time.perf_counter()
    for j, row in enumerate(host):
        w[j], p[j], _ = cases.scipy_row(row[c1], row[c2], np.float32)
    return (time.perf_counter() - t0) / len(host), w, p


def shape(label, ps, calls, copy_gbs, slice_rows, with_ranksum=False):
    J, S = ps.shape
    P = S // 2
    dev = ps.device
    c1, c2 = np.arange(0, 2 * P, 2, dtype=np.int32), np.arange(1, 2 * P, 2, dtype=np.int32)
    d1, d2 = torch.from_numpy(c1).to(dev), torch.from_numpy(c2).to(dev)
    n_out, st = torch.empty((J, 3), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev)
    sp = native.stream_ptr()
    run = lambda: native.call(                                          # noqa: E731
        "sd_signedrank_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, P, native.ptr(d1),
        native.ptr(d2), 0, J, native.ptr(n_out), 3, native.ptr(st), 4, sp)
    extra = {}
    if with_ranksum:
        n_rs, st_rs = torch.empty((J, 2), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev)
        run_rs = lambda: native.call(                                   # noqa: E731
            "sd_ranksum_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, P, native.ptr(d1),
            P, native.ptr(d2), 0, J, native.ptr(n_rs), 2, native.ptr(st_rs), 4, sp)
        for _ in range(2):
            run()
            run_rs()
        ms, ms_rs = timed_pair(run, run_rs, calls)
        extra = {"ranksum_split": [P, P], "ranksum_kernel_ms": ms_rs, "signedrank_over_ranksum": ms / ms_rs}
    else:
        run()
        run()
        ms = timed(run, calls)
    res = ops.signedrank_rows(ps, c1, c2)
    torch.cuda.synchronize()
    if not (torch.equal(res["n"], n_out[:, 0]) and torch.equal(res["p"].view(torch.int64), st[:, 3].view(torch.int64))):
        raise SystemExit(f"{label}: ops.signedrank_rows differs from the timed call")
    method = n_out[:, 2].cpu().numpy()
    read = J * 2 * P * ps.element_size()
    written = J * (3 * 4 + 4 * 8)
    floor_ms = (read + written) / (copy_gbs * 1e9) * 1e3
    rows = min(slice_rows, J)
    host = ps[:rows].cpu().numpy()
    per_event_s, w_ref, p_ref = scipy_loop(host, c1, c2)
    got = {k: v[:rows].cpu().numpy() for k, v in res.items()}
    p_err = 0.0
    for j in range(rows):
        n, c, mode, W, P_rule = cases.signed_rank_row(host[j, c1], host[j, c2], np.float32)
        if (got["n"][j], got["c"][j], got["method"][j]) != (n, c, mode):
            raise SystemExit(f"{label}: row {j}: n / c / method differ from the row rule")
        if mode == 0:
            if not (np.isnan(got["W"][j]) and np.isnan(got["p"][j])):
                raise SystemExit(f"{label}: row {j}: untested row has a statistic")
            continue
        if got["W"][j] != W or got["W"][j] != w_ref[j]:
            raise SystemExit(f"{label}: row {j}: W differs ({got['W'][j]}, rule {W}, scipy {w_ref[j]})")
        if mode == 1 and not (got["p"][j] == P_rule == p_ref[j]):
            raise SystemExit(f"{label}: row {j}: exact p differs ({got['p'][j]}, rule {P_rule}, scipy {p_ref[j]})")
        if mode == 2 and p_ref[j] > 1e-300:
            p_err = max(p_err, abs(got["p"][j] - p_ref[j]) / p_ref[j])
    if p_err > 1e-12:
        raise SystemExit(f"{label}: normal-approximation p differs from scipy by {p_err} relative")
    return {"shape": label, "events": J, "samples": S, "pairs": P,
            "rows_per_method": {str(m): int((method == m).sum()) for m in (0, 1, 2)},
            "kernel_ms": ms, "events_per_s": J / (ms * 1e-3), **extra,
            "bytes_read": read, "bytes_written": written, "hbm_floor_ms": floor_ms, "kernel_over_floor": ms / floor_ms,
            "scipy_slice_events": rows, "scipy_slice_rows_per_method":
                {str(m): int((got["method"] == m).sum()) for m in (0, 1, 2)},
            "scipy_s_per_event": per_event_s, "scipy_loop_s_extrapolated_to_all_events": per_event_s * J,
            "speedup_over_scipy_loop": per_event_s * J / (ms * 1e-3),
            "exact_p_bit_identical_to_scipy": True, "max_rel_normal_p_err_vs_scipy": p_err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=9)
    ap.add_argument("--slice", type=int, default=2000, help="events in the timed scipy loop (300 for 12 pairs)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.calls < 5:
        raise SystemExit("--calls must be at least 5")
    ops.require_cuda()
    dev = torch.device("cuda", 0)
    info = card()
    copy_gbs = ops.probe_copy(1 << 30, dev)
    shapes = []
    ps = torch.round(ps_matrix(400_000, 1000, SEED, SEED + 1, dev), decimals=3)
    shapes.append(shape("400k x 1,000 (configs[1], 3 decimals) as 500 pairs; rank sum 500 / 500", ps, args.calls,
                        copy_gbs, args.slice, with_ranksum=True))
    del ps
    shapes.append(shape("400k x 100 uniform float32 as 50 pairs (untied)", uniform(400_000, 100, SEED + 20, None, dev),
                        args.calls, copy_gbs, args.slice))
    shapes.append(shape("400k x 24 uniform, 2 decimals, as 12 pairs (tied)", uniform(400_000, 24, SEED + 21, 2, dev),
                        args.calls, copy_gbs, min(args.slice, 300)))
    shapes.append(shape("200k x 64 (pairwise width) as 32 pairs", ps_matrix(200_000, 64, SEED + 7, SEED + 8, dev),
                        args.calls, copy_gbs, args.slice))
    res = {"tool": "tools/signedrank_bench.py", **info,
           "timing": f"median of {args.calls} per-call CUDA-event times after two warm-up calls (K8 and K6 "
                     "alternating on the first shape); scipy loop: host wall clock, one process on one core",
           "method_codes": "0 untested, 1 exact count (exact null or sign-flip enumeration), 2 normal approximation",
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
