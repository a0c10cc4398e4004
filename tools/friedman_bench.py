"""Time sd_friedman_rows (compare_repeated) on two shapes, with sd_kruskal_rows (compare_conditions) on the
same columns as groups, and print one JSON line:

  * 400,000 events x 1,000 samples: float32 PS of bench.py's configs[1] (synth counts -> quant_ps, seed
    SEED / SEED + 1) as 250 subjects x 4 conditions (column c: subject c // 4, condition c % 4); K7 takes
    the same columns as 4 groups of 250 (column c in group c % 4).  1.6 GB of PS, far beyond the 126 MB
    L2, so every pass reads it from HBM;
  * 200,000 x 64 as 16 subjects x 4 conditions (the pairwise width; junctions SEED + 7, counts SEED + 8).
    51 MB of PS fits in the L2, so after the first call this shape reads mostly from there.

These are tools/ranksum_bench.py's matrices.  Per shape: the median CUDA-event time of each library call
after two warm-up calls (the two alternate call by call; device column lists built once), events/s, the
HBM floor (bytes read + written over sd_probe_copy's rate from the same run) and kernel / floor, and the
scipy.stats.friedmanchisquare loop on the first ~2,000 events timed on this host in the same run (one
core: the loop is serial), with the kernel's Q on those events checked bit for bit against the exact
fraction oracle and within 1e-13 of scipy's scale, and p against chdtrc.  ``--out FILE`` also writes
the line."""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np
import torch
from scipy.special import chdtrc
from scipy.stats import friedmanchisquare

sys.path.insert(0, ".")
from splicedice_b200 import native, ops                       # noqa: E402
from tests import friedman_cases as cases                     # noqa: E402
from tools.kruskal_bench import timed_pair                    # noqa: E402
from tools.ranksum_bench import SEED, card, ps_matrix          # noqa: E402


def scipy_loop(ps_host, blocks):
    """(seconds per event, Q) of scipy.stats.friedmanchisquare(..., nan_policy='omit') over the rows of
    ps_host"""
    q = np.full(len(ps_host), np.nan)
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for j, row in enumerate(ps_host):
            try:
                q[j] = friedmanchisquare(*row[blocks].T, nan_policy="omit")[0]
            except ValueError:
                pass
    return (time.perf_counter() - t0) / len(ps_host), q


def shape(label, J, S, k, junction_seed, count_seed, calls, copy_gbs, slice_rows, dev, l2_note):
    ps = ps_matrix(J, S, junction_seed, count_seed, dev)
    nb = S // k
    blocks = np.arange(nb * k, dtype=np.int32).reshape(nb, k)          # column c: subject c // k, condition c % k
    groups = [np.arange(g, nb * k, k, dtype=np.int32) for g in range(k)]
    d_cols = torch.from_numpy(np.ascontiguousarray(blocks.T).reshape(-1)).to(dev)
    d_kw_cols = torch.from_numpy(np.concatenate(groups)).to(dev)
    d_group = torch.from_numpy(np.repeat(np.arange(k, dtype=np.int32), nb)).to(dev)
    n_fr, mean_fr, st_fr = (torch.empty(J, dtype=torch.int32, device=dev),
                            torch.empty((J, k), dtype=torch.float64, device=dev),
                            torch.empty((J, 2), dtype=torch.float64, device=dev))
    n_kw, mean_kw, st_kw = (torch.empty((J, k), dtype=torch.int32, device=dev),
                            torch.empty((J, k), dtype=torch.float64, device=dev),
                            torch.empty((J, 2), dtype=torch.float64, device=dev))
    sp = native.stream_ptr()
    # both arms are the bare library call on device lists built once, so neither times host-side checks
    # or copies (ops.friedman_rows lists the columns condition-major, as here)
    run_fr = lambda: native.call(                                       # noqa: E731
        "sd_friedman_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, k, nb, native.ptr(d_cols),
        0, J, native.ptr(n_fr), native.ptr(mean_fr), k, native.ptr(st_fr), 2, sp)
    run_kw = lambda: native.call(                                       # noqa: E731
        "sd_kruskal_rows", J, S, native.ptr(ps), ps.stride(0), native.SD_RANKSUM_F32, k, d_kw_cols.numel(),
        native.ptr(d_kw_cols), native.ptr(d_group), 0, J, native.ptr(n_kw), k, native.ptr(mean_kw), k,
        native.ptr(st_kw), 2, sp)
    for _ in range(2):
        run_fr()
        run_kw()
    ms_fr, ms_kw = timed_pair(run_fr, run_kw, calls)
    res = ops.friedman_rows(ps, blocks)
    torch.cuda.synchronize()
    if not (torch.equal(res["n"], n_fr) and torch.equal(res["Q"].view(torch.int64), st_fr[:, 0].view(torch.int64))):
        raise SystemExit(f"{label}: ops.friedman_rows differs from the timed call")
    read = J * S * ps.element_size()
    written = J * (4 + k * 8 + 2 * 8)
    floor_ms = (read + written) / (copy_gbs * 1e9) * 1e3
    rows = min(slice_rows, J)
    # scipy computes in float32 for float32 input; the kernel compares the float32 cells, whose order is
    # that of their float64 widening, so the reference is scipy on the same values as float64
    host = ps[:rows].cpu().numpy().astype(np.float64)
    per_event_s, q_ref = scipy_loop(host, blocks)
    q = res["Q"][:rows].cpu().numpy()
    p = res["p"][:rows].cpu().numpy()
    n = res["n"][:rows].cpu().numpy()
    q_exact = np.full(rows, np.nan)
    scale = np.full(rows, np.nan)                      # 3 n (k + 1) / c: scipy's Q cancels at this size
    n_ref = np.zeros(rows, dtype=np.int64)
    for j in range(rows):
        d, n_ref[j], t = cases.block_terms(host[j][blocks])
        e = cases.exact_q(d, n_ref[j], k, t)
        if e is not None:
            q_exact[j] = float(e)
            scale[j] = 3 * n_ref[j] * (k + 1) / cases.tie_factor(n_ref[j], k, t)
    if not np.array_equal(n, n_ref) or not np.array_equal(np.isnan(q), np.isnan(q_exact)):
        raise SystemExit(f"{label}: n or the NaN pattern differs from the exact oracle")
    ok = ~np.isnan(q_exact)
    q_bits = int((q[ok].view(np.uint64) != q_exact[ok].view(np.uint64)).sum())
    fin = ok & np.isfinite(q_ref)
    q_scipy = float((np.abs(q[fin] - q_ref[fin]) / scale[fin]).max(initial=0))
    want_p = chdtrc(k - 1, q[ok])
    big = want_p > 1e-300
    p_err = float((np.abs(p[ok][big] - want_p[big]) / want_p[big]).max(initial=0))
    if q_bits or q_scipy > 1e-13 or p_err > 1e-12:
        raise SystemExit(f"{label}: kernel differs (Q off the exact fraction in {q_bits} rows, vs scipy {q_scipy} "
                         f"of its scale, p rel {p_err})")
    return {"shape": label, "events": J, "samples": S, "subjects": nb, "conditions": k,
            "complete_block_fraction": float(res["n"].double().mean().item() / nb),
            "kernel_ms": ms_fr, "events_per_s": J / (ms_fr * 1e-3),
            "kruskal_same_columns_kernel_ms": ms_kw, "friedman_over_kruskal": ms_fr / ms_kw,
            "bytes_read": read, "bytes_written": written, "hbm_floor_ms": floor_ms,
            "kernel_over_floor": ms_fr / floor_ms, "cache_note": l2_note,
            "scipy_slice_events": rows, "scipy_tested_events": int(ok.sum()), "scipy_s_per_event": per_event_s,
            "scipy_loop_s_extrapolated_to_all_events": per_event_s * J,
            "speedup_over_scipy_loop": per_event_s * J / (ms_fr * 1e-3),
            "q_rows_not_bit_identical_to_exact": q_bits, "max_abs_q_err_vs_scipy_over_its_scale": q_scipy,
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
    shapes = [shape("400k x 1,000 (configs[1]), 250 subjects x 4 conditions; K7 on 4 x 250", 400_000, 1000, 4,
                    SEED, SEED + 1, args.calls, copy_gbs, args.slice, dev,
                    "1.6 GB of PS: every call reads it from HBM"),
              shape("200k x 64 (pairwise width), 16 subjects x 4 conditions; K7 on 4 x 16", 200_000, 64, 4,
                    SEED + 7, SEED + 8, args.calls, copy_gbs, args.slice, dev,
                    "51 MB of PS fits in the 126 MB L2: after the warm-up calls it is read mostly from L2, so "
                    "kernel_over_floor understates how close to the HBM floor the kernel runs")]
    res = {"tool": "tools/friedman_bench.py", **info,
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
