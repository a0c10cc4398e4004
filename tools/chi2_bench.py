"""Time sd_chi2_pairwise (pairwise --chi2) on the configs[2] inputs of bench.py (200,000 junctions x
64 samples = 2,016 pairs, built as bench.py builds them) and print one JSON line: the median CUDA-event
kernel time, tests/s, bytes written per kernel time against sd_probe_copy from the same run, the
fraction of tables scipy would refuse (zero margins), the Fisher kernel on the same inputs, and
chi2 + per-column Benjamini-Hochberg.  ``--out FILE`` also writes the line to FILE."""
import argparse
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from splicedice_b200 import ops, synth            # noqa: E402

SEED = 20261018                                   # bench.py's seed; configs[2] draws from SEED + 7, + 8, + 9


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--junctions", type=int, default=200_000)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--calls", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.calls < 5:
        raise SystemExit("--calls must be at least 5")
    ops.require_cuda()
    dev = torch.device("cuda", 0)
    J, S = args.junctions, args.samples
    cl = ops.cluster_build(*synth.junction_arrays(J, SEED + 7)[:4], device=dev)
    inc = (ops.synth_counts(SEED + 8, 0, J, S, logical_cols=S, device=dev) +
           ops.synth_counts(SEED + 9, 0, J, S, logical_cols=S, device=dev))
    exc = ops.quant_ps(inc, cl["row_ptr"], cl["col_idx"], want_f32=False, want_exc=True)["exc"]
    pa, pb = ops.all_pairs(S)
    d_pa, d_pb = torch.from_numpy(pa).to(dev), torch.from_numpy(pb).to(dev)
    P = len(pa)
    tests = J * P
    out = torch.empty((J, P), dtype=torch.float64, device=dev)   # 3.2 GB: far beyond the 126 MB L2

    refused = torch.full((1,), -1, dtype=torch.int64, device=dev)
    ops.chi2_pairwise(inc, exc, d_pa, d_pb, out=out, refused=refused)        # warm-up
    ops.chi2_pairwise(inc, exc, d_pa, d_pb, out=out)
    chi2_ms = timed(lambda: ops.chi2_pairwise(inc, exc, d_pa, d_pb, out=out, refused=refused), args.calls)
    chi2_null_ms = timed(lambda: ops.chi2_pairwise(inc, exc, d_pa, d_pb, out=out), args.calls)

    # refused / all-zero fractions, counted with torch in row blocks (not timed)
    n_refused = n_zero = 0
    for r0 in range(0, J, 20_000):
        i, e = inc[r0:r0 + 20_000].long(), exc[r0:r0 + 20_000]
        a, b, c, d = i[:, d_pa], i[:, d_pb], e[:, d_pa], e[:, d_pb]
        n = a + b + c + d
        margin0 = ((a + b) == 0) | ((c + d) == 0) | ((a + c) == 0) | ((b + d) == 0)
        n_zero += int((n == 0).sum())
        n_refused += int((margin0 & (n > 0)).sum())
    nan = int(torch.isnan(out).sum())
    if nan != n_refused + n_zero:
        raise SystemExit(f"NaN count {nan} != refused {n_refused} + all-zero {n_zero}")

    def chi2_bh():
        ops.chi2_pairwise(inc, exc, d_pa, d_pb, out=out)
        ops.bh_adjust(out, "pairwise", out=out)
    chi2_bh()
    chi2_bh_ms = timed(chi2_bh, args.calls)

    bound = int((inc.long() + exc).max())
    ops.fisher_pairwise(inc, exc, d_pa, d_pb, out=out, max_cell_bound=bound)
    fisher_ms = timed(lambda: ops.fisher_pairwise(inc, exc, d_pa, d_pb, out=out, max_cell_bound=bound), args.calls)

    copy_gbs = ops.probe_copy(1 << 30, dev)
    fp64_gflops = ops.probe_fp64(dev)
    written = tests * 8
    write_gbs = written / (chi2_ms * 1e-3) / 1e9
    res = {"tool": "tools/chi2_bench.py", **card(),
           "workload": f"pairwise --chi2 on configs[2]: {J} junctions x {S} samples ({P} pairs), seed {SEED}",
           "timing": f"median of {args.calls} per-call CUDA-event times after a warm-up",
           "chi2_kernel_ms": chi2_ms, "chi2_kernel_ms_without_refusal_tracking": chi2_null_ms,
           "tests_per_s": tests / (chi2_ms * 1e-3),
           "bytes_written": written, "write_gbs": write_gbs,
           "copy_probe_gbs": copy_gbs, "copy_probe_note": "sd_probe_copy: device-to-device copy, read + write bytes",
           "write_frac_of_copy_probe": write_gbs / copy_gbs,
           "fp64_probe_gflops": fp64_gflops,
           "refused_fraction": n_refused / tests, "all_zero_fraction": n_zero / tests,
           "first_refused": int(refused.item()),
           "fisher_kernel_ms": fisher_ms, "fisher_over_chi2": fisher_ms / chi2_ms,
           "chi2_plus_bh_pairwise_ms": chi2_bh_ms}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
