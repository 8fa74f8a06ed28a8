"""Cost of the bias-corrected salience intervals against the plain percentile intervals, in one process on one GPU.

    python tools/time_percentile_bc.py [--p 200000] [--R 5000] [--reps 7] [--out FILE]

The streamed salience intervals of the mct bench shape: 300 rows x p voxels (X is 480 MB at p = 200 000, larger than
the L2), K = 12, R bootstraps -- 2.4 M series of 5000.  `Engine.salience_percentiles` (plain) and
`Engine.salience_percentiles_bc` (bias-corrected, `prop` too) run the same chunk loop over the explicit salience chunks;
only the percentile kernel differs (one binary search and four normal-distribution evaluations per series).
1. Whole calls, the two alternated rep by rep after one warm-up each: CUDA events around a call; median / min / max.
2. Kernel times from torch.profiler in a phase of its own (mean per launch and total per call, both variants).
The GPU's name, power limit and clocks are recorded with the numbers.  Data: seeded standard normal."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.time_collapsed import gpu_info  # noqa: E402


def _kernels(fn, reps):
    """Per-call device time (us) of every kernel `fn` launches, and its launches per call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    rows = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.count > 0 and "kernel" in e.key:
            rows[e.key.split("(")[0].replace("void ", "")] = {"us_per_call": round(t / reps, 1),
                                                              "launches_per_call": e.count / reps,
                                                              "us_per_launch": round(t / e.count, 2)}
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--p", type=int, default=200_000)
    ap.add_argument("--R", type=int, default=5000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from plspy_b200.engine import Engine
    N, K, p, R = 300, 12, a.p, a.R
    rs = np.random.RandomState(0)
    eng = Engine(rs.standard_normal((N, p)))
    E = eng.to_device(rs.standard_normal((N, K)) / np.sqrt(N), torch.float64)
    idx = eng.to_device(rs.randint(0, N, size=(R, N)).astype(np.int32), torch.int32)
    ident = eng.to_device(np.arange(N, dtype=np.int32)[None, :], torch.int32)
    orig = eng.salience(E, ident)[0]                       # the salience of the undrawn rows: p x K
    conf = (0.025, 0.975)
    fns = {"plain": lambda: eng.salience_percentiles(E, idx, conf),
           "bias_corrected": lambda: eng.salience_percentiles_bc(E, idx, orig, conf)}

    def timed(fn):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    outs = {k: timed(fn)[1] for k, fn in fns.items()}      # warm-up; keeps one result of each
    ts = {k: [] for k in fns}
    for _ in range(a.reps):
        for k, fn in fns.items():
            ts[k].append(timed(fn)[0])
    whole = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "reps_ms": v}
             for k, v in ts.items()}
    lo, hi = outs["plain"]
    blo, bhi, prop = outs["bias_corrected"]
    kern = {k: _kernels(fn, 2) for k, fn in fns.items()}

    def pc_us(k):
        return sum(v["us_per_call"] for name, v in kern[k].items() if "percentile_kernel" in name)
    rec = {
        "shape": {"N": N, "p": p, "K": K, "R": R, "series": p * K, "x_bytes": N * p * 8},
        "gpu": gpu_info(),
        "whole_call": whole,
        "whole_call_extra_pct": 100.0 * (whole["bias_corrected"]["median_ms"] / whole["plain"]["median_ms"] - 1.0),
        "kernels": kern,
        "percentile_kernel_ms_per_call": {k: pc_us(k) / 1e3 for k in fns},
        "percentile_kernel_extra_pct": 100.0 * (pc_us("bias_corrected") / pc_us("plain") - 1.0),
        "check": {"prop_mean": float(prop.mean()), "nan_bounds": int(torch.isnan(blo).sum() + torch.isnan(bhi).sum()),
                  "plain_width_mean": float((hi - lo).mean()), "bc_width_mean": float((bhi - blo).nanmean())},
    }
    line = json.dumps(rec, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
