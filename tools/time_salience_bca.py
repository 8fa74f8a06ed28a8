"""Cost of the BCa salience intervals against the bias-corrected ones, in one process on one GPU.

    python tools/time_salience_bca.py [--p 200000] [--nboot 5000] [--reps 3] [--out FILE]

Two shapes: the bench task workload (mct, groups (25, 25, 25) x 4 conditions x p voxels, K = 12) and cfg 3 (cst,
3 x 25 subjects x 4 conditions x p voxels, 3 contrasts), nboot bootstraps each, X float64 (480 MB at p = 200 000,
larger than the L2).  `salience_bias_corrected_intervals()` and `salience_bca_intervals()` run the same chunk loop over
the explicit bootstrap salience chunks (default budget, 4 GiB); BCa adds per chunk the jackknife pass over the voxel
window of X (75 subjects), the acceleration kernel and the BCa levels in the sort, and once per call the host build of
the jackknife coefficients.
1. Whole result-side calls (host arrays out), the two alternated rep by rep after one warm-up each, each timed on the
   host around a call that ends in a device synchronise; median / min / max.
2. Kernel times from torch.profiler in a phase of its own: per call, and per chunk for the jackknife pass and the
   acceleration kernel.
The GPU's name, power limit and SM clocks are read in the same call (nvidia-smi, and NVML sampled during phase 1)."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools._clocks import Clocks  # noqa: E402
from tools.time_collapsed import gpu_info  # noqa: E402
from tools.time_percentile_bc import _kernels  # noqa: E402

SHAPES = {
    "bench_mct": dict(method="mct", groups=(25, 25, 25), C=4),
    "cfg3_cst": dict(method="cst", groups=(25, 25, 25), C=4, ncontrast=3),
}


def run_shape(name, p, nboot, reps):
    import torch
    import bench
    import plspy_b200
    sh = SHAPES[name]
    groups, C = sh["groups"], sh["C"]
    X = bench.make_data(groups=groups, C=C, p=p)
    kw = {}
    if sh["method"] == "cst":
        kw["contrasts"] = np.random.RandomState(3).standard_normal((len(groups) * C, sh["ncontrast"]))
    np.random.seed(1234)
    res = plspy_b200.PLS(X, groups, C, num_perm=0, num_boot=nboot, pls_method=sh["method"], **kw)
    rt = res.resample_tests
    K = int(rt.boot_ratios.shape[1])
    J, N = sum(groups), X.shape[0]
    fns = {"bias_corrected": rt.salience_bias_corrected_intervals, "bca": rt.salience_bca_intervals}

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0), out

    outs = {k: timed(fn)[1] for k, fn in fns.items()}       # warm-up; keeps one result of each
    clocks = Clocks()
    clocks.start()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            ts[k].append(timed(fn)[0])
    clk = clocks.summary()
    whole = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "reps_ms": v}
             for k, v in ts.items()}
    kern = {k: _kernels(fn, 1) for k, fn in fns.items()}
    jack = {n: v for n, v in kern["bca"].items() if "12, true, true" in n or "jack_accel" in n}
    chunks = max(int(v["launches_per_call"]) for n, v in jack.items())
    flops = 2.0 * p * N * K * J
    jt = sum(v["us_per_call"] for n, v in jack.items() if "salience_kernel" in n)
    lo, hi, prop, accel = outs["bca"]
    bprop = outs["bias_corrected"][2]
    live = np.isfinite(lo) & np.isfinite(hi)
    return {
        "shape": {"method": sh["method"], "groups": groups, "C": C, "N": N, "p": p, "K": K, "nboot": nboot,
                  "subjects_J": J, "x_bytes": N * p * 8},
        "whole_call": whole,
        "whole_call_extra_pct": 100.0 * (whole["bca"]["median_ms"] / whole["bias_corrected"]["median_ms"] - 1.0),
        "clocks_during_whole_calls": clk,
        "kernels": kern,
        "jackknife": {"chunks": chunks, "flops": flops,
                      "pass_ms_per_call": jt / 1e3, "pass_ms_per_chunk": jt / 1e3 / chunks,
                      "pass_tflops": flops / (jt * 1e-6) / 1e12 if jt > 0 else None,
                      "accel_ms_per_call": sum(v["us_per_call"] for n, v in jack.items() if "jack_accel" in n) / 1e3},
        "check": {"prop_equal_to_bc": bool(np.array_equal(prop, bprop, equal_nan=True)),
                  "accel_abs_mean": float(np.nanmean(np.abs(accel))), "accel_abs_max": float(np.nanmax(np.abs(accel))),
                  "finite_bounds_share": float(live.mean())},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--p", type=int, default=200_000)
    ap.add_argument("--nboot", type=int, default=5000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rec = {"gpu": gpu_info(), "shapes": {}}
    for name in a.shapes.split(","):
        rec["shapes"][name] = run_shape(name, a.p, a.nboot, a.reps)
        print(name, json.dumps({k: rec["shapes"][name][k] for k in ("whole_call_extra_pct", "jackknife")}), flush=True)
    rec["gpu_after"] = gpu_info()
    line = json.dumps(rec, indent=1, default=float)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
