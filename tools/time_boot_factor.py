"""The three exact bootstrap routes of the task methods, alternated in one process on one GPU, at the benchmark workload
and at the cfg-3 shape:

    direct    -- coefficient pack + moment GEMM over the B bootstraps + finalize (boot_algo="direct")
    nxn       -- N x N covariance build + quadratic form + finalize (boot_algo="collapsed" on draws without the
                 subject structure)
    factored  -- draw counts + their Gram matrix + one-CTA factor + pack + moment GEMM over the ns - G pseudo-resamples
                 + finalize (boot_algo="collapsed", and "auto" when B > N)

    python tools/time_boot_factor.py [--reps 5] [--out profiles/time_boot_factor_r06.json]

Per shape: CUDA-event times of each stage and of its GEMM kernel alone, the flops each route needs with the resulting
TFLOP/s and share of the measured DGEMM figure (profiles/FP64_PEAKS.json), the largest relative differences of
std_errs / boot_ratios against the direct route, and the GPU's name, power limit and NVML clocks read in the same run.
Inputs: bench.make_data() (seeded); X resident on the device (480 MB, larger than L2)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.time_collapsed import DGEMM_TFLOPS, gpu_info  # noqa: E402


def run_shape(method, groups, C, p, nboot, reps, contrasts=None):
    import torch
    import bench
    import oracle.pls_oracle as po
    from plspy_b200 import bootstrap_permutation as bp, resample
    from plspy_b200.engine import Engine

    X = bench.make_data(groups=groups, C=C, p=p)
    co = np.array([[n] * C for n in groups])
    N, G, ns = X.shape[0], len(groups), sum(groups)
    a = po.analysis(method, X, groups, C, contrasts=contrasts, mctype=0)
    _, _, E = bp._task_operators(method, co, 0, a["U"], a.get("contrast"))
    K = E.shape[1]
    np.random.seed(1234)
    idx_h = resample.bootstrap_indices(method, nboot, co)[0]
    eng = Engine(torch.from_numpy(X).to(torch.device("cuda", 0)))
    idx = eng.to_device(idx_h, torch.int32)
    V = eng.to_device(a["V"], torch.float64)
    numer = V * eng.to_device(a["s"], torch.float64) if method == "mct" else V
    plan = bp._factor_plan(eng, method, a["U"], a.get("contrast"), co, 0, nboot, idx)
    assert plan is not None

    routes = {
        "direct": lambda: eng.boot_finalize(*eng.boot_moments(E, idx, pivot=numer), nboot, numer=numer),
        "nxn": lambda: eng.boot_finalize(torch.zeros(eng.p, K, dtype=torch.float64, device=eng.device),
                                         bp._collapsed_sumsq(eng, E, idx, nboot, 0, nboot), nboot, numer=numer),
        "factored": lambda: eng.boot_finalize(torch.zeros(eng.p, K, dtype=torch.float64, device=eng.device),
                                              bp._collapsed_sumsq(eng, E, idx, nboot, 0, nboot, factor=plan), nboot,
                                              numer=numer),
    }
    kname = {"direct": "boot_moments", "nxn": "boot_quad", "factored": "boot_moments"}

    def timed(fn):
        eng.kernel_events = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); out = fn(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for fn in routes.values():                          # warm-up: module loads, allocator
        timed(fn)
    stage = {k: [] for k in routes}
    kern = {k: [] for k in routes}
    outs = {}
    for _ in range(reps):
        for name, fn in routes.items():
            t, outs[name] = timed(fn)
            stage[name].append(t)
            kern[name].append(sum(eng.kernel_ms(kname[name])))
    host = {k: eng.to_host(*v) for k, v in outs.items()}
    live = np.abs(a["s"]) > 1e-8 * np.abs(a["s"]).max()

    def rel(x, y):
        return float(np.max(np.abs(x[:, live] - y[:, live]) / np.maximum(np.abs(y[:, live]), 1e-300)))

    med = lambda v: float(np.median(v))   # noqa: E731
    flops = {"direct": 2.0 * p * N * K * nboot, "nxn": 2.0 * p * N * N * K, "factored": 2.0 * p * N * K * (ns - G)}
    rec = {"workload": f"{method} PLS mctype=0, {G} groups x {groups[0]} subj x {C} cond (N={N}, ns={ns}) x {p} "
                       f"voxels, K={K}, {nboot} bootstraps",
           "stage_ms": {k: {"median": med(v), "all": [round(x, 3) for x in v]} for k, v in stage.items()},
           "gemm_kernel_ms": {k: {"kernel": kname[k] + "_kernel", "median": med(v), "all": [round(x, 3) for x in v]}
                              for k, v in kern.items()},
           "gemm_flops": flops,
           "gemm_tflops": {k: flops[k] / med(kern[k]) / 1e9 for k in routes},
           "gemm_fraction_of_dgemm": {k: flops[k] / med(kern[k]) / 1e9 / DGEMM_TFLOPS for k in routes},
           "dgemm_tflops": DGEMM_TFLOPS,
           "stage_speedup_over_direct": {k: med(stage["direct"]) / med(stage[k]) for k in routes},
           "max_rel_diff_vs_direct": {k: {"std_errs": rel(host[k][0], host["direct"][0]),
                                          "boot_ratios": rel(host[k][1], host["direct"][1])} for k in ("nxn", "factored")},
           "live_lvs": int(live.sum())}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_boot_factor_r06.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_boot_factor.py needs a CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from tools._clocks import Clocks
    try:
        clk = Clocks(0); clk.start()
    except Exception:  # noqa: BLE001  (NVML missing: nvidia-smi's snapshot below still names the card)
        clk = None
    rec = {"gpu_before": gpu_info()}
    rec["bench_mct"] = run_shape("mct", (25, 25, 25), 4, 200_000, 5000, args.reps)
    contrasts = np.linalg.qr(np.random.RandomState(3).standard_normal((12, 3)))[0]
    rec["cfg3_cst"] = run_shape("cst", (25, 25, 25), 4, 200_000, 5000, args.reps, contrasts=contrasts)
    rec["gpu_after"] = gpu_info()
    rec["clocks_under_load"] = clk.summary() if clk is not None else None
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
