"""Direct vs collapsed exact bootstrap (boot_algo="direct" / "collapsed") at the benchmark workload and at the cfg-3
shape, alternated in one process on one GPU.

    python tools/time_collapsed.py [--reps 5] [--calls 3] [--out profiles/time_collapsed_r03.json]

Per shape it records CUDA-event times of the bootstrap stage (direct: coefficient pack + moment GEMM + finalize;
collapsed: covariance build + quadratic form + finalize), of the covariance build and of the two GEMM kernels alone,
wall times of whole plspy_b200.PLS(...) calls in both modes, the algorithmic flops of each formulation with the
resulting TFLOP/s and share of the measured DGEMM figure (profiles/FP64_PEAKS.json), the largest relative difference
between the modes' std_errs / boot_ratios, and the GPU's name, power limit and SM clock read in the same run.
Inputs: bench.make_data() (seeded); X resident on the device for the stage timings (480 MB, larger than L2)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DGEMM_TFLOPS = json.load(open(os.path.join(ROOT, "profiles", "FP64_PEAKS.json")))["fp64_cublas_dgemm_tflops"]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {"nvidia-smi": "unavailable"}


def run_shape(method, groups, C, p, nboot, reps, calls, contrasts=None):
    import torch
    import bench
    import oracle.pls_oracle as po
    import plspy_b200
    from plspy_b200 import bootstrap_permutation as bp, resample
    from plspy_b200.engine import Engine

    X = bench.make_data(groups=groups, C=C, p=p)
    co = np.array([[n] * C for n in groups])
    N = X.shape[0]
    a = po.analysis(method, X, groups, C, contrasts=contrasts, mctype=0)
    _, _, E = bp._task_operators(method, co, 0, a["U"], a.get("contrast"))
    K = E.shape[1]
    np.random.seed(1234)
    idx_h = resample.bootstrap_indices(method, nboot, co)[0]
    dev = torch.device("cuda", 0)
    eng = Engine(torch.from_numpy(X).to(dev))
    eng.kernel_events = {}
    idx = eng.to_device(idx_h, torch.int32)
    V = eng.to_device(a["V"], torch.float64)
    numer = V * eng.to_device(a["s"], torch.float64) if method == "mct" else V

    def direct():
        s1, s2 = eng.boot_moments(E, idx, pivot=numer)
        return eng.boot_finalize(s1, s2, nboot, numer=numer)

    def collapsed():
        s2 = bp._collapsed_sumsq(eng, E, idx, nboot, 0, nboot)
        return eng.boot_finalize(torch.zeros_like(s2), s2, nboot, numer=numer)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); out = fn(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for fn in (direct, collapsed):                      # warm-up: module loads, allocator
        timed(fn)
    eng.kernel_events = {}
    stage = {"direct": [], "collapsed": [], "cov_build": []}
    for _ in range(reps):
        t, out_d = timed(direct); stage["direct"].append(t)
        t, out_c = timed(collapsed); stage["collapsed"].append(t)
        t, _ = timed(lambda: eng.boot_cov(E, idx)); stage["cov_build"].append(t)
    kern = {"boot_moments": eng.kernel_ms("boot_moments"), "boot_quad": eng.kernel_ms("boot_quad")}
    (se_d, br_d), (se_c, br_c) = [eng.to_host(*o) for o in (out_d, out_c)]
    live = np.abs(a["s"]) > 1e-8 * np.abs(a["s"]).max()

    def rel(x, y):
        return float(np.max(np.abs(x[:, live] - y[:, live]) / np.maximum(np.abs(y[:, live]), 1e-300)))

    # whole PLS(...) calls, alternated (host analysis, index draws, upload of X, permutations, bootstraps)
    kw = dict(num_perm=nboot, num_boot=nboot, pls_method=method, mctype=0)
    if contrasts is not None:
        kw["contrasts"] = contrasts
    wall = {"direct": [], "collapsed": []}
    for rep in range(calls + 1):
        for algo in ("direct", "collapsed"):
            np.random.seed(99)
            torch.cuda.synchronize(); t0 = time.perf_counter()
            plspy_b200.PLS(X, groups, C, boot_algo=algo, **kw)
            torch.cuda.synchronize()
            if rep:
                wall[algo].append(time.perf_counter() - t0)

    med = lambda v: float(np.median(v)) if v else float("nan")   # noqa: E731
    f_direct = 2.0 * p * N * K * nboot
    f_quad = 2.0 * p * N * N * K
    f_cov = 2.0 * N * N * K * nboot
    t_mom, t_quad = med(kern["boot_moments"]), med(kern["boot_quad"])
    return {
        "workload": f"{method} PLS mctype=0, {len(groups)} groups x {groups[0]} subj x {C} cond (N={N}) x {p} voxels, "
                    f"K={K}, {nboot} bootstraps (stage) / {nboot} perm + {nboot} boot (whole call)",
        "stage_ms": {k: {"median": med(v), "all": [round(x, 3) for x in v]} for k, v in stage.items()},
        "kernel_ms": {"boot_moments_kernel": {"median": t_mom, "all": [round(x, 3) for x in kern["boot_moments"]]},
                      "boot_quad_kernel": {"median": t_quad, "all": [round(x, 3) for x in kern["boot_quad"]]}},
        "stage_speedup": med(stage["direct"]) / med(stage["collapsed"]),
        "cov_build_over_quad_kernel": med(stage["cov_build"]) / t_quad,
        "pls_call_s": {k: {"median": med(v), "all": [round(x, 4) for x in v]} for k, v in wall.items()},
        "flops": {"direct_2pNKB": f_direct, "collapsed_quad_2pN2K": f_quad, "collapsed_cov_2N2KB": f_cov,
                  "ratio_direct_over_collapsed": f_direct / (f_quad + f_cov)},
        "tflops": {"boot_moments_kernel": f_direct / t_mom / 1e9, "boot_quad_kernel": f_quad / t_quad / 1e9},
        "fraction_of_dgemm": {"dgemm_tflops": DGEMM_TFLOPS,
                              "boot_moments_kernel": f_direct / t_mom / 1e9 / DGEMM_TFLOPS,
                              "boot_quad_kernel": f_quad / t_quad / 1e9 / DGEMM_TFLOPS},
        "max_rel_diff_collapsed_vs_direct": {"std_errs": rel(se_c, se_d), "boot_ratios": rel(br_c, br_d),
                                             "live_lvs": int(live.sum())},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_collapsed_r03.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_collapsed.py needs a CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from tools._clocks import Clocks
    try:
        clk = Clocks(0); clk.start()
    except Exception:  # noqa: BLE001  (NVML missing: nvidia-smi's snapshot below still names the card)
        clk = None
    rec = {"gpu_before": gpu_info()}
    rec["bench_mct"] = run_shape("mct", (25, 25, 25), 4, 200_000, 5000, args.reps, args.calls)
    contrasts = np.linalg.qr(np.random.RandomState(3).standard_normal((12, 3)))[0]
    rec["cfg3_cst"] = run_shape("cst", (25, 25, 25), 4, 200_000, 5000, args.reps, args.calls,
                                contrasts=contrasts)
    rec["gpu_after"] = gpu_info()
    rec["clocks_under_load"] = clk.summary() if clk is not None else None
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) or "stage_ms" not in v else
                          {kk: v[kk] for kk in ("stage_ms", "kernel_ms", "stage_speedup", "tflops",
                                                "fraction_of_dgemm", "max_rel_diff_collapsed_vs_direct",
                                                "cov_build_over_quad_kernel", "pls_call_s")})
                      for k, v in rec.items()}, indent=1))


if __name__ == "__main__":
    main()
