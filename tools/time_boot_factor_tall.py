"""The exact bootstrap of BASELINE config 5 at its per-GPU shape, direct against factored, alternated in one process on
one GPU: mct, 4 groups x 50 subjects x 6 conditions (N = 1200), 10^6 voxels, K = 24, X resident (9.6 GB, larger than
L2), draws of resample.bootstrap_indices.

    direct_1250   -- pack + moment GEMM over 1250 bootstraps (one rank's share at 8 GPUs) + finalize
    direct_10000  -- the same over all 10 000 bootstraps (the whole job on one GPU)
    factored      -- draw counts of the 10 000 bootstraps + their Gram matrix + one-CTA factor + pack + moment GEMM
                     over the ns - G = 196 pseudo-resamples + finalize (boot_algo="collapsed")

    python tools/time_boot_factor_tall.py [--reps 3] [--out profiles/time_boot_factor_tall_r07.json]

Records CUDA-event times of each stage and of its GEMM launch, the flops each needs (2 p N K x resamples) with the
resulting TFLOP/s and share of the measured DGEMM figure (profiles/FP64_PEAKS.json), the largest relative differences
of std_errs / boot_ratios of the factored stage against direct_10000 (the same draws), per-kernel device times of one
factored stage from torch.profiler in a separate run, boot_factor_kernel alone at J = 196 and at J = 118 (the largest
factor of tests/test_gpu_boot_factor_tall.py), and the GPU's name, power limit and NVML clocks read in the same run.
X is drawn on the device (seeded), so that the 9.6 GB never cross PCIe."""
import argparse
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.time_collapsed import DGEMM_TFLOPS, gpu_info  # noqa: E402

GROUPS, C, P, NBOOT, SHARE = (50, 50, 50, 50), 6, 1_000_000, 10_000, 1250


def _events_ms(fn, n=1):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def factor_kernel_ms(groups, C, nboot, launches=20):
    """boot_factor_kernel alone (CUDA events over `launches` launches) for the draws of one design: J = ns - G."""
    import torch
    from plspy_b200 import bootstrap_permutation as bp, resample
    from plspy_b200.engine import Engine
    co = np.array([[n] * C for n in groups])
    N = int(co.sum())
    eng = Engine(torch.zeros(N, 256, dtype=torch.float64, device="cuda"))
    U = np.linalg.qr(np.random.RandomState(0).standard_normal((len(groups) * C, len(groups) * C)))[0]
    np.random.seed(5)
    idx = eng.to_device(resample.bootstrap_indices("mct", nboot, co)[0], torch.int32)
    plan = bp._factor_plan(eng, "mct", U, None, co, 0, nboot, None)
    Mg = eng.boot_count_gram(idx, plan["layout"])
    gstart = eng.to_device(plan["gstart"], torch.int32)
    eng.boot_factor(Mg, nboot, gstart)                                      # warm-up
    ms, _ = _events_ms(lambda: eng.boot_factor(Mg, nboot, gstart), launches)
    return {"J": sum(groups) - len(groups), "ms_per_launch": ms, "launches": launches}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_boot_factor_tall_r07.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_boot_factor_tall.py needs a CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from plspy_b200 import bootstrap_permutation as bp, resample
    from plspy_b200.engine import Engine
    from tools._clocks import Clocks
    try:
        clk = Clocks(0); clk.start()
    except Exception:  # noqa: BLE001  (NVML missing: nvidia-smi's snapshot below still names the card)
        clk = None
    rec = {"gpu_before": gpu_info()}

    dev = torch.device("cuda", 0)
    co = np.array([[n] * C for n in GROUPS])
    G, ns, N = len(GROUPS), sum(GROUPS), int(co.sum())
    gen = torch.Generator(device=dev).manual_seed(20260007)
    X = torch.randn(N, P, dtype=torch.float64, device=dev, generator=gen)
    X[:GROUPS[0] * C, : P // 20] += 0.5                                    # an effect in the first group
    eng = Engine(X)
    # the mct analysis (mctype 0) on the device: M = Lop X (24 x p), U s V^T = M through the 24 x 24 Gram matrix
    Lop, _, _ = bp._task_operators("mct", co, 0, np.eye(G * C), None)
    M = torch.from_numpy(Lop).to(dev) @ X
    w, U = torch.linalg.eigh(M @ M.T)
    order = torch.argsort(w, descending=True)
    w, U = w[order].clamp_min(0), U[:, order]
    s = w.sqrt()
    live_t = s > 1e-8 * s.max()
    V = (M.T @ U) / torch.where(live_t, s, torch.ones_like(s))
    del M
    U_h, s_h = U.cpu().numpy(), s.cpu().numpy()
    _, _, E = bp._task_operators("mct", co, 0, U_h, None)
    K = E.shape[1]
    numer = V * s
    np.random.seed(1234)
    idx = eng.to_device(resample.bootstrap_indices("mct", NBOOT, co)[0], torch.int32)
    idx_share = idx[:SHARE].contiguous()
    plan = bp._factor_plan(eng, "mct", U_h, None, co, 0, NBOOT, None)
    zeros = torch.zeros(eng.p, K, dtype=torch.float64, device=dev)
    routes = {
        "direct_1250": lambda: eng.boot_finalize(*eng.boot_moments(E, idx_share, pivot=numer), SHARE, numer=numer),
        "direct_10000": lambda: eng.boot_finalize(*eng.boot_moments(E, idx, pivot=numer), NBOOT, numer=numer),
        "factored": lambda: eng.boot_finalize(zeros, bp._collapsed_sumsq(eng, E, idx, NBOOT, 0, NBOOT, factor=plan),
                                              NBOOT, numer=numer),
    }
    resamples = {"direct_1250": SHARE, "direct_10000": NBOOT, "factored": ns - G}

    def timed(fn):
        eng.kernel_events = {}
        return _events_ms(fn)

    for name in ("direct_1250", "factored"):         # warm-up: module loads, allocator (direct_10000: same kernels)
        timed(routes[name])
    stage = collections.defaultdict(list)
    gemm = collections.defaultdict(list)
    outs = {}
    for _ in range(args.reps):
        for name, fn in routes.items():
            t, outs[name] = timed(fn)
            stage[name].append(t)
            gemm[name].append(sum(eng.kernel_ms("boot_moments")))
            outs[name] = tuple(o.cpu().numpy() for o in outs[name])
    eng.kernel_events = None
    live = live_t.cpu().numpy()

    def rel(x, y):
        return float(np.max(np.abs(x[:, live] - y[:, live]) / np.maximum(np.abs(y[:, live]), 1e-300)))

    med = lambda v: float(np.median(v))   # noqa: E731
    flops = {k: 2.0 * P * N * K * r for k, r in resamples.items()}
    rec["workload"] = (f"mct PLS mctype=0, {G} groups x {GROUPS[0]} subj x {C} cond (N={N}, ns={ns}) x {P} voxels, "
                       f"K={K}, {NBOOT} bootstraps; X resident ({X.numel() * 8 / 1e9:.1f} GB)")
    rec["resamples_in_gemm"] = resamples
    rec["stage_ms"] = {k: {"median": med(v), "all": [round(x, 3) for x in v]} for k, v in stage.items()}
    rec["gemm_launch_ms"] = {k: {"median": med(v), "all": [round(x, 3) for x in v]} for k, v in gemm.items()}
    rec["gemm_flops"] = flops
    rec["gemm_tflops"] = {k: flops[k] / med(gemm[k]) / 1e9 for k in routes}
    rec["gemm_fraction_of_dgemm"] = {k: flops[k] / med(gemm[k]) / 1e9 / DGEMM_TFLOPS for k in routes}
    rec["dgemm_tflops"] = DGEMM_TFLOPS
    rec["stage_speedup_of_factored"] = {k: med(stage[k]) / med(stage["factored"]) for k in ("direct_1250",
                                                                                           "direct_10000")}
    rec["factored_max_rel_diff_vs_direct_10000"] = {"std_errs": rel(outs["factored"][0], outs["direct_10000"][0]),
                                                    "boot_ratios": rel(outs["factored"][1], outs["direct_10000"][1]),
                                                    "live_lvs": int(live.sum())}
    if clk is not None:
        rec["clocks_under_load"] = clk.summary(stop=False)

    # per-kernel device times of one factored stage and one direct_1250 stage (runs of their own: tracing slows the
    # host), and the GEMM kernel's rate from them (the launch times above include the image of X)
    from torch.profiler import ProfilerActivity, profile
    for name in ("factored", "direct_1250"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            routes[name]()
            torch.cuda.synchronize()
        kern = collections.defaultdict(float)
        for evt in prof.key_averages():
            if evt.device_type == torch.autograd.DeviceType.CUDA:
                t = getattr(evt, "device_time_total", None)
                kern[evt.key.replace("void ", "").replace("plsb::", "").split("(")[0]] += \
                    (t if t is not None else evt.cuda_time_total) / 1e3
        rec[f"{name}_kernels_ms_profiler"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]))
        gk = sum(v for k, v in kern.items() if k.startswith("boot_moments_os_kernel"))
        rec[f"{name}_gemm_kernel_profiler"] = {"ms": gk, "tflops": flops[name] / gk / 1e9 if gk else None,
                                               "fraction_of_dgemm": flops[name] / gk / 1e9 / DGEMM_TFLOPS if gk
                                               else None}
    del routes, outs, X, eng, idx, idx_share, V, numer, zeros
    torch.cuda.empty_cache()

    rec["boot_factor_kernel"] = [factor_kernel_ms(GROUPS, C, NBOOT), factor_kernel_ms((60, 60), 3, 130)]
    rec["gpu_after"] = gpu_info()
    if clk is not None:
        rec["clocks_whole_run"] = clk.summary()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
