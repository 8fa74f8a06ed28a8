"""Float32-resident X (x_storage="fp32") against the float64 default, alternated in one process on one GPU.

    python tools/time_x32.py [--reps 5] [--calls 3] [--out profiles/time_x32_r04.json]

Cases: the benchmark workload (mct, 300 x 200 000, 5000 permutations + 5000 bootstraps) in the exact and the fast
mode, the same with boot_algo="collapsed", and the config-5 row count (1200 rows) at 200 000 voxels (1000 + 1000
resamples, exact mode).  Per case and storage it records torch.cuda.max_memory_allocated over a whole
plspy_b200.PLS(...) call (above what was allocated before it), the bytes of X on the device, the CUDA-event time of
every engine pass that reads X (median over --reps), the device time of each CUDA kernel inside those passes
(torch.profiler, in a phase of its own after the event timings: a pass such as the tall-design bootstrap GEMM is an
image kernel that reads X followed by a GEMM that does not), the wall time of whole calls (median over --calls), whether the
two storages gave bit-identical std_errs / boot_ratios / permute_ratio, the GPU's name, power limit and NVML clocks.
Inputs: bench.make_data() (seeded) rounded to float32, so that both storages analyse the same matrix; X is larger
than the L2 in every case."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.time_collapsed import gpu_info  # noqa: E402

CASES = [
    # name, groups, C, voxels, perms, boots, PLS keywords
    ("bench_exact", (25, 25, 25), 4, 200_000, 5000, 5000, {}),
    ("bench_fast", (25, 25, 25), 4, 200_000, 5000, 5000, {"precision": "tf32x3"}),
    ("bench_collapsed", (25, 25, 25), 4, 200_000, 5000, 5000, {"boot_algo": "collapsed"}),
    ("rows1200_exact", (100, 100, 100), 4, 200_000, 1000, 1000, {}),
]
STORAGES = ("fp64", "fp32")


def _event_ms(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(); fn(); e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def _passes(X32, groups, C, nboot, kw, storage):
    """Engine passes that read X, as {name: callable}, on an engine holding X resident in `storage`."""
    import torch
    import oracle.pls_oracle as po
    from plspy_b200 import bootstrap_permutation as bp, resample
    from plspy_b200._lib import lib
    from plspy_b200.engine import Engine
    Xw = X32.astype(np.float64)
    co = np.array([[n] * C for n in groups])
    a = po.analysis("mct", Xw, groups, C, mctype=0)
    _, _, E = bp._task_operators("mct", co, 0, a["U"], None)
    np.random.seed(1234)
    idx_h = resample.bootstrap_indices("mct", nboot, co)[0]
    eng = Engine(torch.from_numpy(X32 if storage == "fp32" else Xw).cuda(), precision=kw.get("precision", "fp64"),
                 x_storage=storage)
    idx = eng.to_device(idx_h, torch.int32)
    E = eng.to_device(E, torch.float64)
    V = eng.to_device(a["V"], torch.float64)
    N, p, x32 = eng.N, eng.p, storage == "fp32"
    t = {"xv": lambda: eng.xv(V)}
    if eng.precision == "fp64":
        t["gram_f64"] = lambda: eng.gram_of(eng.X)
    if kw.get("boot_algo") == "collapsed":
        S1, S2 = eng.boot_cov(E, idx)
        Sig = S2 - S1.T[:, :, None] * S1.T[:, None, :] / nboot
        t["boot_quad"] = lambda: eng.boot_quad(Sig)
    elif eng.precision == "tf32x3":
        split = lib.plsb200_tf32_split_x32 if x32 else lib.plsb200_tf32_split_x
        img = eng._ws(lib.plsb200_tf32_ximage_bytes(N, p))
        t["tf32_split_x"] = lambda: split(eng._xp(0), N, p, eng.ldx, img.data_ptr(), eng._stream())
        gsplit = lib.plsb200_gram_tf32_split_x32 if x32 else lib.plsb200_gram_tf32_split
        gimg = eng._ws(lib.plsb200_gram_tf32_image_bytes(N, p))
        t["gram_tf32_split"] = lambda: gsplit(eng._xp(0), N, p, eng.ldx, gimg.data_ptr(), eng._stream())
        t["boot_moments_tf32 (planes cached)"] = lambda: eng.boot_moments(E, idx)
    elif N <= 320:
        t["boot_moments_f64"] = lambda: eng.boot_moments(E, idx)          # boot_moments_kernel, A in registers
        series = lib.plsb200_salience_series_x32_f64 if x32 else lib.plsb200_salience_series_f64
        vc = 8192
        cube = eng._empty(vc, E.shape[1], nboot)
        t[f"salience_series ({vc} voxels)"] = lambda: series(eng._xp(0), N, vc, eng.ldx, E.data_ptr(), int(E.shape[1]),
                                                             idx.data_ptr(), nboot, cube.data_ptr(), eng._stream())
    else:
        t["boot_moments_f64 (os_ximage + os GEMM)"] = lambda: eng.boot_moments(E, idx)
    return eng, t


def kernel_times(X32, groups, C, nboot, kw, reps):
    """Both storages' engines side by side; every pass timed with the storages alternated, first pass = warm-up."""
    engs, fns = {}, {}
    for s in STORAGES:
        engs[s], fns[s] = _passes(X32, groups, C, nboot, kw, s)
    ms = {s: {k: [] for k in fns[s]} for s in STORAGES}
    for rep in range(reps + 1):
        for k in fns["fp64"]:
            for s in STORAGES:
                t = _event_ms(fns[s][k])
                if rep:
                    ms[s][k].append(t)
    out = {s: {k: {"median_ms": float(np.median(v)), "all_ms": [round(x, 4) for x in v]} for k, v in ms[s].items()}
           for s in STORAGES}
    for s in STORAGES:
        out[s]["x_on_device_bytes"] = engs[s].X.numel() * engs[s].X.element_size()
        out[s]["kernels_us"] = kernel_profile(fns[s], reps)
    return out


def kernel_profile(fns, reps):
    """Mean device time (us) of every CUDA kernel launched by each pass, from torch.profiler over `reps` calls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for k, fn in fns.items():
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
                rows[e.key.split("(")[0].replace("void ", "")] = round(t / e.count, 2)
        out[k] = rows
    return out


def whole_calls(X32, groups, C, nperm, nboot, kw, calls):
    import torch
    import plspy_b200
    Xw = X32.astype(np.float64)
    wall = {s: [] for s in STORAGES}
    peak = {s: [] for s in STORAGES}
    res = {}
    for rep in range(calls + 1):
        for s in STORAGES:
            np.random.seed(99)
            torch.cuda.synchronize(); torch.cuda.empty_cache()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            t0 = time.perf_counter()
            r = plspy_b200.PLS(Xw if s == "fp64" else X32, groups, C, num_perm=nperm, num_boot=nboot,
                               pls_method="mct", x_storage=s, **kw)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            peak[s].append(int(torch.cuda.max_memory_allocated() - base))
            if rep:
                wall[s].append(dt)
            res[s] = r.resample_tests
            del r
    same = {f: bool(np.array_equal(getattr(res["fp32"], f), getattr(res["fp64"], f)))
            for f in ("std_errs", "boot_ratios", "permute_ratio")}
    return ({s: {"median_s": float(np.median(v)), "all_s": [round(x, 4) for x in v]} for s, v in wall.items()},
            {s: max(v) for s, v in peak.items()}, same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_x32_r04.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_x32.py needs a CUDA device")
    import bench
    from tools._clocks import Clocks
    clocks = Clocks()
    clocks.start()
    out = {"gpu": gpu_info(), "cases": {}}
    for name, groups, C, p, nperm, nboot, kw in CASES:
        if name not in args.cases.split(","):
            continue
        X32 = bench.make_data(groups=groups, C=C, p=p).astype(np.float32)
        mark = clocks.mark()
        kern = kernel_times(X32, groups, C, nboot, kw, args.reps)
        torch.cuda.empty_cache()
        wall, peak, same = whole_calls(X32, groups, C, nperm, nboot, kw, args.calls)
        out["cases"][name] = {
            "workload": f"mct, {len(groups)} groups x {groups[0]} subj x {C} cond (N={sum(groups) * C}) x {p} voxels, "
                        f"{nperm} perm + {nboot} boot, {kw or 'exact mode'}",
            "kernel_ms": kern, "pls_call_s": wall, "max_memory_allocated_bytes": peak,
            "bit_identical_fp32_vs_fp64_on_widened": same,
            "clocks": clocks.summary(since=mark, stop=False),
        }
        print(name, json.dumps(out["cases"][name]), flush=True)
    out["clocks_all"] = clocks.summary()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
