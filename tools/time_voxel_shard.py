"""The two multi-process layouts of X, shard="resamples" (X replicated) and shard="voxels" (each rank holds
dist.voxel_shard of the columns), alternated in one process group over the GPUs of one box.

    python tools/time_voxel_shard.py [--voxels 1000000 --perms 10000 --boots 10000 --reps 3]
        [--precisions fp64,tf32x3] [--out profiles/time_voxel_shard_r05.json]

Default workload: config 5 (mct, 4 groups x 50 subjects x 6 conditions = 1200 rows, 10^6 voxels, 10 000 permutations +
10 000 bootstraps), analysis="device" so that the whole call stays on the GPUs, on every GPU of the box over NCCL.
On a box with one GPU two processes share it over gloo (collectives staged through the host); that run checks the
layouts and their memory, not their speed, and the record says so (`speed_claim: false`).

Per rank, layout and precision: the bytes of X on the device, the bytes of the bootstrap GEMM workspace (which holds
the tile-major image of X of the tall-design kernel), torch.cuda.max_memory_allocated over a whole PLS call, the
CUDA-event times of the Gram passes, of the bootstrap moment GEMM and of the collectives (all-reduce / all-gather
calls of plspy_b200.dist, events on the calling stream), the wall time of the whole call between two barriers
(median over --reps), the largest relative difference of std_errs / boot_ratios between the layouts and whether the
permutation p-values agree; rank 0 adds the GPU name, power limit and NVML clocks.  X is a seeded host matrix
(identical on every rank), pinned, so that both layouts take their fastest upload path."""
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

LAYOUTS = ("resamples", "voxels")


def _timed(owner, name, label, acc):
    """Wrap owner.name so that every call is bracketed by CUDA events on the current stream, collected under label."""
    import torch
    fn = getattr(owner, name)

    def wrapper(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn(*a, **k)
        e1.record()
        acc.setdefault(label, []).append((e0, e1))
        return out
    setattr(owner, name, wrapper)


def _worker(rank, world, port, backend, args, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import plspy_b200
        from plspy_b200 import dist as pd
        from plspy_b200._lib import lib
        from plspy_b200.engine import Engine
        acc = {}
        for owner, name, label in ((Engine, "gram_of", "gram"), (Engine, "_gram_tf32", "gram"),
                                   (Engine, "boot_moments", "boot_gemm"), (pd, "allreduce_sum_", "collectives"),
                                   (pd, "allreduce_packed_", "collectives"), (pd, "gather_spans", "collectives")):
            _timed(owner, name, label, acc)
        engines = []
        init = Engine.__init__

        def keep(self, *a, **k):
            init(self, *a, **k)
            engines.append(self)
        Engine.__init__ = keep
        groups, C, p = (50, 50, 50, 50), 6, args.voxels
        N = sum(groups) * C
        g = torch.Generator(); g.manual_seed(20260005)                   # the same matrix on every rank
        X = torch.randn(N, p, dtype=torch.float64, generator=g)
        X[:200, : p // 20] += 0.5
        X = X.pin_memory()
        rec = {}
        for prec in args.precisions.split(","):
            runs = {lay: [] for lay in LAYOUTS}
            last = {}
            for rep in range(args.reps + 1):                              # rep 0: warm-up, not recorded
                for lay in LAYOUTS:
                    acc.clear(); engines.clear()
                    import gc
                    gc.collect(); torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats()
                    base = torch.cuda.memory_allocated()
                    np.random.seed(1234)
                    dist.barrier(); torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = plspy_b200.PLS(X, groups, C, num_perm=args.perms, num_boot=args.boots, pls_method="mct",
                                         analysis="device", precision=prec, shard=lay)
                    se = res.resample_tests.std_errs
                    torch.cuda.synchronize(); dist.barrier()
                    wall = time.perf_counter() - t0
                    eng = engines[0]
                    K = int(se.shape[1])
                    ms = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in acc.items()}
                    row = {"step_s": wall, "peak_bytes": torch.cuda.max_memory_allocated() - base,
                           "x_bytes": eng._X.numel() * eng._X.element_size(), "voxel_range": list(eng.voxel_range),
                           "boot_gemm_workspace_bytes": int(lib.plsb200_boot_moments_f64_workspace(
                               N, max(eng.p, 1), min(K, Engine.KMAX), args.boots)) if prec == "fp64" else None,
                           "tf32_x_image_bytes": int(lib.plsb200_tf32_ximage_bytes(N, max(eng.p, 1)))
                           if prec == "tf32x3" else None,
                           **{f"{k}_ms": v for k, v in ms.items()}}
                    if rep:
                        runs[lay].append(row)
                    last[lay] = (np.asarray(se), np.asarray(res.resample_tests.boot_ratios),
                                 np.asarray(res.resample_tests.permute_ratio))
                    del res, eng, se
                    engines.clear()
            a, b = last["resamples"], last["voxels"]
            live = np.abs(a[1]).max(axis=0) > 0
            rel = lambda x, y: float(np.max(np.abs(x[:, live] - y[:, live]) / np.maximum(np.abs(x[:, live]), 1e-300)))
            rec[prec] = {lay: {"runs": runs[lay],
                               "median": {k: statistics.median(r[k] for r in runs[lay])
                                          for k in runs[lay][0] if isinstance(runs[lay][0][k], (int, float))}}
                         for lay in LAYOUTS}
            rec[prec]["std_errs_max_rel_diff"] = rel(a[0], b[0])
            rec[prec]["boot_ratios_max_rel_diff"] = rel(a[1], b[1])
            rec[prec]["permute_ratio_equal"] = bool(np.array_equal(a[2], b[2]))
        q.put((rank, rec))
    except BaseException:
        import traceback
        q.put((rank, {"error": traceback.format_exc()}))
        raise
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--voxels", type=int, default=1_000_000)
    ap.add_argument("--perms", type=int, default=10_000)
    ap.add_argument("--boots", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--precisions", default="fp64,tf32x3")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_voxel_shard_r05.json"))
    args = ap.parse_args()
    import socket
    import torch
    import torch.multiprocessing as mp
    from tools.time_collapsed import gpu_info
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ngpu = torch.cuda.device_count()
    backend, world = ("nccl", ngpu) if ngpu >= 2 else ("gloo", 2)
    clocks = None
    try:
        from tools._clocks import Clocks
        clocks = Clocks(0); clocks.start()
    except Exception:  # noqa: BLE001  (NVML missing: the record says so)
        clocks = None
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, args, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    per_rank = {}
    for _ in range(world):
        rank, rec = q.get()
        if "error" in rec:
            for pr in procs:
                pr.terminate()
            raise SystemExit(f"rank {rank} failed:\n{rec['error']}")
        per_rank[rank] = rec
    for pr in procs:
        pr.join()
    out = {
        "workload": f"mct, 4 x 50 subjects x 6 conditions (N = 1200) x {args.voxels} voxels, {args.perms} permutations + "
                    f"{args.boots} bootstraps, analysis='device', {args.reps} timed repetitions per layout "
                    "(alternated) after one warm-up",
        "processes": world, "gpus": ngpu, "backend": backend,
        "speed_claim": backend == "nccl",
        "note": ("one rank per GPU over NCCL" if backend == "nccl" else
                 "two processes share ONE GPU over gloo (collectives staged through the host): the record shows what "
                 "each layout holds on the device and that the results agree; its times are not a speed comparison"),
        "gpu": gpu_info(), "clocks": clocks.summary() if clocks is not None else "NVML unavailable",
        "per_rank": {str(r): per_rank[r] for r in sorted(per_rank)},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for prec, rec in per_rank[0].items():
        for lay in LAYOUTS:
            m = rec[lay]["median"]
            print(f"{prec:7s} {lay:9s} step {m['step_s']:.3f} s  X {m['x_bytes'] / 1e9:.2f} GB  "
                  f"peak {m['peak_bytes'] / 1e9:.2f} GB  gemm {m.get('boot_gemm_ms', 0):.1f} ms  "
                  f"collectives {m.get('collectives_ms', 0):.1f} ms")
        print(f"{prec:7s} std_errs max rel diff {rec['std_errs_max_rel_diff']:.2e}, "
              f"permute_ratio equal {rec['permute_ratio_equal']}")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
