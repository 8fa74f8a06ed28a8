"""Cost of streaming the whole per-bootstrap salience cube to the host with `right_sv_sampled_chunks()`.

    python tools/time_right_sv_chunks.py [--max-bytes 1073741824] [--out profiles/time_right_sv_chunks_r11.json]
                                         [--trace-dir DIR]

Two shapes, 1000 bootstraps each, data seeded like bench.make_data:
  * BASELINE cfg 2: rb, 2 groups x 20 subjects x 3 conditions (N = 120) x 50 000 voxels, 4 behaviours (K = 24): 9.6 GB;
  * the bench task workload: mct, 3 groups x 25 subjects x 4 conditions (N = 300) x 200 000 voxels (K = 12): 19.2 GB.
Each stream is consumed twice: once touching one element per chunk (the stream itself) and once with a reduction of
every element of the chunk on the host (np.sum), so the host never holds the cube.  Recorded in the same process: the
GPU's name and power limit, the device-to-pinned-host bandwidth of a 1 GiB copy (CUDA events), the kernel time of every
chunk (CUDA events around the chunk's launch), the copy time that bandwidth gives for a chunk, and the whole stream's
GB/s (host clock from the first step to the end).  `--trace-dir`: one more stream of each shape under torch.profiler,
whose chrome trace is written there and summarised (gaps between consecutive device-to-host copies, kernel time per
chunk from the trace)."""
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

from tools.time_collapsed import gpu_info  # noqa: E402


def d2h_bandwidth(nbytes=1 << 30, reps=5):
    import torch
    d = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    h = torch.empty(nbytes // 8, dtype=torch.float64, pin_memory=True)
    ts = []
    for _ in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); h.copy_(d, non_blocking=True); e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts[1:])
    return {"bytes": nbytes, "median_ms": ms, "GB_per_s": nbytes / ms / 1e6, "reps_ms": ts[1:]}


def _result(method):
    """the resampling result of one shape: PLS(..., num_perm=0, num_boot=1000) on the device"""
    import bench
    import plspy_b200
    if method == "rb":
        groups, C, p, nb = (20, 20), 3, 50_000, 4
        X = bench.make_data(groups=groups, C=C, p=p, seed=20260002)
        Y = np.random.RandomState(3).standard_normal((X.shape[0], nb)) + 0.3 * X[:, :nb]
        kw = dict(Y=Y)
    else:
        groups, C, p = bench.GROUPS, bench.C, bench.P_VOX
        X = bench.make_data()
        kw = dict(mctype=0)
    np.random.seed(7)
    res = plspy_b200.PLS(X, groups, C, num_perm=0, num_boot=1000, pls_method=method, **kw)
    return {"method": method, "groups": groups, "C": C, "p": p, "N": X.shape[0]}, res.resample_tests


class _KernelEvents:
    """Engine.stream_chunks with CUDA events around every chunk's launch"""

    def __enter__(self):
        import torch
        from plspy_b200.engine import Engine
        self.events, orig = [], Engine.stream_chunks
        self._orig = orig

        def stream_chunks(eng, fill, B, K, max_bytes, v_offset=0):
            def timed(v0, v1, out):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fill(v0, v1, out); e1.record()
                self.events.append((v1 - v0, e0, e1))
            yield from orig(eng, timed, B, K, max_bytes, v_offset)
        Engine.stream_chunks = stream_chunks
        return self

    def __exit__(self, *exc):
        from plspy_b200.engine import Engine
        Engine.stream_chunks = self._orig

    def ms(self):
        return [e0.elapsed_time(e1) for _, e0, e1 in self.events]


def _stream(rt, max_bytes, consume):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nbytes, n, host_ms = 0, 0, 0.0
    for v0, v1, chunk in rt.right_sv_sampled_chunks(max_bytes):
        h0 = time.perf_counter()
        consume(chunk)
        host_ms += (time.perf_counter() - h0) * 1e3
        nbytes += chunk.nbytes
        n += 1
    s = time.perf_counter() - t0
    return {"chunks": n, "bytes": nbytes, "stream_s": s, "GB_per_s": nbytes / s / 1e9, "host_consume_ms": host_ms}


def _trace_summary(path):
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    copies = sorted((e["ts"], e["dur"]) for e in ev if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", ""))
    kernels = sorted((e["ts"], e["dur"], e["name"]) for e in ev if e.get("cat") == "kernel")
    big = [c for c in copies if c[1] > 1000]                     # the chunk copies (> 1 ms)
    gaps = [b[0] - (a[0] + a[1]) for a, b in zip(big, big[1:])]
    names = {}
    for _, d, nm in kernels:
        key = nm.split("<")[0].split("(")[0]
        names[key] = names.get(key, 0.0) + d / 1e3
    return {"chunk_copies": len(big), "copy_ms": [d / 1e3 for _, d in big],
            "gaps_between_chunk_copies_ms": [g / 1e3 for g in gaps], "kernel_ms_by_name": names}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-bytes", type=int, default=1 << 30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_right_sv_chunks_r11.json"))
    ap.add_argument("--trace-dir", default=None)
    ap.add_argument("--shapes", default="rb,mct")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    rec = {"gpu": gpu_info(), "max_bytes": args.max_bytes, "d2h_pinned": d2h_bandwidth()}
    bw = rec["d2h_pinned"]["GB_per_s"]
    for method in args.shapes.split(","):
        shape, rt = _result(method)
        first = next(rt.right_sv_sampled_chunks(args.max_bytes))       # warm-up: coefficients, module loads
        B, _, K = first[2].shape
        del first
        shape.update(B=B, K=K, cube_GB=B * shape["p"] * K * 8 / 1e9)
        out = {"shape": shape, "path": getattr(rt._engine, "last_rb_path", None) if method == "rb" else "salience_f64"}
        with _KernelEvents() as kev:
            out["touch_one_element"] = _stream(rt, args.max_bytes, lambda c: float(c[0, 0, 0]))
        kms, widths = kev.ms(), [w for w, _, _ in kev.events]
        copy_ms = [B * w * K * 8 / bw / 1e6 for w in widths]
        out["kernel_ms_per_chunk"] = kms
        out["copy_ms_per_chunk_at_measured_bandwidth"] = copy_ms
        out["kernel_over_copy_median"] = statistics.median(k / c for k, c in zip(kms, copy_ms))
        out["copy_bound_stream_s"] = sum(copy_ms) / 1e3
        out["sum_every_element"] = _stream(rt, args.max_bytes, lambda c: float(np.sum(c)))
        if args.trace_dir:
            from torch.profiler import ProfilerActivity, profile
            os.makedirs(args.trace_dir, exist_ok=True)
            path = os.path.join(args.trace_dir, f"right_sv_chunks_{method}.json")
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                _stream(rt, args.max_bytes, lambda c: float(c[0, 0, 0]))
            prof.export_chrome_trace(path)
            out["trace"] = {"file": os.path.basename(path), **_trace_summary(path)}
        rec[method] = out
        print(json.dumps({method: out}, default=str)[:2000], flush=True)
        del rt
        torch.cuda.empty_cache()
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1, default=str)


if __name__ == "__main__":
    main()
