"""Device time of the exact FP64 Gram launch (csrc/gram.cu: partial kernel + split reduction) at the shapes the
package runs it at, with CUDA events over many launches, and optionally of its probe modes.

    python tools/time_gram.py [--probes] [--out profiles/time_gram_rNN.json] [--save-dir DIR]

Shapes: the benchmark's stack [X; V^T] (300 + 12 rows x 200 000 voxels, plsb200_gram_stacked_f64), X alone at that
size (plsb200_gram_f64), config 1 (60 x 10 000), config 5 per GPU (1200 x 1 000 000) and the float32-resident twin of
the bench matrix (plsb200_gram_x32_f64).  Inputs are seeded normal matrices generated on the device; every shape but
config 1 is larger than the 126 MB L2.  --probes also times the probe modes of the partial kernel (PLSB200_GRAM_PROBE,
see gram.cu) at the benchmark stack, from a copy of the library whose gram.cu is compiled with -DPLSB_PROBES into a
temporary directory.  --save-dir writes each shape's G as .npy, so that two builds can be compared bit for bit.
Records the GPU's name, power limit and NVML clocks of the same run."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.time_collapsed import gpu_info  # noqa: E402

SHAPES = [
    # name, rows of X, rows stacked below X, voxels, storage
    ("bench_stack", 300, 12, 200_000, "fp64"),
    ("bench_x", 300, 0, 200_000, "fp64"),
    ("cfg1", 60, 0, 10_000, "fp64"),
    ("cfg5_per_gpu", 1200, 0, 1_000_000, "fp64"),
    ("bench_x_fp32", 300, 0, 200_000, "fp32"),
]
PROBES = {0: "as is", 1: "operands resident (no cp.async after the ring is first filled)",
          2: "feed only (no fragment loads or DMMAs)"}


def probe_library(tmp):
    """libplsb200 with gram.cu compiled with -DPLSB_PROBES (the other objects are the in-tree ones build() made)."""
    from plspy_b200 import build as b
    b.build()
    o = os.path.join(tmp, "gram_probe.o")
    subprocess.check_call(["nvcc", *b.NVCC_FLAGS, "-DPLSB_PROBES", "-c", os.path.join(b.CSRC, "gram.cu"), "-o", o])
    objs = [os.path.join(b.CSRC, os.path.splitext(s)[0] + ".o") for s in b.SOURCES if s != "gram.cu"]
    so = os.path.join(tmp, "libplsb200_probe.so")
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so, *objs, o,
                           "-lcudart"])
    lib = ctypes.CDLL(so)
    from plspy_b200._lib import SIGNATURES
    for name, (res, args) in SIGNATURES.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib


def time_launches(fn, min_ms=300.0, windows=5):
    """Median and minimum device time of one launch (ms) over `windows` windows of back-to-back launches."""
    import torch
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n = max(3, int(min_ms / max(e0.elapsed_time(e1), 1e-3)))
    per = []
    for _ in range(windows):
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        per.append(e0.elapsed_time(e1) / n)
    return {"median_ms": statistics.median(per), "min_ms": min(per), "launches_per_window": n}


def gram_call(lib, X, n1, X2=None):
    """A closure that forms the Gram matrix of X (or of the stack [X; X2]) into G, and G."""
    import torch
    from plspy_b200._lib import check
    p = int(X.shape[1])
    n = n1 + (int(X2.shape[0]) if X2 is not None else 0)
    nb = lib.plsb200_gram_f64_workspace(n, p)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=X.device)
    G = torch.empty((n, n), dtype=torch.float64, device=X.device)
    st = torch.cuda.current_stream().cuda_stream
    if X2 is not None:
        f = lambda: check(lib.plsb200_gram_stacked_f64(X.data_ptr(), n1, X.stride(0), X2.data_ptr(), int(X2.shape[0]),
                                                       X2.stride(0), p, G.data_ptr(), ws.data_ptr(), nb, st), "stk")
    elif X.dtype == torch.float32:
        f = lambda: check(lib.plsb200_gram_x32_f64(X.data_ptr(), n1, p, X.stride(0), G.data_ptr(), ws.data_ptr(), nb,
                                                   st), "x32")
    else:
        f = lambda: check(lib.plsb200_gram_f64(X.data_ptr(), n1, p, X.stride(0), G.data_ptr(), ws.data_ptr(), nb, st),
                          "f64")
    return f, G


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--probes", action="store_true")
    ap.add_argument("--out")
    ap.add_argument("--save-dir")
    ap.add_argument("--shapes", help="comma-separated subset of " + ",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    import torch
    from plspy_b200._lib import lib
    from tools._clocks import Clocks
    dev = torch.device("cuda", 0)
    rec = {"gpu": gpu_info(), "shapes": []}
    clk = Clocks(); clk.start()
    want = set(args.shapes.split(",")) if args.shapes else None
    for name, n1, n2, p, storage in SHAPES:
        if want and name not in want:
            continue
        g = torch.Generator(device=dev); g.manual_seed(n1 * 7 + n2 + p)
        X = torch.randn((n1, p), dtype=torch.float64, device=dev, generator=g) + 0.5
        if storage == "fp32":
            X = X.float()
        X2 = torch.randn((n2, p), dtype=torch.float64, device=dev, generator=g) if n2 else None
        f, G = gram_call(lib, X, n1, X2)
        mark = clk.mark()
        t = time_launches(f)
        n = n1 + n2
        flops_tri = float(n) * (n + 1) * p        # the upper triangle (with the diagonal) of the n x n product
        r = {"name": name, "rows": n1, "stacked_rows": n2, "voxels": p, "storage": storage, **t,
             "upper_triangle_tflops": flops_tri / t["median_ms"] * 1e-9,
             "clocks": clk.summary(since=mark, stop=False)}
        if args.save_dir:
            os.makedirs(args.save_dir, exist_ok=True)
            np.save(os.path.join(args.save_dir, f"G_{name}.npy"), G.cpu().numpy())
        print(json.dumps(r), flush=True)
        rec["shapes"].append(r)
        del X, X2, G
        torch.cuda.empty_cache()
    if args.probes:
        with tempfile.TemporaryDirectory() as tmp:
            plib = probe_library(tmp)
            name, n1, n2, p, _ = SHAPES[0]
            g = torch.Generator(device=dev); g.manual_seed(n1 * 7 + n2 + p)
            X = torch.randn((n1, p), dtype=torch.float64, device=dev, generator=g) + 0.5
            X2 = torch.randn((n2, p), dtype=torch.float64, device=dev, generator=g)
            f, _ = gram_call(plib, X, n1, X2)
            rec["probes"] = []
            for mode, what in PROBES.items():
                os.environ["PLSB200_GRAM_PROBE"] = str(mode)
                r = {"shape": name, "probe": mode, "what": what, **time_launches(f)}
                print(json.dumps(r), flush=True)
                rec["probes"].append(r)
            os.environ.pop("PLSB200_GRAM_PROBE")
    rec["clocks"] = clk.summary()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rec, fh, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "clocks": rec["clocks"]}))


if __name__ == "__main__":
    main()
