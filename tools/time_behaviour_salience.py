"""Cost of the per-bootstrap salience export (`right_sv_sampled` of rb / csb / mb / cmb) in one process on one GPU.

    python tools/time_behaviour_salience.py --baseline-lib PATH [--reps 7] [--out profiles/time_behaviour_salience_r08.json]

--baseline-lib: libplsb200.so built from the commit before the export (for example `git worktree add /tmp/base HEAD~1
&& python -m plspy_b200.build` there).  Its entry points are bound with this tree's signatures; the one the engine
calls that it lacks, `plsb200_rb_boot*_vs_f64`, is routed to the plain entry point, which exists in both.

1. Default path, baseline library against this tree's, alternated rep by rep: the bootstrap stage of the behaviour
   method (`_bootstrap_behaviour`, BASELINE cfg 2: rb 2 x 20 x 3 rows x 50 000 voxels, 4 behaviours, 1000
   bootstraps) and of the multiblock method (`_boot_multiblock`, the cfg 4 shape: mb 2 x 30 x 4 rows x 200 000 voxels,
   bscan [1, 2], 4 behaviours, 500 of its 2000 bootstraps).  Host clock around the stage, which ends in a device
   synchronise (its results are copied to the host); median / min / max over --reps, and whether the two libraries
   gave bit-identical std_errs, boot_ratios and LVcorr.
2. One read of the cube: rb, 2 x 20 x 3 rows, 4 behaviours (K = 24), 10 000 voxels, 1000 bootstraps (1.79 GiB): the
   whole read (coefficients, p-space pass with the store, copy to the host) and, with CUDA events, the p-space pass
   with the store next to the moment-only pass on the same inputs.
The GPU's name, power limit and clocks are recorded with the numbers.  Data: seeded standard normal (bench.make_data
style); X is larger than the L2 in the cfg 2 / cfg 4 cases."""
import argparse
import ctypes
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


class _Baseline:
    """The baseline library with this tree's ctypes signatures; `_vs` entry points map to the plain ones (VS NULL)."""

    def __init__(self, path):
        from plspy_b200 import _lib
        self._so = ctypes.CDLL(path)
        for name, (res, args) in _lib.SIGNATURES.items():
            if hasattr(self._so, name):
                f = getattr(self._so, name)
                f.restype, f.argtypes = res, args

    def __getattr__(self, name):
        if name.endswith("_vs_f64") and not hasattr(self._so, name):
            plain = getattr(self._so, name[: -len("_vs_f64")] + "_f64")

            def call(*a):           # (..., T, nrm2, VS, workspace, workspace_bytes, stream)
                assert a[-4] is None, "the baseline library cannot export the saliences"
                return plain(*a[:-4], *a[-3:])
            return call
        return getattr(self._so, name)


def _stats(ts):
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts), "reps_ms": ts}


def _shape(method, groups, C, p, nb, nboot, bscan=None, seed=0):
    import oracle.pls_oracle as po
    from plspy_b200 import resample
    rs = np.random.RandomState(seed)
    N = sum(groups) * C
    X = rs.standard_normal((N, p))
    X[: groups[0], : p // 20] += 0.5
    Y = rs.standard_normal((N, nb)) + 0.3 * X[:, :nb]
    co = np.array([[n] * C for n in groups])
    a = po.analysis(method, X, groups, C, Y=Y, mctype=0, bscan=bscan)
    np.random.seed(seed + 1)
    idx = resample.bootstrap_indices(method, nboot, co, Y=Y, bscan=a.get("bscan"), Ybscan=a.get("Ybscan"))
    return X, Y, co, a, idx


def _stage(method, eng, Y, co, a, idx, nboot):
    """The bootstrap stage as PLS(...) runs it; returns the arrays compared between the libraries."""
    from plspy_b200 import bootstrap_permutation as bp
    if method == "rb":
        ci, se, br, lv, _ = bp._ResampleTestPLS._bootstrap_behaviour(eng, Y, a["U"], a["s"].copy(), a["V"], co, nboot,
                                                                      "rb", None, a["lvcorrs_orig"], 0.95, idx[0])
    else:
        ci, _, se, br, lv, _ = bp._boot_multiblock(eng, a["U"], a["s"].copy(), a["V"], co, 0, nboot, "mb", None,
                                                   a["bscan"], a["Ybscan"], a["lvcorrs_orig"], a["Tvsc_orig"], 0.95,
                                                   idx)
    return se, br, lv


def time_default_path(libs, reps):
    import torch
    from plspy_b200 import engine as engmod
    from plspy_b200.engine import Engine
    out = {}
    for name, method, groups, C, p, nb, nboot, bscan in (
            ("cfg2_rb", "rb", (20, 20), 3, 50_000, 4, 1000, None),
            ("cfg4_mb", "mb", (30, 30), 4, 200_000, 4, 500, [1, 2])):
        X, Y, co, a, idx = _shape(method, groups, C, p, nb, nboot, bscan)
        eng = Engine(torch.from_numpy(X).cuda())
        times = {k: [] for k in libs}
        results = {}
        for k, lib in libs.items():          # warm-up: module loads, workspaces, the cached block-standardised X
            engmod.lib = lib
            results[k] = [np.asarray(r) for r in _stage(method, eng, Y, co, a, idx, nboot)]
        for _ in range(reps):
            for k, lib in libs.items():
                engmod.lib = lib
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _stage(method, eng, Y, co, a, idx, nboot)
                torch.cuda.synchronize()
                times[k].append((time.perf_counter() - t0) * 1e3)
        engmod.lib = libs["this_tree"]
        out[name] = {"shape": dict(method=method, groups=groups, C=C, p=p, behaviours=nb, nboot=nboot, bscan=bscan),
                     "path": eng.last_rb_path,
                     **{k: _stats(v) for k, v in times.items()},
                     "bit_identical_std_errs_boot_ratios_LVcorr": all(
                         np.array_equal(x, y) for x, y in zip(results["baseline"], results["this_tree"]))}
        del eng
        torch.cuda.empty_cache()
    return out


def time_cube_read(reps):
    import torch
    from plspy_b200 import bootstrap_permutation as bp
    from plspy_b200.engine import Engine
    groups, C, p, nb, nboot = (20, 20), 3, 10_000, 4, 1000
    X, Y, co, a, idx = _shape("rb", groups, C, p, nb, nboot, seed=5)
    eng = Engine(torch.from_numpy(X).cuda())
    _, se, _, _, debug = bp._ResampleTestPLS._bootstrap_behaviour(eng, Y, a["U"], a["s"].copy(), a["V"], co, nboot, "rb",
                                                                  None, a["lvcorrs_orig"], 0.95, idx[0])
    K = a["U"].shape[1]
    cells = bp._cell_offsets(co)
    Xc = bp._behaviour_state(eng, cells)["Xc"]
    Q, W, _ = eng.rb_coef(Y, eng.to_device(idx[0], torch.int32), cells, a["U"], scatter=True)
    cube = torch.empty(nboot, p, K, dtype=torch.float64, device=eng.device)

    def ev(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    export, moments = [], []
    for _ in range(reps + 1):              # the first of each is the warm-up
        export.append(ev(lambda: eng.rb_boot(Xc, Q, W, cells, want_t=False, vs_out=cube)))
        moments.append(ev(lambda: eng.rb_boot(Xc, Q, W, cells, want_t=False)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    right = debug["right_sv_sampled"]
    read_ms = (time.perf_counter() - t0) * 1e3
    std_rel = float(np.max(np.abs(np.std(right, axis=0) - se) / np.maximum(np.abs(se), 1e-300)))
    return {"shape": dict(method="rb", groups=groups, C=C, p=p, behaviours=nb, K=K, nboot=nboot),
            "cube_gib": right.nbytes / 2**30, "path": eng.last_rb_path,
            "first_read_ms (coefficients + p-space pass with the store + copy to the host)": read_ms,
            "p_space_pass_with_store": _stats(export[1:]), "p_space_pass_moments_only": _stats(moments[1:]),
            "max_rel_diff_std_of_cube_vs_std_errs": std_rel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_behaviour_salience_r08.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from plspy_b200._lib import lib
    libs = {"baseline": _Baseline(os.path.abspath(args.baseline_lib)), "this_tree": lib}
    rec = {"gpu": gpu_info(), "reps": args.reps,
           "default_path": time_default_path(libs, args.reps),
           "cube_read": time_cube_read(args.reps)}
    rec["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1, default=str)
    print(json.dumps(rec, indent=1, default=str))


if __name__ == "__main__":
    main()
