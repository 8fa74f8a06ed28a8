"""shard="voxels" on the GPU: two ranks that each hold only their columns of X must reproduce the single-process run
on the same seed -- p-values, step-down ratios and index matrices identically, the rest to summation-order accuracy.

The two ranks share cuda:0 and exchange over gloo (staged through the host), which is how the multi-process path runs
on a box with one GPU; the NCCL variant needs two GPUs.  One spawn runs every case (`_run_cases`)."""
import gc
import os
import socket
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GROUPS, C = (7, 6), 3
NPERM, NBOOT = 41, 37          # odd: ragged resample shards

CASES = {
    "mct": dict(p=1500),
    "cst": dict(p=1500, method="cst"),
    "collapsed": dict(p=1500, kw=dict(boot_algo="collapsed")),
    "tf32x3": dict(p=1500, kw=dict(precision="tf32x3")),
    "tf32x3+gram": dict(p=1500, kw=dict(precision="tf32x3+gram")),
    "fp32": dict(p=1500, kw=dict(x_storage="fp32")),
    "fp64_widened": dict(p=1500, widen=True),
    "tall": dict(p=1500, groups=(60, 60)),                  # N = 360: the output-stationary bootstrap GEMM
    "device": dict(p=1500, kw=dict(analysis="device")),
    "device_cst": dict(p=1500, method="cst", kw=dict(analysis="device")),
    "split": dict(p=1500, kw=dict(num_split=5, lv=1)),
    "cst_split": dict(p=1500, method="cst", kw=dict(num_split=5, lv=1, x_storage="fp32")),
    "p300": dict(p=300),                                    # ragged slices: 256 + 44 voxels
    "p200": dict(p=200, kw=dict(analysis="device")),        # rank 1 holds no voxel
    "p200_collapsed": dict(p=200, kw=dict(boot_algo="collapsed")),
    "mem": dict(p=200_000),                                 # a wide X, for the peak device memory (both layouts)
}
NCCL_CASES = ("mct", "collapsed", "tall", "device", "p300", "p200")


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _inputs(case):
    c = CASES[case]
    groups = c.get("groups", GROUPS)
    rs = np.random.RandomState(3)
    X = rs.standard_normal((sum(groups) * C, c["p"])); X[:7, :80] += 1.0
    if c.get("widen"):
        X = X.astype(np.float32).astype(np.float64)
    kw = dict(num_perm=NPERM, num_boot=NBOOT, pls_method=c.get("method", "mct"), **c.get("kw", {}))
    if kw["pls_method"] == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(groups) * C, 2))
    return X, groups, kw


def _outputs(res, lazy=True):
    rt = res.resample_tests
    out = dict(pr=rt.permute_ratio, sr=rt.stepdown_ratio, sl=rt.perm_debug_dict["s_list"], se=rt.std_errs,
               br=rt.boot_ratios, lo=rt.conf_ints[0], hi=rt.conf_ints[1], left=rt.boot_debug_dict["left_sv_sampled"],
               td=rt.boot_debug_dict["Tdistrib"], s=res.s, brain=res.U, xl=res.X_latent,
               pidx=rt.perm_debug_dict["indices"], bidx=rt.boot_debug_dict["indices"])
    for k in ("X_mc", "X_means", "R"):
        if hasattr(res, k):
            out[k] = np.asarray(getattr(res, k))
    if hasattr(res, "pls_repro_tt"):
        out["sh_test"] = res.pls_repro_tt["pls_s_test"]
        out["sh_test_null"] = res.pls_repro_tt["pls_s_test_null"]
        out["sh_u"] = res.pls_repro_sh["pls_dist_u"]
    if lazy:        # collectives under voxel sharding: every rank asks
        out["right"] = rt.boot_debug_dict["right_sv_sampled"]
        out["pct_lo"], out["pct_hi"] = rt.salience_percentile_intervals()
    return out


def _run(case, **extra):
    import plspy_b200
    X, groups, kw = _inputs(case)
    kw.update(extra)
    np.random.seed(11)      # same seed on every rank -> identical index matrices
    return plspy_b200.PLS(X, groups, C, **kw)


def _run_cases(rank, world, port, q, backend, cases):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from plspy_b200 import dist as pd
        for case in cases:
            res = _run(case, shard="voxels")
            eng = res.resample_tests._engine
            X, groups, kw = _inputs(case)
            N, p = X.shape
            v0, v1 = pd.voxel_shard(p, rank, world)
            es = 4 if kw.get("x_storage") == "fp32" else 8
            assert eng.voxel_sharded and eng.voxel_range == (v0, v1) and eng.p == v1 - v0 and eng.p_total == p
            assert tuple(eng._X.shape) == (N, v1 - v0) and eng._X.numel() * eng._X.element_size() == N * (v1 - v0) * es
            assert eng.h2d_bytes == N * (v1 - v0) * es
            q.put((rank, case, _outputs(res)))
            del res, eng
        # memory: the device never holds a full-width copy of X (a wide X, where X dominates the peak)
        peaks = {}
        for shard in ("resamples", "voxels"):
            gc.collect(); torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats()
            res = _run("mem", shard=shard)
            torch.cuda.synchronize()
            peaks[shard] = torch.cuda.max_memory_allocated()
            del res
        q.put((rank, "peaks", peaks))
    except BaseException:
        q.put((rank, "error", traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def _spawn(backend, cases, world=2):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_run_cases, args=(r, world, port, q, backend, cases)) for r in range(world)]
    for pr in procs:
        pr.start()
    got = {}
    for _ in range(world * (len(cases) + 1)):
        rank, case, out = q.get(timeout=900)
        if case == "error":             # the other rank may be waiting in a collective: stop both
            for pr in procs:
                pr.terminate()
                pr.join(timeout=60)
            raise AssertionError(f"rank {rank} failed:\n{out}")
        got[(rank, case)] = out
    for pr in procs:
        pr.join(timeout=300)
        assert pr.exitcode == 0
    return got


@pytest.fixture(scope="module")
def gloo_runs():
    return _spawn("gloo", [c for c in CASES if c != "mem"])


_SINGLE = {}


def _single(case):
    if case not in _SINGLE:
        _SINGLE[case] = _outputs(_run(case))
    return _SINGLE[case]


def _assert_matches(multi, single, case):
    live = np.abs(single["s"]) > 1e-8
    for k in ("pr", "sr", "pidx", "bidx"):
        np.testing.assert_array_equal(multi[k], single[k], err_msg=k)
    sl_tol = 1e-6 if case == "tf32x3+gram" else 1e-12    # the TF32 Gram matrix: partial sums of other ranges
    np.testing.assert_allclose(multi["sl"][:, live], single["sl"][:, live], rtol=sl_tol, err_msg="s_list")
    np.testing.assert_allclose(multi["s"], single["s"], rtol=1e-12, atol=1e-12 * single["s"].max())
    for k, tol in (("se", 1e-10), ("br", 1e-10), ("lo", 1e-9), ("hi", 1e-9), ("right", 1e-10), ("pct_lo", 1e-10),
                   ("pct_hi", 1e-10), ("brain", 1e-10)):
        a, b = np.asarray(multi[k]), np.asarray(single[k])
        assert a.shape == b.shape, k
        np.testing.assert_allclose(a[..., live], b[..., live], rtol=tol, atol=tol * np.abs(b).max(), err_msg=k)
    for k in ("left", "td", "xl", "X_mc", "X_means", "R", "sh_test", "sh_test_null", "sh_u"):
        if k in single:
            a, b = np.asarray(multi[k]), np.asarray(single[k])
            if k in ("left", "td", "xl"):   # latent variables last; a null one's design side is any vector of the null
                a, b = a[..., live], b[..., live]       # space (analysis="device"), so only the live ones compare
            elif k.startswith("sh_"):       # split-half cubes (LV x LV x split): a half's null latent variables are
                # just as undetermined -- a 1e-14 relative perturbation of X moves them by O(1) in the float64 oracle too
                a, b = a[live][:, live], b[live][:, live]
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-11 * max(np.abs(b).max(), 1e-300), err_msg=k)


@pytest.mark.parametrize("case", [c for c in CASES if c != "mem"])
def test_voxel_sharded_run_matches_single_process(gloo_runs, case):
    single = _single(case)
    for rank in range(2):
        _assert_matches(gloo_runs[(rank, case)], single, case)


def test_voxel_sharded_float32_equals_voxel_sharded_float64_on_the_widened_matrix(gloo_runs):
    for rank in range(2):
        a, b = gloo_runs[(rank, "fp32")], gloo_runs[(rank, "fp64_widened")]
        assert a.keys() == b.keys()
        for k in a:
            np.testing.assert_array_equal(np.asarray(a[k]), np.asarray(b[k]), err_msg=k)


def test_voxel_sharded_peak_memory_is_below_the_replicated_run(gloo_runs):
    for rank in range(2):
        pk = gloo_runs[(rank, "peaks")]
        X = _inputs("mem")[0]
        # at least a quarter of X less: the replicated rank holds all of X, the voxel-sharded one half of it
        assert pk["voxels"] + X.nbytes // 4 < pk["resamples"], pk


def test_one_process_voxels_is_the_default_bit_for_bit():
    """World size 1: shard="voxels" is the same computation as the default."""
    for case in ("mct", "collapsed", "device"):
        a = _outputs(_run(case, shard="voxels"))
        b = _single(case)
        for k in a:
            np.testing.assert_array_equal(np.asarray(a[k]), np.asarray(b[k]), err_msg=f"{case} {k}")


def test_two_gpu_nccl_voxel_sharded_run_matches_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    got = _spawn("nccl", list(NCCL_CASES))
    for case in NCCL_CASES:
        for rank in range(2):
            _assert_matches(got[(rank, case)], _single(case), case)
