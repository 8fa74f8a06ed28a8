"""The factored collapsed bootstrap: the standard errors of mct / cst from the covariance of the subjects' draw counts
(boot_counts / boot_factor kernels + the bootstrap GEMM over ns - G pseudo-resamples), and boot_algo="auto".  Checked
against the explicit N x N covariance, the direct formulation, both storages of X, both upload paths, two processes in
both layouts, and draws without the subject structure (which take the N x N route)."""
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN_DIR

pytestmark = pytest.mark.gpu


def _load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _design(seed, groups, C, p, offset=0.0):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((sum(groups) * C, p))
    X[:groups[0], : p // 10] += 0.7
    return X + offset


def _pls(X, groups, C, seed, **kw):
    import plspy_b200
    np.random.seed(seed)
    return plspy_b200.PLS(X, groups, C, **kw)


# ---- the device factor against the N x N build ------------------------------------------------------------------
@pytest.mark.parametrize("name", ["mct_m0_bal", "mct_m1_unbal", "mct_m2_unbal", "mct_m3_bal", "cst_bal", "cst_unbal"])
def test_device_factor_rebuilds_the_nxn_covariance(name):
    import torch
    from plspy_b200 import bootstrap_permutation as bp
    from plspy_b200.engine import Engine
    g = _load(name)
    method, X = str(g["method"]), g["X"]
    groups, C = tuple(int(n) for n in g["groups"]), int(g["C"])
    co = np.array([[n] * C for n in groups])
    rs = np.random.RandomState(0)
    U = np.linalg.qr(rs.standard_normal((len(groups) * C, len(groups) * C)))[0]
    contrast = g["contrasts_in"] if "contrasts_in" in g else None
    idx = g["boot_idx"]
    R = idx.shape[0]
    eng = Engine(X)
    plan = bp._factor_plan(eng, method, U, contrast, co, int(g["mctype"]), R, idx)
    ns, G = sum(groups), len(groups)
    if R <= ns - G:
        assert plan is None                                # too few draws for the factor: the N x N route
        return
    assert plan is not None
    _, _, E = bp._task_operators(method, co, int(g["mctype"]), U, contrast)
    Mg = eng.boot_count_gram(eng.to_device(idx, torch.int32), plan["layout"])
    L = eng.boot_factor(Mg, R, plan["gstart"]).cpu().numpy()
    S1, S2 = eng.boot_cov(E, eng.to_device(idx, torch.int32))
    Sig = (S2 - S1.T[:, :, None] * S1.T[:, None, :] / R).cpu().numpy()
    sid = plan["sid"].cpu().numpy()
    Sf = np.einsum("nk,nj,mj,mk->knm", E, L[sid], L[sid], E)
    assert np.max(np.abs(Sf - Sig)) <= 1e-13 * np.max(np.abs(Sig))


# ---- against the direct formulation -------------------------------------------------------------------------------
def test_factored_matches_direct_at_benchmark_shape():
    import bench
    X = bench.make_data()
    out = {}
    for algo in ("direct", "auto"):
        res = _pls(X, bench.GROUPS, bench.C, 3, num_perm=0, num_boot=500, pls_method="mct", boot_algo=algo)
        out[algo] = res.resample_tests
    assert out["auto"].boot_algo == "collapsed" and out["direct"].boot_algo == "direct"
    live = np.abs(res.s) > 1e-8
    for f in ("std_errs", "boot_ratios"):
        assert _rel(getattr(out["auto"], f)[:, live], getattr(out["direct"], f)[:, live]) <= 1e-11, f


@pytest.mark.parametrize("case", ["offset_golden", "baseline_1e4", "cst"])
def test_factored_matches_direct_with_large_baselines(case):
    if case == "offset_golden":
        g = _load("mct_m0_offset")
        X, groups, C = g["X"], tuple(int(n) for n in g["groups"]), int(g["C"])
        kw, tol = dict(pls_method="mct", mctype=int(g["mctype"])), 1e-9
    elif case == "baseline_1e4":
        groups, C = (9, 7, 8), 3
        X = _design(5, groups, C, 3000) + 1e4 * np.random.RandomState(6).uniform(0.5, 1.5, 3000)
        kw, tol = dict(pls_method="mct", mctype=0), 1e-9
    else:
        groups, C = (10, 8), 3
        X = _design(7, groups, C, 3000)
        kw = dict(pls_method="cst", contrasts=np.random.RandomState(1).standard_normal((len(groups) * C, 3)))
        tol = 1e-11
    res = {}
    for algo in ("direct", "collapsed"):
        res[algo] = _pls(X.copy(), groups, C, 9, num_perm=0, num_boot=200, boot_algo=algo, **kw)
    live = np.abs(res["direct"].s) > 1e-8 * np.abs(res["direct"].s).max()
    for f in ("std_errs", "boot_ratios"):
        a, b = getattr(res["collapsed"].resample_tests, f), getattr(res["direct"].resample_tests, f)
        assert _rel(a[:, live], b[:, live]) <= tol, (f, _rel(a[:, live], b[:, live]))


def test_float32_storage_equals_widened_float64():
    groups, C = (9, 7, 8), 3
    X32 = _design(5, groups, C, 5000).astype(np.float32)
    kw = dict(num_perm=0, num_boot=150, pls_method="mct")
    a = _pls(X32, groups, C, 2, x_storage="fp32", **kw).resample_tests
    b = _pls(X32.astype(np.float64), groups, C, 2, **kw).resample_tests
    assert a.boot_algo == b.boot_algo == "collapsed"
    np.testing.assert_array_equal(a.std_errs, b.std_errs)
    np.testing.assert_array_equal(a.boot_ratios, b.boot_ratios)


def test_pipelined_upload_is_bit_identical_to_resident():
    import torch
    from plspy_b200.engine import Engine
    groups, C = (10, 10), 3
    X = _design(9, groups, C, 140_000)
    assert X.nbytes >= Engine.PIPELINED_UPLOAD_MIN_BYTES
    out = {}
    for tag in ("pinned", "resident"):
        kw = dict(num_perm=20, num_boot=70, pls_method="mct")
        if tag == "resident":
            kw["engine"] = Engine(torch.from_numpy(X).cuda())
            Xa = X
        else:
            Xa = torch.from_numpy(X).pin_memory()
        out[tag] = _pls(Xa, groups, C, 4, **kw).resample_tests
    assert out["pinned"].boot_algo == "collapsed"
    np.testing.assert_array_equal(out["pinned"].std_errs, out["resident"].std_errs)
    np.testing.assert_array_equal(out["pinned"].boot_ratios, out["resident"].boot_ratios)
    np.testing.assert_array_equal(out["pinned"].permute_ratio, out["resident"].permute_ratio)


# ---- draws without the subject structure take the N x N route ----------------------------------------------------
def test_unstructured_draws_fall_back_and_match_direct():
    import torch
    from plspy_b200 import bootstrap_permutation as bp, resample
    groups, C = (9, 7, 8), 3
    co = np.array([[n] * C for n in groups])
    X = _design(5, groups, C, 2000)
    np.random.seed(1)
    idx = resample.bootstrap_indices("mct", 120, co)[0].copy()
    idx[7, 3] = idx[7, 3 + 9]                               # row 3 draws from another cell
    idx[50, 9 + 2], idx[50, 9 + 3] = idx[50, 9 + 3], idx[50, 9 + 2]   # condition 1 uses another subject map
    res = {}
    for algo, ind in (("direct", idx), ("collapsed", idx), ("collapsed_dev", torch.from_numpy(idx).cuda())):
        res[algo] = _pls(X.copy(), groups, C, 2, num_perm=0, num_boot=120, pls_method="mct",
                         boot_algo=algo.split("_")[0], boot_indices=ind).resample_tests
    from plspy_b200.engine import Engine
    eng = Engine(X)
    U = np.linalg.qr(np.random.RandomState(0).standard_normal((9, 9)))[0]
    assert bp._factor_plan(eng, "mct", U, None, co, 0, 120, idx) is None
    assert bp._factor_plan(eng, "mct", U, None, co, 0, 120, torch.from_numpy(idx).cuda()) is None
    good = resample.bootstrap_indices("mct", 120, co)[0]
    assert bp._factor_plan(eng, "mct", U, None, co, 0, 120, good) is not None
    live = res["direct"].std_errs.max(axis=0) > 1e-12
    for key in ("collapsed", "collapsed_dev"):
        assert _rel(res[key].std_errs[:, live], res["direct"].std_errs[:, live]) <= 1e-11


# ---- auto ---------------------------------------------------------------------------------------------------------
def test_auto_resolves_as_specified():
    from plspy_b200.engine import Engine
    groups, C = (6, 6), 3
    X = _design(2, groups, C, 400)
    N = X.shape[0]
    assert _pls(X, groups, C, 1, num_boot=N + 1).resample_tests.boot_algo == "collapsed"
    assert _pls(X, groups, C, 1, num_boot=N).resample_tests.boot_algo == "direct"
    assert _pls(X, groups, C, 1, num_boot=N + 1, precision="tf32x3").resample_tests.boot_algo == "direct"
    assert _pls(X, groups, C, 1, num_boot=N + 1, boot_algo="direct").resample_tests.boot_algo == "direct"
    eng = Engine(X, precision="tf32x3")
    assert _pls(X, groups, C, 1, num_boot=N + 1, engine=eng).resample_tests.boot_algo == "direct"
    Y = np.random.RandomState(0).standard_normal((N, 2))
    assert _pls(X, groups, C, 1, Y=Y, num_boot=N + 1, pls_method="rb").resample_tests.boot_algo == "direct"


# ---- two processes on one GPU (gloo), both layouts ----------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _two_proc_data():
    rs = np.random.RandomState(3)
    groups, C = (7, 6), 3
    X = rs.standard_normal((sum(groups) * C, 20011)); X[:7, :80] += 1.0
    return X, groups, C


def _worker(rank, world, port, q, shard):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import plspy_b200
        X, groups, C = _two_proc_data()
        np.random.seed(11)
        rt = plspy_b200.PLS(X, groups, C, num_perm=0, num_boot=101, pls_method="mct", shard=shard).resample_tests
        se, br = rt.std_errs, rt.boot_ratios
        if rank == 0:
            q.put(dict(algo=rt.boot_algo, se=se, br=br))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("shard", ["resamples", "voxels"])
def test_two_processes_match_one(shard):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, shard)) for r in range(2)]
    for pr in procs:
        pr.start()
    multi = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    X, groups, C = _two_proc_data()
    res = _pls(X, groups, C, 11, num_perm=0, num_boot=101, pls_method="mct")
    rt = res.resample_tests
    assert multi["algo"] == rt.boot_algo == "collapsed"
    live = np.abs(res.s) > 1e-8
    assert _rel(multi["se"][:, live], rt.std_errs[:, live]) <= 1e-12
    assert _rel(multi["br"][:, live], rt.boot_ratios[:, live]) <= 1e-12
