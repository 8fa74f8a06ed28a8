"""boot_algo="collapsed": the bootstrap standard errors of the task methods from the closed form
x_v^T Cov_r(c_rk) x_v (plsb200_boot_quad_f64 + the N-space covariance build) instead of the moments of the B x p x K
salience GEMM.  Checked against an explicit quadratic form, the reference's golden fixtures, the oracle, the direct
formulation at the benchmark shape, both upload paths, two processes and the plug-in."""
import os
import socket

import numpy as np
import pytest

import oracle.pls_oracle as po
from conftest import GOLDEN_DIR, golden_cases

pytestmark = pytest.mark.gpu

TASK_CASES = [c for c in golden_cases() if c.startswith(("mct", "cst"))]


def _load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def _run_golden(g, **extra):
    import plspy_b200
    method = str(g["method"])
    kw = dict(num_perm=int(g["nperm"]), num_boot=int(g["nboot"]), pls_method=method, CI=float(g["CI"]),
              mctype=int(g["mctype"]))
    if "contrasts_in" in g:
        kw["contrasts"] = g["contrasts_in"].copy()
    kw.update(extra)
    np.random.seed(int(g["np_seed"]))
    return plspy_b200.PLS(g["X"].copy(), tuple(int(n) for n in g["groups"]), int(g["C"]), **kw)


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


# ---- the kernel ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4, 37, 60, 300, 320])
@pytest.mark.parametrize("K", [1, 5, 12, 24])
def test_quad_kernel_matches_explicit_quadratic_form(N, K):
    import torch
    from plspy_b200.engine import Engine
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(1000 * N + K)
    for p in (1, 63, 64, 1000, 20011):
        X = torch.randn(N, p, dtype=torch.float64, device=dev, generator=gen)
        A = torch.randn(K, N, N, dtype=torch.float64, device=dev, generator=gen)
        Sig = A + A.transpose(1, 2)                                     # symmetric, indefinite
        q = Engine(X).boot_quad(Sig)
        ref = (X[None] * (Sig @ X)).sum(dim=1).T                        # einsum('nv,knm,mv->vk')
        err = float((q - ref).abs().max() / ref.abs().max())
        assert err <= 1e-12, (N, p, K, err)
        # a voxel sub-range writes exactly the rows of the whole call's result for those voxels
        if p >= 64:
            sub = Engine(X).boot_quad(Sig, 5, p - 3)
            assert float((sub - ref[5:p - 3]).abs().max() / ref.abs().max()) <= 1e-12


def test_quad_kernel_rejects_tall_designs():
    from plspy_b200 import _lib
    assert _lib.lib.plsb200_boot_quad_coef_bytes(321, 12) == 0
    assert _lib.lib.plsb200_boot_quad_f64_workspace(321, 1000, 12) == 0
    assert _lib.lib.plsb200_boot_quad_coef_bytes(300, 25) == 0


# ---- golden fixtures: the reference's values, and the direct run's -------------------------------------------
@pytest.mark.parametrize("name", TASK_CASES)
def test_collapsed_matches_golden_and_direct(name):
    g = _load(name)
    live = np.abs(g["s"]) > 1e-8
    d = _run_golden(g).resample_tests
    c = _run_golden(g, boot_algo="collapsed").resample_tests
    assert c.boot_algo == "collapsed" and d.boot_algo == "direct"
    for f in ("std_errs", "boot_ratios"):
        assert _rel(getattr(c, f)[:, live], g[f][:, live]) <= 1e-8, f
        # X + a large offset (mct_m0_offset): the offset cancels inside the quadratic form, not before it
        assert _rel(getattr(c, f)[:, live], getattr(d, f)[:, live]) <= (1e-9 if "offset" in name else 1e-11), f
    np.testing.assert_array_equal(c.permute_ratio, d.permute_ratio)
    np.testing.assert_array_equal(c.stepdown_ratio, d.stepdown_ratio)
    np.testing.assert_array_equal(c.permute_ratio, g["permute_ratio"])
    for i in range(2):
        np.testing.assert_array_equal(c.conf_ints[i], d.conf_ints[i])
    for key in ("Tdistrib", "left_sv_sampled"):
        np.testing.assert_array_equal(c.boot_debug_dict[key], d.boot_debug_dict[key])


# ---- oracle on seeded larger designs -------------------------------------------------------------------------
def _design(seed, groups, C, p, offset=0.0):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((sum(groups) * C, p))
    X[:groups[0], : p // 10] += 0.7
    return X + offset


ORACLE_CASES = [
    ("mct", 0, (9, 7, 8), 3, 0.0),
    ("mct", 1, (9, 7, 8), 3, 0.0),
    ("mct", 2, (9, 7, 8), 3, 0.0),
    ("mct", 3, (9, 9), 4, 0.0),
    ("cst", 0, (10, 8), 3, 0.0),
    ("mct", 0, (9, 7, 8), 3, 100.0),
    ("mct", 0, (4, 4, 4, 4, 4), 6, 0.0),     # K = 30 > 24: the quadratic form is split by column
]


@pytest.mark.parametrize("method,mctype,groups,C,offset", ORACLE_CASES)
def test_collapsed_matches_oracle(method, mctype, groups, C, offset):
    import plspy_b200
    X = _design(5, groups, C, 2000, offset)
    kw = dict(num_perm=0, num_boot=60, pls_method=method, mctype=mctype)
    if method == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(groups) * C, 3))
    np.random.seed(7)
    d = plspy_b200.PLS(X.copy(), groups, C, **kw).resample_tests
    np.random.seed(7)
    res = plspy_b200.PLS(X.copy(), groups, C, boot_algo="collapsed", **kw)
    c = res.resample_tests
    live = np.abs(res.s) > 1e-8 * np.abs(res.s).max()
    a = po.analysis(method, X.copy(), groups, C, contrasts=kw.get("contrasts"), mctype=mctype)
    o = po.bootstrap_test(method, X, None, a["U"], a["s"], a["V"], a["cond_order"], mctype,
                          c.boot_debug_dict["indices"], contrast=a.get("contrast"), Tvsc_orig=a["Tvsc_orig"],
                          keep_right=False)
    tol = 1e-7 if offset else 1e-9
    assert _rel(c.std_errs[:, live], o["std_errs"][:, live]) <= tol
    assert _rel(c.std_errs[:, live], d.std_errs[:, live]) <= tol
    assert _rel(c.boot_ratios[:, live], d.boot_ratios[:, live]) <= tol


# ---- benchmark shape -----------------------------------------------------------------------------------------
def test_collapsed_matches_direct_at_benchmark_shape():
    import bench
    import plspy_b200
    X = bench.make_data()
    d = {}
    for algo in ("direct", "collapsed"):
        np.random.seed(3)
        res = plspy_b200.PLS(X, bench.GROUPS, bench.C, num_perm=0, num_boot=500, pls_method="mct", boot_algo=algo)
        d[algo] = res.resample_tests
    live = np.abs(res.s) > 1e-8
    for f in ("std_errs", "boot_ratios"):
        assert _rel(getattr(d["collapsed"], f)[:, live], getattr(d["direct"], f)[:, live]) <= 1e-10, f


# ---- upload paths: pinned host X (pipelined upload, early bootstrap) vs a resident copy -------------------------
def test_pipelined_upload_gives_the_resident_result():
    import torch
    import plspy_b200
    from plspy_b200.engine import Engine
    groups, C = (10, 10), 3
    X = _design(9, groups, C, 140_000)                    # 67 MB: above the pipelined-upload threshold
    assert X.nbytes >= Engine.PIPELINED_UPLOAD_MIN_BYTES
    out = {}
    for tag, Xa in (("pinned", torch.from_numpy(X).pin_memory()), ("resident", None)):
        kw = dict(num_perm=20, num_boot=40, pls_method="mct", boot_algo="collapsed")
        if Xa is None:
            kw["engine"] = Engine(torch.from_numpy(X).cuda())
            Xa = X
        np.random.seed(4)
        out[tag] = plspy_b200.PLS(Xa, groups, C, **kw).resample_tests
    live = np.abs(out["resident"].std_errs).max(axis=0) > 0
    for f in ("std_errs", "boot_ratios"):
        assert _rel(getattr(out["pinned"], f)[:, live], getattr(out["resident"], f)[:, live]) <= 1e-12, f
    np.testing.assert_array_equal(out["pinned"].permute_ratio, out["resident"].permute_ratio)


# ---- lazy fields -------------------------------------------------------------------------------------------
def test_lazy_fields_still_recompute_from_the_indices():
    import plspy_b200
    X = _design(2, (6, 6), 3, 300)
    np.random.seed(8)
    rt = plspy_b200.PLS(X, (6, 6), 3, num_perm=0, num_boot=25, boot_algo="collapsed").resample_tests
    right = rt.boot_debug_dict["right_sv_sampled"]
    assert right.shape == (25, 300, rt.std_errs.shape[1])
    live = rt.std_errs.max(axis=0) > 1e-12
    assert _rel(rt.std_errs[:, live], right.std(axis=0)[:, live]) <= 1e-10
    np.random.seed(8)
    rd = plspy_b200.PLS(X, (6, 6), 3, num_perm=0, num_boot=25).resample_tests
    lo, hi = rt.salience_percentile_intervals()
    lo_d, hi_d = rd.salience_percentile_intervals()
    np.testing.assert_array_equal(lo, lo_d)
    np.testing.assert_array_equal(hi, hi_d)


# ---- validation with an engine that is already there ---------------------------------------------------------
def test_collapsed_needs_an_exact_engine():
    import plspy_b200
    from plspy_b200.engine import Engine
    X = _design(2, (6, 6), 3, 300)
    with pytest.raises(ValueError):
        plspy_b200.PLS(X, (6, 6), 3, num_boot=5, boot_algo="collapsed", engine=Engine(X, precision="tf32x3"))


# ---- plug-in through the reference's own PLS -----------------------------------------------------------------
def test_plugin_collapsed_matches_drop_in():
    import baseline
    if not baseline.reference_available():
        pytest.skip("baseline/_ref not installed (python -m baseline.install_ref)")
    import contextlib
    import io
    import warnings
    import plspy_b200
    g = _load("mct_m0_bal")
    mod = baseline.import_reference()
    plspy_b200.install(mod, boot_algo="collapsed")
    try:
        np.random.seed(int(g["np_seed"]))
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = mod.PLS(g["X"].copy(), tuple(int(n) for n in g["groups"]), int(g["C"]), num_perm=int(g["nperm"]),
                          num_boot=int(g["nboot"]), pls_method="mct", mctype=int(g["mctype"]), CI=float(g["CI"]))
    finally:
        plspy_b200.uninstall()
    rt = ref.resample_tests
    assert rt.boot_algo == "collapsed"
    own = _run_golden(g, boot_algo="collapsed").resample_tests
    live = np.abs(g["s"]) > 1e-8
    assert _rel(rt.std_errs[:, live], own.std_errs[:, live]) <= 1e-12
    np.testing.assert_array_equal(rt.permute_ratio, own.permute_ratio)


# ---- two processes on one GPU (gloo) ---------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _two_proc_data(p):
    rs = np.random.RandomState(3)
    groups, C = (7, 6), 3
    X = rs.standard_normal((sum(groups) * C, p)); X[:7, :80] += 1.0
    return X, groups, C


def _worker(rank, world, port, q, p):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import plspy_b200
        X, groups, C = _two_proc_data(p)
        np.random.seed(11)
        res = plspy_b200.PLS(X, groups, C, num_perm=41, num_boot=37, pls_method="mct", boot_algo="collapsed")
        rt = res.resample_tests
        if rank == 0:
            q.put(dict(pr=rt.permute_ratio, se=rt.std_errs, br=rt.boot_ratios, lo=rt.conf_ints[0]))
    finally:
        dist.destroy_process_group()


def test_two_processes_match_the_single_process_collapsed_run():
    import torch.multiprocessing as mp
    import plspy_b200
    p = 20011                                      # ragged voxel shares; 37 bootstraps: ragged resample shards
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, p)) for r in range(2)]
    for pr in procs:
        pr.start()
    multi = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    X, groups, C = _two_proc_data(p)
    np.random.seed(11)
    res = plspy_b200.PLS(X, groups, C, num_perm=41, num_boot=37, pls_method="mct", boot_algo="collapsed")
    rt = res.resample_tests
    live = np.abs(res.s) > 1e-8
    np.testing.assert_array_equal(multi["pr"], rt.permute_ratio)
    assert _rel(multi["se"][:, live], rt.std_errs[:, live]) <= 1e-10
    assert _rel(multi["br"][:, live], rt.boot_ratios[:, live]) <= 1e-10
    np.testing.assert_allclose(multi["lo"][:, live], rt.conf_ints[0][:, live], rtol=1e-9)
