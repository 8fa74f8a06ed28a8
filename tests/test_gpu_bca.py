"""Bias-corrected and accelerated (BCa) percentile intervals (DESIGN.md section 5.8): `percentile_kernel<GLOBAL, PC_BCA>`
against a numpy restatement of the definition, and the streamed `salience_bca_intervals()` of the task methods against
the explicit `right_sv_sampled` cube and the oracle's leave-one-subject-out jackknife -- in voxel chunks, with float32
X, voxel-sharded over two processes and through the plug-in.

Restatement: prop and z0 = Phi^-1(prop) as in the bias-corrected interval (`test_gpu_bias_corrected._ref_bc`); with
w = z0 + Phi^-1(q) the level is Phi(z0 + w / (1 - a w)), NaN where 1 - a w <= 0; q = 0 / 1 keep the minimum / maximum;
the bound is the percentile interpolation (`_interp`) at that level.  The acceleration is `test_bca_host.accel_ref` of
`test_bca_host.jackknife_values`."""
import os
import socket
import traceback

import numpy as np
import pytest
from scipy.stats import norm

from test_bca_host import accel_ref, jackknife_values
from test_gpu_bias_corrected import _interp, _ref_bc
from test_gpu_parity import _load, _run_product

pytestmark = pytest.mark.gpu


def _ref_bca(M, theta, accel, conf):
    """(lower, upper, prop) of a (B x ...) stack with original values `theta` and accelerations `accel`"""
    M = np.asarray(M, dtype=float)
    B = M.shape[0]
    shape = M.shape[1:]
    _, _, prop = _ref_bc(M, theta, conf)
    prop = prop.reshape(-1)
    a = np.broadcast_to(np.asarray(accel, dtype=float), shape).reshape(-1)
    S = np.sort(M.reshape(B, -1), axis=0)
    out = []
    for q in conf:
        b = np.full(prop.shape, np.nan)
        for j in range(prop.size):
            if not 0 < prop[j] < 1:
                continue
            if q in (0.0, 1.0):
                level = q
            else:
                z0 = norm.ppf(prop[j])
                w = z0 + norm.ppf(q)
                den = 1.0 - a[j] * w
                if not den > 0:
                    continue
                level = norm.cdf(z0 + w / den)
            b[j] = _interp(S[:, j], level)
        out.append(b.reshape(shape))
    return out[0], out[1], prop.reshape(shape)


def _assert_bca(got, M, theta, accel, conf, tol=1e-11):
    lo, hi, prop = (np.asarray(g) for g in got[:3])
    rlo, rhi, rprop = _ref_bca(M, theta, accel, conf)
    np.testing.assert_array_equal(prop, rprop)                       # an exact count over B
    np.testing.assert_array_equal(np.isnan(lo), np.isnan(rlo))
    np.testing.assert_array_equal(np.isnan(hi), np.isnan(rhi))
    np.testing.assert_allclose(lo, rlo, rtol=tol, atol=tol)
    np.testing.assert_allclose(hi, rhi, rtol=tol, atol=tol)


def _engine():
    from plspy_b200.engine import Engine
    return Engine(np.random.RandomState(0).standard_normal((4, 8)))


def _launches():
    from plspy_b200 import _lib
    return _lib.launch_count()


# ---- the kernel ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [2, 7, 100, 513, 1000, 5000, 16384, 20000])
def test_kernel_matches_the_definition(B):
    """series lengths on both sides of the padding boundaries, incl. the global-memory path (> 16384 samples), on a
    strided (B x m x n) stack: prop 0 and 1, a NaN theta, accelerations of both signs, 0, NaN, and ones large enough
    that 1 - a w <= 0 for one bound"""
    rs = np.random.RandomState(B + 7)
    m, n = 3, 4
    M = rs.standard_normal((B, m, n)) * 3.0 + 1.0
    theta = M[rs.randint(0, B), :, :] + 0.1 * rs.standard_normal((m, n))
    accel = 0.05 * rs.standard_normal((m, n))
    theta[0, 1] = M[:, 0, 1].min() - 1.0                     # prop 0
    theta[0, 2] = M[:, 0, 2].max()                           # prop 1
    theta[1, 2] = np.nan
    S = np.sort(M, axis=0)
    theta[1, 1], theta[2, 0] = (0.5 * (S[(B - 1) // 2, i, j] + S[B // 2, i, j]) for i, j in ((1, 1), (2, 0)))
    accel[1, 0] = 0.0
    accel[1, 1] = 0.6                    # theta at the median (z0 ~ 0): 1 - a w <= 0 for the upper bound (w ~ +2)
    accel[2, 0] = -0.6                   # ... and for the lower bound (w ~ -2)
    accel[2, 1] = np.nan
    eng = _engine()
    for conf in ((0.025, 0.975), (0.0, 1.0), (0.1, 0.9), (0.3, 0.31)):
        _assert_bca(eng.to_host(*eng.percentile_interval_bca(M, theta, accel, conf)), M, theta, accel, conf)
    lo, hi, prop = eng.to_host(*eng.percentile_interval_bca(M, theta, accel, (0.025, 0.975)))
    assert prop[0, 1] == 0 and prop[0, 2] == 1 and np.isnan(prop[1, 2])
    assert np.isnan(lo[0, 1]) and np.isnan(hi[0, 2]) and np.isnan(lo[1, 2]) and np.isnan(lo[2, 1])
    assert np.isnan(hi[1, 1]) and not np.isnan(lo[1, 1])
    assert np.isnan(lo[2, 0]) and not np.isnan(hi[2, 0])
    # q = 0 / 1: the minimum / maximum, whatever the acceleration
    lo, hi, prop = eng.to_host(*eng.percentile_interval_bca(M, theta, accel, (0.0, 1.0)))
    live = (prop > 0) & (prop < 1)
    np.testing.assert_array_equal(lo[live], M.min(axis=0)[live])
    np.testing.assert_array_equal(hi[live], M.max(axis=0)[live])


@pytest.mark.parametrize("B", [2, 1000, 5000, 20000])
def test_zero_acceleration_gives_the_bias_corrected_interval(B):
    rs = np.random.RandomState(B + 3)
    M = rs.standard_normal((B, 3, 5))
    theta = M[rs.randint(0, B)] + 0.2 * rs.standard_normal((3, 5))
    theta[0, 0] = np.nan
    theta[1, 1] = M[:, 1, 1].max() + 1
    eng = _engine()
    for conf in ((0.025, 0.975), (0.0, 1.0), (0.2, 0.7)):
        got = eng.to_host(*eng.percentile_interval_bca(M, theta, np.zeros((3, 5)), conf))
        bc = eng.to_host(*eng.percentile_interval_bc(M, theta, conf))
        for x, y in zip(got, bc):
            np.testing.assert_array_equal(x, y)


def test_kernel_argument_errors():
    from plspy_b200._lib import PlsB200Error
    eng = _engine()
    M = np.random.RandomState(1).standard_normal((50, 2, 2))
    with pytest.raises(PlsB200Error):
        eng.percentile_interval_bca(M, M[0], M[1], (-0.1, 0.9))
    with pytest.raises(ValueError):
        eng.percentile_interval_bca(M, M[0], M[1, 0], (0.1, 0.9))


# ---- the brain saliences -------------------------------------------------------------------------------------------
GROUPS, C, P, NBOOT = (7, 6), 3, 700, 150


def _chunk(rt):
    """a budget of 256 voxels for the bootstrap and jackknife chunks together: chunks of 256, 256 and 188 voxels"""
    return (NBOOT + sum(GROUPS)) * rt.boot_ratios.shape[1] * 8 * 256 + 13


def _data():
    X = np.random.RandomState(11).standard_normal((sum(GROUPS) * C, P)); X[:7, :80] += 1.0
    X[:, 100:200] = np.exp(X[:, 100:200])                 # skewed voxels: accelerations well away from 0
    return X


def _task_run(method, X=None, mctype=0, **kw):
    import plspy_b200
    if X is None:
        X = _data()
    if method == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(GROUPS) * C, 2))
    else:
        kw["mctype"] = mctype
    np.random.seed(5)
    return plspy_b200.PLS(X.copy(), GROUPS, C, num_perm=0, num_boot=NBOOT, pls_method=method, **kw)


def _design_weights(res, method):
    """theta (the numerator of boot_ratios), the design weights the saliences are projected on, and the live latent
    variables: a column of U whose singular value is 0 has saliences (and jackknife values) of rounding size only,
    whose acceleration is that of the rounding"""
    import oracle
    if method == "mct":
        s = np.asarray(res.s, dtype=float)
        return res.U * s, res.V, np.abs(s) > 1e-8 * np.abs(s).max()
    K = res.U.shape[1]
    return res.U, oracle.normalize(np.random.RandomState(1).standard_normal((len(GROUPS) * C, 2))), np.ones(K, bool)


def _assert_salience_bca(got, cube, theta, a_ref, conf, live):
    """the live latent variables against the restatement; prop of every one against the count on the cube"""
    np.testing.assert_allclose(got[3][:, live], a_ref[:, live], rtol=1e-10, atol=1e-10)
    _assert_bca([g[:, live] for g in got[:3]], cube[:, :, live], theta[:, live], a_ref[:, live], conf, tol=1e-11)
    np.testing.assert_array_equal(got[2], _ref_bc(cube, theta, conf)[2])


@pytest.mark.parametrize("method, mctype", [("mct", 0), ("mct", 1), ("mct", 2), ("mct", 3), ("cst", 0)])
def test_salience_intervals_match_the_restatement(method, mctype):
    res = _task_run(method, mctype=mctype)
    rt = res.resample_tests
    cube = np.asarray(rt.boot_debug_dict["right_sv_sampled"])
    theta, Ucoef, live = _design_weights(res, method)
    assert live.sum() >= 2
    co = np.asarray(res.cond_order)
    jv = jackknife_values(method, _data(), co, mctype, Ucoef)
    a_ref = accel_ref(jv, np.concatenate(([0], np.cumsum(co[:, 0]))), theta)
    assert np.abs(a_ref[:, live]).max() > 0.05
    for conf in (None, (0.1, 0.9), (0.0, 1.0)):
        got = rt.salience_bca_intervals(conf, max_bytes=_chunk(rt))
        assert len(got) == 4 and all(a.shape == theta.shape for a in got)
        _assert_salience_bca(got, cube, theta, a_ref, rt._default_conf(conf), live)
        bc = rt.salience_bias_corrected_intervals(conf, max_bytes=_chunk(rt))
        np.testing.assert_array_equal(got[2], bc[2])
    one = rt.salience_bca_intervals(max_bytes=1 << 30)
    for x, y in zip(one, rt.salience_bca_intervals(max_bytes=_chunk(rt))):
        np.testing.assert_array_equal(x, y)


def test_float32_x_is_bit_identical_to_float64_on_the_widened_matrix():
    rs = np.random.RandomState(11)
    X = rs.standard_normal((sum(GROUPS) * C, P)).astype(np.float32)
    a = _task_run("mct", X=X, x_storage="fp32").resample_tests
    b = _task_run("mct", X=X.astype(np.float64)).resample_tests
    assert a._engine.X.dtype.itemsize == 4
    for x, y in zip(a.salience_bca_intervals(max_bytes=_chunk(a)), b.salience_bca_intervals(max_bytes=_chunk(b))):
        np.testing.assert_array_equal(x, y)


def test_error_paths_launch_nothing():
    import plspy_b200
    from plspy_b200 import exceptions
    rs = np.random.RandomState(2)
    rb = _run_product(_load("rb_bal"), num_perm=0, num_boot=40).resample_tests
    no_boot = plspy_b200.PLS(rs.standard_normal((30, 50)), (5, 5), 3, num_perm=5, num_boot=0, pls_method="mct")
    rt = _task_run("mct").resample_tests
    np.random.seed(3)
    lone = plspy_b200.PLS(rs.standard_normal((7 * C, 40)), (6, 1), C, num_perm=0, num_boot=20,
                          pls_method="mct").resample_tests           # a group of one subject: no jackknife
    n0 = _launches()
    with pytest.raises(exceptions.NotImplementedError):
        rb.salience_bca_intervals()
    with pytest.raises(exceptions.MissingParameterError):
        no_boot.resample_tests.salience_bca_intervals()
    for conf in ((-0.1, 0.9), (0.1, 1.5)):
        with pytest.raises(ValueError):
            rt.salience_bca_intervals(conf)
    with pytest.raises(exceptions.NotImplementedError, match="group 1 has 1 subject"):
        lone.salience_bca_intervals()
    assert _launches() == n0


# ---- voxel sharding: two processes on one GPU over gloo ------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _rank(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out = {}
        for method in ("mct", "cst"):
            rt = _task_run(method, shard="voxels").resample_tests
            assert rt._engine.voxel_sharded
            out[method] = rt.salience_bca_intervals(max_bytes=_chunk(rt))
        q.put((rank, out))
    except BaseException:
        q.put((rank, traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def test_voxel_sharded_salience_intervals_equal_the_single_process_ones():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    got = {}
    try:
        for _ in range(2):
            rank, out = q.get(timeout=900)
            if isinstance(out, str):
                raise AssertionError(f"rank {rank} failed:\n{out}")
            got[rank] = out
    finally:
        for pr in procs:
            pr.join(timeout=300)
            if pr.is_alive():
                pr.terminate()
                pr.join(timeout=60)
    assert all(pr.exitcode == 0 for pr in procs)
    for method in ("mct", "cst"):
        rt = _task_run(method).resample_tests
        single = rt.salience_bca_intervals(max_bytes=_chunk(rt))
        for rank in range(2):
            for a, b in zip(got[rank][method], single):
                np.testing.assert_array_equal(a, b)


# ---- the plug-in ---------------------------------------------------------------------------------------------------
def test_plugin_result_has_the_bca_intervals():
    """Through the reference's own `PLS` once plspy_b200.install() has replaced its resampling class"""
    import baseline
    import plspy_b200
    from plspy_b200 import plugin
    if not baseline.reference_available():
        pytest.skip("the reference (baseline/_ref) is not installed")
    import contextlib
    import io
    import warnings
    rs = np.random.RandomState(11)
    X = rs.standard_normal((sum(GROUPS) * C, P)); X[:7, :80] += 1.0
    mod = baseline.import_reference()
    plspy_b200.install(mod)
    try:
        np.random.seed(5)
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = mod.PLS(X.copy(), GROUPS, C, num_perm=0, num_boot=NBOOT, pls_method="mct")
        rt = res.resample_tests
        assert isinstance(rt, plugin.PINNED["mct"])
        got = rt.salience_bca_intervals(max_bytes=_chunk(rt))
        cube = np.asarray(rt.boot_debug_dict["right_sv_sampled"])
        theta, Ucoef, live = _design_weights(res, "mct")
    finally:
        plspy_b200.uninstall()
    co = np.array([[n] * C for n in GROUPS])
    a_ref = accel_ref(jackknife_values("mct", X, co, 0, Ucoef), np.concatenate(([0], np.cumsum(GROUPS))), theta)
    _assert_salience_bca(got, cube, theta, a_ref, (0.025, 0.975), live)
