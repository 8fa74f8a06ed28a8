"""Bias-corrected percentile intervals (Efron) and `prop`, the share of bootstrap samples at or below the original value
(DESIGN.md section 5.8): `percentile_kernel<GLOBAL, true>` against a numpy restatement of the definition, the
design-side `bias_corrected_conf_ints()` of all six methods, and the streamed `salience_bias_corrected_intervals()` of
the task methods -- in voxel chunks, with float32 X, voxel-sharded over two processes and through the plug-in.

Restatement: prop = mean(samples <= theta); prop 0 or 1 (or theta NaN) gives NaN bounds; otherwise the bounds are the
percentile interval (the interpolation of `test_gpu_percentile._ref_ci`) at the levels Phi(2 Phi^-1(prop) +
Phi^-1(q)).  Tolerance 1e-12: the sort and the count are exact; CUDA's normcdf / normcdfinv and scipy's differ in the
last bits, which moves an interpolation weight by about B ulp."""
import os
import socket
import traceback

import numpy as np
import pytest
from scipy.stats import norm

from test_gpu_parity import _load, _run_product

pytestmark = pytest.mark.gpu


def _interp(sorted_series, level):
    B = sorted_series.shape[0]
    x = np.concatenate(([0], (np.arange(0.5, B - 0.5 + 1) / B) * 100, [100]))
    y = np.concatenate(([sorted_series[0]], sorted_series, [sorted_series[-1]]))
    return np.interp(level * 100, x, y)


def _ref_bc(M, theta, conf):
    """(lower, upper, prop) of a (B x ...) stack with original values `theta` shaped like M[0]"""
    M = np.asarray(M, dtype=float)
    B = M.shape[0]
    flat = M.reshape(B, -1)
    th = np.broadcast_to(np.asarray(theta, dtype=float), M.shape[1:]).reshape(-1)
    prop = (flat <= th).mean(axis=0)
    prop[np.isnan(th)] = np.nan
    lo = np.full(th.shape, np.nan); hi = np.full(th.shape, np.nan)
    S = np.sort(flat, axis=0)
    for j in range(flat.shape[1]):
        if 0 < prop[j] < 1:
            z0 = norm.ppf(prop[j])
            lo[j] = _interp(S[:, j], norm.cdf(2 * z0 + norm.ppf(conf[0])))
            hi[j] = _interp(S[:, j], norm.cdf(2 * z0 + norm.ppf(conf[1])))
    return lo.reshape(M.shape[1:]), hi.reshape(M.shape[1:]), prop.reshape(M.shape[1:])


def _assert_bc(got, M, theta, conf, tol=1e-12):
    lo, hi, prop = (np.asarray(g) for g in got)
    rlo, rhi, rprop = _ref_bc(M, theta, conf)
    np.testing.assert_array_equal(prop, rprop)                       # an exact count over B
    np.testing.assert_array_equal(np.isnan(lo), np.isnan(rlo))
    np.testing.assert_array_equal(np.isnan(hi), np.isnan(rhi))
    np.testing.assert_allclose(lo, rlo, rtol=tol, atol=tol)
    np.testing.assert_allclose(hi, rhi, rtol=tol, atol=tol)


def _engine():
    from plspy_b200.engine import Engine
    return Engine(np.random.RandomState(0).standard_normal((4, 8)))


# ---- the kernel ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 2, 7, 100, 511, 512, 513, 1000, 5000, 8192, 10000, 16384, 20000])
def test_kernel_matches_the_definition(B):
    """series lengths on both sides of every padding boundary, incl. the global-memory path (> 16384 samples), on a
    strided (B x m x n) stack: heavy ties with theta on a tied value, a constant series, theta below the minimum, at
    the maximum, above it and NaN"""
    rs = np.random.RandomState(B)
    m, n = (3, 4) if B <= 5000 else (2, 3)
    M = rs.standard_normal((B, m, n)) * 3.0 + 1.0
    theta = M[rs.randint(0, B), :, :] + 0.1 * rs.standard_normal((m, n))
    M[:, 0, 0] = np.round(M[:, 0, 0])                        # heavy ties, theta one of the tied values
    theta[0, 0] = np.sort(M[:, 0, 0])[B // 3]
    if B > 2:
        M[:, 1, 1] = 7.0                                     # a constant series at theta: prop 1
        theta[1, 1] = 7.0
    theta[0, 1] = M[:, 0, 1].min() - 1.0                     # prop 0
    theta[0, 2] = M[:, 0, 2].max()                           # prop 1
    theta[1, 0] = M[:, 1, 0].max() + 1.0
    theta[1, 2] = np.nan
    eng = _engine()
    for conf in ((0.025, 0.975), (0.0, 1.0), (0.1, 0.9), (0.3, 0.31)):
        _assert_bc(eng.to_host(*eng.percentile_interval_bc(M, theta, conf)), M, theta, conf)
    lo, hi, prop = eng.to_host(*eng.percentile_interval_bc(M, theta, (0.025, 0.975)))
    assert prop[0, 1] == 0 and prop[0, 2] == 1 and prop[1, 0] == 1 and np.isnan(prop[1, 2])
    assert np.isnan(lo[0, 1]) and np.isnan(hi[0, 2]) and np.isnan(lo[1, 2])


@pytest.mark.parametrize("B", [2, 100, 1000, 5000, 8192, 20000])
def test_theta_at_the_median_gives_the_plain_percentile_interval(B):
    """prop = 1/2 exactly (theta between the two middle samples): z0 = 0 and the levels are the quantiles"""
    rs = np.random.RandomState(B + 1)
    M = rs.standard_normal((B, 3, 5))
    S = np.sort(M, axis=0)
    theta = 0.5 * (S[B // 2 - 1] + S[B // 2])
    eng = _engine()
    for conf in ((0.025, 0.975), (0.0, 1.0), (0.2, 0.7)):
        lo, hi, prop = eng.to_host(*eng.percentile_interval_bc(M, theta, conf))
        plo, phi = eng.to_host(*eng.percentile_interval(M, conf))
        assert (prop == 0.5).all()
        np.testing.assert_allclose(lo, plo, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(hi, phi, rtol=1e-12, atol=1e-12)


def test_kernel_argument_errors():
    from plspy_b200._lib import PlsB200Error
    eng = _engine()
    M = np.random.RandomState(1).standard_normal((50, 2, 2))
    with pytest.raises(PlsB200Error):
        eng.percentile_interval_bc(M, M[0], (-0.1, 0.9))
    with pytest.raises(ValueError):
        eng.percentile_interval_bc(M, M[0, 0], (0.1, 0.9))


# ---- the design side -----------------------------------------------------------------------------------------------
DESIGNS = ["mct_m0_bal", "cst_bal", "rb_bal", "csb_square", "mb_bscan", "cmb_full"]


@pytest.mark.parametrize("name", DESIGNS)
def test_design_side_intervals_match_the_definition(name):
    """the golden designs with 200 bootstraps; the centres are those of the normal-theory intervals"""
    g = _load(name)
    res = _run_product(g, num_perm=0, num_boot=200)
    rt = res.resample_tests
    method = str(g["method"])
    centres = {}
    if method in ("mct", "cst", "mb", "cmb"):
        centres["Tdistrib"] = rt._Tvsc_orig
        ci = rt.conf_ints_T if method in ("mb", "cmb") else rt.conf_ints
        np.testing.assert_allclose(0.5 * (ci[0] + ci[1]), rt._Tvsc_orig, rtol=1e-12, atol=1e-12)
    if method in ("rb", "csb", "mb", "cmb"):
        centres["left_sv_sampled"] = rt._lvcorrs_orig
        np.testing.assert_allclose(rt._lvcorrs_orig, res.lvintercorrs if method == "csb" else res.lvcorrs, rtol=0)
        ci = rt.conf_ints
        np.testing.assert_allclose(0.5 * (ci[0] + ci[1]), np.broadcast_to(rt._lvcorrs_orig, ci[0].shape),
                                   rtol=1e-12, atol=1e-12)
    for conf in (None, (0.05, 0.95)):
        got = rt.bias_corrected_conf_ints(conf)
        assert set(got) == set(centres)
        c = rt._default_conf(conf)
        for key, theta in centres.items():
            _assert_bc(got[key], rt.boot_debug_dict[key], theta, c)
            assert 0 < np.nanmean(got[key][2]) < 1


# ---- the brain saliences -------------------------------------------------------------------------------------------
GROUPS, C, P, NBOOT = (7, 6), 3, 700, 150


def _task_run(method, X=None, **kw):
    import plspy_b200
    rs = np.random.RandomState(11)
    if X is None:
        X = rs.standard_normal((sum(GROUPS) * C, P)); X[:7, :80] += 1.0
    if method == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(GROUPS) * C, 2))
    np.random.seed(5)
    return plspy_b200.PLS(X.copy(), GROUPS, C, num_perm=0, num_boot=NBOOT, pls_method=method, **kw)


def _numerator(res, method):
    """the numerator of boot_ratios from the result fields: the brain saliences (`U` of the result) x s for mct, the
    brain saliences for cst"""
    return res.U * res.s if method == "mct" else res.U


CHUNK = NBOOT * 8 * 8 * 256          # at most 256 voxels of K <= 8 per chunk: three or more chunks of 700 voxels


@pytest.mark.parametrize("method", ["mct", "cst"])
def test_salience_intervals_match_the_explicit_cube(method):
    res = _task_run(method)
    rt = res.resample_tests
    cube = np.asarray(rt.boot_debug_dict["right_sv_sampled"])
    theta = _numerator(res, method)
    assert cube.shape[1:] == theta.shape
    for conf in (None, (0.1, 0.9), (0.0, 1.0)):
        got = rt.salience_bias_corrected_intervals(conf, max_bytes=CHUNK)
        assert all(a.shape == theta.shape for a in got)
        _assert_bc(got, cube, theta, rt._default_conf(conf), tol=1e-11)
    # one chunk: the same values
    one = rt.salience_bias_corrected_intervals(max_bytes=1 << 30)
    for a, b in zip(one, rt.salience_bias_corrected_intervals(max_bytes=CHUNK)):
        np.testing.assert_array_equal(a, b)


def test_float32_x_is_bit_identical_to_float64_on_the_widened_matrix():
    X = np.random.RandomState(11).standard_normal((sum(GROUPS) * C, P)).astype(np.float32)
    a = _task_run("mct", X=X, x_storage="fp32").resample_tests
    b = _task_run("mct", X=X.astype(np.float64)).resample_tests
    assert a._engine.X.dtype.itemsize == 4
    for x, y in zip(a.salience_bias_corrected_intervals(max_bytes=CHUNK),
                    b.salience_bias_corrected_intervals(max_bytes=CHUNK)):
        np.testing.assert_array_equal(x, y)
    ga, gb = a.bias_corrected_conf_ints(), b.bias_corrected_conf_ints()
    assert ga.keys() == gb.keys()
    for key in ga:
        for x, y in zip(ga[key], gb[key]):
            np.testing.assert_array_equal(x, y)


def test_error_paths():
    import plspy_b200
    from plspy_b200 import exceptions
    g = _load("rb_bal")
    rt = _run_product(g, num_perm=0, num_boot=40).resample_tests
    with pytest.raises(exceptions.NotImplementedError):
        rt.salience_bias_corrected_intervals()
    rs = np.random.RandomState(2)
    res = plspy_b200.PLS(rs.standard_normal((30, 50)), (5, 5), 3, num_perm=5, num_boot=0, pls_method="mct")
    with pytest.raises(exceptions.MissingParameterError):
        res.resample_tests.bias_corrected_conf_ints()
    with pytest.raises(exceptions.MissingParameterError):
        res.resample_tests.salience_bias_corrected_intervals()
    rt = _task_run("mct").resample_tests
    for conf in ((-0.1, 0.9), (0.1, 1.5)):
        with pytest.raises(ValueError):
            rt.bias_corrected_conf_ints(conf)
        with pytest.raises(ValueError):
            rt.salience_bias_corrected_intervals(conf)


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
            out[method] = rt.salience_bias_corrected_intervals(max_bytes=CHUNK)
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
        single = _task_run(method).resample_tests.salience_bias_corrected_intervals(max_bytes=CHUNK)
        for rank in range(2):
            for a, b in zip(got[rank][method], single):
                np.testing.assert_array_equal(a, b)


# ---- the plug-in ---------------------------------------------------------------------------------------------------
def test_plugin_result_has_the_bias_corrected_intervals():
    """Through the reference's own `PLS` when it is installed; otherwise through the registered class with the
    reference's positional signature (what its `ResampleTest._create` calls)."""
    import baseline
    import plspy_b200
    from plspy_b200 import plugin
    rs = np.random.RandomState(11)
    X = rs.standard_normal((sum(GROUPS) * C, P)); X[:7, :80] += 1.0
    if baseline.reference_available():
        import contextlib
        import io
        import warnings
        mod = baseline.import_reference()
        plspy_b200.install(mod)
        try:
            np.random.seed(5)
            with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = mod.PLS(X.copy(), GROUPS, C, num_perm=0, num_boot=NBOOT, pls_method="mct")
            rt, theta = res.resample_tests, res.U * res.s
            assert isinstance(rt, plugin.PINNED["mct"])
            got = rt.salience_bias_corrected_intervals(max_bytes=CHUNK)
            cube = np.asarray(rt.boot_debug_dict["right_sv_sampled"])
        finally:
            plspy_b200.uninstall()
    else:
        ref = _task_run("mct")                 # the result's U / V are the brain / design saliences: swapped here
        U, s, V = ref.V.copy(), np.array(ref.s, dtype=float), ref.U.copy()
        np.random.seed(5)
        try:
            rt = plugin.PINNED["mct"](X.copy(), None, U, s, V, ref.cond_order, ref.mctype, nperm=0, nboot=NBOOT,
                                      Tvsc_orig=ref.resample_tests._Tvsc_orig, CI=0.95)
            got = rt.salience_bias_corrected_intervals(max_bytes=CHUNK)
            cube = np.asarray(rt.boot_debug_dict["right_sv_sampled"])
            dc = rt.bias_corrected_conf_ints()
            _assert_bc(dc["Tdistrib"], rt.boot_debug_dict["Tdistrib"], ref.resample_tests._Tvsc_orig,
                       rt._default_conf(None))
        finally:
            plugin._drop_engine()
        theta = V * s
    _assert_bc(got, cube, theta, (0.025, 0.975), tol=1e-11)
