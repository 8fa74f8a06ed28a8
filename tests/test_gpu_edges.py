"""Edge cases of the CUDA path against the oracle: ragged/odd designs, wide column counts, tiny voxel
counts, single resamples.  Same tolerances as test_gpu_parity.py."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


def _data(groups, C, p, nb=0, seed=0):
    rs = np.random.RandomState(seed)
    N = sum(groups) * C
    X = rs.standard_normal((N, p)) + 2.0
    X[: groups[0], : max(1, p // 8)] += 1.0
    Y = rs.standard_normal((N, nb)) + 0.4 * X[:, :nb] if nb else None
    return X, Y


def _both(method, groups, C, p, nb=0, L=0, mctype=0, bscan=None, nperm=9, nboot=9, nsplit=0, lv=1, seed=0):
    import plspy_b200
    X, Y = _data(groups, C, p, nb, seed)
    rs = np.random.RandomState(seed + 1)
    G = len(groups)
    contrasts = None
    if L:
        K = {"cst": G * C, "csb": G * C * nb, "cmb": G * (C + C * nb)}[method]
        contrasts = np.linalg.qr(rs.standard_normal((K, L)))[0]
    np.random.seed(100 + seed)
    o = oracle.run_full(method, X.copy(), groups, C, Y=None if Y is None else Y.copy(), contrasts=contrasts,
                        mctype=mctype, bscan=bscan, nperm=nperm, nboot=nboot, nsplit=nsplit, lv=lv)
    kw = dict(num_perm=nperm, num_boot=nboot, pls_method=method)
    if method in ("mct", "cst", "mb", "cmb"):
        kw["mctype"] = mctype
    if Y is not None:
        kw["Y"] = Y.copy()
    if contrasts is not None:
        kw["contrasts"] = contrasts.copy()
    if bscan is not None:
        kw["bscan"] = list(bscan)
    if nsplit:
        kw.update(num_split=nsplit, lv=lv)
    np.random.seed(100 + seed)
    res = plspy_b200.PLS(X.copy(), groups, C, **kw)
    return o, res


def _check(o, res, nsplit=0):
    rt = res.resample_tests
    live = np.abs(o["s"]) > 1e-8
    if "perm" in o:
        np.testing.assert_array_equal(rt.permute_ratio, o["perm"]["permute_ratio"])
        np.testing.assert_array_equal(rt.stepdown_ratio, o["perm"]["stepdown_ratio"])
    if "boot" in o:
        np.testing.assert_allclose(rt.std_errs[:, live], o["boot"]["std_errs"][:, live], rtol=1e-8)
        np.testing.assert_allclose(rt.boot_ratios[:, live], o["boot"]["boot_ratios"][:, live], rtol=1e-8)
        np.testing.assert_allclose(rt.conf_ints[0][:, live], o["boot"]["conf_ints"][0][:, live], rtol=1e-7, atol=1e-9)
        if "LVcorr" in o["boot"]:
            np.testing.assert_allclose(rt.LVcorr[:, :, live], o["boot"]["LVcorr"][:, :, live], rtol=1e-7, atol=1e-9)
    if nsplit:
        nl = max(1, int(live.sum()) - 1)
        a, b = res.pls_repro_tt["pls_s_test"], o["tt"]["pls_s_test"]
        d = np.arange(min(nl, a.shape[0]))
        np.testing.assert_allclose(a[d, d, :], b[d, d, :], rtol=1e-7, atol=1e-9)
        a, b = res.pls_repro_sh["pls_dist_u"], o["sh"]["pls_dist_u"]
        np.testing.assert_allclose(np.abs(a[d, d, :]), np.abs(b[d, d, :]), rtol=1e-7, atol=1e-9)
        a, b = res.pls_repro_sh["pls_dist_null_v"], o["sh"]["pls_dist_null_v"]
        np.testing.assert_allclose(np.abs(a[d, d, :]), np.abs(b[d, d, :]), rtol=1e-7, atol=1e-9)


def test_odd_group_sizes_split_half_mct():
    o, res = _both("mct", (5, 7, 3), 3, 300, nsplit=6, lv=2, seed=1)      # halves of 2/3, 3/4, 1/2 subjects
    _check(o, res, nsplit=6)


def test_odd_group_sizes_split_half_rb():
    o, res = _both("rb", (9, 7), 2, 200, nb=2, nsplit=5, lv=1, seed=2)   # halves 4/5 and 3/4: full-rank blocks
    _check(o, res, nsplit=5)


def test_wide_behaviour_design_k48():
    """rb with 3 groups x 4 conditions x 4 behaviours: 48 latent variables (> 24 columns per launch)."""
    o, res = _both("rb", (9, 8, 9), 4, 400, nb=4, nperm=7, nboot=7, seed=3)
    _check(o, res)


def test_wide_behaviour_design_k48_split_half():
    """the same 48-LV design with num_split > 0: the split-half SVDs go through the CTA-level Jacobi solver
    (np.linalg.svd in the reference has no size limit: class_functions.py:122, split_half_resampling.py:194, 612)."""
    # (groups of 11-12 subjects: every half block keeps >= 5 subjects, so the 4 behaviours of a block stay full rank
    # and all 48 latent variables of the halves are live)
    o, res = _both("rb", (12, 11, 12), 4, 400, nb=4, nperm=3, nboot=3, nsplit=4, lv=2, seed=3)
    _check(o, res, nsplit=4)


def test_tiny_voxel_counts():
    for p in (1, 7, 65):
        o, res = _both("mct", (6, 6), 2, p, nperm=5, nboot=5, seed=10 + p)
        rt = res.resample_tests
        np.testing.assert_array_equal(rt.permute_ratio, o["perm"]["permute_ratio"])
        live = np.abs(o["s"]) > 1e-8
        np.testing.assert_allclose(rt.std_errs[:, live], o["boot"]["std_errs"][:, live], rtol=1e-8, atol=1e-12)


def test_single_resample():
    o, res = _both("mct", (6, 5), 3, 120, nperm=1, nboot=1, seed=4)
    np.testing.assert_array_equal(res.resample_tests.permute_ratio, o["perm"]["permute_ratio"])
    # std over one bootstrap is exactly 0; streaming moments leave sqrt(eps)-level noise relative to |VS - pivot|
    assert np.all(res.resample_tests.std_errs[:, np.abs(o["s"]) > 1e-8] < 1e-7)


def test_multiblock_mctype3_bscan_single():
    o, res = _both("mb", (6, 7), 3, 250, nb=2, mctype=3, bscan=(1,), nperm=8, nboot=8, nsplit=4, lv=1, seed=5)
    _check(o, res, nsplit=4)


def test_cst_single_contrast_and_cmb():
    o, res = _both("cst", (7, 7), 3, 180, L=1, nperm=8, nboot=8, nsplit=4, lv=1, seed=6)
    _check(o, res, nsplit=4)
    o, res = _both("cmb", (6, 6), 2, 160, nb=2, L=2, nperm=6, nboot=6, seed=7)
    _check(o, res)


@pytest.mark.parametrize("groups,C,p", [((60, 60), 3, 300), ((40, 45, 35), 6, 300), ((40, 45, 35), 6, 301),
                                        ((150, 160, 150), 3, 140)])
def test_tall_designs(groups, C, p):
    """N > 320 rows (360, 720, 720 with an odd voxel count, 1380): the output-stationary bootstrap GEMM
    (boot_os.cu), both operands staged through shared memory."""
    o, res = _both("mct", groups, C, p, nperm=4, nboot=11, seed=8)
    _check(o, res)


def test_wide_k_fails_loudly():
    """more than 24 columns per launch are split by the engine, but the kernels themselves refuse K > 24"""
    from plspy_b200 import _lib
    assert _lib.lib.plsb200_boot_coef_bytes(300, 25, 10) == 0


def test_pinned_tensor_input_and_float32_storage():
    """X assembled by plspy_b200.io into pinned host memory is uploaded as it is; float32 storage (half the PCIe
    bytes, widened on the device) gives the results of the float64 analysis of the same numbers"""
    import plspy_b200
    from plspy_b200 import io
    rs = np.random.RandomState(5)
    sizes, C, p = (6, 5), 3, 700
    groups = [[[rs.standard_normal(p).astype(np.float32) for _ in range(C)] for _ in range(n)] for n in sizes]
    X64, gs, nc = io.assemble_pinned(groups, dtype=np.float64)
    X32, _, _ = io.assemble_pinned(groups, dtype=np.float32)
    assert X64.is_pinned() and X32.is_pinned()
    out = []
    for X in (X64.numpy().copy(), X64, X32):
        np.random.seed(3)
        out.append(plspy_b200.PLS(X, gs, nc, num_perm=20, num_boot=20, pls_method="mct", analysis="device"))
    ref = out[0].resample_tests
    for r in out[1:]:
        np.testing.assert_array_equal(r.resample_tests.permute_ratio, ref.permute_ratio)
        np.testing.assert_allclose(r.resample_tests.std_errs, ref.std_errs, rtol=1e-12)
        np.testing.assert_allclose(r.s, out[0].s, rtol=1e-12)
    np.random.seed(3)
    host = plspy_b200.PLS(X64, gs, nc, num_perm=20, num_boot=20, pls_method="mct")      # host analysis on the numpy view
    np.testing.assert_array_equal(host.resample_tests.permute_ratio, ref.permute_ratio)


@pytest.mark.parametrize("N,p,threads", [(7, 1000, 8), (300, 5000, 4), (33, 70001, 3), (2, 64, 2)])
def test_staged_upload_of_a_pageable_matrix_is_exact(N, p, threads, monkeypatch):
    """Engine._upload_pageable (pinned staging buffers filled by several host threads): forced onto small matrices --
    fewer rows than threads, several blocks per staging buffer, odd widths -- and compared bit for bit"""
    from plspy_b200.engine import Engine
    X = np.random.RandomState(N + p).standard_normal((N, p))
    monkeypatch.setattr(Engine, "PIPELINED_UPLOAD_MIN_BYTES", 1)
    monkeypatch.setattr(Engine, "PAGEABLE_UPLOAD_THREADS", threads)
    monkeypatch.setattr(Engine, "STAGING_BLOCK_BYTES", 64 * 1024)
    for _ in range(2):                                   # second engine: staging buffers reused
        eng = Engine(X)
        assert np.array_equal(eng.X.cpu().numpy(), X)
    np.testing.assert_allclose(eng.G.cpu().numpy(), X @ X.T, rtol=1e-12, atol=1e-10)
