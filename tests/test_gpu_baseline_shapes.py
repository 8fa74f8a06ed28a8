"""Oracle parity AT the BASELINE.json shapes (SURVEY.md section 8, table of configs), with the iteration counts cut to
what the numpy oracle finishes in seconds on the box's host cores -- the shapes (rows, voxels, latent variables,
behaviours, bscan, contrasts) are the full ones, so every kernel runs on the tile counts / k-steps / paddings of the
real workloads:

* cfg 3   cst, 3 x 25 x 4 (N = 300) x 200 000 voxels, L = 3 contrasts          16 perm + 16 boot
* cfg 3m  mct (the north-star target), same design, K = 12                      16 perm + 16 boot
* cfg 4   mb, bscan = [1, 2], 2 x 30 x 4 (N = 240 + 120 bscan rows) x 200 000 voxels, 4 behaviours, K = 24
                                                                                 3 perm + 3 boot + 2 splits (lv = 1)
* cfg 5 shape (rows): mct 4 x 50 x 6 (N = 1200, K = 24) x 200 000 voxels -- the output-stationary DMMA kernel
  `boot_os` that only tall designs reach                                          3 perm + 4 boot

Both sides draw their indices from numpy's global stream after the same seed (the product through its native
generator), so index generation is part of the check.  Tolerances are those of tests/test_gpu_parity.py: p-values and
stepdown ratios exact, permuted singular values 1e-10 (1e-9 for the multiblock rescale), standard errors / bootstrap
ratios 1e-8 for the task methods and 1e-6 for multiblock (BASELINE.json: 1e-4), split-half 1e-7."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


def _planted(seed, groups, C, p, nb=0):
    rs = np.random.RandomState(seed)
    N = sum(groups) * C
    X = rs.standard_normal((N, p))
    ne = p // 20
    row = 0
    for g in groups:
        for _ in range(C):
            X[row:row + g, :ne] += 0.5 * rs.standard_normal(ne)
            row += g
    Y = (rs.standard_normal((N, nb)) + 0.3 * X[:, :nb]) if nb else None
    return rs, X, Y


def _compare_task(res, o, tol=1e-8):
    rt = res.resample_tests
    s = np.asarray(o["s"])
    live = np.abs(s) > 1e-8 * np.abs(s).max()
    np.testing.assert_allclose(res.s[live], s[live], rtol=1e-10)
    np.testing.assert_array_equal(rt.perm_debug_dict["indices"], o["perm_idx_task"])
    np.testing.assert_array_equal(rt.boot_debug_dict["indices"], o["boot_idx"])
    # p-values on the live latent variables: for a rank-deficient design (mctype 0: G (C - 1) of G C) LAPACK's null
    # singular values land at ~1e-11 for 200 000 voxels, above the reference's 1e-12 zero threshold
    # (bootstrap_permutation.py:295), so the reference itself compares rounding noise with rounding noise there --
    # the documented tie class (DESIGN.md section 7)
    np.testing.assert_array_equal(rt.permute_ratio[live], o["perm"]["permute_ratio"][live])
    np.testing.assert_array_equal(rt.stepdown_ratio[live], o["perm"]["stepdown_ratio"][live])
    np.testing.assert_allclose(rt.perm_debug_dict["s_list"][:, live], o["perm"]["s_hat"][:, live], rtol=1e-10)
    np.testing.assert_allclose(rt.std_errs[:, live], o["boot"]["std_errs"][:, live], rtol=tol)
    # (voxels whose original salience is ~0 carry V entries at LAPACK's rounding level, which differ between the two
    # sides' own SVDs of the original data: absolute floor 1e-9 on ratios that are O(1..10) where they matter)
    np.testing.assert_allclose(rt.boot_ratios[:, live], o["boot"]["boot_ratios"][:, live], rtol=tol, atol=1e-9)
    for i in (0, 1):
        np.testing.assert_allclose(rt.conf_ints[i][:, live], o["boot"]["conf_ints"][i][:, live], rtol=1e-8, atol=1e-9)
    np.testing.assert_allclose(rt.boot_debug_dict["Tdistrib"][:, :, live], o["boot"]["Tdistrib"][:, :, live],
                               rtol=1e-8, atol=1e-9)
    return live


def test_cfg3_cst_200k_matches_oracle():
    import plspy_b200
    groups, C, p, L = (25, 25, 25), 4, 200_000, 3
    rs, X, _ = _planted(20260003, groups, C, p)
    contrasts = np.linalg.qr(rs.standard_normal((len(groups) * C, L)))[0]
    np.random.seed(1237)
    o = oracle.run_full("cst", X, groups, C, contrasts=contrasts.copy(), mctype=0, nperm=16, nboot=16)
    np.random.seed(1237)
    res = plspy_b200.PLS(X, groups, C, contrasts=contrasts.copy(), num_perm=16, num_boot=16, mctype=0,
                         pls_method="cst")
    _compare_task(res, o)


def test_cfg3m_mct_200k_matches_oracle():
    import plspy_b200
    groups, C, p = (25, 25, 25), 4, 200_000
    _, X, _ = _planted(20260003, groups, C, p)
    np.random.seed(1237)
    o = oracle.run_full("mct", X, groups, C, mctype=0, nperm=16, nboot=16)
    np.random.seed(1237)
    res = plspy_b200.PLS(X, groups, C, num_perm=16, num_boot=16, mctype=0, pls_method="mct")
    live = _compare_task(res, o)
    rt = res.resample_tests
    np.testing.assert_allclose(rt.boot_debug_dict["left_sv_sampled"][:, :, live],
                               o["boot"]["left_sv_sampled"][:, :, live], rtol=1e-8, atol=1e-9)
    # fast mode on the same resamples: identical p-values, bootstrap ratios inside the north-star 1e-4
    np.random.seed(1237)
    fast = plspy_b200.PLS(X, groups, C, num_perm=16, num_boot=16, mctype=0, pls_method="mct", precision="tf32x3")
    np.testing.assert_array_equal(fast.resample_tests.permute_ratio[live], o["perm"]["permute_ratio"][live])
    np.testing.assert_allclose(fast.resample_tests.boot_ratios[:, live], o["boot"]["boot_ratios"][:, live], rtol=1e-4,
                               atol=1e-9)


def test_cfg5_rows_mct_n1200_matches_oracle():
    """N = 1200 rows (4 x 50 x 6, K = 24): the exact bootstrap GEMM takes the output-stationary kernel
    (csrc/boot_os.cu)."""
    import plspy_b200
    groups, C, p = (50, 50, 50, 50), 6, 200_000
    _, X, _ = _planted(20260005, groups, C, p)
    np.random.seed(1239)
    o = oracle.run_full("mct", X, groups, C, mctype=0, nperm=3, nboot=4)
    np.random.seed(1239)
    res = plspy_b200.PLS(X, groups, C, num_perm=3, num_boot=4, mctype=0, pls_method="mct")
    live = _compare_task(res, o)
    # fast mode, same resamples.  With only 4 bootstraps some voxels draw nearly identical saliences (std_errs a
    # thousandth of the column's typical value), where a RELATIVE bound on 1 / std_errs is meaningless: the standard
    # errors are held to the north-star 1e-4 of the column scale (observed 6e-5 with 4 bootstraps of 1200 rows; the
    # per-bootstrap rounding of the 3xTF32 products averages down with the number of bootstraps: 6e-6 at 5000) and
    # the ratios to 2e-4 wherever the standard error is not degenerate
    np.random.seed(1239)
    fast = plspy_b200.PLS(X, groups, C, num_perm=3, num_boot=4, mctype=0, pls_method="mct", precision="tf32x3")
    se, se_f = o["boot"]["std_errs"][:, live], fast.resample_tests.std_errs[:, live]
    scale = np.median(se, axis=0)
    assert np.max(np.abs(se_f - se) / scale) < 1e-4
    ok = se > 0.5 * scale
    np.testing.assert_allclose(fast.resample_tests.boot_ratios[:, live][ok], o["boot"]["boot_ratios"][:, live][ok],
                               rtol=2e-4, atol=1e-9)


def test_cfg4_mb_bscan_200k_with_splits_matches_oracle():
    import plspy_b200
    groups, C, p, nb, bscan = (30, 30), 4, 200_000, 4, [1, 2]
    _, X, Y = _planted(20260004, groups, C, p, nb)
    np.random.seed(1238)
    o = oracle.run_full("mb", X, groups, C, Y=Y.copy(), mctype=0, bscan=bscan, nperm=3, nboot=3, nsplit=2, lv=1)
    np.random.seed(1238)
    res = plspy_b200.PLS(X, groups, C, Y=Y.copy(), num_perm=3, num_boot=3, num_split=2, lv=1, mctype=0, bscan=bscan,
                         pls_method="mb")
    rt = res.resample_tests
    s = np.asarray(o["s"])
    live = np.abs(s) > 1e-8 * np.abs(s).max()
    assert res.s.shape == (24,)
    np.testing.assert_allclose(res.s[live], s[live], rtol=1e-10)
    np.testing.assert_array_equal(rt.permute_ratio, o["perm"]["permute_ratio"])
    np.testing.assert_array_equal(rt.stepdown_ratio, o["perm"]["stepdown_ratio"])
    np.testing.assert_allclose(rt.perm_debug_dict["s_list"][:, live], o["perm"]["s_hat"][:, live], rtol=1e-9)
    np.testing.assert_allclose(rt.std_errs[:, live], o["boot"]["std_errs"][:, live], rtol=1e-6)
    np.testing.assert_allclose(rt.boot_ratios[:, live], o["boot"]["boot_ratios"][:, live], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(rt.LVcorr[:, :, live], o["boot"]["LVcorr"][:, :, live], rtol=1e-7, atol=1e-9)
    for i in (0, 1):
        np.testing.assert_allclose(rt.conf_ints[i][:, live], o["boot"]["conf_ints"][i][:, live], rtol=1e-7, atol=1e-9)
        np.testing.assert_allclose(rt.conf_ints_T[i][:, live], o["boot"]["conf_ints_T"][i][:, live], rtol=1e-7, atol=1e-9)
    tt, sh = res.pls_repro_tt, res.pls_repro_sh
    ott, osh = o["tt"], o["sh"]
    nl = int(live.sum())
    d = np.arange(nl - 1)
    for k in ("pls_s_test", "pls_s_test_null"):
        np.testing.assert_allclose(tt[k][d, d, :], ott[k][d, d, :], rtol=1e-7, atol=1e-9, err_msg=k)
    for k in ("pls_s_train", "pls_s_train_null"):
        np.testing.assert_allclose(tt[k][:, :nl - 1, :], ott[k][:, :nl - 1, :], rtol=1e-9, atol=1e-10, err_msg=k)
    for k in ("pls_dist_u", "pls_dist_v", "pls_dist_null_u", "pls_dist_null_v"):
        np.testing.assert_allclose(np.abs(sh[k][d, d, :]), np.abs(osh[k][d, d, :]), rtol=1e-7, atol=1e-8, err_msg=k)
    for k in ("pls_rep_mean_u", "pls_rep_mean_v", "pls_null_mean_u", "pls_null_mean_v"):
        np.testing.assert_allclose(np.asarray(sh[k]), np.asarray(osh[k]), rtol=1e-7, atol=1e-9, err_msg=k)
