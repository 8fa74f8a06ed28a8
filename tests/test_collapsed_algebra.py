"""The identity behind boot_algo="collapsed", on the CPU with the oracle: for the task methods every bootstrap salience
is linear in the draw, VS_r[v,k] = x_v^T c_rk with C_r = scatter(E, idx_r), so

    std_errs[v,k]^2 = Var_r(x_v^T c_rk) = x_v^T S_k x_v / R,    S_k = sum_r d_rk d_rk^T - s1_k s1_k^T / R,

with d_r = C_r - E (pivot at the original coefficients) and s1_k = sum_r d_rk.  Checked against the standard errors
the reference recorded for every mct / cst golden fixture, with the fixtures' own bootstrap indices.  Also the
argument validation of the option, which runs before any GPU work."""
import os

import numpy as np
import pytest

import oracle.pls_oracle as po
from conftest import GOLDEN_DIR

FIXTURES = ["mct_m0_bal", "mct_m1_unbal", "mct_m2_unbal", "mct_m3_bal", "mct_m0_1grp", "mct_m0_offset",
            "cst_bal", "cst_unbal"]


def load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def collapsed_std_errs(g):
    method, X = str(g["method"]), g["X"]
    groups, C, mctype = tuple(int(n) for n in g["groups"]), int(g["C"]), int(g["mctype"])
    a = po.analysis(method, X.copy(), groups, C, contrasts=g.get("contrasts_in"), mctype=mctype)
    co = a["cond_order"]
    N = X.shape[0]
    # the row-space operator of the cross-block matrix (M = Lop X): the oracle applied to the identity
    Lop = po.mean_centre(np.eye(N), co, mctype) if method == "mct" else po.group_condition_means(np.eye(N), co)
    E = Lop.T @ a["U"]                                            # N x K
    idx = g["boot_idx"]
    R, K = idx.shape[0], E.shape[1]
    S1 = np.zeros((N, K)); S2 = np.zeros((K, N, N))
    for r in range(R):
        Cr = np.zeros_like(E)
        np.add.at(Cr, idx[r], E)                                  # C_r = scatter(E, idx_r)
        d = Cr - E
        S1 += d
        S2 += np.einsum("nk,mk->knm", d, d)
    Sig = S2 - np.einsum("nk,mk->knm", S1, S1) / R
    q = np.einsum("nv,knm,mv->vk", X, Sig, X)
    return np.sqrt(np.maximum(q / R, 0.0)), Sig


@pytest.mark.parametrize("name", FIXTURES)
def test_collapsed_std_errs_match_reference(name):
    g = load(name)
    se, Sig = collapsed_std_errs(g)
    live = np.abs(g["s"]) > 1e-8
    ref = g["std_errs"][:, live]
    rel = np.max(np.abs(se[:, live] - ref) / np.abs(ref))
    assert rel <= (1e-8 if name == "mct_m0_offset" else 1e-10), rel
    # every row of the operators sums to zero, so a per-voxel offset of X cancels inside the quadratic form
    assert np.max(np.abs(Sig.sum(axis=2))) <= 1e-12 * max(1.0, np.max(np.abs(Sig)))


# ---- argument validation (before any GPU work) --------------------------------------------------------------
def test_boot_algo_validation():
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import check_boot_algo
    check_boot_algo("direct", "rb", "tf32x3", 10000)
    check_boot_algo("collapsed", "mct", "fp64", 320)
    check_boot_algo("collapsed", "cst", "fp64", 4)
    with pytest.raises(ValueError):
        check_boot_algo("fast", "mct", "fp64", 30)
    for prec in ("tf32x3", "tf32x3+gram"):
        with pytest.raises(ValueError):
            check_boot_algo("collapsed", "mct", prec, 30)
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            check_boot_algo("collapsed", m, "fp64", 30)
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        check_boot_algo("collapsed", "mct", "fp64", 321)


def test_pls_rejects_collapsed_before_gpu_work():
    import plspy_b200
    from plspy_b200 import exceptions
    rng = np.random.default_rng(0)
    X = rng.standard_normal((24, 40))
    Y = rng.standard_normal((24, 2))
    with pytest.raises(ValueError):
        plspy_b200.PLS(X, [12], 2, num_boot=5, boot_algo="exact")
    with pytest.raises(ValueError):
        plspy_b200.PLS(X, [12], 2, num_boot=5, boot_algo="collapsed", precision="tf32x3")
    with pytest.raises(exceptions.NotImplementedError):
        plspy_b200.PLS(X, [12], 2, Y=Y, num_boot=5, boot_algo="collapsed", pls_method="rb")
    Xt = rng.standard_normal((330, 8))
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        plspy_b200.PLS(Xt, [165], 2, num_boot=5, boot_algo="collapsed")


def test_plugin_install_rejects_bad_boot_algo():
    from plspy_b200 import plugin
    with pytest.raises(ValueError):
        plugin.install(object(), boot_algo="exact")
    with pytest.raises(ValueError):
        plugin.install(object(), precision="tf32x3", boot_algo="collapsed")
    assert not plugin.installed()
