"""The identity behind the factored collapsed bootstrap, on the CPU with the oracle.  A draw of
resample.bootstrap_indices keeps every row in its cell and uses one subject map for all conditions, and
E = Lop^T Ucoef is constant within a cell, so C_r = scatter(E, idx_r) = D_E P m_r (m_r: draws of each subject) and

    S_k = sum_r d_rk d_rk^T - s1_k s1_k^T / R = D_k P M P^T D_k,   M = sum_r (m_r - 1)(m_r - 1)^T - s1 s1^T / R.

M has rank <= ns - G; its factor L (ns x (ns - G)) is built as boot_factor_kernel builds it (Cholesky without the last
subject of each group, dropped rows = minus the sum of the group's other rows), and the standard errors become a sum of
squares over the ns - G columns of L.  Also the resolution of boot_algo="auto"."""
import os

import numpy as np
import pytest

import oracle.pls_oracle as po
from conftest import GOLDEN_DIR

FIXTURES = ["mct_m0_bal", "mct_m1_unbal", "mct_m2_unbal", "mct_m3_bal", "mct_m0_1grp", "mct_m0_offset",
            "cst_bal", "cst_unbal"]


def load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def operators(method, X, groups, C, mctype, contrasts=None):
    a = po.analysis(method, X.copy(), groups, C, contrasts=contrasts, mctype=mctype)
    N = X.shape[0]
    Lop = po.mean_centre(np.eye(N), a["cond_order"], mctype) if method == "mct" else po.group_condition_means(
        np.eye(N), a["cond_order"])
    return a, Lop.T @ a["U"]


def subjects(groups, C):
    """sid[n] (subject of row n) and the group offsets of the subjects, rows ordered group, condition, subject."""
    gstart = np.concatenate(([0], np.cumsum(groups)))
    sid = np.concatenate([gstart[g] + np.arange(n) for g, n in enumerate(groups) for _ in range(C)])
    return sid, gstart


def count_cov(idx, sid, ns):
    """M from the draws: m_r[s] = draws of subject s (counted in any one condition; here all, divided by C)."""
    R = idx.shape[0]
    C = len(sid) // ns
    m = np.stack([np.bincount(sid[idx[r]], minlength=ns) for r in range(R)]) / C - 1.0
    s1 = m.sum(axis=0)
    return m.T @ m - np.outer(s1, s1) / R


def factor(M, gstart):
    """boot_factor_kernel in numpy."""
    G = len(gstart) - 1
    ns = int(gstart[-1])
    keep = np.array([s for g in range(G) for s in range(gstart[g], gstart[g + 1] - 1)])
    Lk = np.linalg.cholesky(M[np.ix_(keep, keep)])
    L = np.zeros((ns, len(keep)))
    L[keep] = Lk
    for g in range(G):
        L[gstart[g + 1] - 1] = -Lk[(keep >= gstart[g]) & (keep < gstart[g + 1])].sum(axis=0)
    return L


def nxn(E, idx):
    R, (N, K) = idx.shape[0], E.shape
    S1 = np.zeros((N, K)); S2 = np.zeros((K, N, N))
    for r in range(R):
        Cr = np.zeros_like(E)
        np.add.at(Cr, idx[r], E)
        d = Cr - E
        S1 += d
        S2 += np.einsum("nk,mk->knm", d, d)
    return S2 - np.einsum("nk,mk->knm", S1, S1) / R


@pytest.mark.parametrize("name", FIXTURES)
def test_factored_covariance_equals_the_nxn_build(name):
    g = load(name)
    method, X = str(g["method"]), g["X"]
    groups, C, mctype = tuple(int(n) for n in g["groups"]), int(g["C"]), int(g["mctype"])
    a, E = operators(method, X, groups, C, mctype, g.get("contrasts_in"))
    cells = np.concatenate(([0], np.cumsum(np.asarray(a["cond_order"]).reshape(-1))))
    for lo, hi in zip(cells[:-1], cells[1:]):
        assert (E[lo:hi] == E[lo]).all()                  # bit-identical within each cell
    sid, gstart = subjects(groups, C)
    ns = int(gstart[-1])
    idx = g["boot_idx"]
    M = count_cov(idx, sid, ns)
    Sig = nxn(E, idx)
    P = np.eye(ns)[sid]                                   # N x ns subject indicator
    Sf = np.einsum("nk,ns,st,mt,mk->knm", E, P, M, P, E)
    assert np.max(np.abs(Sf - Sig)) <= 1e-13 * np.max(np.abs(Sig))
    if idx.shape[0] > ns - len(groups):                   # the factor needs more draws than its columns
        L = factor(M, gstart)
        assert np.max(np.abs(L @ L.T - M)) <= 1e-13 * np.max(np.abs(M))
        q = sum((X.T @ (E * L[sid, j][:, None])) ** 2 for j in range(L.shape[1]))
        se = np.sqrt(np.maximum(q / idx.shape[0], 0.0))
        live = np.abs(g["s"]) > 1e-8
        ref = g["std_errs"][:, live]
        assert np.max(np.abs(se[:, live] - ref) / np.abs(ref)) <= (1e-8 if "offset" in name else 1e-10)


def test_factored_std_errs_match_direct_on_a_large_baseline():
    """3 groups (5, 4, 6) x 3 conditions, 500 voxels with a per-voxel baseline of +100, 400 bootstraps."""
    import plspy_b200.resample as resample
    groups, C = (5, 4, 6), 3
    rs = np.random.RandomState(3)
    N = sum(groups) * C
    X = rs.standard_normal((N, 500)) + 100.0
    X[:5, :50] += 0.7
    a, E = operators("mct", X, groups, C, 0)
    old = resample.USE_NATIVE_RNG
    resample.USE_NATIVE_RNG = False                      # numpy's own draws: no native library needed
    try:
        np.random.seed(5)
        idx = resample.bootstrap_indices("mct", 400, a["cond_order"])[0]
    finally:
        resample.USE_NATIVE_RNG = old
    sid, gstart = subjects(groups, C)
    L = factor(count_cov(idx, sid, int(gstart[-1])), gstart)
    q = sum((X.T @ (E * L[sid, j][:, None])) ** 2 for j in range(L.shape[1]))
    se = np.sqrt(q / idx.shape[0])
    VS = np.stack([X[idx[r]].T @ E for r in range(idx.shape[0])])      # the direct per-bootstrap saliences
    ref = VS.std(axis=0)
    live = np.abs(a["s"]) > 1e-8 * np.abs(a["s"]).max()
    assert np.max(np.abs(se[:, live] - ref[:, live]) / ref[:, live]) <= 1e-12


def test_auto_resolution():
    from plspy_b200.bootstrap_permutation import check_boot_algo
    assert check_boot_algo("auto", "mct", "fp64", 300, 5000) == "collapsed"
    assert check_boot_algo("auto", "cst", "fp64", 300, 301) == "collapsed"
    assert check_boot_algo("auto", "mct", "fp64", 300, 300) == "direct"          # B must exceed N
    assert check_boot_algo("auto", "mct", "fp64", 24, 12) == "direct"            # the golden fixtures stay direct
    assert check_boot_algo("auto", "mct", "fp64", 321, 5000) == "direct"         # beyond the collapsed kernels
    assert check_boot_algo("auto", "mct", "tf32x3", 300, 5000) == "direct"
    assert check_boot_algo("auto", "mct", "tf32x3+gram", 300, 5000) == "direct"
    for m in ("rb", "csb", "mb", "cmb"):
        assert check_boot_algo("auto", m, "fp64", 300, 5000) == "direct"
    assert check_boot_algo("auto", "mct", "fp64", None, 5000) == "direct"
    assert check_boot_algo("direct", "mct", "fp64", 300, 5000) == "direct"
    assert check_boot_algo("collapsed", "mct", "fp64", 300, 10) == "collapsed"


def test_plugin_install_accepts_auto():
    from plspy_b200 import plugin
    assert plugin._options["boot_algo"] == "auto"
    with pytest.raises(ValueError):
        plugin.install(object(), boot_algo="automatic")
    assert not plugin.installed()
