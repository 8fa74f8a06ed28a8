"""Host side of the BCa salience intervals (DESIGN.md section 5.8), no GPU: the leave-one-subject-out jackknife
coefficients against an independent restatement through the oracle, the stratified acceleration against the textbook
single-group formula, the preconditions, and the argument checks of the new entry points.

`accel_ref` and `jackknife_values` are the restatement `test_gpu_bca.py` compares the kernels with."""
import numpy as np
import pytest

import oracle

GOLDEN = ["mct_m0_1grp", "mct_m0_bal", "mct_m0_offset", "mct_m1_unbal", "mct_m2_unbal", "mct_m3_bal", "cst_bal",
          "cst_unbal"]


def _load(name):
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    return dict(np.load(os.path.join(here, "golden", name + ".npz"), allow_pickle=False))


def subject_rows(cond_order, g, sub):
    """The C rows of subject `sub` of group g (rows are group -> condition -> subject)"""
    starts, sizes = oracle.cell_layout(cond_order)
    C = np.asarray(cond_order).shape[1]
    return np.array([starts[g * C + c] + sub for c in range(C)])


def jackknife_values(method, X, cond_order, mctype, Ucoef):
    """theta_(-gs) for every subject, J x p x K (group-major): the oracle's mean-centring (mct) or cell means (cst) of
    X without the subject's rows, projected on the original design weights"""
    co = np.asarray(cond_order)
    out = []
    for g in range(co.shape[0]):
        co_r = co.copy(); co_r[g] -= 1
        for sub in range(co[g, 0]):
            keep = np.ones(X.shape[0], dtype=bool); keep[subject_rows(co, g, sub)] = False
            M = (oracle.mean_centre(X[keep], co_r, mctype) if method == "mct"
                 else oracle.group_condition_means(X[keep], co_r))
            out.append(M.T @ Ucoef)
    return np.stack(out)


def accel_ref(jv, goff, theta):
    """The stratified jackknife acceleration of every element of the J x ... stack jv, groups [goff[g], goff[g+1])"""
    d = np.asarray(jv, dtype=float) - np.asarray(theta, dtype=float)
    num = np.zeros(d.shape[1:]); den = np.zeros(d.shape[1:])
    for g in range(len(goff) - 1):
        blk = d[goff[g]:goff[g + 1]]
        n = blk.shape[0]
        l = (n - 1) * (blk.mean(axis=0) - blk)
        num += (l ** 3).sum(axis=0) / n ** 3
        den += (l ** 2).sum(axis=0) / n ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, num / (6.0 * den ** 1.5), 0.0)


def _design(g):
    method = str(g["method"])
    groups = tuple(int(n) for n in g["groups"])
    a = oracle.analysis(method, g["X"], groups, int(g["C"]), contrasts=g.get("contrasts_in"), mctype=int(g["mctype"]))
    return method, a["cond_order"], int(g["mctype"]), a["U"]


@pytest.mark.parametrize("name", GOLDEN)
def test_jackknife_coefficients_match_the_oracle(name):
    """X^T C_gs equals the oracle's centring / cell means of X without subject (g, s), projected on U (or the
    normalised contrasts), for every subject; C_gs is zero on the subject's rows"""
    from plspy_b200.bootstrap_permutation import _jackknife_coefficients
    g = _load(name)
    X = g["X"]
    method, co, mctype, Ucoef = _design(g)
    jack, goff = _jackknife_coefficients(method, co, mctype, Ucoef)
    J = int(co[:, 0].sum())
    assert jack.shape == (J, X.shape[0], Ucoef.shape[1])
    np.testing.assert_array_equal(goff, np.concatenate(([0], np.cumsum(co[:, 0]))))
    ref = jackknife_values(method, X, co, mctype, Ucoef)
    got = np.einsum("np,jnk->jpk", X, jack)
    scale = np.abs(ref).max()
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12 * scale)
    j = 0
    for grp in range(co.shape[0]):
        for sub in range(co[grp, 0]):
            assert not jack[j, subject_rows(co, grp, sub)].any()
            j += 1


def test_acceleration_is_the_textbook_formula_for_one_group():
    """one group: a = sum d^3 / (6 (sum d^2)^(3/2)), d = mean(theta_(-i)) - theta_(-i) (Efron & Tibshirani 14.15)"""
    g = _load("mct_m0_1grp")
    method, co, mctype, Ucoef = _design(g)
    assert co.shape[0] == 1
    jv = jackknife_values(method, g["X"], co, mctype, Ucoef)
    theta = oracle.mean_centre(g["X"], co, mctype).T @ Ucoef
    d = jv.mean(axis=0) - jv
    textbook = (d ** 3).sum(axis=0) / (6.0 * ((d ** 2).sum(axis=0)) ** 1.5)
    got = accel_ref(jv, [0, jv.shape[0]], theta)
    np.testing.assert_allclose(got, textbook, rtol=1e-12, atol=1e-15)
    assert np.abs(got).max() > 1e-3
    # the pivot only conditions the sums: a does not depend on it
    np.testing.assert_allclose(accel_ref(jv, [0, jv.shape[0]], 0.0), got, rtol=1e-10, atol=1e-14)


def test_acceleration_is_zero_without_spread():
    jv = np.ones((6, 3, 2))
    np.testing.assert_array_equal(accel_ref(jv, [0, 2, 6], 0.5), 0.0)


@pytest.mark.parametrize("cond_order, missing", [
    ([[5, 4, 5], [6, 6, 6]], "unequal subject counts across conditions"),
    ([[6, 6, 6], [1, 1, 1]], "group 1 has 1 subject(s)"),
    ([[1, 1]], "group 0 has 1 subject(s)"),
])
def test_preconditions_raise_on_the_host(cond_order, missing):
    """raised by the host builder that runs before any GPU work, naming what the design lacks"""
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import _jackknife_coefficients
    Ucoef = np.ones((np.asarray(cond_order).size, 2))
    for method in ("mct", "cst"):
        with pytest.raises(exceptions.NotImplementedError, match=missing.replace("(", r"\(").replace(")", r"\)")):
            _jackknife_coefficients(method, cond_order, 0, Ucoef)


def test_entry_point_argument_errors_without_a_gpu():
    """null pointers are reported by the host-side checks"""
    from plspy_b200 import _lib
    lib = _lib.lib
    rc = lib.plsb200_percentile_bca_f64(None, 10, 4, 1, 10, None, None, 0.05, 0.95, None, None, None, None, 0, None)
    assert rc == -1 and b"percentile_bca_f64: null pointer" in lib.plsb200_last_error()
    rc = lib.plsb200_jack_accel_f64(None, 4, 10, None, 2, None, None, None)
    assert rc == -1 and b"jack_accel_f64: null pointer" in lib.plsb200_last_error()
    for name in ("plsb200_salience_coef_series_f64", "plsb200_salience_coef_series_x32_f64"):
        rc = getattr(lib, name)(None, 10, 100, 100, None, 3, 5, None, None)
        assert rc == -1 and b"null pointer" in lib.plsb200_last_error()
