"""boot_algo="collapsed" beyond 320 rows, on the host: only the factored route exists there, so its conditions on the
design (a cond_order with every group the same size in each of its conditions, more bootstraps than ns - G) are
checked before any GPU work, by check_boot_algo and by PLS(...)."""
import numpy as np
import pytest


def _co(groups, C):
    return np.array([[n] * C for n in groups])


def test_collapsed_beyond_320_rows_needs_the_factored_layout():
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import check_boot_algo
    co = _co((60, 60), 3)                                   # N = 360, ns - G = 118
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        check_boot_algo("collapsed", "mct", "fp64", 360, 500)                     # no cond_order
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        check_boot_algo("collapsed", "mct", "fp64", 360, None, co)                # no bootstrap count
    unbalanced = np.array([[60, 60, 61], [60, 60, 59]])
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        check_boot_algo("collapsed", "mct", "fp64", 360, 500, unbalanced)
    for nboot in (5, 117, 118):
        with pytest.raises(exceptions.NotImplementedError, match="ns - G"):
            check_boot_algo("collapsed", "cst", "fp64", 360, nboot, co)
    assert check_boot_algo("collapsed", "mct", "fp64", 360, 119, co) == "collapsed"
    assert check_boot_algo("collapsed", "cst", "fp64", 360, 500, co.tolist()) == "collapsed"
    # groups of different sizes, each balanced across its conditions: ns - G = 117
    co = _co((40, 45, 35), 6)
    assert check_boot_algo("collapsed", "mct", "fp64", 720, 118, co) == "collapsed"
    with pytest.raises(exceptions.NotImplementedError):
        check_boot_algo("collapsed", "mct", "fp64", 720, 117, co)
    # one subject per group: no pseudo-resamples at all
    with pytest.raises(exceptions.NotImplementedError):
        check_boot_algo("collapsed", "mct", "fp64", 400, 10_000, _co((1,) * 400, 1))


def test_the_other_refusals_are_unchanged_beyond_320_rows():
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import check_boot_algo
    co = _co((60, 60), 3)
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            check_boot_algo("collapsed", m, "fp64", 360, 500, co)
    for prec in ("tf32x3", "tf32x3+gram"):
        with pytest.raises(ValueError):
            check_boot_algo("collapsed", "mct", prec, 360, 500, co)


def test_auto_stays_direct_beyond_320_rows():
    from plspy_b200.bootstrap_permutation import check_boot_algo
    co = _co((200, 200), 3)
    assert check_boot_algo("auto", "mct", "fp64", 1200, 10_000, co) == "direct"
    assert check_boot_algo("auto", "cst", "fp64", 321, 10_000, _co((107,), 3)) == "direct"


def test_pls_checks_the_tall_layout_before_gpu_work():
    import plspy_b200
    from plspy_b200 import exceptions
    rng = np.random.default_rng(0)
    X = rng.standard_normal((360, 8))
    with pytest.raises(exceptions.NotImplementedError, match="ns - G"):
        plspy_b200.PLS(X, [60, 60], 3, num_boot=118, boot_algo="collapsed")
    with pytest.raises(exceptions.NotImplementedError, match="320"):
        plspy_b200.PLS(X, [60, 60], 3, cond_order=np.array([[60, 60, 61], [60, 60, 59]]), num_boot=500,
                       boot_algo="collapsed")
    with pytest.raises(exceptions.NotImplementedError, match="ns - G"):
        plspy_b200.PLS(X, [60, 60], 3, None, None, 0, 100, boot_algo="collapsed")       # positional num_boot


def test_boot_layout_reads_the_call_as_the_class_does():
    from plspy_b200.pls import _boot_layout
    nboot, co = _boot_layout("mct", (np.zeros((360, 4)), [60, 60], 3), {"pls_alg": "mct"})
    assert nboot == 1000
    np.testing.assert_array_equal(co, _co((60, 60), 3))
    given = np.array([[50, 50], [60, 60]])
    nboot, co = _boot_layout("cst", (np.zeros((220, 4)), [50, 60], 2), {"num_boot": 7, "cond_order": given})
    assert nboot == 7 and co is given
    assert _boot_layout("nope", (), {}) == (None, None)
