"""x_storage="fp32" without a GPU: every validation error is raised before any GPU work, and the host-side steps see
X.astype(float32) widened to float64 (a float64 input rounded once, a float32 input used as it is)."""
import numpy as np
import pytest


@pytest.fixture
def no_gpu_work(monkeypatch):
    """Fails the test if an Engine (the only owner of device work) is constructed."""
    from plspy_b200 import engine

    def refuse():
        raise AssertionError("GPU work started before the arguments were validated")
    monkeypatch.setattr(engine, "_require_cuda", refuse)


def _design(seed=0, n=24, p=40):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, p)), rng.standard_normal((n, 2))


def test_check_x_storage():
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import check_x_storage
    for m in ("mct", "cst", "rb", "csb", "mb", "cmb"):
        check_x_storage("fp64", m)
    check_x_storage("fp32", "mct")
    check_x_storage("fp32", "cst")
    for bad in ("float32", "f32", None, 32):
        with pytest.raises(ValueError):
            check_x_storage(bad, "mct")
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            check_x_storage("fp32", m)


def test_pls_rejects_before_gpu_work(no_gpu_work):
    import plspy_b200
    from plspy_b200 import exceptions
    X, Y = _design()
    with pytest.raises(ValueError):
        plspy_b200.PLS(X, [12], 2, num_boot=5, x_storage="float32")
    for m in ("rb", "csb", "mb", "cmb"):
        kw = dict(pls_method=m, num_boot=5, x_storage="fp32")
        if m in ("csb", "cmb"):
            kw["contrasts"] = np.ones((4, 1))
        with pytest.raises(exceptions.NotImplementedError):
            plspy_b200.PLS(X, [12], 2, Y=Y, **kw)


def test_pls_classes_reject_before_gpu_work(no_gpu_work):
    """The method classes validate too (they are reachable without `PLS`), and an engine's storage must match."""
    from plspy_b200 import exceptions, pls_classes
    X, Y = _design()
    with pytest.raises(exceptions.NotImplementedError):
        pls_classes.PLSBase._create("rb", X, [12], 2, Y=Y, num_boot=5, pls_alg="rb", x_storage="fp32")
    with pytest.raises(ValueError):
        pls_classes.PLSBase._create("mct", X, [12], 2, num_boot=5, pls_alg="mct", x_storage="fp16")

    class FakeEngine:
        x_storage, precision, N = "fp64", "fp64", 24
    with pytest.raises(ValueError, match="engine"):
        pls_classes.PLSBase._create("mct", X, [12], 2, num_boot=5, pls_alg="mct", x_storage="fp32",
                                    engine=FakeEngine())


def test_resample_test_rejects_before_gpu_work(no_gpu_work):
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import ResampleTest
    X, Y = _design()
    co = np.array([[12, 12]])
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            ResampleTest._create(m, X, Y, None, np.ones(2), None, co, 0, nperm=5, nboot=5, x_storage="fp32")
    with pytest.raises(ValueError):
        ResampleTest._create("mct", X, None, None, np.ones(2), None, co, 0, nperm=5, nboot=5, x_storage="half")


def test_plugin_rejects_before_gpu_work(no_gpu_work):
    from plspy_b200 import exceptions, plugin
    with pytest.raises(ValueError):
        plugin.install(object(), x_storage="float32")
    assert not plugin.installed()
    X, Y = _design()
    co = np.array([[12, 12]])
    old = dict(plugin._options)
    plugin._options["x_storage"] = "fp32"           # what install(x_storage="fp32") sets
    try:
        for m in ("rb", "csb", "mb", "cmb"):
            with pytest.raises(exceptions.NotImplementedError):
                plugin.PINNED[m](X, Y, None, np.ones(2), None, co, 0, nperm=5, nboot=5)
    finally:
        plugin._options.update(old)


def _host_only(X, **kw):
    """A PLS call without resampling runs on the host only (no engine is built)."""
    import plspy_b200
    return plspy_b200.PLS(X, [6, 6], 3, num_perm=0, num_boot=0, **kw)


@pytest.mark.parametrize("method", ["mct", "cst"])
def test_host_analysis_sees_the_rounded_values(no_gpu_work, method):
    rng = np.random.default_rng(5)
    X = rng.standard_normal((36, 50)) * 7.0 + 3.0
    kw = {"pls_method": method}
    if method == "cst":
        kw["contrasts"] = rng.standard_normal((6, 2))
    a = _host_only(X.copy(), x_storage="fp32", **kw)
    b = _host_only(X.astype(np.float32).astype(np.float64), **kw)
    assert a.X.dtype == np.float64
    np.testing.assert_array_equal(a.X, X.astype(np.float32).astype(np.float64))
    for k, v in vars(b).items():
        if isinstance(v, np.ndarray) and not k.startswith("_"):
            np.testing.assert_array_equal(getattr(a, k), v, err_msg=k)
    # the engine would upload the float32 matrix, rounded once from the float64 input
    assert a._x_tensor.dtype == np.float32
    np.testing.assert_array_equal(a._x_tensor, X.astype(np.float32))


def test_float32_input_is_not_copied_for_the_device(no_gpu_work):
    X32 = np.random.default_rng(6).standard_normal((36, 50)).astype(np.float32)
    a = _host_only(X32, x_storage="fp32")
    assert a._x_tensor is X32                       # handed to the engine as it is
    np.testing.assert_array_equal(a.X, X32.astype(np.float64))      # the one widened copy: the host analysis's


def test_float32_torch_input(no_gpu_work):
    import torch
    X = np.random.default_rng(7).standard_normal((36, 50))
    t64 = torch.from_numpy(X.copy())
    a = _host_only(t64, x_storage="fp32")
    assert a._x_tensor.dtype == torch.float32
    np.testing.assert_array_equal(a.X, X.astype(np.float32).astype(np.float64))
    t32 = torch.from_numpy(X.astype(np.float32))
    b = _host_only(t32, x_storage="fp32")
    assert b._x_tensor is t32
    np.testing.assert_array_equal(b.X, a.X)


def test_default_storage_is_unchanged(no_gpu_work):
    X = np.random.default_rng(8).standard_normal((36, 50))
    a = _host_only(X)
    assert a.X is X and not hasattr(a, "_x_tensor")


def test_split_half_without_resampling_gets_a_float32_engine(monkeypatch):
    """With no resampling engine, the split-half functions are handed one engine built from the float32 matrix
    (they would otherwise each upload the widened float64 host copy)."""
    import plspy_b200
    from plspy_b200 import engine, split_half_resampling
    built, seen = [], []

    class FakeEngine:
        def __init__(self, X, device=None, precision="fp64", x_storage="fp64"):
            built.append((X, precision, x_storage))
    monkeypatch.setattr(engine, "Engine", FakeEngine)

    def record(*args, engine=None, **kw):
        seen.append(engine)
        return {}
    monkeypatch.setattr(split_half_resampling, "split_half_test_train", record)
    monkeypatch.setattr(split_half_resampling, "split_half", record)
    X = np.random.default_rng(9).standard_normal((36, 50))
    plspy_b200.PLS(X, [6, 6], 3, num_perm=0, num_boot=0, num_split=5, lv=1, x_storage="fp32")
    assert len(built) == 1 and len(seen) == 2 and seen[0] is seen[1] and isinstance(seen[0], FakeEngine)
    Xe, prec, xs = built[0]
    assert xs == "fp32" and prec == "fp64" and Xe.dtype == np.float32
    np.testing.assert_array_equal(Xe, X.astype(np.float32))
    # the default storage keeps the split-half functions' own engines
    built.clear(); seen.clear()
    plspy_b200.PLS(X, [6, 6], 3, num_perm=0, num_boot=0, num_split=5, lv=1)
    assert built == [] and seen == [None, None]
