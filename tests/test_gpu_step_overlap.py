"""The order of one task-method resampling step: X V out of the Gram launch (Engine.prepare_xv) where the stack
[X; V^T] adds no 64-row tile, and, on the collapsed bootstrap route, the moment stage with the copy of the p x K
results to the host enqueued before the N-space work of both tests."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _data(N, p, seed=0):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((N, p))
    X[: N // 3, : p // 10] += 0.5
    return X


def _engine_and_v(N, p, K, **kw):
    import torch
    from plspy_b200.engine import Engine
    X = _data(N, p)
    V = np.linalg.qr(np.random.RandomState(1).standard_normal((p, K)))[0]
    dev = torch.device("cuda", 0)
    Xd = torch.from_numpy(X).to(dev)
    if kw.get("x_storage") == "fp32":
        Xd = Xd.float()
    return Engine(Xd, device=dev, **kw), torch.from_numpy(np.ascontiguousarray(V)).to(dev)


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize("N,K", [(300, 12), (300, 3), (250, 6)])
def test_stacked_gram_gives_g_bit_identical_and_xv(N, K):
    eng, Vd = _engine_and_v(N, 40000 + 6, K)
    ref, _ = _engine_and_v(N, 40000 + 6, K)
    assert eng.prepare_xv(Vd)
    G = eng.G.cpu().numpy()
    np.testing.assert_array_equal(G, ref.gram_of(ref.X).cpu().numpy())
    xv = eng.xv(Vd)
    assert xv is eng._xv_done[1]                       # the product of the Gram launch, no pass of its own
    assert _rel(xv.cpu().numpy(), ref.xv(Vd).cpu().numpy()) <= 1e-13


@pytest.mark.parametrize("N,K,kw", [(60, 6, {}), (300, 21, {}), (300, 12, {"x_storage": "fp32"}),
                                    (300, 12, {"precision": "tf32x3+gram"})])
def test_stacked_gram_falls_back(N, K, kw):
    """A stack that adds a tile (60 + 6, 300 + 21 rows), float32 X and the TF32 Gram keep the separate X V pass."""
    eng, Vd = _engine_and_v(N, 5000, K, **kw)
    ref, _ = _engine_and_v(N, 5000, K, **kw)
    assert not eng.prepare_xv(Vd)
    np.testing.assert_array_equal(eng.G.cpu().numpy(), ref.G.cpu().numpy())
    np.testing.assert_array_equal(eng.xv(Vd).cpu().numpy(), ref.xv(Vd).cpu().numpy())


def test_xv_before_g_forms_the_stacked_gram():
    eng, Vd = _engine_and_v(300, 6000, 12)
    ref, _ = _engine_and_v(300, 6000, 12)
    assert eng.prepare_xv(Vd)
    xv = eng.xv(Vd)
    assert eng._G is not None
    np.testing.assert_array_equal(eng.G.cpu().numpy(), ref.G.cpu().numpy())
    assert _rel(xv.cpu().numpy(), ref.xv(Vd).cpu().numpy()) <= 1e-13


def test_collapsed_step_copies_p_sized_results_before_the_nspace_work(monkeypatch):
    import torch
    from plspy_b200 import bootstrap_permutation as bp, class_functions as cf, resample
    from plspy_b200.engine import Engine
    groups, C, p = (12, 10, 8), 3, 8000
    N = sum(groups) * C
    X = _data(N, p, seed=3)
    co = np.array([[n] * C for n in groups])
    _, X_mc = cf._mean_centre(X, co, 0)
    U, s, V = cf._run_pls(X_mc)
    Tvsc = cf._get_group_condition_means(X @ V, co)
    np.random.seed(4)
    ip = resample.permutation_indices("mct", 200, co)[0]
    ib = resample.bootstrap_indices("mct", 400, co)[0]
    dev = torch.device("cuda", 0)
    Xd = torch.from_numpy(X).to(dev)
    Vd = torch.from_numpy(np.ascontiguousarray(V)).to(dev)

    log = []
    for name in ("to_host_async", "nspace", "gram_of", "gram_stacked", "xv"):
        fn = getattr(Engine, name)

        def w(self, *a, _fn=fn, _name=name, **k):
            shape = tuple(a[0].shape) if (a and torch.is_tensor(a[0])) else None
            log.append((_name, shape))
            return _fn(self, *a, **k)
        monkeypatch.setattr(Engine, name, w)

    def run(algo):
        log.clear()
        eng = Engine(Xd, device=dev)
        rt = bp.ResampleTest._create("mct", Xd, None, U, s.copy(), Vd, co, 0, preprocess=cf._mean_centre, nperm=200,
                                     nboot=400, Tvsc_orig=Tvsc, CI=0.95, perm_indices=ip, boot_indices=ib,
                                     engine=eng, boot_algo=algo)
        return rt, list(log)

    rt_c, log_c = run("collapsed")
    rt_d, log_d = run("direct")
    assert rt_c.boot_algo == "collapsed" and rt_d.boot_algo == "direct"
    p_copy = next(i for i, (n, sh) in enumerate(log_c) if n == "to_host_async" and sh == (p, V.shape[1]))
    first_nspace = next(i for i, (n, _) in enumerate(log_c) if n == "nspace")
    first_gram_x = next(i for i, (n, sh) in enumerate(log_c) if n in ("gram_of", "gram_stacked") and sh == (N, p))
    assert p_copy < first_nspace and p_copy < first_gram_x
    # X V came out of the Gram launch of the stack [X; V^T] in both routes
    assert ("gram_stacked", (N, p)) in log_c and ("gram_stacked", (N, p)) in log_d
    assert not any(n == "gram_of" and sh == (N, p) for n, sh in log_c + log_d)

    # the same N-space outputs bit for bit; the standard errors to rounding (two formulations of the same moments)
    np.testing.assert_array_equal(rt_c.permute_ratio, rt_d.permute_ratio)
    np.testing.assert_array_equal(rt_c.stepdown_ratio, rt_d.stepdown_ratio)
    np.testing.assert_array_equal(rt_c.perm_debug_dict["s_list"], rt_d.perm_debug_dict["s_list"])
    for key in ("Tdistrib", "left_sv_sampled"):
        np.testing.assert_array_equal(rt_c.boot_debug_dict[key], rt_d.boot_debug_dict[key])
    np.testing.assert_array_equal(rt_c.conf_ints[0], rt_d.conf_ints[0])
    live = np.abs(s) > 1e-8 * np.abs(s).max()
    for f in ("std_errs", "boot_ratios"):
        a, b = getattr(rt_c, f)[:, live], getattr(rt_d, f)[:, live]
        assert float(np.max(np.abs(a - b) / np.abs(b))) <= 1e-11, f
