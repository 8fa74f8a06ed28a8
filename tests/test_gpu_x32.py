"""x_storage="fp32": X held as float32 on the device, widened where each kernel loads it.  Every float32-input entry
point must give exactly (np.testing.assert_array_equal) what its FP64 twin gives on the widened matrix, and every
result field of PLS(X, ..., x_storage="fp32") must equal that of PLS(X.astype(float32).astype(float64), ...)."""
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN_DIR, golden_cases

pytestmark = pytest.mark.gpu

TASK_CASES = [c for c in golden_cases() if c.startswith(("mct", "cst"))]


def _widened(X):
    return np.asarray(X).astype(np.float32).astype(np.float64)


def _assert_same(a, b, path="res"):
    """Every public array / scalar field of two result objects, bit for bit (resample_tests and split-half too)."""
    for k, v in vars(b).items():
        if k.startswith("_") or "debug" in k:
            continue
        w = getattr(a, k)
        if k == "resample_tests":
            _assert_same(w, v, path + "." + k)
        elif isinstance(v, dict):
            assert set(w) == set(v), (path, k)
            for kk in v:
                np.testing.assert_array_equal(np.asarray(w[kk]), np.asarray(v[kk]), err_msg=f"{path}.{k}[{kk}]")
        elif isinstance(v, (np.ndarray, float, int, str)) or (isinstance(v, (list, tuple)) and
                                                             all(isinstance(x, np.ndarray) for x in v)):
            if isinstance(v, (list, tuple)):
                assert len(w) == len(v)
                for i, (x, y) in enumerate(zip(w, v)):
                    np.testing.assert_array_equal(x, y, err_msg=f"{path}.{k}[{i}]")
            else:
                np.testing.assert_array_equal(w, v, err_msg=f"{path}.{k}")


# ---- the ABI: every *_x32 entry point against its FP64 twin on the widened matrix ----------------------------
def _pair(N, p, off, ldx, seed):
    """X32 (float32 view at voxel offset `off`, pitch `ldx`) and the same values widened to float64 (same layout)."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.randn(N, ldx, generator=g, device="cuda", dtype=torch.float32) * 3.0 + 0.5
    return base[:, off:off + p], base.double()[:, off:off + p]


def _ws(nbytes):
    import torch
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device="cuda")


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _ok(rc, what):
    from plspy_b200 import _lib
    _lib.check(rc, what)


# odd offsets / pitches (4-byte aligned rows: element loads), and two 16-byte aligned layouts with ldx % 4 == 0 (the
# 16-byte cp.async of the Gram kernel, the 16-byte loads of the Gram TF32 split)
SHAPES = [(N, p, off, p + off + extra) for N, p, off, extra in
          [(4, 1001, 3, 5), (37, 2053, 1, 2), (300, 4099, 5, 3), (320, 1027, 7, 1), (360, 1203, 3, 9),
           (1380, 517, 1, 6), (37, 2045, 4, 7), (300, 4096, 0, 4)]]


@pytest.mark.parametrize("N,p,off,ldx", SHAPES)
def test_gram_xv_salience_and_splits_match_the_fp64_twins(N, p, off, ldx):
    import torch
    from plspy_b200._lib import lib
    X32, X64 = _pair(N, p, off, ldx, seed=N + p)
    ws = _ws(lib.plsb200_gram_f64_workspace(N, p))
    G = [torch.empty(N, N, dtype=torch.float64, device="cuda") for _ in range(2)]
    _ok(lib.plsb200_gram_x32_f64(X32.data_ptr(), N, p, ldx, G[0].data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "g")
    _ok(lib.plsb200_gram_f64(X64.data_ptr(), N, p, ldx, G[1].data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "g")
    torch.testing.assert_close(G[1], (X64 @ X64.T), rtol=1e-12, atol=1e-9)
    np.testing.assert_array_equal(G[0].cpu().numpy(), G[1].cpu().numpy())
    for K in (1, 12, 24, 30):
        V = torch.randn(p, K, dtype=torch.float64, device="cuda")
        ws = _ws(lib.plsb200_xv_f64_workspace(N, p, K))
        out = [torch.empty(N, K, dtype=torch.float64, device="cuda") for _ in range(2)]
        _ok(lib.plsb200_xv_x32_f64(X32.data_ptr(), N, p, ldx, V.data_ptr(), K, out[0].data_ptr(), ws.data_ptr(),
                                   ws.numel(), _stream()), "xv")
        _ok(lib.plsb200_xv_f64(X64.data_ptr(), N, p, ldx, V.data_ptr(), K, out[1].data_ptr(), ws.data_ptr(),
                               ws.numel(), _stream()), "xv")
        np.testing.assert_array_equal(out[0].cpu().numpy(), out[1].cpu().numpy())
    if N <= 320:
        K, R = 12, 3
        E = torch.randn(N, K, dtype=torch.float64, device="cuda")
        idx = torch.randint(0, N, (R, N), dtype=torch.int32, device="cuda")
        for series, (f32, f64) in enumerate([(lib.plsb200_salience_x32_f64, lib.plsb200_salience_f64),
                                             (lib.plsb200_salience_series_x32_f64, lib.plsb200_salience_series_f64)]):
            out = [torch.empty(R * p * K, dtype=torch.float64, device="cuda") for _ in range(2)]
            _ok(f32(X32.data_ptr(), N, p, ldx, E.data_ptr(), K, idx.data_ptr(), R, out[0].data_ptr(), _stream()), "s")
            _ok(f64(X64.data_ptr(), N, p, ldx, E.data_ptr(), K, idx.data_ptr(), R, out[1].data_ptr(), _stream()), "s")
            np.testing.assert_array_equal(out[0].cpu().numpy(), out[1].cpu().numpy(), err_msg=f"series={series}")
        img = [_ws(lib.plsb200_gram_tf32_image_bytes(N, p)) for _ in range(2)]
        _ok(lib.plsb200_gram_tf32_split_x32(X32.data_ptr(), N, p, ldx, img[0].data_ptr(), _stream()), "gs")
        _ok(lib.plsb200_gram_tf32_split(X64.data_ptr(), N, p, ldx, img[1].data_ptr(), _stream()), "gs")
        assert torch.equal(img[0], img[1])
    img = [_ws(lib.plsb200_tf32_ximage_bytes(N, p)) for _ in range(2)]
    for t in img:
        t.zero_()
    _ok(lib.plsb200_tf32_split_x32(X32.data_ptr(), N, p, ldx, img[0].data_ptr(), _stream()), "ts")
    _ok(lib.plsb200_tf32_split_x(X64.data_ptr(), N, p, ldx, img[1].data_ptr(), _stream()), "ts")
    assert torch.equal(img[0], img[1])


@pytest.mark.parametrize("N,p,off,ldx", SHAPES)
@pytest.mark.parametrize("K", [1, 12, 24])
def test_boot_moments_and_quad_match_the_fp64_twins(N, p, off, ldx, K):
    """Register-resident kernels for N <= 320, the tile-major image (os_ximage_kernel) above."""
    import torch
    from plspy_b200._lib import lib
    from plspy_b200.engine import Engine
    X32, X64 = _pair(N, p, off, ldx, seed=7 * N + K)
    eng = Engine(X64.contiguous())
    R = 37
    E = torch.randn(N, K, dtype=torch.float64, device="cuda")
    idx = torch.randint(0, N, (R, N), dtype=torch.int32, device="cuda")
    pivot = torch.randn(p, K, dtype=torch.float64, device="cuda")
    coef = eng.pack_coef(E, idx)["coef"]
    ws = _ws(lib.plsb200_boot_moments_f64_workspace(N, p, K, R))
    outs = []
    for fn, X in ((lib.plsb200_boot_moments_x32_f64, X32), (lib.plsb200_boot_moments_f64, X64)):
        s1 = torch.empty(p, K, dtype=torch.float64, device="cuda"); s2 = torch.empty_like(s1)
        _ok(fn(X.data_ptr(), N, p, ldx, coef.data_ptr(), K, R, pivot.data_ptr(), s1.data_ptr(), s2.data_ptr(),
               ws.data_ptr(), ws.numel(), _stream()), "boot_moments")
        outs.append((s1.cpu().numpy(), s2.cpu().numpy()))
    np.testing.assert_array_equal(outs[0][0], outs[1][0])
    np.testing.assert_array_equal(outs[0][1], outs[1][1])
    if N > 320:
        return
    A = torch.randn(K, N, N, dtype=torch.float64, device="cuda")
    S = (A + A.transpose(1, 2)).contiguous()
    qc = _ws(lib.plsb200_boot_quad_coef_bytes(N, K))
    _ok(lib.plsb200_boot_quad_coef_pack_f64(S.data_ptr(), N, K, qc.data_ptr(), _stream()), "quad_pack")
    ws = _ws(lib.plsb200_boot_quad_f64_workspace(N, p, K))
    q = []
    for fn, X in ((lib.plsb200_boot_quad_x32_f64, X32), (lib.plsb200_boot_quad_f64, X64)):
        out = torch.empty(p, K, dtype=torch.float64, device="cuda")
        _ok(fn(X.data_ptr(), N, p, ldx, qc.data_ptr(), K, out.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "q")
        q.append(out.cpu().numpy())
    np.testing.assert_array_equal(q[0], q[1])


@pytest.mark.parametrize("N", [37, 300, 360])
def test_engine_column_split_and_fast_mode(N):
    """K = 30 goes through the engine's column split; the fast mode's TF32 planes come from float32 X."""
    import torch
    from plspy_b200.engine import Engine
    X32, X64 = _pair(N, 3001, 0, 3001, seed=N)
    E = torch.randn(N, 30, dtype=torch.float64, device="cuda")
    idx = torch.randint(0, N, (45, N), dtype=torch.int32, device="cuda")
    for prec in ("fp64", "tf32x3"):
        a = Engine(X32.contiguous(), precision=prec, x_storage="fp32")
        b = Engine(X64.contiguous(), precision=prec)
        assert a.X.dtype == torch.float32 and a.h2d_bytes == 0
        for x, y in zip(a.boot_moments(E, idx), b.boot_moments(E, idx)):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy())
    a = Engine(X32.contiguous(), precision="tf32x3+gram", x_storage="fp32")
    b = Engine(X64.contiguous(), precision="tf32x3+gram")
    np.testing.assert_array_equal(a.G.cpu().numpy(), b.G.cpu().numpy())


def test_behaviour_kernels_refuse_float32_x():
    import torch
    from plspy_b200._lib import PlsB200Error
    from plspy_b200.engine import Engine
    eng = Engine(torch.randn(12, 100, device="cuda"), x_storage="fp32")
    with pytest.raises(PlsB200Error, match="float64"):
        eng.cell_standardize(np.array([0, 6, 12]))
    with pytest.raises(PlsB200Error, match="float64"):
        eng.gram_stacked(eng.X, eng.X)


# ---- whole analyses ------------------------------------------------------------------------------------------
def _load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def _run_golden(g, X, **extra):
    import plspy_b200
    method = str(g["method"])
    kw = dict(num_perm=int(g["nperm"]), num_boot=int(g["nboot"]), pls_method=method, CI=float(g["CI"]),
              mctype=int(g["mctype"]))
    if "contrasts_in" in g:
        kw["contrasts"] = g["contrasts_in"].copy()
    kw.update(extra)
    np.random.seed(int(g["np_seed"]))
    return plspy_b200.PLS(X, tuple(int(n) for n in g["groups"]), int(g["C"]), **kw)


VARIANTS = {
    "fp64": {},
    "tf32x3": {"precision": "tf32x3"},
    "tf32x3+gram": {"precision": "tf32x3+gram"},
    "collapsed": {"boot_algo": "collapsed"},
    "device": {"analysis": "device"},
    "split": {"num_split": 6, "lv": 1},
}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("name", TASK_CASES)
def test_golden_fixtures_bit_identical(name, variant):
    g = _load(name)
    kw = VARIANTS[variant]
    a = _run_golden(g, g["X"].copy(), x_storage="fp32", **kw)
    b = _run_golden(g, _widened(g["X"]), **kw)
    assert a.resample_tests._engine.X.dtype.itemsize == 4 and b.resample_tests._engine.X.dtype.itemsize == 8
    _assert_same(a, b)
    if variant == "split":
        assert hasattr(a, "pls_repro_sh")


@pytest.mark.parametrize("method", ["mct", "cst"])
def test_split_half_without_resampling_keeps_x_float32(method, monkeypatch):
    """num_perm = num_boot = 0 with num_split > 0: the split-half engine holds the float32 matrix too."""
    import torch
    import plspy_b200
    from plspy_b200.engine import Engine
    stored = []
    upload = Engine._upload_x

    def recording(self, X):
        out = upload(self, X)
        stored.append(out.dtype)
        return out
    monkeypatch.setattr(Engine, "_upload_x", recording)
    groups, C = (9, 8), 3
    X = _design(12, groups, C, 3001)
    kw = dict(num_perm=0, num_boot=0, num_split=7, lv=1, pls_method=method)
    if method == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(groups) * C, 2))
    res = []
    for Xa, xs in ((X, "fp32"), (_widened(X), "fp64")):
        stored.clear()
        np.random.seed(13)
        res.append(plspy_b200.PLS(Xa, groups, C, x_storage=xs, **kw))
        if xs == "fp32":
            assert stored == [torch.float32]                 # one engine, float32, for both split-half functions
    _assert_same(*res)


@pytest.mark.parametrize("name", ["mct_m0_bal", "cst_unbal"])
def test_percentile_intervals_and_lazy_fields(name):
    g = _load(name)
    a = _run_golden(g, g["X"].copy(), x_storage="fp32").resample_tests
    b = _run_golden(g, _widened(g["X"])).resample_tests
    for x, y in zip(a.salience_percentile_intervals(), b.salience_percentile_intervals()):
        np.testing.assert_array_equal(x, y)
    for x, y in zip(a.percentile_conf_ints(), b.percentile_conf_ints()):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a.boot_debug_dict["right_sv_sampled"], b.boot_debug_dict["right_sv_sampled"])


def _design(seed, groups, C, p):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((sum(groups) * C, p))
    X[: groups[0], : p // 7] += 0.8
    return X


def test_pinned_float32_pipelined_upload():
    """A pinned float32 tensor of >= 64 MB is uploaded in voxel ranges (float32 bytes) with the bootstrap starting on
    the first range; the result equals the pipelined float64 upload of the widened matrix."""
    import torch
    import plspy_b200
    from plspy_b200.engine import Engine
    groups, C = (10, 10), 3
    X = _design(9, groups, C, 290_000).astype(np.float32)
    assert X.nbytes >= Engine.PIPELINED_UPLOAD_MIN_BYTES
    out = {}
    for tag, Xa, kw in (("fp32", torch.from_numpy(X).pin_memory(), {"x_storage": "fp32"}),
                        ("fp64", torch.from_numpy(X.astype(np.float64)).pin_memory(), {})):
        for algo in ("direct", "collapsed"):
            np.random.seed(4)
            out[tag, algo] = plspy_b200.PLS(Xa, groups, C, num_perm=20, num_boot=40, boot_algo=algo, **kw)
    assert out["fp32", "direct"].resample_tests._engine.h2d_bytes == X.nbytes
    for algo in ("direct", "collapsed"):
        _assert_same(out["fp32", algo], out["fp64", algo])


def test_tall_design():
    import plspy_b200
    groups, C = (120, 120), 3                     # N = 720: output-stationary moments, FP64 image from float32 X
    X = _design(5, groups, C, 4001)
    res = []
    for Xa, kw in ((X, {"x_storage": "fp32"}), (_widened(X), {})):
        np.random.seed(6)
        res.append(plspy_b200.PLS(Xa, groups, C, num_perm=15, num_boot=20, **kw))
    _assert_same(*res)


def test_benchmark_shape_memory_and_results():
    """At the benchmark shape X dominates device memory: with "fp32" no float64 copy of it is ever allocated."""
    import torch
    import bench
    import plspy_b200
    from plspy_b200.engine import Engine
    X = bench.make_data()
    x32_bytes = X.size * 4
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    eng = Engine(X, x_storage="fp32")
    eng.G
    torch.cuda.synchronize()
    assert eng.X.dtype == torch.float32
    assert torch.cuda.memory_allocated() - base < x32_bytes + (64 << 20)
    assert torch.cuda.max_memory_allocated() - base < 1.5 * x32_bytes          # a float64 X would be 2 x32_bytes
    del eng
    res = {}
    for tag, Xa, kw in (("fp32", X, {"x_storage": "fp32"}), ("fp64", _widened(X), {})):
        np.random.seed(3)
        res[tag] = plspy_b200.PLS(Xa, bench.GROUPS, bench.C, num_perm=50, num_boot=200, pls_method="mct", **kw)
    _assert_same(res["fp32"], res["fp64"])


# ---- plug-in through the reference's own PLS -----------------------------------------------------------------
def test_plugin_x32_matches_fp64_on_float32_data():
    import baseline
    if not baseline.reference_available():
        pytest.skip("baseline/_ref not installed (python -m baseline.install_ref)")
    import contextlib
    import io
    import warnings
    import plspy_b200
    g = _load("mct_m0_bal")
    Xw = _widened(g["X"])
    mod = baseline.import_reference()
    out = {}
    for xs in ("fp32", "fp64"):
        plspy_b200.install(mod, x_storage=xs)
        try:
            np.random.seed(int(g["np_seed"]))
            with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                out[xs] = mod.PLS(Xw.copy(), tuple(int(n) for n in g["groups"]), int(g["C"]), num_perm=int(g["nperm"]),
                                  num_boot=int(g["nboot"]), pls_method="mct", mctype=int(g["mctype"]), CI=float(g["CI"]))
        finally:
            plspy_b200.uninstall()
    assert out["fp32"].resample_tests._engine.X.dtype.itemsize == 4
    for f in ("std_errs", "boot_ratios", "permute_ratio"):
        np.testing.assert_array_equal(getattr(out["fp32"].resample_tests, f), getattr(out["fp64"].resample_tests, f))


# ---- two processes on one GPU (gloo) ---------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _two_proc_data(p):
    rs = np.random.RandomState(3)
    groups, C = (7, 6), 3
    X = rs.standard_normal((sum(groups) * C, p)); X[:7, :80] += 1.0
    return X, groups, C


def _fields(rt):
    return dict(pr=rt.permute_ratio, se=rt.std_errs, br=rt.boot_ratios, lo=rt.conf_ints[0], hi=rt.conf_ints[1])


def _worker(rank, world, port, q, p):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import plspy_b200
        X, groups, C = _two_proc_data(p)
        out = {}
        for tag, Xa, kw in (("fp32", X, {"x_storage": "fp32"}), ("fp64", _widened(X), {})):
            np.random.seed(11)
            out[tag] = _fields(plspy_b200.PLS(Xa, groups, C, num_perm=41, num_boot=37, pls_method="mct",
                                              **kw).resample_tests)
        if rank == 0:
            q.put(out)
    finally:
        dist.destroy_process_group()


def test_two_processes_match():
    import torch.multiprocessing as mp
    import plspy_b200
    p = 70_001                                   # ragged shares; >= 4096 voxels per rank: per-rank partial Gram
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, p)) for r in range(2)]
    for pr in procs:
        pr.start()
    multi = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    for k in multi["fp32"]:                      # the float32 share + all-gather == the widened float64 run
        np.testing.assert_array_equal(multi["fp32"][k], multi["fp64"][k], err_msg=k)
    X, groups, C = _two_proc_data(p)
    np.random.seed(11)
    single = _fields(plspy_b200.PLS(X, groups, C, num_perm=41, num_boot=37, pls_method="mct",
                                    x_storage="fp32").resample_tests)
    np.testing.assert_array_equal(multi["fp32"]["pr"], single["pr"])
    live = np.abs(single["se"]).max(axis=0) > 0
    for k in ("se", "br", "lo", "hi"):           # the all-reduce orders sums differently from one process
        np.testing.assert_allclose(multi["fp32"][k][:, live], single[k][:, live], rtol=1e-9, atol=1e-12, err_msg=k)
