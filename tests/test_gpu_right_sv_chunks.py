"""The per-bootstrap brain saliences in voxel chunks, `right_sv_sampled_chunks()`, for all six methods: bit-identical to
the lazy `boot_debug_dict["right_sv_sampled"]` on the golden fixtures and on both behaviour / multiblock kernels (DMMA
and the FMA fallback), against the oracle, above the in-memory bound, with float32 X, voxel-sharded over two processes,
with no GPU work before the first step and after an early close, and through the plug-in."""
import os
import socket
import traceback

import numpy as np
import pytest

import oracle
from test_gpu_parity import _load, _run_product

pytestmark = pytest.mark.gpu

GOLDEN = ["mct_m0_bal", "cst_bal", "rb_bal", "csb_square", "mb_bscan", "cmb_full"]


def _launches():
    from plspy_b200 import _lib
    return _lib.launch_count()


def _ragged_budget(B, p, K):
    """a max_bytes that gives at least three chunks and a shorter last one"""
    vc = max(1, p // 3)
    while vc > 1 and p % vc == 0:
        vc -= 1
    assert -(-p // vc) >= 3 and (p % vc != 0 or vc == 1)
    return B * K * 8 * vc + 7


def _stream(rt, max_bytes=1 << 30):
    """(the chunks laid side by side, the (v0, v1) spans); every chunk is copied before the next step"""
    parts, spans = [], []
    for v0, v1, chunk in rt.right_sv_sampled_chunks(max_bytes):
        assert chunk.dtype == np.float64 and chunk.shape[1] == v1 - v0
        assert chunk.nbytes <= max_bytes or v1 - v0 == 1
        parts.append(chunk.copy())
        spans.append((v0, v1))
    return np.concatenate(parts, axis=1), spans


def _assert_tiles(spans, v0, v1):
    assert spans[0][0] == v0 and spans[-1][1] == v1
    assert all(a[1] == b[0] and a[0] < a[1] for a, b in zip(spans, spans[1:]))


@pytest.mark.parametrize("name", GOLDEN)
def test_chunks_equal_the_lazy_cube_on_the_golden_fixtures(name):
    g = _load(name)
    rt = _run_product(g).resample_tests
    cube = rt.boot_debug_dict["right_sv_sampled"]
    B, p, K = cube.shape
    budget = _ragged_budget(B, p, K)
    got, spans = _stream(rt, budget)
    _assert_tiles(spans, 0, p)
    assert len(spans) >= 3 and spans[-1][1] - spans[-1][0] < spans[0][1] - spans[0][0]
    np.testing.assert_array_equal(got, cube)


def _behaviour_case(method):
    """test_gpu_behaviour_salience's oracle case: rb with K = 27 (two column passes of the DMMA kernel), mb with a
    bscan subset; 30 bootstraps (not a multiple of 8)"""
    rs = np.random.RandomState(31 if method == "rb" else 32)
    groups, C, p, nb, B = (8, 7, 9), 3, 2500, 3 if method == "rb" else 2, 30
    N = sum(groups) * C
    X = rs.standard_normal((N, p)) + 5.0
    X[:, :40] += rs.standard_normal((N, 1))
    Y = rs.standard_normal((N, nb)) + 0.4 * X[:, :nb]
    bscan = [0, 2] if method == "mb" else None
    np.random.seed(17)
    o = oracle.run_full(method, X.copy(), groups, C, Y=Y.copy(), bscan=bscan, nboot=B)
    return X, Y, groups, C, bscan, B, o


@pytest.mark.parametrize("fma", [False, True], ids=["dmma", "fma"])
@pytest.mark.parametrize("method", ["rb", "mb"])
def test_both_kernels_match_the_lazy_cube_and_the_oracle(method, fma):
    import torch
    import plspy_b200
    from plspy_b200.engine import Engine
    X, Y, groups, C, bscan, B, o = _behaviour_case(method)
    eng = Engine(torch.from_numpy(X.copy()).cuda())
    eng.force_rb_fma = fma
    kw = dict(Y=Y.copy(), num_perm=0, num_boot=B, pls_method=method, engine=eng)
    if method == "mb":
        kw.update(bscan=bscan, mctype=0, boot_indices=(o["boot_idx"], o["boot_idx_beh"]))
    else:
        kw.update(boot_indices=o["boot_idx"])
    rt = plspy_b200.PLS(X.copy(), groups, C, **kw).resample_tests
    cube = rt.boot_debug_dict["right_sv_sampled"]
    want = o["boot"]["right_sv_sampled"]
    assert cube.shape == want.shape
    if method == "rb":
        assert want.shape[2] == 27
    p = X.shape[1]
    got, spans = _stream(rt, _ragged_budget(B, p, cube.shape[2]))
    assert eng.last_rb_path == ("fma" if fma else "dmma")
    _assert_tiles(spans, 0, p)
    np.testing.assert_array_equal(got, cube)
    live = np.abs(o["s"]) > 1e-8              # (the tolerance and the live columns of test_gpu_behaviour_salience)
    np.testing.assert_allclose(got[:, :, live], want[:, :, live], rtol=1e-8, atol=1e-11)
    # one chunk: the same values
    np.testing.assert_array_equal(_stream(rt)[0], cube)


@pytest.mark.parametrize("name", ["mct_m0_bal", "rb_bal", "mb_bscan"])
def test_streaming_works_above_the_in_memory_bound(name, monkeypatch):
    from plspy_b200 import bootstrap_permutation as bp
    g = _load(name)
    cube = _run_product(g).resample_tests.boot_debug_dict["right_sv_sampled"]     # the same run, read within the bound
    rt = _run_product(g).resample_tests
    monkeypatch.setattr(bp, "RIGHT_SV_MAX_BYTES", 1024)
    with pytest.raises(MemoryError, match="right_sv_sampled would need"):
        rt.boot_debug_dict["right_sv_sampled"]
    got, spans = _stream(rt, 64 << 10)
    assert got.nbytes > 1024
    _assert_tiles(spans, 0, cube.shape[1])
    np.testing.assert_array_equal(got, cube)


GROUPS, C, P, NBOOT = (7, 6), 3, 700, 150


def _task_run(method="mct", X=None, **kw):
    import plspy_b200
    rs = np.random.RandomState(11)
    if X is None:
        X = rs.standard_normal((sum(GROUPS) * C, P)); X[:7, :80] += 1.0
    if method == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(GROUPS) * C, 2))
    np.random.seed(5)
    return plspy_b200.PLS(X.copy(), GROUPS, C, num_perm=0, num_boot=NBOOT, pls_method=method, **kw)


def test_float32_x_chunks_equal_that_runs_cube():
    X = np.random.RandomState(11).standard_normal((sum(GROUPS) * C, P)).astype(np.float32)
    rt = _task_run("mct", X=X, x_storage="fp32").resample_tests
    assert rt._engine.X.dtype.itemsize == 4
    cube = rt.boot_debug_dict["right_sv_sampled"]
    got, spans = _stream(rt, _ragged_budget(*cube.shape))
    _assert_tiles(spans, 0, P)
    np.testing.assert_array_equal(got, cube)


def test_no_gpu_work_before_the_first_step_and_a_second_stream_after_an_early_close():
    import torch
    for name in ("mct_m0_bal", "rb_bal", "mb_bscan"):
        rt = _run_product(_load(name)).resample_tests
        torch.cuda.synchronize()
        n0 = _launches()
        gen = rt.right_sv_sampled_chunks(4096)
        assert _launches() == n0
        v0, v1, first = next(gen)
        assert _launches() > n0 and v0 == 0
        first = first.copy()
        gen.close()
        cube = rt.boot_debug_dict["right_sv_sampled"]
        np.testing.assert_array_equal(first, cube[:, v0:v1])
        for _ in rt.right_sv_sampled_chunks(4096):
            break                                   # an abandoned generator is closed when it is dropped
        got, spans = _stream(rt, 4096)
        _assert_tiles(spans, 0, cube.shape[1])
        np.testing.assert_array_equal(got, cube)


def test_error_paths():
    import torch
    import plspy_b200
    from plspy_b200 import exceptions
    rs = np.random.RandomState(2)
    res = plspy_b200.PLS(rs.standard_normal((30, 50)), (5, 5), 3, num_perm=5, num_boot=0, pls_method="mct")
    rt = _run_product(_load("rb_bal")).resample_tests
    torch.cuda.synchronize()
    n0 = _launches()
    with pytest.raises(exceptions.MissingParameterError):
        res.resample_tests.right_sv_sampled_chunks()
    for bad in (0, -1):
        with pytest.raises(ValueError):
            rt.right_sv_sampled_chunks(bad)
    assert _launches() == n0


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
            got, spans = _stream(rt, NBOOT * 8 * 8 * 100)
            out[method] = (rt._engine.voxel_range, spans, got)
        q.put((rank, out))
    except BaseException:
        q.put((rank, traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def test_voxel_sharded_ranks_stream_their_own_voxels():
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
        single = _task_run(method).resample_tests.boot_debug_dict["right_sv_sampled"]
        ranges = [got[r][method][0] for r in range(2)]
        assert ranges[0][0] == 0 and ranges[0][1] == ranges[1][0] and ranges[1][1] == P
        for r in range(2):
            (v0, v1), spans, part = got[r][method]
            _assert_tiles(spans, v0, v1)
            np.testing.assert_array_equal(part, single[:, v0:v1])


# ---- the plug-in ---------------------------------------------------------------------------------------------------
def test_reference_result_object_streams_the_cube_through_the_plugin():
    import baseline
    if not baseline.reference_available():
        pytest.skip("baseline/_ref not installed (python -m baseline.install_ref)")
    import plspy_b200
    from plspy_b200 import plugin
    from test_gpu_plugin import _run_reference
    mod = baseline.import_reference()
    plspy_b200.install(mod)
    try:
        for name in ("rb_unbal", "mct_m0_bal"):
            g = _load(name)
            rt = _run_reference(mod, g).resample_tests
            assert isinstance(rt, plugin._InstalledResampleTest)
            cube = rt.boot_debug_dict["right_sv_sampled"]
            got, spans = _stream(rt, _ragged_budget(*cube.shape))
            _assert_tiles(spans, 0, cube.shape[1])
            np.testing.assert_array_equal(got, cube)
    finally:
        plspy_b200.uninstall()
