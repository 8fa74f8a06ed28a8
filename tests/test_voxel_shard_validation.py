"""shard="voxels" without a GPU: every validation error is raised before any GPU work, and dist.voxel_shard cuts the
voxel range into aligned contiguous slices (empty ones included) that dist.gather_spans reassembles."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


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


def test_check_shard():
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import check_shard
    for m in ("mct", "cst", "rb", "csb", "mb", "cmb"):
        check_shard("resamples", m)
    check_shard("voxels", "mct")
    check_shard("voxels", "cst")
    for bad in ("voxel", "columns", None, 1):
        with pytest.raises(ValueError):
            check_shard(bad, "mct")
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            check_shard("voxels", m)


def _method_kw(m):
    kw = dict(pls_method=m, num_boot=5, shard="voxels")
    if m in ("csb", "cmb"):
        kw["contrasts"] = np.ones((4, 1))
    return kw


def test_pls_rejects_before_gpu_work(no_gpu_work):
    import plspy_b200
    from plspy_b200 import exceptions
    X, Y = _design()
    with pytest.raises(ValueError):
        plspy_b200.PLS(X, [12], 2, num_boot=5, shard="rows")
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            plspy_b200.PLS(X, [12], 2, Y=Y, **_method_kw(m))


def test_pls_classes_reject_before_gpu_work(no_gpu_work):
    """The method classes validate too (they are reachable without `PLS`), and an engine's layout must match."""
    from plspy_b200 import exceptions, pls_classes
    X, Y = _design()
    for m in ("rb", "csb", "mb", "cmb"):
        kw = _method_kw(m)
        kw["pls_alg"] = kw.pop("pls_method")
        with pytest.raises(exceptions.NotImplementedError):
            pls_classes.PLSBase._create(m, X, [12], 2, Y=Y, **kw)
    with pytest.raises(ValueError):
        pls_classes.PLSBase._create("mct", X, [12], 2, num_boot=5, pls_alg="mct", shard="all")

    class FakeEngine:
        x_storage, precision, N, shard = "fp64", "fp64", 24, "resamples"
    with pytest.raises(ValueError, match="engine"):
        pls_classes.PLSBase._create("mct", X, [12], 2, num_boot=5, pls_alg="mct", shard="voxels",
                                    engine=FakeEngine())
    FakeEngine.shard = "voxels"
    with pytest.raises(ValueError, match="engine"):
        pls_classes.PLSBase._create("mct", X, [12], 2, num_boot=5, pls_alg="mct", shard="resamples",
                                    engine=FakeEngine())
    with pytest.raises(exceptions.NotImplementedError):     # the layout of an engine given without the option
        pls_classes.PLSBase._create("rb", X, [12], 2, Y=Y, num_boot=5, pls_alg="rb", engine=FakeEngine())


def test_resample_test_rejects_before_gpu_work(no_gpu_work):
    from plspy_b200 import exceptions
    from plspy_b200.bootstrap_permutation import ResampleTest
    X, Y = _design()
    co = np.array([[12, 12]])
    for m in ("rb", "csb", "mb", "cmb"):
        with pytest.raises(exceptions.NotImplementedError):
            ResampleTest._create(m, X, Y, None, np.ones(2), None, co, 0, nperm=5, nboot=5, shard="voxels")
    with pytest.raises(ValueError):
        ResampleTest._create("mct", X, None, None, np.ones(2), None, co, 0, nperm=5, nboot=5, shard="rows")

    class FakeEngine:
        x_storage, precision, N, shard = "fp64", "fp64", 24, "voxels"
    with pytest.raises(ValueError, match="engine"):
        ResampleTest._create("mct", X, None, None, np.ones(2), None, co, 0, nperm=5, nboot=5, shard="resamples",
                             engine=FakeEngine())


def test_plugin_rejects_before_gpu_work(no_gpu_work):
    from plspy_b200 import exceptions, plugin
    with pytest.raises(ValueError):
        plugin.install(object(), shard="voxel")
    assert not plugin.installed()
    assert plugin._options["shard"] == "resamples"
    X, Y = _design()
    co = np.array([[12, 12]])
    old = dict(plugin._options)
    plugin._options["shard"] = "voxels"               # what install(shard="voxels") sets
    try:
        for m in ("rb", "csb", "mb", "cmb"):
            with pytest.raises(exceptions.NotImplementedError):
                plugin.PINNED[m](X, Y, None, np.ones(2), None, co, 0, nperm=5, nboot=5)
            with pytest.raises(exceptions.NotImplementedError):
                plugin._split_half_test_train(m, X, Y, co, 3)
    finally:
        plugin._options.update(old)


def test_split_half_without_resampling_gets_a_voxel_sharded_engine(monkeypatch):
    """With no resampling engine, the split-half functions of a shard="voxels" analysis share one engine built with
    that layout (they would otherwise each upload the whole of X)."""
    import plspy_b200
    from plspy_b200 import engine, split_half_resampling
    built, seen = [], []

    class FakeEngine:
        def __init__(self, X, device=None, precision="fp64", x_storage="fp64", shard="resamples"):
            built.append((X, x_storage, shard))
    monkeypatch.setattr(engine, "Engine", FakeEngine)

    def record(*args, engine=None, **kw):
        seen.append(engine)
        return {}
    monkeypatch.setattr(split_half_resampling, "split_half_test_train", record)
    monkeypatch.setattr(split_half_resampling, "split_half", record)
    X = np.random.default_rng(9).standard_normal((36, 50))
    for xs in ("fp64", "fp32"):
        built.clear(); seen.clear()
        plspy_b200.PLS(X, [6, 6], 3, num_perm=0, num_boot=0, num_split=5, lv=1, shard="voxels", x_storage=xs)
        assert len(built) == 1 and len(seen) == 2 and seen[0] is seen[1] and isinstance(seen[0], FakeEngine)
        Xe, xs_e, sh = built[0]
        assert sh == "voxels" and xs_e == xs
        np.testing.assert_array_equal(Xe, X if xs == "fp64" else X.astype(np.float32))


@pytest.mark.parametrize("size", range(1, 9))
@pytest.mark.parametrize("p", [0, 1, 200, 255, 256, 300, 511, 2048, 20011, 10 ** 6])
def test_voxel_shard_partitions_voxels(p, size):
    from plspy_b200 import dist as pd
    spans = [pd.voxel_shard(p, r, size) for r in range(size)]
    assert spans[0][0] == 0 and spans[-1][1] == p
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))                # contiguous, in rank order
    assert all(lo <= hi for lo, hi in spans)
    assert all(lo % 256 == 0 or lo == p for lo, _ in spans)                   # aligned cut points
    sizes = [hi - lo for lo, hi in spans]
    blocks = [-(-s // 256) for s in sizes]                                    # balanced in 256-voxel blocks
    assert max(blocks) - min(blocks) <= 1
    if p < 256 * size:                                                        # ranks beyond the voxels: empty
        assert sum(s == 0 for s in sizes) == size - -(-p // 256)
    if size == 1:
        assert spans == [(0, p)]


def test_voxel_shard_defaults_to_this_process():
    from plspy_b200 import dist as pd
    assert pd.voxel_shard(1000) == (0, 1000)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _gather_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from plspy_b200 import dist as pd
        res = {}
        for p in (1000, 300, 200):                      # ragged, and one rank without voxels at p = 200 and world 3
            full = torch.arange(p * 3, dtype=torch.float64).reshape(p, 3)
            spans = [pd.voxel_shard(p, r, world) for r in range(world)]
            v0, v1 = pd.voxel_shard(p)
            got = pd.gather_spans(full[v0:v1].clone(), spans)
            res[p] = bool(torch.equal(got, full))
        # the resample gather still reassembles shards in order
        n = 11
        lo, hi = pd.shard(n)
        rows = torch.arange(n, dtype=torch.float64)[:, None].repeat(1, 2)
        res["rows"] = bool(torch.equal(pd.gather_rows(rows[lo:hi].clone(), n, lo), rows))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_gather_spans_world3():
    world = 3
    mgr = mp.get_context("spawn").Manager()
    out = mgr.dict()
    mp.spawn(_gather_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        assert all(out[r].values()), out[r]
