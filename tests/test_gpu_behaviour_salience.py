"""Per-bootstrap brain saliences `boot_debug_dict["right_sv_sampled"]` (B x p x K) of the behaviour and multiblock
methods (rb, csb, mb, cmb): against the voxel subsample the real reference recorded in the golden fixtures, against the
oracle at larger shapes on both bootstrap kernels (DMMA and the FMA fallback) with several column passes and several
bootstrap chunks, against the standard errors of the same run, and for laziness, the shared memory bound, a
multi-process run and the reference-side plug-in."""
import os
import socket

import numpy as np
import pytest

import oracle
from test_gpu_parity import _load, _run_product

pytestmark = pytest.mark.gpu

GOLDEN = ["rb_bal", "rb_unbal", "csb_square", "mb_full", "mb_bscan", "cmb_full"]


def _launches():
    from plspy_b200 import _lib
    return _lib.launch_count()


@pytest.mark.parametrize("name", GOLDEN)
def test_cube_matches_reference_golden_and_the_standard_errors(name):
    g = _load(name)
    rt = _run_product(g).resample_tests
    live = np.abs(g["s"]) > 1e-8
    p = g["X"].shape[1]
    right = rt.boot_debug_dict["right_sv_sampled"]
    assert right.shape == (int(g["nboot"]), p, g["right_sv_sub"].shape[2])
    np.testing.assert_allclose(right[:, :: max(1, p // 16), :][:, :, live], g["right_sv_sub"][:, :, live],
                               rtol=1e-8, atol=1e-9)
    # the cube is the distribution whose moments gave the standard errors
    np.testing.assert_allclose(np.std(right, axis=0)[:, live], rt.std_errs[:, live], rtol=1e-10)


def _chunked_rb_boot(monkeypatch, per_launch):
    """Engine.rb_boot with a workspace budget of about `per_launch` bootstraps, so that every p-space pass (the
    bootstrap's and the cube's) runs in several launches; records the bootstrap counts it saw."""
    from plspy_b200 import engine as engmod
    from plspy_b200._lib import lib
    orig = engmod.Engine.rb_boot
    seen = []

    def rb_boot(self, Xc, Q, W, cell_start, *a, unit_cells=0, want_t=True, X2=None, **k):
        N, K, p = int(Q.shape[1]), int(Q.shape[2]), int(Xc.shape[1])
        cs = np.ascontiguousarray(np.asarray(cell_start, dtype=np.int32))
        per = lib.plsb200_rb_boot_dmma_f64_workspace(N, p, K, 1, cs.ctypes.data, cs.size - 1, int(unit_cells),
                                                     int(want_t))
        if not per or getattr(self, "force_rb_fma", False):
            per = lib.plsb200_rb_boot_f64_workspace(N, p, K, 1)
        seen.append(int(Q.shape[0]))
        return orig(self, Xc, Q, W, cell_start, *a, unit_cells=unit_cells, want_t=want_t, X2=X2,
                    max_ws_bytes=per_launch * per, **k)
    monkeypatch.setattr(engmod.Engine, "rb_boot", rb_boot)
    return seen


@pytest.mark.parametrize("fma", [False, True], ids=["dmma", "fma"])
@pytest.mark.parametrize("method", ["rb", "mb"])
def test_cube_matches_oracle_on_both_kernels(method, fma, monkeypatch):
    """rb: 3 groups x 3 conditions x 3 behaviours (K = 27: two column passes of 24); mb: a bscan subset.  30
    bootstraps in launches of about 7, same index matrices as the oracle."""
    import torch
    import plspy_b200
    from plspy_b200.engine import Engine
    rs = np.random.RandomState(31 if method == "rb" else 32)
    groups, C, p, nb, B = (8, 7, 9), 3, 2500, 3 if method == "rb" else 2, 30
    N = sum(groups) * C
    X = rs.standard_normal((N, p)) + 5.0
    X[:, :40] += rs.standard_normal((N, 1))
    Y = rs.standard_normal((N, nb)) + 0.4 * X[:, :nb]
    bscan = [0, 2] if method == "mb" else None
    np.random.seed(17)
    o = oracle.run_full(method, X.copy(), groups, C, Y=Y.copy(), bscan=bscan, nboot=B)
    seen = _chunked_rb_boot(monkeypatch, 7)
    eng = Engine(torch.from_numpy(X.copy()).cuda())
    eng.force_rb_fma = fma
    kw = dict(Y=Y.copy(), num_perm=0, num_boot=B, pls_method=method, engine=eng)
    if method == "mb":
        kw.update(bscan=bscan, mctype=0, boot_indices=(o["boot_idx"], o["boot_idx_beh"]))
    else:
        kw.update(boot_indices=o["boot_idx"])
    rt = plspy_b200.PLS(X.copy(), groups, C, **kw).resample_tests
    right = rt.boot_debug_dict["right_sv_sampled"]
    assert eng.last_rb_path == ("fma" if fma else "dmma")
    assert seen and all(n == B for n in seen)
    want = o["boot"]["right_sv_sampled"]
    assert right.shape == want.shape == (B, p, want.shape[2])
    if method == "rb":
        assert want.shape[2] == 27
    # (mb: the centred task rows leave G columns of U in the null space, singular value 0, where either analysis may
    # pick any basis -- compared on the live columns like the golden tests)
    live = np.abs(o["s"]) > 1e-8
    assert live.sum() >= want.shape[2] - len(groups)
    np.testing.assert_allclose(right[:, :, live], want[:, :, live], rtol=1e-8, atol=1e-11)


@pytest.mark.parametrize("name", ["rb_bal", "mb_bscan"])
def test_cube_is_built_on_first_read_only(name):
    g = _load(name)
    rt = _run_product(g).resample_tests
    d = rt.boot_debug_dict
    assert "right_sv_sampled" in d
    n0 = _launches()
    d["left_sv_sampled"], rt.LVcorr, d["indices"]
    if name.startswith("mb"):
        d["indices_behaviour"]
    assert _launches() == n0
    cube = d["right_sv_sampled"]
    n1 = _launches()
    assert n1 > n0
    assert d["right_sv_sampled"] is cube and _launches() == n1


@pytest.mark.parametrize("name", ["mct_m0_bal", "rb_bal", "mb_bscan"])
def test_cube_above_the_shared_bound_raises_before_any_work(name, monkeypatch):
    import torch
    from plspy_b200 import bootstrap_permutation as bp
    rt = _run_product(_load(name)).resample_tests
    monkeypatch.setattr(bp, "RIGHT_SV_MAX_BYTES", 1024)
    torch.cuda.synchronize()
    n0, m0 = _launches(), torch.cuda.memory_allocated()
    with pytest.raises(MemoryError, match="right_sv_sampled would need"):
        rt.boot_debug_dict["right_sv_sampled"]
    assert _launches() == n0 and torch.cuda.memory_allocated() == m0


def _mp_data():
    rs = np.random.RandomState(8)
    groups, C, p = (7, 6), 3, 1500
    N = sum(groups) * C
    X = rs.standard_normal((N, p)); X[:7, :80] += 1.0
    Y = rs.standard_normal((N, 2)) + 0.3 * X[:, :2]
    return X, Y, groups, C


def _mp_run(X, Y, groups, C):
    import plspy_b200
    np.random.seed(23)      # same seed on every rank -> identical index matrices
    return plspy_b200.PLS(X, groups, C, Y=Y, num_perm=0, num_boot=37, pls_method="rb").resample_tests


def _mp_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rt = _mp_run(*_mp_data())
        if rank == 1:           # one rank alone: the read involves no collective
            q.put(rt.boot_debug_dict["right_sv_sampled"])
    finally:
        dist.destroy_process_group()


def test_one_rank_of_two_processes_reads_the_single_process_cube():
    """Two processes on cuda:0 over gloo (as in test_gpu_multi): rank 1 alone reads the cube; the same kernels on the
    same draws in the same launches give the single-process cube bit for bit."""
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_mp_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    multi = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    single = _mp_run(*_mp_data()).boot_debug_dict["right_sv_sampled"]
    assert multi.shape == single.shape == (37, 1500, 12)
    assert np.array_equal(multi, single)


def test_reference_result_object_carries_the_cube_through_the_plugin():
    import baseline
    if not baseline.reference_available():
        pytest.skip("baseline/_ref not installed (python -m baseline.install_ref)")
    import plspy_b200
    from test_gpu_plugin import _run_reference
    mod = baseline.import_reference()
    plspy_b200.install(mod)
    try:
        g = _load("rb_unbal")
        rt = _run_reference(mod, g).resample_tests
        assert isinstance(rt, mod.core.bootstrap_permutation.ResampleTest)
        live = np.abs(g["s"]) > 1e-8
        p = g["X"].shape[1]
        right = rt.boot_debug_dict["right_sv_sampled"]
        np.testing.assert_allclose(right[:, :: max(1, p // 16), :][:, :, live], g["right_sv_sub"][:, :, live],
                                   rtol=1e-8, atol=1e-9)
    finally:
        plspy_b200.uninstall()
