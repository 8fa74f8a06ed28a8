"""The factored collapsed bootstrap beyond 320 rows: the factored pack in the layout of the output-stationary bootstrap
GEMM (boot_os.cu), and boot_algo="collapsed" for tall mct / cst designs against the direct formulation, across both
storages and both upload paths of X, two processes in both layouts, PLSB200_EXACT=os at N <= 320, and draws without
the subject structure (which have no other route there and are refused)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _design(seed, groups, C, p, offset=0.0):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((sum(groups) * C, p))
    X[:groups[0], : p // 10] += 0.7
    return X + offset


def _pls(X, groups, C, seed, **kw):
    import plspy_b200
    np.random.seed(seed)
    return plspy_b200.PLS(X, groups, C, **kw)


# ---- the kernel: pack + moment GEMM over J pseudo-resamples, against numpy ------------------------------------------
@pytest.mark.parametrize("N", [321, 360, 720, 1380])
@pytest.mark.parametrize("K,J", [(1, 196), (5, 7), (12, 49), (24, 196), (24, 1)])
def test_factored_pack_in_the_output_stationary_layout(N, K, J):
    import torch
    from plspy_b200.engine import Engine
    rs = np.random.RandomState(N + 31 * K + J)
    p = 1001                                                 # odd: a partial voxel tile
    ns = N // 3
    X = rs.standard_normal((N, p))
    E = rs.standard_normal((N, K))
    L = rs.standard_normal((ns, J))
    sid = rs.randint(0, ns, N).astype(np.int32)
    C = E[:, :, None] * L[sid][:, None, :]                    # c_jk[n] = E[n,k] L[sid[n], j]: N x K x J
    want = (np.einsum("nv,nkj->vkj", X, C) ** 2).sum(axis=2)
    # relative to sum_j (|x_v|^T |c_jk|)^2: a single product (J = 1) can cancel to near zero, where any summation
    # order differs from numpy's by more than 1e-12 of the result itself
    scale = (np.einsum("nv,nkj->vkj", np.abs(X), np.abs(C)) ** 2).sum(axis=2)
    q = Engine(X).boot_factor_quad(E, torch.from_numpy(L).cuda(), sid).cpu().numpy()
    err = float(np.max(np.abs(q - want) / scale))
    assert err <= 1e-12, err
    # float32 storage: bit-identical to float64 storage of the widened matrix
    X32 = X.astype(np.float32)
    L_d = torch.from_numpy(L).cuda()
    q32 = Engine(X32, x_storage="fp32").boot_factor_quad(E, L_d, sid).cpu().numpy()
    q64 = Engine(X32.astype(np.float64)).boot_factor_quad(E, L_d, sid).cpu().numpy()
    np.testing.assert_array_equal(q32, q64)


# ---- whole calls against the direct formulation ---------------------------------------------------------------------
TALL = {
    "mct_60x60x3": dict(groups=(60, 60), C=3, kw=dict(pls_method="mct")),
    "mct_40_45_35x6": dict(groups=(40, 45, 35), C=6, kw=dict(pls_method="mct", mctype=1)),
    "cst_40_45_35x6": dict(groups=(40, 45, 35), C=6, kw=dict(pls_method="cst")),
    "mct_60x60x3_offset": dict(groups=(60, 60), C=3, kw=dict(pls_method="mct"), offset=1000.0),
}


@pytest.mark.parametrize("case", sorted(TALL))
def test_tall_collapsed_matches_direct(case):
    c = TALL[case]
    groups, C = c["groups"], c["C"]
    X = _design(5, groups, C, 3001, offset=c.get("offset", 0.0))
    kw = dict(c["kw"])
    if kw["pls_method"] == "cst":
        kw["contrasts"] = np.random.RandomState(1).standard_normal((len(groups) * C, 4))
    assert X.shape[0] > 320 and 150 > sum(groups) - len(groups)
    res = {algo: _pls(X.copy(), groups, C, 9, num_perm=30, num_boot=150, boot_algo=algo, **kw)
           for algo in ("direct", "collapsed")}
    a, b = res["collapsed"].resample_tests, res["direct"].resample_tests
    assert a.boot_algo == "collapsed" and b.boot_algo == "direct"
    s = np.abs(res["direct"].s)
    live = s > 1e-8 * s.max()
    for f in ("std_errs", "boot_ratios"):
        d = _rel(getattr(a, f)[:, live], getattr(b, f)[:, live])
        assert d <= 1e-12, (f, d)
    np.testing.assert_array_equal(a.permute_ratio, b.permute_ratio)


def test_tall_upload_paths_and_storage_are_bit_identical():
    import torch
    from plspy_b200.engine import Engine
    groups, C = (60, 60), 3
    X = _design(9, groups, C, 30_001)
    assert X.nbytes >= Engine.PIPELINED_UPLOAD_MIN_BYTES
    kw = dict(num_perm=20, num_boot=130, pls_method="mct", boot_algo="collapsed")
    pinned = _pls(torch.from_numpy(X).pin_memory(), groups, C, 4, **kw).resample_tests
    resident = _pls(X, groups, C, 4, engine=Engine(torch.from_numpy(X).cuda()), **kw).resample_tests
    assert pinned.boot_algo == resident.boot_algo == "collapsed"
    np.testing.assert_array_equal(pinned.std_errs, resident.std_errs)
    np.testing.assert_array_equal(pinned.boot_ratios, resident.boot_ratios)
    X32 = X.astype(np.float32)
    a = _pls(X32, groups, C, 4, x_storage="fp32", **kw).resample_tests
    b = _pls(X32.astype(np.float64), groups, C, 4, **kw).resample_tests
    np.testing.assert_array_equal(a.std_errs, b.std_errs)
    np.testing.assert_array_equal(a.boot_ratios, b.boot_ratios)


def test_tall_draws_without_subject_structure_are_refused():
    import torch
    from plspy_b200 import exceptions, resample
    groups, C = (60, 60), 3
    co = np.array([[n] * C for n in groups])
    X = _design(5, groups, C, 500)
    np.random.seed(1)
    idx = resample.bootstrap_indices("mct", 130, co)[0].copy()
    idx[7, 3] = idx[7, 3 + 60]                               # row 3 draws from another cell
    for ind in (idx, torch.from_numpy(idx).cuda()):
        with pytest.raises(exceptions.NotImplementedError, match="320"):
            _pls(X.copy(), groups, C, 2, num_perm=0, num_boot=130, pls_method="mct", boot_algo="collapsed",
                 boot_indices=ind)
    # the same draws run with the direct formulation
    rt = _pls(X.copy(), groups, C, 2, num_perm=0, num_boot=130, pls_method="mct", boot_indices=idx).resample_tests
    assert rt.boot_algo == "direct"


# ---- PLSB200_EXACT=os: every design through boot_os.cu, the factored route included -----------------------------
_EXACT_OS_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import plspy_b200
rs = np.random.RandomState(3)
groups, C = (25, 25, 25), 4
X = rs.standard_normal((sum(groups) * C, 4001)); X[:25, :400] += 0.7
np.random.seed(8)
res = plspy_b200.PLS(X, groups, C, num_perm=0, num_boot=200, pls_method="mct", boot_algo="collapsed")
rt = res.resample_tests
np.savez(sys.argv[2], se=rt.std_errs, br=rt.boot_ratios, s=res.s)
print(json.dumps({"algo": rt.boot_algo}))
"""


def test_exact_os_runs_the_factored_route(tmp_path):
    out = tmp_path / "os.npz"
    env = dict(os.environ, PLSB200_EXACT="os")
    r = subprocess.run([sys.executable, "-c", _EXACT_OS_SCRIPT, ROOT, str(out)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["algo"] == "collapsed"
    got = np.load(out)
    rs = np.random.RandomState(3)
    groups, C = (25, 25, 25), 4
    X = rs.standard_normal((sum(groups) * C, 4001)); X[:25, :400] += 0.7
    res = _pls(X, groups, C, 8, num_perm=0, num_boot=200, pls_method="mct", boot_algo="collapsed")
    live = np.abs(res.s) > 1e-8 * np.abs(res.s).max()
    assert _rel(got["se"][:, live], res.resample_tests.std_errs[:, live]) <= 1e-13
    assert _rel(got["br"][:, live], res.resample_tests.boot_ratios[:, live]) <= 1e-13


# ---- two processes on one GPU (gloo), both layouts, at a tall design ----------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _two_proc_data():
    rs = np.random.RandomState(3)
    groups, C = (40, 45, 35), 3
    X = rs.standard_normal((sum(groups) * C, 20011)); X[:40, :80] += 1.0
    return X, groups, C


def _worker(rank, world, port, q, shard):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import plspy_b200
        X, groups, C = _two_proc_data()
        np.random.seed(11)
        rt = plspy_b200.PLS(X, groups, C, num_perm=0, num_boot=131, pls_method="mct", boot_algo="collapsed",
                            shard=shard).resample_tests
        se, br = rt.std_errs, rt.boot_ratios
        if rank == 0:
            q.put(dict(algo=rt.boot_algo, se=se, br=br))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("shard", ["resamples", "voxels"])
def test_two_processes_match_one_tall(shard):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, shard)) for r in range(2)]
    for pr in procs:
        pr.start()
    multi = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    X, groups, C = _two_proc_data()
    res = _pls(X, groups, C, 11, num_perm=0, num_boot=131, pls_method="mct", boot_algo="collapsed")
    rt = res.resample_tests
    assert X.shape[0] > 320
    assert multi["algo"] == rt.boot_algo == "collapsed"
    live = np.abs(res.s) > 1e-8
    assert _rel(multi["se"][:, live], rt.std_errs[:, live]) <= 1e-12
    assert _rel(multi["br"][:, live], rt.boot_ratios[:, live]) <= 1e-12
