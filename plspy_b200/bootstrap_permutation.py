"""GPU-backed permutation and bootstrap tests with the reference's plugin seam.

Mirrors plspy/core/bootstrap_permutation.py: an abstract `ResampleTest` with a registry
(`_register_subclass`, `_create`, :14-63) and one implementation registered for the six method keys
(:66-72) whose constructor has the reference's signature (:139-159) and sets the reference's result
attributes (`permute_ratio, stepdown_ratio, perm_debug_dict, conf_ints, [conf_ints_T], std_errs,
boot_ratios, [LVcorr], boot_debug_dict, CI`; "NA" placeholders when a test is skipped, :181-182,
:261-263).  The per-iteration Python loops (:323-452, :537-675) are replaced by batched CUDA kernels
(plspy_b200/csrc) driven through the C ABI; there is no CPU path.

Extra keyword-only arguments (not in the reference): `perm_indices`, `boot_indices` (index matrices
generated elsewhere -- each an int array, or a (task, behaviour) tuple for mb/cmb), `engine`
(an `Engine` that already holds X on the device), `device` (CUDA device of the engine built here), `precision` ("fp64" exact mode, or "tf32x3": the
bootstrap moment GEMM of the task methods on the tcgen05 tensor cores; p-values stay FP64-exact), `boot_algo`
("auto", default: "collapsed" where it does fewer flops, else "direct"; "direct": the bootstrap moments from the
B x p x K salience GEMM; "collapsed": mct / cst in the exact mode only, the same standard errors from the closed form
x_v^T Cov_r(c_rk) x_v -- see `check_boot_algo`; `boot_algo` of the result is the one that ran), `shard`
("resamples", default, or "voxels": the layout of X in a multi-process run -- see `check_shard`).
"""
import abc
import functools

import numpy as np
import torch
from scipy.stats import norm

from . import class_functions, dist, exceptions, resample
from .engine import Engine, check_choice

VERBOSE = False


def _log(*a):
    if VERBOSE:
        print(*a)


class ResampleTest(abc.ABC):
    _subclasses = {}
    pls_alg = None
    _pls_types = {
        "mct": "Mean-Centering Task PLS",
        "cst": "Contrast Task PLS",
        "rb": "Regular Behaviour PLS",
        "mb": "Multiblock PLS",
        "csb": "Contrast Behaviour PLS",
        "cmb": "Contrast Multiblock PLS",
    }

    @abc.abstractmethod
    def __str__(self):
        pass

    @abc.abstractmethod
    def __repr__(self):
        pass

    @classmethod
    def _register_subclass(cls, pls_method):
        def decorator(subclass):
            cls._subclasses[pls_method] = subclass
            return subclass
        return decorator

    @classmethod
    def _create(cls, pls_method, *args, **kwargs):
        if pls_method not in cls._subclasses and pls_method in cls._pls_types:
            raise exceptions.NotImplementedError(
                f"Specified PLS/Resample method {cls._pls_types[pls_method]} has not yet been implemented.")
        elif pls_method not in cls._subclasses:
            raise ValueError(f"Invalid PLS/Resample method {pls_method}")
        cls.pls_alg = pls_method
        return cls._subclasses[pls_method](*args, **kwargs)


class _LazyDebugDict(dict):
    """Debug dictionary whose expensive entries (e.g. the B x p x K `right_sv_sampled` cube the reference
    always materialises, bootstrap_permutation.py:497) are computed on first access."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self._lazy = {}

    def set_lazy(self, key, fn):
        self._lazy[key] = fn

    def __getitem__(self, key):
        if not dict.__contains__(self, key) and key in self._lazy:
            dict.__setitem__(self, key, self._lazy.pop(key)())
        return dict.__getitem__(self, key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in self._lazy

    def keys(self):
        return list(dict.keys(self)) + list(self._lazy.keys())

    # every other read access sees the lazy entries too (the reference returns a plain dict with every key present)
    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return dict.__len__(self) + len(self._lazy)

    def get(self, key, default=None):
        return self[key] if key in self else default

    def materialize(self):
        """Compute every pending entry (may be large: `right_sv_sampled` is B x p x K)."""
        for key in list(self._lazy):
            self[key]
        return self

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def values(self):
        return [self[k] for k in self.keys()]

    def copy(self):
        return dict(self.items())


class _DeviceResult:
    """A result matrix that is still on the device.  In a multi-process run every rank holds the same all-reduced
    results; only rank 0 copies the two p x K matrices (std_errs, boot_ratios) to the host eagerly -- eight ranks
    pulling the same 38 MB through one host at the same time ran at 12 GB/s each instead of 52 (3.3 ms of a 32.6 ms
    step at 8 GPUs) -- and the other ranks fetch theirs on first access (`_ResampleTestPLS.std_errs` / `.boot_ratios`)."""

    def __init__(self, eng, tensor):
        self.eng, self.tensor = eng, tensor

    def fetch(self):
        return self.eng.to_host(self.tensor)


def _p_sized_to_host(eng, *tensors):
    """(std_errs, boot_ratios, ...) as numpy arrays on rank 0 / in single-process runs, `_DeviceResult` elsewhere."""
    if dist.world()[1] > 1 and dist.world()[0] != 0:
        return [_DeviceResult(eng, t) for t in tensors]
    out = eng.to_host(*tensors)
    return out if isinstance(out, (list, tuple)) else [out]


def _p_sized_to_host_async(eng, *tensors):
    """`_p_sized_to_host` with the copies on the side stream, so that they overlap the kernels enqueued next: returns a
    function that waits for them and hands back what `_p_sized_to_host` would."""
    if dist.world()[1] > 1 and dist.world()[0] != 0:
        out = [_DeviceResult(eng, t) for t in tensors]
        return lambda: out
    fetch = eng.to_host_async(*tensors, side=True)
    return lambda: list(fetch()) if len(tensors) > 1 else [fetch()]


# Largest `right_sv_sampled` cube (B x p x K float64) a read builds.  The bootstrap itself never stores the cube: it
# accumulates the moments on the fly, and the lazy entry rebuilds the saliences only when asked for.
RIGHT_SV_MAX_BYTES = 2 << 30


def _check_right_sv_bytes(niter, p, K):
    """Raises MemoryError, before anything is allocated, when the niter x p x K cube exceeds RIGHT_SV_MAX_BYTES."""
    nbytes = niter * p * K * 8
    if nbytes > RIGHT_SV_MAX_BYTES:
        raise MemoryError(f"right_sv_sampled would need {nbytes / 2**30:.1f} GiB; the B200 path "
                          "accumulates its moments on the fly instead of storing it")


def _stepdown_tail(s):
    return np.cumsum((np.asarray(s, dtype=float) ** 2)[::-1])[::-1].copy()


def _index_shard(eng, indices, niter, lo, hi):
    """Rows [lo, hi) of the first `niter` index vectors as an int32 device tensor; `indices` may be a
    numpy array, a host tensor (pinned or not) or a device tensor."""
    if torch.is_tensor(indices):
        return eng.to_device(indices[lo:min(hi, niter)], torch.int32)
    return eng.to_device(np.asarray(indices)[lo:min(hi, niter)], torch.int32)


def _indices_to_host(indices, niter):
    if torch.is_tensor(indices):
        return indices[:niter].cpu().numpy()
    return np.asarray(indices)[:niter]


def _cell_offsets(cond_order):
    """int32 offsets of the (group, condition) blocks of rows."""
    sizes = np.asarray(cond_order).reshape(-1)
    return np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)


def _behaviour_state(eng, cells):
    """Per-engine cache of the block-centred X, its z-scored copy's Gram matrix (Gz = Z Z^T)."""
    st = getattr(eng, "_behaviour", None)
    key = tuple(int(c) for c in cells)
    if st is None or st["key"] != key:
        Xc, Z = eng.cell_standardize(cells)
        st = {"key": key, "Xc": Xc, "Gz": eng.gram_of(Z)}
        del Z
        eng._behaviour = st
    return st


def _multiblock_state(eng, cond_order, bscan, keep_zb=False):
    """Per-engine cache for mb/cmb: the bscan rows of X block-centred (Xcb) and z-scored (Zb), the Gram matrix Gw
    of the row stack W1 = [X; Zb] (permutations; formed from the two matrices, the stack is never built) and the
    column maps of the multiblock row order (per group: C task rows, then |bscan|*nb behaviour rows,
    class_functions.py:496-514).  The bootstraps work on the stack W2 = [Xcb; X], likewise as two row segments."""
    co = np.asarray(cond_order)
    key = ("mb", tuple(co.reshape(-1).tolist()), tuple(bscan))
    st = getattr(eng, "_multiblock", None)
    if st is not None and st["key"] == key and (not keep_zb or "Zb" in st):
        return st
    rows_b = np.concatenate([np.full(co[g, c], c in list(bscan), dtype=bool)
                             for g in range(co.shape[0]) for c in range(co.shape[1])]).nonzero()[0]
    cells_b = _cell_offsets(co[:, bscan])
    Xb = eng.X.index_select(0, torch.as_tensor(rows_b, device=eng.device))
    Xcb, Zb = eng.cell_standardize(cells_b, M=Xb)
    st = {"key": key, "rows_b": rows_b, "cells_b": cells_b, "Xcb": Xcb, "Nb": int(Xb.shape[0]),
          "Gw": eng.gram_stacked(eng.X, Zb)}
    if keep_zb:         # the device-side original analysis projects on Zb once more (device_analysis.multiblock)
        st["Zb"] = Zb
    del Zb, Xb
    eng._multiblock = st
    return st


def _multiblock_columns(cond_order, bscan, nb):
    co = np.asarray(cond_order)
    G, C = co.shape
    nbs = len(bscan)
    Kg = C + nbs * nb
    task = np.array([g * Kg + c for g in range(G) for c in range(C)])
    beh = np.array([g * Kg + C + cb * nb + j for g in range(G) for cb in range(nbs) for j in range(nb)])
    return task, beh, G * Kg


def _multiblock_indices(pls_alg, indices, niter, cond_order, bscan, Ybscan, boot):
    if indices is None:
        gen = resample.bootstrap_indices if boot else resample.permutation_indices
        indices = gen(pls_alg, niter, cond_order, bscan=bscan, Ybscan=Ybscan)
    if not isinstance(indices, tuple) or len(indices) != 2:
        raise ValueError("multiblock resampling needs a (task, behaviour) pair of index matrices")
    return indices


def _perm_multiblock(eng, X, U, s, cond_order, mctype, niter, pls_alg, contrast, bscan, Xbscan, Ybscan, indices,
                     rotate_method=2):
    """bootstrap_permutation.py:305-312, 342-347, 391-393, 413-433 for mb / cmb.  Task rows come from the
    task-permuted X, behaviour rows from the ORIGINAL bscan rows of X with globally permuted Ybscan; every
    row is L2-normalised.  With W = [X; Zb] all of it is N-space: row norms and projected norms are
    quadratic forms in Gw = W W^T."""
    st = _multiblock_state(eng, cond_order, bscan)
    nb = Ybscan.shape[1]
    tcol, bcol, K = _multiblock_columns(cond_order, bscan, nb)
    idx_t, idx_b = _multiblock_indices(pls_alg, indices, niter, cond_order, bscan, Ybscan, boot=False)
    Lop = (class_functions._cell_mean_operator(cond_order) if pls_alg == "cmb"
           else class_functions._centring_operator(cond_order, mctype))
    N, Nb = eng.N, st["Nb"]
    # rescaled observed singular values (:305-312): ||un-normalised multiblock of the original data||_F^2 is the sum
    # of the quadratic forms of its rows' coefficients in Gw
    C0 = np.zeros((N + Nb, K))
    C0[:N, tcol] = Lop.T
    C0[N:, bcol] = class_functions._behaviour_coefficients(Ybscan, np.asarray(cond_order)[:, list(bscan)])
    raw_sq = float(eng.nspace_coef(st["Gw"], eng.to_device(C0[None], torch.float64))[0].sum())   # sum_k C0_k^T Gw C0_k
    org_s = np.sqrt(s ** 2 / np.sum(s ** 2) * raw_sq)
    totcov_org = _stepdown_tail(org_s)
    Ucoef = _ucoef(U, contrast)
    Kc = Ucoef.shape[1]
    lo, hi = dist.shard(niter)
    it = _index_shard(eng, idx_t, niter, lo, hi); ib = _index_shard(eng, idx_b, niter, lo, hi)
    R = hi - lo
    Ct = eng.scatter_coef(np.ascontiguousarray(Lop.T), it)                          # R x N x GC
    Qb, _, _ = eng.rb_coef(Ybscan, ib, st["cells_b"], np.eye(len(bcol)), scatter=False)   # R x Nb x Kb
    C1 = torch.zeros(R, N + Nb, K, dtype=torch.float64, device=eng.device)
    C1[:, :N, torch.as_tensor(tcol, device=eng.device)] = Ct
    C1[:, N:, torch.as_tensor(bcol, device=eng.device)] = Qb
    d2row, _ = eng.nspace_coef(st["Gw"], C1)                                        # squared row norms
    total = d2row.sum(dim=1)                                                        # ||un-normalised multiblock||_F^2
    if rotate_method == 0:      # singular values of the permuted (row-normalised) multiblock matrix itself
        C2 = eng.coef_project(C1, d2row, np.eye(K))
        d2, _ = eng.sym_eig(eng.nspace_coef_gram(st["Gw"], C2))
        d2 = torch.clamp(d2, min=0.0)
    else:
        C2 = eng.coef_project(C1, d2row, Ucoef)
        d2, _ = eng.nspace_coef(st["Gw"], C2)
    if pls_alg == "mb":     # s_hat^4 rescale, compared with org_s (:419-427)
        counts, s_hat = eng.perm_count(d2, org_s, totcov_org, 0.0, mb_total=total)
    else:                   # cmb: raw s for the counts, rescaled org_s for the stepdown baseline (:433, :316-319)
        counts, s_hat = eng.perm_count(d2, s, totcov_org, 0.0)
    dist.allreduce_sum_(counts)
    s_hat = dist.gather_rows(s_hat, niter, lo)
    counts, s_list = eng.to_host(counts, s_hat)
    counts = counts.astype(float)
    debug = _LazyDebugDict()
    debug["s_list"] = s_list
    debug["sum_perm"] = np.sum(s_list ** 2, axis=1)
    debug["org_s"] = org_s
    debug.set_lazy("indices", lambda: _indices_to_host(idx_t, niter))
    debug.set_lazy("indices_behaviour", lambda: _indices_to_host(idx_b, niter))
    return counts[:Kc] / (niter + 1), counts[Kc:] / (niter + 1), debug


def _multiblock_boot_coef(eng, st, Lop, Ucoef, Ybscan, bscan, cond_order, it, ib, want_yz=False):
    """Row coefficients of pass 2 of the mb / cmb bootstrap for the draws (it, ib), rows ordered like W2 = [Xcb; X]:
    task rows (scatter of Lop^T, squared norms through G), behaviour rows (raw correlation rows, squared norms from
    pass 1), each row normalised and projected on Ucoef.  Returns (C2, Wfull, cells2, Yz); Yz only with want_yz.  The
    bootstrap and the lazy `right_sv_sampled` both build their coefficients here, so the cube comes from exactly the
    coefficients the moments used."""
    nb = Ybscan.shape[1]
    tcol, bcol, K = _multiblock_columns(cond_order, bscan, nb)
    N, Nb, dev = eng.N, st["Nb"], eng.device
    R = int(it.shape[0])
    tcol_d = torch.as_tensor(tcol, device=dev); bcol_d = torch.as_tensor(bcol, device=dev)
    # task rows: coefficients over the rows of X and their squared norms through G
    Ct = eng.scatter_coef(np.ascontiguousarray(Lop.T), it)                          # R x N x GC
    d2t, _ = eng.nspace_coef(eng.G, Ct)
    # behaviour rows: raw (un-normalised) correlation rows and pass 1 for their squared norms
    Qraw, Wb, Yz = eng.rb_coef(Ybscan, ib, st["cells_b"], np.eye(len(bcol)), scatter=True, want_yz=want_yz)
    _, _, _, nrm_b = eng.rb_boot(st["Xcb"], Qraw, Wb, st["cells_b"], want_t=False)
    d2row = torch.zeros(R, K, dtype=torch.float64, device=dev)
    d2row[:, tcol_d] = d2t
    d2row[:, bcol_d] = nrm_b
    C1 = torch.zeros(R, Nb + N, K, dtype=torch.float64, device=dev)                 # rows ordered like W2 = [Xcb; X]
    C1[:, :Nb, bcol_d] = Qraw
    C1[:, Nb:, tcol_d] = Ct
    C2 = eng.coef_project(C1, d2row, Ucoef)                                         # R x (Nb+N) x Kc
    Wfull = torch.cat([Wb, torch.zeros(R, N, dtype=torch.float64, device=dev)], dim=1)
    cells2 = np.concatenate([st["cells_b"], [Nb + N]]).astype(np.int32)
    return C2, Wfull, cells2, Yz


def _boot_multiblock(eng, U, s, V, cond_order, mctype, niter, pls_alg, contrast, bscan, Ybscan, lvcorrs_orig,
                     Tvsc_orig, CI, indices):
    """bootstrap_permutation.py:545-554, 609-675, 695-766 for mb / cmb: independent bootstrap draws for the
    task block (rows of X) and the behaviour block (bscan rows).  Two p-space passes per bootstrap batch:
    (1) squared norms of the behaviour rows (their per-voxel std depends on the draw), (2) the projected
    cross-block matrix VS = permuted^T U of the row-normalised multiblock, with fused moments and the
    latent products [Xcb; X] @ VS needed for LVcorr and Tdistrib."""
    st = _multiblock_state(eng, cond_order, bscan)
    nb = Ybscan.shape[1]
    idx_t, idx_b = _multiblock_indices(pls_alg, indices, niter, cond_order, bscan, Ybscan, boot=True)
    Lop = (class_functions._cell_mean_operator(cond_order) if pls_alg == "cmb"
           else class_functions._centring_operator(cond_order, mctype))
    Abar = class_functions._cell_mean_operator(cond_order)
    Ucoef = _ucoef(U, contrast)
    Nb = st["Nb"]
    numer = _numerator(eng, V, s, contrast)
    lo, hi = dist.shard(niter)
    it = _index_shard(eng, idx_t, niter, lo, hi); ib = _index_shard(eng, idx_b, niter, lo, hi)
    C2, Wfull, cells2, Yz = _multiblock_boot_coef(eng, st, Lop, Ucoef, Ybscan, bscan, cond_order, it, ib, want_yz=True)
    s1, s2, T, nrm2 = eng.rb_boot(st["Xcb"], C2, Wfull, cells2, pivot=numer, unit_cells=1, X2=eng.X)   # pass 2
    dist.allreduce_packed_([s1, s2])
    std_errs, boot_ratios = eng.boot_finalize(s1, s2, niter, numer=numer)
    LV = eng.rb_lvcorr(T[:, :Nb, :].contiguous(), nrm2, Yz, ib, st["cells_b"], nb)  # (:650, :674)
    XV = T[:, Nb:, :].contiguous()                                                  # X @ VS_b per bootstrap
    if pls_alg == "mb":      # cellmeans(smeanmat(X_new_T) @ V_hat) (:654-656)
        Lop2 = Abar @ class_functions._smeanmat_operator(cond_order, mctype)
        Td = eng.uhat(XV, Lop2, it)
    else:                    # cmb: cellmeans(X @ norm_crossblock) (:665-666)
        Td = eng.uhat(XV, Abar, None)
    inv = torch.where(nrm2 > 0, 1.0 / torch.sqrt(nrm2), torch.zeros_like(nrm2))
    Td = Td * inv[:, None, :]
    LV = dist.gather_rows(LV, niter, lo); Td = dist.gather_rows(Td, niter, lo)
    std_L, std_T, LV_h, Td_h = eng.to_host(eng.colstd(LV), eng.colstd(Td), LV, Td)
    std_errs_h, boot_ratios_h = _p_sized_to_host(eng, std_errs, boot_ratios)
    z = norm.ppf(1 - (1 - CI) / 2)
    conf_int = (lvcorrs_orig - std_L * z, lvcorrs_orig + std_L * z)                 # (:723-725)
    conf_int_T = (Tvsc_orig - std_T * z, Tvsc_orig + std_T * z)                     # (:732-734)
    debug = _LazyDebugDict()
    debug["left_sv_sampled"] = LV_h
    debug["Tdistrib"] = Td_h
    debug.set_lazy("indices", lambda: _indices_to_host(idx_t, niter))
    debug.set_lazy("indices_behaviour", lambda: _indices_to_host(idx_b, niter))

    def _right():   # the reference's B x p x K cube, only on request: every draw on this rank, no collective
        _check_right_sv_bytes(niter, eng.p, Ucoef.shape[1])
        st_ = _multiblock_state(eng, cond_order, bscan)
        it_all = _index_shard(eng, idx_t, niter, 0, niter); ib_all = _index_shard(eng, idx_b, niter, 0, niter)
        C2_, W_, cells_, _ = _multiblock_boot_coef(eng, st_, Lop, Ucoef, Ybscan, bscan, cond_order, it_all, ib_all)
        VS = torch.empty(niter, eng.p, Ucoef.shape[1], dtype=torch.float64, device=eng.device)
        eng.rb_boot(st_["Xcb"], C2_, W_, cells_, unit_cells=1, X2=eng.X, want_t=False, vs_out=VS)
        return VS.cpu().numpy()
    debug.set_lazy("right_sv_sampled", _right)

    def _right_chunks(max_bytes):   # the same cube in voxel chunks: pass 1 over all of X, then windows of pass 2
        st_ = _multiblock_state(eng, cond_order, bscan)
        it_all = _index_shard(eng, idx_t, niter, 0, niter); ib_all = _index_shard(eng, idx_b, niter, 0, niter)
        C2_, W_, cells_, _ = _multiblock_boot_coef(eng, st_, Lop, Ucoef, Ybscan, bscan, cond_order, it_all, ib_all)
        fill = eng.rb_salience(st_["Xcb"], C2_, W_, cells_, unit_cells=1, X2=eng.X)
        yield from eng.stream_chunks(fill, niter, Ucoef.shape[1], max_bytes)
    debug.right_sv_chunks = _right_chunks
    return conf_int, conf_int_T, std_errs_h, boot_ratios_h, LV_h, debug


def _ucoef(U, contrast):
    """The design-side weights the saliences are projected on: U, or the normalised contrasts (:385-389, :620)."""
    if contrast is None:
        return np.asarray(U, dtype=float)
    return class_functions._normalize(np.asarray(contrast, dtype=float))


def _numerator(eng, V, s, contrast):
    """Numerator of the bootstrap ratios, the original salience (:700-703): V s, or V with contrasts; also the pivot
    that keeps the running sums of squares well conditioned.  V may already be a device tensor."""
    Vd = eng.to_device(V, torch.float64)
    return Vd * eng.to_device(np.asarray(s, dtype=float), torch.float64) if contrast is None else Vd


def _local_numerator(eng, V, s, contrast):
    """`_numerator`, its rows of the voxels this engine holds."""
    numer, (v0, v1) = _numerator(eng, V, s, contrast), eng.voxel_range
    return numer[v0:v1].contiguous() if eng.voxel_sharded else numer


def _task_operators(pls_alg, cond_order, mctype, U, contrast):
    """Row-space pull-back of the design-side weights: E = Lop^T @ Ucoef (N x K).
    mct: Lop = centring operator, Ucoef = U (bootstrap_permutation.py:385-387, 404);
    cst: Lop = cell-mean operator, Ucoef = normalised contrasts (:389, :430-432, :620)."""
    if pls_alg == "mct":
        Lop = class_functions._centring_operator(cond_order, mctype)
        Ucoef = _ucoef(U, None)
    else:
        Lop = class_functions._cell_mean_operator(cond_order)
        Ucoef = _ucoef(U, contrast)
    return Lop, Ucoef, Lop.T @ Ucoef


def _jackknife_coefficients(pls_alg, cond_order, mctype, Ucoef):
    """The leave-one-subject-out jackknife of the task-method saliences, in row space (DESIGN.md section 5.8).  The
    jackknife unit is the subject that resample.bootstrap_indices draws: group g, subject s, in every condition.
    Without it the design has n_g - 1 subjects in group g, and its saliences are X_(-gs)^T Lop'^T Ucoef with Lop' the
    method's operator for that design (centring for mct, cell means for cst) and Ucoef the original design weights
    (U, or the normalised contrasts): no re-SVD, as for the bootstrap samples.  In row space that is X^T C_gs, C_gs
    (N x K) zero on the C removed rows.  Lop' depends on the group only, so one product per group is scattered.

    Returns (C, goff): C (J x N x K), J the number of subjects, group-major in the order of the rows; goff (G + 1,
    int32) the offsets of the groups in C.  Raises exceptions.NotImplementedError (host only, before any GPU work)
    unless every group has the same number of subjects in each condition and at least two subjects."""
    missing = _balance_missing(cond_order)
    co = np.asarray(cond_order) if missing is None else None
    if missing is None and (co[:, 0] < 2).any():
        g = int(np.flatnonzero(co[:, 0] < 2)[0])
        missing = f"group {g} has {int(co[g, 0])} subject(s)"
    if missing is not None:
        raise exceptions.NotImplementedError(
            "BCa salience intervals need a leave-one-subject-out jackknife: a cond_order in which every group has the "
            f"same number of subjects in each condition, and at least two subjects in every group ({missing})")
    G, C = co.shape
    n = co[:, 0].astype(np.int64)
    N, K = int(co.sum()), int(Ucoef.shape[1])
    goff = np.concatenate(([0], np.cumsum(n))).astype(np.int32)
    gstart = np.concatenate(([0], np.cumsum(n * C)))
    jack = np.zeros((int(n.sum()), N, K))
    for g in range(G):
        co_r = co.copy()
        co_r[g] -= 1
        Lop = (class_functions._centring_operator(co_r, mctype) if pls_alg == "mct"
               else class_functions._cell_mean_operator(co_r))
        E_r = Lop.T @ Ucoef                                   # (N - C) x K, the rows of the reduced design
        for sub in range(n[g]):
            keep = np.ones(N, dtype=bool)
            keep[gstart[g] + np.arange(C) * n[g] + sub] = False   # subject `sub` of group g in every condition
            jack[goff[g] + sub, keep] = E_r
    return jack, goff


BOOT_ALGOS = ("auto", "direct", "collapsed")


def _balance_missing(cond_order):
    """None when `cond_order` gives every group the same number of subjects in each condition, else what is missing."""
    if cond_order is None:
        return "no cond_order"
    co = np.asarray(cond_order)
    if co.ndim != 2 or co.size == 0 or (co != co[:, :1]).any():
        return "unequal subject counts across conditions"
    return None


def _factor_layout_missing(cond_order, nboot):
    """What the design lacks for the factored collapsed bootstrap (None: nothing): a `cond_order` with every group the
    same size in each condition, and more bootstraps than the ns - G columns of the factor (else M is singular)."""
    missing = _balance_missing(cond_order)
    if missing is not None:
        return missing
    co = np.asarray(cond_order)
    ns_g = int(co[:, 0].sum()) - co.shape[0]
    if nboot is None or not nboot > ns_g >= 1:
        return f"num_boot={nboot}, ns - G = {ns_g}"
    return None


def _no_collapsed_route(N, missing):
    return exceptions.NotImplementedError(
        f'boot_algo="collapsed" for a design of {N} rows: the N x N covariance route is limited to '
        f'{Engine.QUAD_MAX_ROWS} rows, and the factored route needs a cond_order in which every group has the same '
        'number of subjects in each condition, more bootstraps than ns - G (subjects minus groups), design weights '
        'constant within each cell and bootstrap draws with the subject structure of resample.bootstrap_indices (each '
        f'row drawn from its own cell, one subject map for all conditions) ({missing}); use boot_algo="direct"')


def check_boot_algo(boot_algo, pls_alg, precision, N, nboot=None, cond_order=None):
    """Validates the bootstrap formulation before any GPU work and returns the one that runs.

    "direct" accumulates the moments of the B x p x K bootstrap saliences VS_r = X^T C_r.  "collapsed" uses that every
    task-method salience is linear in the draw: Var_r(x_v^T c_rk) = x_v^T Cov_r(c_rk) x_v.  When the draws have the
    subject structure of resample.bootstrap_indices, the covariance factors through the draw counts of the ns subjects
    (DESIGN.md section 3) and the standard errors come from the bootstrap GEMM over ns - G pseudo-resamples
    (2 p N K (ns - G) flops instead of 2 p N K B); otherwise, for N <= 320, from K covariance matrices of N x N and one
    p x K quadratic form (2 p N^2 K flops).  Exact FP64 like the direct form; results agree to rounding.
    Beyond 320 rows only the factored route exists, so "collapsed" there needs `cond_order` (G x C subject counts)
    with every group the same size in each of its conditions (groups may differ) and more bootstraps (`nboot`, the
    whole run's) than ns - G; draws passed in must also have the subject structure (checked on the device).
    "auto" (default) is "collapsed" for mct / cst with precision="fp64", N <= 320 and more bootstraps than rows, else
    "direct"."""
    check_choice("boot_algo", boot_algo, BOOT_ALGOS)
    if boot_algo == "auto":
        fits = N is not None and N <= Engine.QUAD_MAX_ROWS and nboot is not None and nboot > N
        return "collapsed" if (pls_alg in ("mct", "cst") and precision == "fp64" and fits) else "direct"
    if boot_algo == "direct":
        return boot_algo
    if precision != "fp64":
        raise ValueError(f'boot_algo="collapsed" is an exact (precision="fp64") formulation, got precision={precision!r}')
    if pls_alg not in ("mct", "cst"):
        raise exceptions.NotImplementedError(
            'boot_algo="collapsed" applies to the task methods (mct, cst): the block standardisation of the behaviour '
            'and multiblock methods makes their saliences non-linear in the bootstrap draw')
    if N is not None and N > Engine.QUAD_MAX_ROWS:
        missing = _factor_layout_missing(cond_order, nboot)
        if missing is not None:
            raise _no_collapsed_route(N, missing)
    return boot_algo


def check_x_storage(x_storage, pls_alg):
    """Validates the device storage of X before any GPU work.

    "fp64" (default) holds X as float64.  "fp32" analyses X.astype(float32): the device holds that float32 matrix
    (half the memory and half the bytes of every pass over X) and every kernel widens an element where it loads it,
    so all results equal, bit for bit, those of the "fp64" run on the widened matrix.  Task methods (mct, cst) only:
    the block standardisation kernels of the behaviour and multiblock methods read float64."""
    check_choice("x_storage", x_storage, Engine.X_STORAGES)
    if x_storage == "fp32" and pls_alg not in ("mct", "cst"):
        raise exceptions.NotImplementedError(
            'x_storage="fp32" applies to the task methods (mct, cst); the behaviour and multiblock methods keep X '
            'in float64')


def check_shard(shard, pls_alg):
    """Validates the multi-process layout of X before any GPU work.

    "resamples" (default): every rank holds the whole of X and takes a share of the resamples.  "voxels": every rank
    holds only its columns of X (dist.voxel_shard: 1/world of the device memory for X and for the tall-design image of
    the bootstrap GEMM) and runs every bootstrap on them; the permutations and the per-bootstrap N-space outputs stay
    resample-sharded through the all-reduced Gram matrix, and the p x K results are gathered.  Task methods (mct,
    cst): the behaviour and multiblock bootstraps reduce over voxels per resample.  One process: the two are the
    same."""
    check_choice("shard", shard, Engine.SHARDS)
    if shard == "voxels" and pls_alg not in ("mct", "cst"):
        raise exceptions.NotImplementedError(
            'shard="voxels" applies to the task methods (mct, cst); the behaviour and multiblock bootstraps need '
            'per-resample norms over all voxels')


def resolve_options(pls_alg, engine=None, X=None, nboot=None, cond_order=None, precision="fp64", boot_algo="auto",
                    x_storage=None, shard=None):
    """The engine options of one analysis, validated before any GPU work: (precision, boot_algo, x_storage, shard).
    A given `engine` sets the precision and row count (else X's rows), and its x_storage and shard, which a value
    passed too must match (None: the engine's, else "fp64" / "resamples").  `boot_algo` None: not checked (a caller
    that does not know `nboot` and `cond_order` yet)."""
    check_choice("precision", precision, Engine.PRECISIONS)
    if engine is not None:
        for name, given in (("x_storage", x_storage), ("shard", shard)):
            if given is not None and given != getattr(engine, name):
                raise ValueError(f"{name}={given!r} but the engine holds X with {name}={getattr(engine, name)!r}")
        precision, N, x_storage, shard = engine.precision, engine.N, engine.x_storage, engine.shard
    else:
        N = int(X.shape[0]) if getattr(X, "shape", None) else None
        x_storage, shard = ("fp64" if x_storage is None else x_storage), ("resamples" if shard is None else shard)
    check_x_storage(x_storage, pls_alg)
    check_shard(shard, pls_alg)
    if boot_algo is not None:
        boot_algo = check_boot_algo(boot_algo, pls_alg, precision, N, nboot, cond_order)
    return precision, boot_algo, x_storage, shard


def _factor_plan(eng, pls_alg, U, contrast, cond_order, mctype, niter, indices):
    """The subject layout for the factored collapsed bootstrap (DESIGN.md section 3), or None when its preconditions
    do not hold and the N x N covariance route runs instead: those of `_factor_layout_missing`, E = Lop^T Ucoef
    bit-identical within each cell, and every draw keeping each row in its cell with one subject map for all
    conditions.  Indices drawn by the library (pass None) have that structure by construction; given ones are checked
    on the device, each rank its shard, with the flag all-reduced.  Designs of more than 320 rows have no N x N route:
    there exceptions.NotImplementedError replaces None (on every rank)."""
    def none_or_raise(missing):
        if eng.N > Engine.QUAD_MAX_ROWS:
            raise _no_collapsed_route(eng.N, missing)
        return None
    missing = _factor_layout_missing(cond_order, niter)
    if missing is not None:
        return none_or_raise(missing)
    co = np.asarray(cond_order)
    sizes = co[:, 0].astype(np.int64)
    G, C = co.shape
    _, _, E = _task_operators(pls_alg, cond_order, mctype, U, contrast)
    cells = _cell_offsets(co)
    if any((E[a:b] != E[a]).any() for a, b in zip(cells[:-1], cells[1:])):
        return none_or_raise("design weights that differ within a cell")
    gstart = np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)
    base = np.repeat(cells[:-1], co.reshape(-1))                         # first row of each row's cell
    sid = np.concatenate([gstart[g] + np.arange(sizes[g]) for g in range(G) for _ in range(C)])
    row0 = np.concatenate([cells[g * C] + np.arange(sizes[g]) for g in range(G)])
    plan = {"layout": eng.to_device(np.concatenate([base, sid, row0]).astype(np.int32), torch.int32),
            "sid": eng.to_device(sid.astype(np.int32), torch.int32), "gstart": gstart}
    if indices is not None:
        if isinstance(indices, tuple):
            indices = indices[0]
        lo, hi = dist.shard(niter)
        bad = (eng.boot_draw_check(_index_shard(eng, indices, niter, lo, hi), plan["layout"]) if hi > lo
               else torch.zeros(1, dtype=torch.int32, device=eng.device)).to(torch.int64)
        dist.allreduce_sum_(bad)
        if int(bad.item()) != 0:
            return none_or_raise("bootstrap draws without the subject structure")
    return plan


def _collapsed_sumsq(eng, E, idx_dev, niter, lo, hi, factor=None):
    """Collapsed bootstrap: q[v,k] = x_v^T S_k x_v with S_k = sum_r (c_rk - e_k)(c_rk - e_k)^T - s1_k s1_k^T / niter
    (= niter . Cov_r(c_rk)): the sum of squares of (VS_r - mean) over all `niter` resamples, p x K, the same on every
    rank.  `factor` (a `_factor_plan`): S_k = D_k P M P^T D_k through the ns x ns covariance M of the subjects' draw
    counts, M = L L^T, and q is the bootstrap GEMM over the ns - G columns of L; else the K N x N matrices S_k.
    Multi-process: one all-reduce of the N-space partial sums ([s1 | M] or [S1 | S2]), each rank evaluates q on its
    share of the voxels and the shares are gathered (a voxel-sharded engine: its own voxels, gathered later)."""
    E = eng.to_device(E, torch.float64)
    eng._x_ranges()          # (starts a deferred upload of X: the covariance build below overlaps it)
    if factor is not None:
        ns = int(factor["gstart"][-1])
        Mg = (eng.boot_count_gram(idx_dev, factor["layout"]) if hi > lo
              else torch.zeros(ns + 1, ns + 1, dtype=torch.float64, device=eng.device))
        dist.allreduce_sum_(Mg)
        L = eng.boot_factor(Mg, niter, factor["gstart"])
        quad = lambda *vox: eng.boot_factor_quad(E, L, factor["sid"], *vox)        # noqa: E731
    else:
        if hi > lo:
            S1, S2 = eng.boot_cov(E, idx_dev)
        else:
            K = E.shape[1]
            S1 = torch.zeros(eng.N, K, dtype=torch.float64, device=eng.device)
            S2 = torch.zeros(K, eng.N, eng.N, dtype=torch.float64, device=eng.device)
        dist.allreduce_packed_([S1, S2])
        s1t = S1.T
        Sig = S2 - s1t[:, :, None] * s1t[:, None, :] / niter
        quad = lambda *vox: eng.boot_quad(Sig, *vox)                                # noqa: E731
    if dist.world()[1] == 1 or eng.voxel_sharded:
        return quad()
    v0, v1 = dist.shard(eng.p)
    return dist.gather_rows(quad(v0, v1), eng.p, v0)


class _TaskPlan:
    """The inputs of one mct / cst bootstrap: operators, this rank's draws (rows [lo, hi); `idx_all`: every draw, for
    the moment stage of a voxel-sharded engine), the resolved `boot_algo` with its `_factor_plan` (None: the N x N
    route), and the `results` once `_boot_results` has run.  `drawn`: the library drew `indices` (no draw check).  V
    reaches the device at its first use: uploaded ahead of the collapsed stage it would hold back a pipelined X."""

    def __init__(self, eng, pls_alg, U, s, V, cond_order, mctype, contrast, niter, indices, boot_algo, drawn=False):
        if isinstance(indices, tuple):
            indices = indices[0]
        self.boot_algo, self.results = boot_algo, None
        self.Lop, self.Ucoef, self.E = _task_operators(pls_alg, cond_order, mctype, U, contrast)
        self.factor = (_factor_plan(eng, pls_alg, U, contrast, cond_order, mctype, niter, None if drawn else indices)
                       if boot_algo == "collapsed" else None)
        self.lo, self.hi = dist.shard(niter)
        self.idx = _index_shard(eng, indices, niter, self.lo, self.hi)
        self.idx_all = _index_shard(eng, indices, niter, 0, niter) if eng.voxel_sharded else self.idx
        self._eng, self._V, self._s, self._contrast = eng, V, s, contrast

    @functools.cached_property
    def V(self):
        return self._eng.to_device(self._V, torch.float64)

    @functools.cached_property
    def numer(self):
        return _local_numerator(self._eng, self.V, self._s, self._contrast)


def _boot_moments(eng, plan, niter, packed=None):
    """The moment stage of the mct / cst bootstrap: sums of VS_r - pivot and of its squares over all `niter` draws,
    complete on every rank (p x K, this engine's voxels); "collapsed": (0, sum of squares about the mean), with no
    p x K all-reduce.  `packed`: a `pack_coef` result for the plan's (E, idx) to reuse."""
    if plan.boot_algo == "collapsed":
        s2 = _collapsed_sumsq(eng, plan.E, plan.idx, niter, plan.lo, plan.hi, factor=plan.factor)
        return torch.zeros_like(s2), s2
    if eng.voxel_sharded:                       # every bootstrap on this rank's voxels: no moment all-reduce
        return eng.boot_moments(plan.E, plan.idx_all, pivot=plan.numer)
    if plan.hi > plan.lo:
        s1, s2 = eng.boot_moments(plan.E, plan.idx, pivot=plan.numer, packed=packed)   # K4
    else:
        s1 = torch.zeros_like(plan.numer); s2 = torch.zeros_like(plan.numer)
    dist.allreduce_packed_([s1, s2])
    return s1, s2


def _boot_results(eng, plan, niter, packed=None):
    """The moment stage of the mct / cst bootstrap, the standard errors and bootstrap ratios from it, and their copy to
    the host started on the side stream; returns the function that waits for [std_errs, boot_ratios]."""
    s1, s2 = _boot_moments(eng, plan, niter, packed)
    std_errs, boot_ratios = eng.boot_finalize(s1, s2, niter, numer=plan.numer)   # (:695-703)
    if eng.voxel_sharded:                                                       # ONE gather of [std_errs | boot_ratios]
        K = int(std_errs.shape[1])
        both = eng.gather_voxels(torch.cat([std_errs, boot_ratios], dim=1))
        std_errs, boot_ratios = both[:, :K], both[:, K:]
    return _p_sized_to_host_async(eng, std_errs, boot_ratios)


@ResampleTest._register_subclass("mct")
@ResampleTest._register_subclass("rb")
@ResampleTest._register_subclass("cst")
@ResampleTest._register_subclass("csb")
@ResampleTest._register_subclass("mb")
@ResampleTest._register_subclass("cmb")
class _ResampleTestPLS(ResampleTest):
    """Runs the permutation and bootstrap tests on the GPU and exposes the reference's result fields."""

    def __init__(self, X, Y, U, s, V, cond_order, mctype, contrast=None, preprocess=None, nperm=1000,
                 nboot=1000, bscan=None, Xbscan=None, Ybscan=None, lvcorrs_orig=None, Tvsc_orig=None,
                 CI=0.95, *, perm_indices=None, boot_indices=None, engine=None, precision="fp64", rotate_method=2,
                 device=None, boot_algo="auto", x_storage=None, shard=None):
        self.CI = CI
        self._Tvsc_orig, self._lvcorrs_orig = Tvsc_orig, lvcorrs_orig     # centres of bias_corrected_conf_ints
        precision, boot_algo, x_storage, shard = resolve_options(self.pls_alg, engine, X, nboot, cond_order, precision,
                                                                 boot_algo, x_storage, shard)
        self.boot_algo = boot_algo
        if rotate_method not in (0, 1, 2):
            raise ValueError("rotate_method must be 0 (SVD), 1 (Procrustes) or 2 (derived)")
        if rotate_method == 0 and self.pls_alg not in ("mct", "rb", "mb"):
            raise exceptions.NotImplementedError(
                "rotate_method=0 (per-permutation SVD) applies to the SVD methods (mct, rb, mb); the contrast methods "
                "have no SVD (class_functions.py:126-162)")
        self.rotate_method = rotate_method
        _log(f"PLS ALG: {self.pls_alg}")
        eng = engine if engine is not None else (
            Engine(X, device=device, precision=precision, x_storage=x_storage, shard=shard)
            if (nperm > 0 or nboot > 0) else None)
        self._engine = eng
        if eng is not None and self.pls_alg in ("mct", "cst") and dist.world()[1] > 1:
            eng.gram_collective()          # all ranks are here: Gram from per-rank voxel ranges + one all-reduce
        perm_pending = None
        plan = None
        if eng is not None and nboot > 0 and self.pls_alg in ("mct", "cst"):
            # the plan checks given draws (one small kernel and one wait) before the permutation work is enqueued;
            # the index matrices are drawn first, in the reference's order
            if nperm > 0:
                s[np.abs(s) < 1e-12] = 0                       # as _permutation_test does before anything reads s
                if perm_indices is None:
                    perm_indices = resample.permutation_indices(self.pls_alg, nperm, cond_order, Y=Y, bscan=bscan,
                                                                Ybscan=Ybscan)
            drawn = boot_indices is None
            if drawn:
                boot_indices = resample.bootstrap_indices(self.pls_alg, nboot, cond_order, Y=Y, bscan=bscan,
                                                          Ybscan=Ybscan)
            plan = _TaskPlan(eng, self.pls_alg, U, s, V, cond_order, mctype, contrast, nboot, boot_indices, boot_algo,
                             drawn=drawn)
            if self.pls_alg == "mct" and not eng.upload_in_flight:
                eng.prepare_xv(plan.V)          # X V for U_hat out of the Gram launch, where that is free
            if plan.boot_algo == "collapsed" or (eng.upload_in_flight and dist.world()[1] == 1):
                # The moment stage runs first, and the copy of its p x K results to the host (38 MB at the bench
                # shape) overlaps the N-space work of both tests.  When X is still crossing PCIe in voxel ranges
                # (Engine._upload_pipelined), the moment stage is also the one that can start on the ranges already
                # there.  The direct route on a resident X keeps it last, where it shares the packed coefficients of
                # the bootstrap's N-space pass.  The bootstrap's N-space outputs come next, so that their copy
                # (Tdistrib, U_hat) overlaps the permutation kernels and the step ends on the small copy of the
                # permutation results.  (The same order on every rank: boot_algo is the whole run's.)
                plan.results = _boot_results(eng, plan, nboot)
        boot_first = nboot > 0 and plan is not None and plan.results is not None
        boot_pending = None
        if boot_first:
            boot_pending = self._bootstrap_test(
                X, Y, U, s, V, cond_order, mctype, nboot, self.pls_alg, preprocess=preprocess, contrast=contrast,
                Tvsc_orig=Tvsc_orig, CI=CI, indices=boot_indices, engine=eng, boot_algo=boot_algo, _plan=plan,
                _defer=True)
        if nperm > 0:
            # the permutation kernels and their device->host copies are enqueued here; the host only waits for
            # them after the bootstrap work has been enqueued too, so the GPU never idles between the two tests
            perm_pending = self._permutation_test(
                X, Y, U, s, V, cond_order, mctype, nperm, self.pls_alg, preprocess=preprocess, contrast=contrast,
                bscan=bscan, Xbscan=Xbscan, Ybscan=Ybscan, indices=perm_indices, engine=eng, _defer=True,
                rotate_method=rotate_method)
        else:
            self.permute_ratio = "NA"
            self.stepdown_ratio = "NA"
        if nboot > 0:
            out = boot_pending() if boot_first else self._bootstrap_test(
                X, Y, U, s, V, cond_order, mctype, nboot, self.pls_alg, preprocess=preprocess, contrast=contrast,
                bscan=bscan, Xbscan=Xbscan, Ybscan=Ybscan, lvcorrs_orig=lvcorrs_orig, Tvsc_orig=Tvsc_orig, CI=CI,
                indices=boot_indices, engine=eng, boot_algo=boot_algo, _plan=plan)
            if self.pls_alg in ("rb", "csb"):
                self.conf_ints, self.std_errs, self.boot_ratios, self.LVcorr, self.boot_debug_dict = out
            elif self.pls_alg in ("mb", "cmb"):
                (self.conf_ints, self.conf_ints_T, self.std_errs, self.boot_ratios, self.LVcorr,
                 self.boot_debug_dict) = out
            else:
                self.conf_ints, self.std_errs, self.boot_ratios, self.boot_debug_dict = out
        else:
            self.conf_ints = ["NA", "NA"]
            self.std_errs = "NA"
            self.boot_ratios = "NA"
        if perm_pending is not None:
            self.permute_ratio, self.stepdown_ratio, self.perm_debug_dict = perm_pending()

    # ------------------------------------------------------------------------------------------
    def _default_conf(self, conf):
        return ((1 - self.CI) / 2, 1 - (1 - self.CI) / 2) if conf is None else (float(conf[0]), float(conf[1]))

    def percentile_conf_ints(self, conf=None):
        """Percentile intervals of the design-side bootstrap distributions: what the reference's commented-out
        `resample.confidence_interval(Tdistrib, conf=dist)` / `(left_sv_sampled, ...)` call sites compute
        (bootstrap_permutation.py:713-731 with resample.py:171-222), next to the normal-theory `conf_ints` it returns.
        conf: (lower, upper) fractions, default from CI.  Returns {name: (lower, upper)} for the distributions of this
        method ("Tdistrib" for the task rows, "left_sv_sampled" for behaviour correlations / design saliences)."""
        if self._engine is None or not hasattr(self, "boot_debug_dict"):
            raise exceptions.MissingParameterError("percentile intervals need a bootstrap test (num_boot > 0)")
        conf = self._default_conf(conf)
        out = {}
        for key in ("Tdistrib", "left_sv_sampled"):
            if key in self.boot_debug_dict:
                a = np.asarray(self.boot_debug_dict[key])
                if a.ndim >= 2 and a.size:
                    out[key] = tuple(self._engine.to_host(*self._engine.percentile_interval(a, conf)))
        return out

    def salience_percentile_intervals(self, conf=None, max_bytes=4 << 30):
        """Percentile interval of every brain salience over the bootstrap samples (element-wise
        `confidence_interval(right_sv_sampled)`), streamed in voxel chunks so the B x p x K cube the reference stores
        (bootstrap_permutation.py:497, 626) never exists.  Task methods (mct, cst).  Returns (lower, upper), p x K.
        With shard="voxels" every rank works on its voxels and the intervals are gathered: every rank must call it."""
        fn = getattr(getattr(self, "boot_debug_dict", None), "salience_percentiles", None)
        if fn is None:
            raise exceptions.NotImplementedError(
                "salience percentile intervals are available for the task methods (mct, cst) after a bootstrap test")
        return fn(self._default_conf(conf), max_bytes)

    def right_sv_sampled_chunks(self, max_bytes=1 << 30):
        """The per-bootstrap brain saliences `boot_debug_dict["right_sv_sampled"]` (B x p x K) at any size, in voxel
        chunks: a generator of (v0, v1, chunk), chunk a float64 array B x (v1 - v0) x K equal, bit for bit, to
        right_sv_sampled[:, v0:v1, :].  The chunks cover the voxels in increasing order, each holds at most `max_bytes`
        (but at least one voxel), and they are computed on the GPU while the previous chunk is copied to the host.

        A yielded array is valid until the next step of the generator (two pinned buffers are reused); copy what you
        keep, e.g. the whole cube to disk:

            out = np.lib.format.open_memmap("right_sv.npy", mode="w+", dtype=np.float64, shape=(B, p, K))
            for v0, v1, chunk in rt.right_sv_sampled_chunks():
                out[:, v0:v1] = chunk

        Nothing runs on the GPU until the first step; closing the generator early waits for the work in flight and
        frees its buffers.  In a multi-process run every rank streams every bootstrap on its own (no collective); with
        shard="voxels" a rank yields only its own voxels (global v0, v1 of its `voxel_range`).  The lazy
        `right_sv_sampled` entry stays bounded by RIGHT_SV_MAX_BYTES; this one is not."""
        fn = getattr(getattr(self, "boot_debug_dict", None), "right_sv_chunks", None)
        if self._engine is None or fn is None:
            raise exceptions.MissingParameterError("right_sv_sampled_chunks needs a bootstrap test (num_boot > 0)")
        if not max_bytes > 0:
            raise ValueError(f"max_bytes must be positive, got {max_bytes}")
        return fn(int(max_bytes))

    def _bc_conf(self, conf):
        if self._engine is None or not hasattr(self, "boot_debug_dict"):
            raise exceptions.MissingParameterError("bias-corrected intervals need a bootstrap test (num_boot > 0)")
        conf = self._default_conf(conf)
        if not all(0.0 <= q <= 1.0 for q in conf):
            raise ValueError(f"conf must hold two fractions in [0, 1], got {conf}")
        return conf

    def bias_corrected_conf_ints(self, conf=None):
        """Bias-corrected percentile intervals (Efron) of the design-side bootstrap distributions, with the share of
        bootstrap samples at or below the original value (the `*_adj` bounds and `prop` of the MATLAB PLS toolbox).
        The original value theta is the centre of the normal-theory interval: `Tvsc_orig` for "Tdistrib" (mct, cst,
        mb, cmb: `conf_ints`, or `conf_ints_T` for mb / cmb), `lvcorrs_orig` for "left_sv_sampled" (rb, csb, mb, cmb:
        `conf_ints`), broadcast against the distribution's elements as there.  prop = #{samples <= theta} / B, and the
        bounds are the samples at the levels Phi(2 Phi^-1(prop) + Phi^-1(q)) (NaN where prop is 0 or 1), interpolated
        like `percentile_conf_ints` (DESIGN.md section 5.8).  conf: (lower, upper) fractions, default from CI.
        Returns {name: (lower, upper, prop)}."""
        conf = self._bc_conf(conf)
        centres = {"Tdistrib": self._Tvsc_orig if self.pls_alg in ("mct", "cst", "mb", "cmb") else None,
                   "left_sv_sampled": self._lvcorrs_orig if self.pls_alg in ("rb", "csb", "mb", "cmb") else None}
        out = {}
        for key, theta in centres.items():
            if theta is None or key not in self.boot_debug_dict:
                continue
            a = np.asarray(self.boot_debug_dict[key])
            if a.ndim >= 2 and a.size:
                theta = np.asarray(theta, dtype=float)
                shape = np.broadcast_shapes(theta.shape, a.shape[1:])
                a, theta = np.broadcast_to(a, a.shape[:1] + shape), np.broadcast_to(theta, shape)
                out[key] = tuple(self._engine.to_host(*self._engine.percentile_interval_bc(a, theta, conf)))
        return out

    def salience_bias_corrected_intervals(self, conf=None, max_bytes=4 << 30):
        """Bias-corrected percentile interval of every brain salience over the bootstrap samples, with prop, as
        `bias_corrected_conf_ints` defines them; theta is the numerator of `boot_ratios` (V s for mct, V for cst).
        Streamed in voxel chunks like `salience_percentile_intervals`.  Task methods (mct, cst).  Returns (lower,
        upper, prop), p x K.  With shard="voxels" every rank works on its voxels and the results are gathered: every
        rank must call it."""
        conf = self._bc_conf(conf)
        fn = getattr(self.boot_debug_dict, "salience_percentiles_bc", None)
        if fn is None:
            raise exceptions.NotImplementedError(
                "bias-corrected salience intervals are available for the task methods (mct, cst)")
        return fn(conf, max_bytes)

    def salience_bca_intervals(self, conf=None, max_bytes=4 << 30):
        """Bias-corrected and accelerated percentile interval (BCa, Efron 1987) of every brain salience over the
        bootstrap samples, with prop and the acceleration.  theta, prop and z0 = Phi^-1(prop) are those of
        `salience_bias_corrected_intervals`.  The acceleration a of every salience comes from its leave-one-subject-out
        jackknife (the subject is the unit resample.bootstrap_indices draws; the saliences without subject (g, s) are
        projected on the original design weights, with no re-SVD), stratified by group: with theta_(-gs) the jackknife
        values and l_gs = (n_g - 1)(mean_s theta_(-gs) - theta_(-gs)),
        a = (1/6) sum_g n_g^-3 sum_s l_gs^3 / (sum_g n_g^-2 sum_s l_gs^2)^(3/2), 0 where the denominator is 0.
        With w = z0 + Phi^-1(q) the bounds are the samples at the levels Phi(z0 + w / (1 - a w)), interpolated like
        `percentile_conf_ints`; they are NaN where 1 - a w <= 0, where prop is 0 or 1 and for a NaN theta, and q = 0 / 1
        give the minimum / maximum.  With a = 0 they are the bias-corrected bounds (DESIGN.md section 5.8).

        Streamed in voxel chunks like `salience_percentile_intervals`; `max_bytes` bounds the bootstrap and the
        jackknife chunks together.  Task methods (mct, cst) on a design in which every group has the same number of
        subjects in each condition and at least two subjects (else exceptions.NotImplementedError, before any GPU work).
        Returns (lower, upper, prop, accel), p x K.  With shard="voxels" every rank works on its voxels and the results
        are gathered: every rank must call it."""
        conf = self._bc_conf(conf)
        fn = getattr(self.boot_debug_dict, "salience_percentiles_bca", None)
        if fn is None:
            raise exceptions.NotImplementedError("BCa salience intervals are available for the task methods (mct, cst)")
        return fn(conf, max_bytes)

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _permutation_test(X, Y, U, s, V, cond_order, mctype, niter, pls_alg, preprocess=None, contrast=None,
                          threshold=1e-12, bscan=None, Xbscan=None, Ybscan=None, indices=None, engine=None,
                          _defer=False, rotate_method=2):
        """bootstrap_permutation.py:265-464.  `s` is thresholded in place like the reference (:295).
        `_defer=True` returns a function that waits for the device results and builds the outputs.

        rotate_method (the option of the older plspy API that survives in docs/_build/html/plspy.html:438-440):
          2 "derived" (the current reference code and the default): s_hat = column norms of permuted^T U;
          1 "Procrustes": [pu, ps, pv] = svd(permuted), rotation Q = v u^T from svd(U^T pv), s_hat = column norms
            of pv ps Q.  U and pv are square orthogonal K x K matrices, so Q = pv^T U exactly and
            s_hat_k^2 = U_k^T (pv ps^2 pv^T) U_k = || permuted^T U_k ||^2: identical to the derived value, and served
            by the same kernels (tests/test_gpu_kernels.py checks this against an explicit numpy Procrustes);
          0 "SVD": s_hat = the singular values of the permuted cross-block matrix itself (mct, rb, mb): K x K Gram
            matrix through G / Gz / Gw (plsb200_nspace_gram_f64, plsb200_nspace_coef_gram_f64) + the Jacobi
            eigensolver (plsb200_sym_eig_f64).
        The bootstrap test always aligns a resample with the original latent variables; there Procrustes (1) and
        derived (2) coincide for the same reason (the rotated salience pv ps Q equals permuted^T U), so
        `rotate_method` does not change any bootstrap output (tests/test_gpu_kernels.py checks an explicit numpy
        SVD + Procrustes bootstrap against it)."""
        eng = engine if engine is not None else Engine(X)
        s[np.abs(s) < threshold] = 0
        if pls_alg in ("mb", "cmb"):
            out = _perm_multiblock(eng, X, U, s, cond_order, mctype, niter, pls_alg, contrast, bscan, Xbscan,
                                   Ybscan, indices, rotate_method=rotate_method)
            return (lambda: out) if _defer else out
        org_s = np.copy(s)
        totcov_org = _stepdown_tail(org_s)
        behaviour = pls_alg in ("rb", "csb")
        if indices is None:
            indices = resample.permutation_indices(pls_alg, niter, cond_order, Y=Y, bscan=bscan, Ybscan=Ybscan)
        if isinstance(indices, tuple):
            indices = indices[1] if behaviour else indices[0]
        lo, hi = dist.shard(niter)
        idx_dev = _index_shard(eng, indices, niter, lo, hi)
        if behaviour:
            # only Y is permuted (:337-340, 395-396): X keeps its block z-scores, so everything lives in
            # N-space through Gz = Z Z^T
            cells = _cell_offsets(cond_order)
            Ucoef = _ucoef(U, contrast)
            K = Ucoef.shape[1]
            Gz = _behaviour_state(eng, cells)["Gz"]
            if rotate_method == 0:
                # singular values of the permuted correlation matrix R_r itself: eigenvalues of R_r R_r^T = Q^T Gz Q
                # with the un-projected row coefficients Q (U = identity)
                Kr = (len(cells) - 1) * Y.shape[1]
                Q, _, _ = eng.rb_coef(Y, idx_dev, cells, np.eye(Kr), scatter=False)
                d2, _ = eng.sym_eig(eng.nspace_coef_gram(Gz, Q))
                d2 = torch.clamp(d2, min=0.0)
                K = Kr
            else:
                Q, _, _ = eng.rb_coef(Y, idx_dev, cells, Ucoef, scatter=False)
                d2, _ = eng.nspace_coef(Gz, Q)
            Lop = None
        else:
            Lop, Ucoef, E = _task_operators(pls_alg, cond_order, mctype, U, contrast)
            K = E.shape[1]
            if rotate_method == 0:
                # squared singular values of M_r = Lop X[idx_r]: eigenvalues of M_r M_r^T = C_r^T G C_r
                Bfull = eng.nspace_gram(np.ascontiguousarray(Lop.T), idx_dev)
                d2, _ = eng.sym_eig(Bfull)
                d2 = torch.clamp(d2, min=0.0)
                K = d2.shape[1]
            else:
                d2, _ = eng.nspace(E, idx_dev)
        counts, s_hat = eng.perm_count(d2, s, totcov_org, threshold if pls_alg in ("mct", "rb") else 0.0)
        dist.allreduce_sum_(counts)
        s_hat = dist.gather_rows(s_hat, niter, lo)
        fetch = eng.to_host_async(counts, s_hat)

        def _sum_sq_crossblock():                              # sum(permuted**2) (:399): trace(Lop S G S^T Lop^T)
            if Lop is None:
                raise exceptions.NotImplementedError("perm_debug_dict['sum_s'] is not provided for behaviour PLS")
            if dist.world()[1] > 1:
                raise RuntimeError("perm_debug_dict['sum_s'] is only available in single-process runs")
            d2f, _ = eng.nspace(np.ascontiguousarray(Lop.T), _index_shard(eng, indices, niter, 0, niter))
            return d2f.sum(dim=1).cpu().numpy()

        def finish():
            counts_h, s_list = fetch()
            counts_h = counts_h.astype(float)
            permute_ratio = counts_h[:K] / (niter + 1)
            stepdown_ratio = counts_h[K:] / (niter + 1)
            _log(f"real s: {s}\nratio: {permute_ratio}\nStepdown perm ratio: {stepdown_ratio}")
            debug = _LazyDebugDict()
            debug["s_list"] = s_list                               # row i = s_hat of permutation i (:439-441)
            debug["sum_perm"] = np.sum(s_list ** 2, axis=1)        # key names swapped in the reference (:459-460)
            debug.set_lazy("indices", lambda: _indices_to_host(indices, niter))
            debug.set_lazy("sum_s", _sum_sq_crossblock)
            return permute_ratio, stepdown_ratio, debug
        return finish if _defer else finish()

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _bootstrap_test(X, Y, U, s, V, cond_order, mctype, niter, pls_alg, preprocess=None, dist_=(0.05, 0.95),
                        contrast=None, bscan=None, Xbscan=None, Ybscan=None, lvcorrs_orig=None, Tvsc_orig=None,
                        CI=0.95, indices=None, engine=None, boot_algo="direct", _plan=None, _defer=False):
        """bootstrap_permutation.py:466-766 for the task methods (mct, cst).  `boot_algo`: see `check_boot_algo`
        ("auto" resolves here).  `_plan`: the `_TaskPlan` of these draws (mct / cst), with its results when its moment
        stage already ran; built here when None.  `_defer=True` (mct / cst) returns a function that waits for the
        device results and builds the outputs.  A voxel-sharded engine
        runs the moment GEMM of ALL bootstraps on its voxels (no moment all-reduce) and gathers the p x K results; the
        lazy `right_sv_sampled` and the salience percentiles are then gathered too, so every rank must ask for them."""
        eng = engine if engine is not None else Engine(X)
        if _plan is None:
            boot_algo = check_boot_algo(boot_algo, pls_alg, eng.precision, eng.N, niter, cond_order)
        if indices is None:
            indices = resample.bootstrap_indices(pls_alg, niter, cond_order, Y=Y, bscan=bscan, Ybscan=Ybscan)
        if pls_alg in ("mb", "cmb"):
            return _boot_multiblock(eng, U, s, V, cond_order, mctype, niter, pls_alg, contrast, bscan, Ybscan,
                                    lvcorrs_orig, Tvsc_orig, CI, indices)
        if isinstance(indices, tuple):
            indices = indices[0]
        if pls_alg in ("rb", "csb"):
            return _ResampleTestPLS._bootstrap_behaviour(eng, Y, U, s, V, cond_order, niter, pls_alg, contrast,
                                                         lvcorrs_orig, CI, indices)
        plan = _plan if _plan is not None else _TaskPlan(eng, pls_alg, U, s, V, cond_order, mctype, contrast, niter,
                                                         indices, boot_algo)
        Lop, Ucoef, E, idx_dev, lo, hi = plan.Lop, plan.Ucoef, plan.E, plan.idx, plan.lo, plan.hi
        Abar = class_functions._cell_mean_operator(cond_order)
        vox = eng.voxel_sharded
        # exact mode, single launch: the packed coefficients serve the N-space pass and the moment GEMM
        packed = (eng.pack_coef(E, idx_dev) if (hi > lo and eng.precision == "fp64" and plan.results is None
                                                and E.shape[1] <= eng.KMAX and not vox) else None)
        d2, Tdist = eng.nspace(E, idx_dev, Lmat=Abar, packed=packed)        # Tdistrib (:633-634, :665-666)
        if pls_alg == "mct":
            XL = eng.xv(plan.V)                                             # X @ V once
            left = eng.uhat(XL, Lop, idx_dev)                               # U_hat (:617, :631)
        else:
            left = None
        # the per-bootstrap N-space outputs are complete here: assemble them across ranks and start their
        # device -> host copies on a second stream, so that they overlap the kernels enqueued next (the moment GEMM, or
        # the permutation test when the moment stage ran first)
        Tdist = dist.gather_rows(Tdist, niter, lo)
        if left is not None:
            left = dist.gather_rows(left, niter, lo)
        # (multi-process runs gather R x K x K per family from every rank -- the whole job's, not the shard's -- so
        # there only the standard deviations cross PCIe now and the distributions follow on first access)
        defer = dist.world()[1] > 1
        fetch_small = (eng.to_host_async(eng.colstd(Tdist), side=True) if defer
                       else eng.to_host_async(eng.colstd(Tdist), Tdist, left, side=True))
        fetch_p = plan.results if plan.results is not None else _boot_results(eng, plan, niter, packed)

        def finish():
            z = norm.ppf(1 - (1 - CI) / 2)                                      # (:709)
            std_errs_h, boot_ratios_h = fetch_p()
            std_T, Tdist_h, left_h = (fetch_small(), None, None) if defer else fetch_small()
            half = std_T * z                                                    # (:715-716)
            conf_int = (Tvsc_orig - half, Tvsc_orig + half)

            debug = _LazyDebugDict()
            if defer:
                debug.set_lazy("Tdistrib", lambda: eng.to_host(Tdist))
                debug.set_lazy("left_sv_sampled", (lambda: eng.to_host(left)) if left is not None
                               else (lambda: np.zeros((niter, Ucoef.shape[0], Ucoef.shape[1]))))
            else:
                debug["left_sv_sampled"] = (left_h if left_h is not None
                                            else np.zeros((niter, Ucoef.shape[0], Ucoef.shape[1])))
                debug["Tdistrib"] = Tdist_h
            debug.set_lazy("indices", lambda: _indices_to_host(indices, niter))

            def _right():   # the reference's B x p x K cube, only on request
                _check_right_sv_bytes(niter, eng.p_total, E.shape[1])
                VS = eng.salience(E, _index_shard(eng, indices, niter, 0, niter))
                if vox:     # voxel-major for the gather
                    VS = eng.gather_voxels(VS.transpose(0, 1).contiguous()).transpose(0, 1).contiguous()
                return VS.cpu().numpy()
            debug.set_lazy("right_sv_sampled", _right)

            def _right_chunks(max_bytes):   # this engine's voxels in chunks (voxel-sharded: no gather)
                fill = eng.salience_window(E, _index_shard(eng, indices, niter, 0, niter))
                yield from eng.stream_chunks(fill, niter, E.shape[1], max_bytes, v_offset=eng.voxel_range[0])
            debug.right_sv_chunks = _right_chunks

            def _to_host_gathered(*parts):       # p x K parts of this engine's voxels; voxel-sharded: one gather
                if vox:
                    K = int(parts[0].shape[1])
                    both = eng.gather_voxels(torch.cat(parts, dim=1))
                    parts = [both[:, i * K:(i + 1) * K] for i in range(len(parts))]
                return tuple(eng.to_host(*parts))

            def _salience_percentiles(conf, max_bytes=4 << 30):
                return _to_host_gathered(*eng.salience_percentiles(E, _index_shard(eng, indices, niter, 0, niter),
                                                                   conf, max_bytes))
            debug.salience_percentiles = _salience_percentiles

            def _salience_percentiles_bc(conf, max_bytes=4 << 30):
                return _to_host_gathered(*eng.salience_percentiles_bc(
                    E, _index_shard(eng, indices, niter, 0, niter), _local_numerator(eng, V, s, contrast), conf,
                    max_bytes))
            debug.salience_percentiles_bc = _salience_percentiles_bc

            def _salience_percentiles_bca(conf, max_bytes=4 << 30):
                jack = _jackknife_coefficients(pls_alg, cond_order, mctype, Ucoef)      # raises before any GPU work
                return _to_host_gathered(*eng.salience_percentiles_bca(
                    E, _index_shard(eng, indices, niter, 0, niter), _local_numerator(eng, V, s, contrast), jack, conf,
                    max_bytes))
            debug.salience_percentiles_bca = _salience_percentiles_bca
            return conf_int, std_errs_h, boot_ratios_h, debug
        return finish if _defer else finish()

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _bootstrap_behaviour(eng, Y, U, s, V, cond_order, niter, pls_alg, contrast, lvcorrs_orig, CI, indices):
        """bootstrap_permutation.py:537-675, 695-766 for rb / csb: X and Y rows are resampled together, the
        block z-scores of X change with every draw, so X is streamed once per bootstrap batch (K5)."""
        cells = _cell_offsets(cond_order)
        Ucoef = _ucoef(U, contrast)
        nb = Y.shape[1]
        numer = _numerator(eng, V, s, contrast)
        Xc = _behaviour_state(eng, cells)["Xc"]
        lo, hi = dist.shard(niter)
        idx_dev = _index_shard(eng, indices, niter, lo, hi)
        if hi > lo:
            Q, W, Yz = eng.rb_coef(Y, idx_dev, cells, Ucoef, scatter=True, want_yz=True)
            s1, s2, T, nrm2 = eng.rb_boot(Xc, Q, W, cells, pivot=numer)
            LV = eng.rb_lvcorr(T, nrm2, Yz, idx_dev, cells, nb)                 # (:636-642, 668-675)
        else:
            s1 = torch.zeros_like(numer); s2 = torch.zeros_like(numer)
            LV = torch.zeros((0, (len(cells) - 1) * nb, Ucoef.shape[1]), dtype=torch.float64, device=eng.device)
        dist.allreduce_packed_([s1, s2])
        std_errs, boot_ratios = eng.boot_finalize(s1, s2, niter, numer=numer)    # (:695-703)
        LV = dist.gather_rows(LV, niter, lo)
        std_L, LV_h = eng.to_host(eng.colstd(LV), LV)
        std_errs_h, boot_ratios_h = _p_sized_to_host(eng, std_errs, boot_ratios)
        z = norm.ppf(1 - (1 - CI) / 2)
        half = std_L * z                                                        # (:723-725)
        conf_int = (lvcorrs_orig - half, lvcorrs_orig + half)
        debug = _LazyDebugDict()
        debug["left_sv_sampled"] = LV_h
        debug.set_lazy("indices", lambda: _indices_to_host(indices, niter))

        def _right():   # the reference's B x p x K cube, only on request: every draw on this rank, no collective
            _check_right_sv_bytes(niter, eng.p, Ucoef.shape[1])
            Xc_ = _behaviour_state(eng, cells)["Xc"]
            Q_, W_, _ = eng.rb_coef(Y, _index_shard(eng, indices, niter, 0, niter), cells, Ucoef, scatter=True)
            VS = torch.empty(niter, eng.p, Ucoef.shape[1], dtype=torch.float64, device=eng.device)
            eng.rb_boot(Xc_, Q_, W_, cells, want_t=False, vs_out=VS)
            return VS.cpu().numpy()
        debug.set_lazy("right_sv_sampled", _right)

        def _right_chunks(max_bytes):   # the same cube in voxel chunks, from the same coefficients
            Xc_ = _behaviour_state(eng, cells)["Xc"]
            Q_, W_, _ = eng.rb_coef(Y, _index_shard(eng, indices, niter, 0, niter), cells, Ucoef, scatter=True)
            fill = eng.rb_salience(Xc_, Q_, W_, cells)
            yield from eng.stream_chunks(fill, niter, Ucoef.shape[1], max_bytes)
        debug.right_sv_chunks = _right_chunks
        return conf_int, std_errs_h, boot_ratios_h, LV_h, debug

    # ------------------------------------------------------------------------------------------
    # std_errs / boot_ratios: plain numpy arrays (or the reference's "NA"); ranks > 0 of a multi-process run hold them on
    # the device until first access (see _DeviceResult)
    def _lazy_get(self, name):
        v = self.__dict__.get(name)
        if isinstance(v, _DeviceResult):
            v = self.__dict__[name] = v.fetch()
        return v

    std_errs = property(lambda self: self._lazy_get("_std_errs"),
                        lambda self, v: self.__dict__.__setitem__("_std_errs", v))
    boot_ratios = property(lambda self: self._lazy_get("_boot_ratios"),
                           lambda self, v: self.__dict__.__setitem__("_boot_ratios", v))

    # ------------------------------------------------------------------------------------------
    def __repr__(self):
        stg = "Permutation Test Results\n------------------------\n\n"
        stg += f"Ratio: {self.permute_ratio}\n\n"
        stg += f"Step Down Ratio: {self.stepdown_ratio}\n\n"
        stg += "Bootstrap Test Results\n----------------------\n\n"
        stg += f"Selected Confidence Interval Level: {self.CI}\n"
        stg += "\nLower CI: \n" + str(self.conf_ints[0])
        stg += "\n\nUpper CI: \n" + str(self.conf_ints[1])
        if self.pls_alg in ["mb", "cmb"] and hasattr(self, "conf_ints_T"):
            stg += "\n\nLower CI (Task): \n" + str(self.conf_ints_T[0])
            stg += "\n\nUpper CI (Task): \n" + str(self.conf_ints_T[1])
        stg += "\n\nStandard Errors:\n" + str(self.std_errs)
        stg += "\n\nBootstrap Ratios:\n" + str(self.boot_ratios)
        return stg

    __str__ = __repr__
