"""The six PLS method classes with the reference's constructor signatures and result fields
(plspy/core/pls_classes.py: mct :74-382, rb :385-646, cst :649-927, csb :930-1202, mb :1205-1557,
cmb :1560-1925; result-field contract SURVEY.md App. D).

Each constructor validates like the reference, runs the one-off analysis step on the host
(`class_functions`), then hands (X, U, s, V, ...) to the GPU resampling engine through the same seam
the reference uses (`ResampleTest._create`, `split_half_resampling.split_half*`), and finally swaps
U and V "to be consistent with matlab" (:323).
"""
import abc
import os

import numpy as np

from . import bootstrap_permutation, class_functions, device_analysis, exceptions, split_half_resampling


class PLSBase(abc.ABC):
    """Registry/factory of PLS variants (pls_classes.py:12-71)."""

    _subclasses = {}
    _pls_types = {
        "mct": "Mean-Centring Task PLS",
        "rb": "Regular Behaviour PLS",
        "cst": "Contrast Task PLS",
        "csb": "Contrast Behaviour PLS",
        "mb": "Multiblock PLS",
        "cmb": "Contrast Multiblock PLS",
    }

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
            raise ValueError(f"Invalid PLS method {pls_method}")
        return cls._subclasses[pls_method](*args, **kwargs)

    # ---- shared helpers -------------------------------------------------------------------
    _ENGINE_KWARGS = ("perm_indices", "boot_indices", "engine", "device", "precision", "rotate_method", "analysis",
                      "boot_algo", "x_storage", "shard")

    def _take_kwargs(self, kwargs):
        self.pls_alg = kwargs["pls_alg"]
        self._user_defined_attrs = set()
        self._engine_kwargs = {}
        for k, v in kwargs.items():
            if k in self._ENGINE_KWARGS:
                self._engine_kwargs[k] = v
                continue
            setattr(self, k, v)
            self._user_defined_attrs.add(k)
        # storage and multi-process layout of X: the options, else those of a given engine (before any GPU work; the
        # bootstrap formulation is resolved with the resampling test, which knows the bootstrap count)
        ek = self._engine_kwargs
        _, _, ek["x_storage"], ek["shard"] = bootstrap_permutation.resolve_options(
            self.pls_alg, ek.get("engine"), precision=ek.get("precision", "fp64"), boot_algo=None,
            x_storage=ek.get("x_storage"), shard=ek.get("shard"))

    def _new_engine(self, device=None, exact=False):
        """An Engine holding X (the copy prepared for the device, else self.X) as the options ask; `exact`: whatever the
        precision option.  No `shard` keyword for the default layout: the same construction as without the option."""
        from .engine import Engine
        ek = self._engine_kwargs
        kw = {} if ek["shard"] == "resamples" else {"shard": ek["shard"]}
        if not exact:
            kw["precision"] = ek.get("precision", "fp64")
        src = getattr(self, "_x_tensor", None)
        return Engine(self.X if src is None else src, device=ek.get("device") if device is None else device,
                      x_storage=ek["x_storage"], **kw)

    @staticmethod
    def _get_groups_info(groups_tuple):
        if groups_tuple is None:
            return ((), 0)
        return (groups_tuple, len(groups_tuple))

    @staticmethod
    def _get_cond_order(X_shape, groups_tuple, num_conditions):
        if sum(groups_tuple) * num_conditions != X_shape[0]:
            raise exceptions.InputMatrixDimensionMismatchError(
                "Derived condition ordering not compatible with input matrix"
                "X's row count. Please specify a custom cond_order field.")
        return np.array([np.array([i] * num_conditions) for i in groups_tuple])

    def _set_design(self, X, Y, groups_sizes, num_conditions, cond_order, need_y):
        if need_y and Y is None:
            raise exceptions.MissingParameterError("Please provide a Y/behavioural matrix.")
        if not need_y and Y is not None:
            raise ValueError(f"Do not provide a Y/behavioural matrix for {self._pls_types[self.pls_alg]}.")
        if len(X.shape) != 2 or (need_y and len(Y.shape) != 2):
            raise exceptions.ImproperShapeError(
                "Input matrices must be 2-dimensional." if need_y else "Input matrix must be 2-dimensional.")
        if hasattr(X, "is_pinned") and hasattr(X, "numpy") and not X.is_cuda:
            # a host tensor from plspy_b200.io.assemble_pinned: the engine uploads the (pinned) tensor itself, the
            # host-side code works on its numpy view (float32 storage: a widened copy, meant for analysis="device")
            if self._engine_kwargs["x_storage"] == "fp32" and X.element_size() != 4:
                X = X.float()                                     # rounded once
            if self._engine_kwargs.get("engine") is None:
                self._x_tensor = X
            X = X.numpy() if X.dtype.is_floating_point and X.element_size() == 8 else X.numpy().astype(np.float64)
        elif self._engine_kwargs["x_storage"] == "fp32":
            # x_storage="fp32": the analysis is that of X.astype(float32).  The engine uploads the float32 matrix (a
            # float32 input as it is); the host-side steps work on its values widened to float64, as the kernels do
            x32 = np.ascontiguousarray(X, dtype=np.float32)
            if self._engine_kwargs.get("engine") is None:
                self._x_tensor = x32
            X = x32.astype(np.float64)
        self.X = X
        if need_y:
            self.Y = Y
        self.groups_sizes, self.num_groups = self._get_groups_info(groups_sizes)
        self.num_conditions = num_conditions
        if cond_order is None:
            self.cond_order = self._get_cond_order(self.X.shape, self.groups_sizes, self.num_conditions)
        else:
            calc_len = sum(groups_sizes) * num_conditions
            if calc_len != self.X.shape[0] or (need_y and calc_len != self.Y.shape[0]):
                raise exceptions.InputMatrixDimensionMismatchError(
                    "Dimension of condition orders does not match dimension of input matrix X and/or Y. "
                    "Please make sure that the sum of the conditions in all groups adds up to the number "
                    "of rows in the input matrices.")
            self.cond_order = cond_order

    def _set_mctype(self, num_conditions, mctype):
        if num_conditions == 1 and mctype != 1:
            print("Because you are running single condition Task PLS, input Mean-Centering Type has to set to 1")
            self.mctype = 1
        else:
            self.mctype = mctype

    def _check_behaviour(self, Y, cond_order):
        if (class_functions._get_group_means(Y, cond_order, return_std=True) == 0).any():
            raise Exception("Please check your behaviour data, and make sure that none of the columns are all "
                            "the same for each group.")

    def _set_bscan(self):
        if "bscan" not in self._user_defined_attrs:
            self.bscan = [i for i in range(self.num_conditions)]
        else:
            if self.bscan != sorted(self.bscan):
                print("provided bscan not in ascending order - conditions in bscan will be correctly reordered")
            if any(b < 0 or b > self.num_conditions - 1 for b in self.bscan):
                print(f"bscan should be a subset of: 1 to {self.num_conditions}")
        mask = []
        for row in self.cond_order:
            for ci, n in enumerate(row):
                mask.append(np.full(n, ci in self.bscan, dtype=bool))
        mask = np.concatenate(mask)
        self.Xbscan = self.X[mask]
        self.Ybscan = self.Y[mask]

    def _prefetch(self, upload):
        """Single-process runs: while this thread does the one-off original analysis, a worker thread (i) uploads X
        (`upload`: host analysis on a host matrix; the pageable copy and the LAPACK SVD both release the GIL) and
        (ii) draws the resampling index matrices in the reference's order (permutations, then bootstraps:
        bootstrap_permutation.py:323-355, 537-572) with the native generator, which releases the GIL too.  Nothing else
        touches numpy's global stream before `_resample` collects the result, so the draws and the stream position are
        the reference's.  Multi-process runs keep everything on the calling thread (the draw sites hold collectives)."""
        from . import dist, resample
        ek = self._engine_kwargs
        if dist.world()[1] > 1 or (self.num_perm <= 0 and self.num_boot <= 0) or os.environ.get("PLSB200_PREFETCH", "1") == "0":
            return
        want_idx = (ek.get("perm_indices") is None and ek.get("boot_indices") is None and resample.USE_NATIVE_RNG
                    and ek.get("rotate_method", 2) == 2)
        want_eng = upload and ek.get("engine") is None
        if not (want_idx or want_eng):
            return
        import concurrent.futures
        import torch
        device = ek.get("device")
        if device is None and torch.cuda.is_available():
            device = torch.device("cuda", torch.cuda.current_device())     # (the current device is per thread)
        Y = getattr(self, "Y", None) if self.pls_alg in ("rb", "csb", "mb", "cmb") else None
        multi = self.pls_alg in ("mb", "cmb")
        bscan, Ybscan = (self.bscan, self.Ybscan) if multi else (None, None)

        def work():
            out = {}
            if want_eng:
                out["engine"] = self._new_engine(device)
            if want_idx:
                if self.num_perm > 0:
                    out["perm_indices"] = resample.permutation_indices(self.pls_alg, self.num_perm, self.cond_order, Y=Y,
                                                                       bscan=bscan, Ybscan=Ybscan)
                if self.num_boot > 0:
                    out["boot_indices"] = resample.bootstrap_indices(self.pls_alg, self.num_boot, self.cond_order, Y=Y,
                                                                     bscan=bscan, Ybscan=Ybscan)
            return out
        pool = concurrent.futures.ThreadPoolExecutor(1)
        self._bg = pool.submit(work)
        pool.shutdown(wait=False)

    def _collect_prefetch(self):
        bg = self.__dict__.pop("_bg", None)
        if bg is not None:
            for k, v in bg.result().items():          # (re-raises what the worker raised, e.g. invalid behaviour data)
                if self._engine_kwargs.get(k) is None:
                    self._engine_kwargs[k] = v

    def _device_analysis(self):
        """True when `analysis="device"` was requested: the one-off analysis then runs through the Gram matrix on the
        GPU (device_analysis.py) and `self._engine_kwargs["engine"]` holds the engine with X.  Also the point where
        every constructor starts the background upload / index drawing (`_prefetch`)."""
        mode = self._engine_kwargs.get("analysis", "host")
        if mode not in ("host", "device"):
            raise ValueError('analysis must be "host" or "device"')
        self._prefetch(upload=(mode == "host"))
        if mode == "host":
            return False
        if self._engine_kwargs.get("engine") is None:
            self._engine_kwargs["engine"] = self._new_engine()
        return True

    def _resample(self, Y, mctype, preprocess, **kw):
        self._collect_prefetch()
        V = getattr(self, "_V_dev", None)
        xt = getattr(self, "_x_tensor", None)
        if xt is not None and self._engine_kwargs.get("engine") is None and (self.num_perm > 0 or self.num_boot > 0):
            self._engine_kwargs["engine"] = self._new_engine()
        self.resample_tests = bootstrap_permutation.ResampleTest._create(
            self.pls_alg, self.X, Y, self.U, self.s, self.V if V is None else V, self.cond_order, mctype, preprocess=preprocess,
            nperm=self.num_perm, nboot=self.num_boot, CI=self.CI,
            perm_indices=self._engine_kwargs.get("perm_indices"),
            boot_indices=self._engine_kwargs.get("boot_indices"),
            engine=self._engine_kwargs.get("engine"), precision=self._engine_kwargs.get("precision", "fp64"),
            rotate_method=self._engine_kwargs.get("rotate_method", 2), device=self._engine_kwargs.get("device"),
            boot_algo=self._engine_kwargs.get("boot_algo", "auto"), x_storage=self._engine_kwargs["x_storage"],
            shard=self._engine_kwargs["shard"], **kw)

    def _split_half(self, Y, mctype, contrasts, **kw):
        """pls_classes.py:285-318 (identical block in every class)."""
        if "num_split" in self._user_defined_attrs:
            self.num_split = int(self.num_split)
            if self.num_split > 0:
                max_lv = min(self.s.shape)
                if self.lv > max_lv:
                    print(f"Warning: Requested lv={self.lv} exceeds maximum possible LVs ({max_lv}). "
                          f"Using lv={max_lv} instead.")
                    self.lv = max_lv
                eng = getattr(self.resample_tests, "_engine", None) or self._engine_kwargs.get("engine")
                if eng is None and (self._engine_kwargs["x_storage"] == "fp32"
                                    or self._engine_kwargs["shard"] == "voxels"):
                    # no resampling engine: the split-half functions would each upload the (widened) host copy as
                    # float64 and whole; one engine holding X as asked (exact mode, as theirs) serves both instead
                    eng = self._new_engine(exact=True)
                self.pls_repro_tt = split_half_resampling.split_half_test_train(
                    self.pls_alg, self.X, Y, self.cond_order, num_split=self.num_split, mctype=mctype,
                    contrasts=contrasts, engine=eng, **kw)
                self.pls_repro_sh = split_half_resampling.split_half(
                    self.pls_alg, self.X, Y, self.cond_order, num_split=self.num_split, mctype=mctype,
                    contrasts=contrasts, lv=self.lv, CI=self.CI, engine=eng, **kw)

    def _finish(self):
        self.U, self.V = self.V, self.U      # pls_classes.py:323

    def __repr__(self):
        stg = f"\nAlgorithm: {self._pls_types[self.pls_alg]}\n\n"
        for k, v in self.__dict__.items():
            if k[0] != "_":
                stg += f"\n{k}:\n\t" + str(v).replace("\n", "\n\t")
        return stg

    __str__ = __repr__


@PLSBase._register_subclass("mct")
class _MeanCentreTaskPLS(PLSBase):
    def __init__(self, X, groups_sizes, num_conditions, Y=None, cond_order=None, num_perm=1000, num_boot=1000,
                 mctype=0, CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        if len(X.shape) != 2:
            raise exceptions.ImproperShapeError("Input matrix must be 2-dimensional.")
        if "contrasts" in kwargs:
            raise ValueError(f"Do not provide a contrast matrix for {self._pls_types[self.pls_alg]}.")
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=False)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        self._set_mctype(num_conditions, mctype)
        if self._device_analysis():
            a = device_analysis.task(self._engine_kwargs["engine"], self.cond_order, self.mctype)
            self.X_means, self.X_mc, self.U, self.s, self.V = a["X_means"], a["X_mc"], a["U"], a["s"], a["V"]
            self.X_latent, Tvsc_orig, self._V_dev = a["X_latent"], a["Tvsc_orig"], a["V_dev"]
        else:
            self.X_means, self.X_mc = class_functions._mean_centre(self.X, self.cond_order, mctype=self.mctype)
            self.U, self.s, self.V = class_functions._run_pls(self.X_mc)
            self.X_latent = class_functions._compute_X_latents(self.X, self.V)
            Tvsc_orig = class_functions._get_group_condition_means(self.X_latent, self.cond_order)
        self._resample(None, self.mctype, class_functions._mean_centre, Tvsc_orig=Tvsc_orig)
        self._split_half(None, self.mctype, None)
        self._finish()


@PLSBase._register_subclass("rb")
class _RegularBehaviourPLS(PLSBase):
    def __init__(self, X, groups_sizes, num_conditions, Y=None, cond_order=None, num_perm=0, num_boot=0,
                 CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        if Y is None:
            raise exceptions.MissingParameterError("Please provide a Y/behavioural matrix.")
        if "contrasts" in kwargs:
            raise ValueError(f"Do not provide a contrast matrix for {self._pls_types[self.pls_alg]}.")
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=True)
        self._check_behaviour(self.Y, self.cond_order)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        if self._device_analysis():
            a = device_analysis.behaviour(self._engine_kwargs["engine"], self.Y, self.cond_order)
            self.R, self.U, self.s, self.V, self.X_latent, self._V_dev = (a["R"], a["U"], a["s"], a["V"], a["X_latent"],
                                                                          a["V_dev"])
        else:
            self.R = class_functions._compute_R(self.X, self.Y, self.cond_order)
            self.U, self.s, self.V = class_functions._run_pls(self.R)
            self.X_latent = class_functions._compute_X_latents(self.X, self.V)
        self.Y_latent = class_functions._compute_Y_latents(self.Y, self.U, self.cond_order)
        self.lvcorrs = class_functions._compute_R(self.X_latent, self.Y, self.cond_order)
        self._resample(self.Y, None, class_functions._compute_R, lvcorrs_orig=self.lvcorrs)
        self._split_half(self.Y, None, None)
        self._finish()


@PLSBase._register_subclass("cst")
class _ContrastTaskPLS(PLSBase):
    def __init__(self, X, groups_sizes, num_conditions, Y=None, cond_order=None, num_perm=1000, num_boot=1000,
                 mctype=0, contrasts=None, CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=False)
        if contrasts is None:
            raise exceptions.MissingParameterError("Please provide a contrast matrix.")
        self.contrasts = class_functions._normalize(contrasts)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        self._set_mctype(num_conditions, mctype)
        if self._device_analysis():
            a = device_analysis.contrast_task(self._engine_kwargs["engine"], self.cond_order, self.contrasts)
            self.R, self.U, self.s, self.V, self.lvintercorrs = a["R"], a["U"], a["s"], a["V"], a["lvintercorrs"]
            self.X_latent, Tvsc_orig, self._V_dev = a["X_latent"], a["Tvsc_orig"], a["V_dev"]
        else:
            self.R = class_functions._get_group_condition_means(self.X, self.cond_order)
            self.U, self.s, self.V = class_functions._run_pls_contrast(self.R, self.contrasts)
            self.lvintercorrs = self.V.T @ self.V
            self.X_latent = class_functions._compute_X_latents(self.X, class_functions._normalize(self.V))
            Tvsc_orig = class_functions._get_group_condition_means(self.X_latent, self.cond_order)
        self._resample(None, self.mctype, class_functions._mean_centre, contrast=self.contrasts,
                       Tvsc_orig=Tvsc_orig)
        self._split_half(None, self.mctype, self.contrasts)
        self._finish()


@PLSBase._register_subclass("csb")
class _ContrastBehaviourPLS(PLSBase):
    def __init__(self, X, groups_sizes, num_conditions, Y=None, cond_order=None, num_perm=1000, num_boot=1000,
                 contrasts=None, CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=True)
        if contrasts is None:
            raise exceptions.MissingParameterError("Please provide a contrast matrix.")
        self.contrasts = class_functions._normalize(contrasts)
        self._check_behaviour(self.Y, self.cond_order)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        if self._device_analysis():
            a = device_analysis.contrast_behaviour(self._engine_kwargs["engine"], self.Y, self.cond_order, self.contrasts)
            self.R, self.U, self.s, self.V, self.lvintercorrs = a["R"], a["U"], a["s"], a["V"], a["lvintercorrs"]
            self.X_latent, self._V_dev = a["X_latent"], a["V_dev"]
        else:
            self.R = class_functions._compute_R(self.X, self.Y, self.cond_order)
            self.U, self.s, self.V = class_functions._run_pls_contrast(self.R, self.contrasts)
            self.lvintercorrs = self.V.T @ self.V
            self.X_latent = class_functions._compute_X_latents(self.X, self.V)
        self.Y_latent = class_functions._compute_Y_latents(self.Y, self.U, self.cond_order)
        self._resample(self.Y, None, class_functions._compute_R, contrast=self.contrasts,
                       lvcorrs_orig=self.lvintercorrs)
        self._split_half(self.Y, None, self.contrasts)
        self._finish()


class _MultiblockCommon(PLSBase):
    def _multiblock_analysis(self, num_conditions, contrasts):
        self._set_bscan()
        self._check_behaviour(self.Ybscan, self.cond_order[:, self.bscan])
        if contrasts is not None:
            # keep the contrast rows of the task block and of the bscan behaviour rows (:1788-1803)
            Ti = np.ones(self.num_conditions)
            Bi = np.zeros((self.Y.shape[1], self.num_conditions))
            Bi[:, self.bscan] = 1
            keep = np.tile(np.concatenate([Ti, Bi.reshape(-1, order="F")]), self.num_groups).astype(bool)
            self.contrasts = class_functions._normalize(contrasts[keep, :])
        self._create_multiblock = class_functions._create_multiblock
        self._compute_corr = class_functions._compute_corr
        if self._device_analysis():
            a = device_analysis.multiblock(self._engine_kwargs["engine"], self.pls_alg, self.cond_order, self.mctype,
                                           self.bscan, self.Ybscan, self.contrasts if contrasts is not None else None)
            self.multiblock, self.U, self.s, self.V, self._V_dev = a["multiblock"], a["U"], a["s"], a["V"], a["V_dev"]
            nrm = np.linalg.norm(self.V, axis=0)
            T_X_latent = a["XV"] * np.where(nrm > 0, 1.0 / np.where(nrm > 0, nrm, 1.0), 0.0)[None, :]
            B_X_latent = a["XV"][a["rows_b"]]                 # Xbscan = the bscan rows of X
        else:
            self.multiblock = class_functions._create_multiblock(
                self.X, self.cond_order, self.pls_alg, self.bscan, self.mctype, Xbscan=self.Xbscan, Ybscan=self.Ybscan)
            if contrasts is not None:
                self.U, self.s, self.V = class_functions._run_pls_contrast(self.multiblock, self.contrasts)
            else:
                self.U, self.s, self.V = class_functions._run_pls(self.multiblock)
            T_X_latent = class_functions._compute_X_latents(self.X, class_functions._normalize(self.V))
            B_X_latent = class_functions._compute_X_latents(self.Xbscan, self.V)
        self.X_latent = np.vstack((np.array(T_X_latent), np.array(B_X_latent)))
        self.usc, self.Tusc, self.Busc = self.X_latent, T_X_latent, B_X_latent
        Tu, Bu = class_functions._get_Tu_Bu(self.U, num_conditions, self.Y.shape[1], self.cond_order, self.bscan)
        self.Tvsc = class_functions._get_Tusc(Tu, num_conditions, self.cond_order)
        self.Bvsc = class_functions._get_Busc(Bu, num_conditions, self.Ybscan, self.cond_order, self.bscan)
        self.Tv, self.Bv = Tu, Bu
        self.Y_latent = np.vstack([self.Tvsc, self.Bvsc])
        self.vsc = self.Y_latent
        self.lvcorrs = class_functions._compute_corr(B_X_latent, self.Ybscan, self.cond_order[:, self.bscan])
        return class_functions._get_group_condition_means(T_X_latent, self.cond_order)


@PLSBase._register_subclass("mb")
class _MultiblockPLS(_MultiblockCommon):
    def __init__(self, X, groups_sizes, num_conditions, mctype=0, Y=None, cond_order=None, num_perm=1000,
                 num_boot=1000, CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        if Y is None:
            raise exceptions.MissingParameterError("Please provide a Y/behavioural matrix.")
        if "contrasts" in kwargs:
            raise ValueError(f"Do not provide a contrast matrix for {self._pls_types[self.pls_alg]}.")
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=True)
        self._set_mctype(num_conditions, mctype)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        Tvsc_orig = self._multiblock_analysis(num_conditions, None)
        self._resample(self.Y, self.mctype, class_functions._create_multiblock, bscan=self.bscan,
                       Xbscan=self.Xbscan, Ybscan=self.Ybscan, lvcorrs_orig=self.lvcorrs, Tvsc_orig=Tvsc_orig)
        self._split_half(self.Y, self.mctype, None, bscan=self.bscan, Xbscan=self.Xbscan, Ybscan=self.Ybscan)
        self._finish()


@PLSBase._register_subclass("cmb")
class _ContrastMultiblockPLS(_MultiblockCommon):
    def __init__(self, X, groups_sizes, num_conditions, mctype=0, Y=None, cond_order=None, num_perm=1000,
                 num_boot=1000, contrasts=None, CI=0.95, **kwargs):
        self._take_kwargs(kwargs)
        if Y is None:
            raise exceptions.MissingParameterError("Please provide a Y/behavioural matrix.")
        self._set_design(X, Y, groups_sizes, num_conditions, cond_order, need_y=True)
        self._set_mctype(num_conditions, mctype)
        self.num_perm, self.num_boot, self.CI = num_perm, num_boot, CI
        if contrasts is None:
            raise exceptions.MissingParameterError("Please provide a contrast matrix.")
        Tvsc_orig = self._multiblock_analysis(num_conditions, contrasts)
        self._resample(self.Y, self.mctype, class_functions._create_multiblock, contrast=self.contrasts,
                       bscan=self.bscan, Xbscan=self.Xbscan, Ybscan=self.Ybscan, lvcorrs_orig=self.lvcorrs,
                       Tvsc_orig=Tvsc_orig)
        self._split_half(self.Y, self.mctype, self.contrasts, bscan=self.bscan, Xbscan=self.Xbscan,
                         Ybscan=self.Ybscan)
        self._finish()
