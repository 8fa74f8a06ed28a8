"""Plug the B200 resampling engine into an installed, UNMODIFIED plspy.

    import plspy, plspy_b200
    plspy_b200.install(plspy)            # or plspy_b200.install(): imports plspy itself
    res = plspy.PLS(X, groups, C, num_perm=5000, num_boot=5000, pls_method="mct")   # the reference's own classes,
                                                                                    # resampling on the GPU
    plspy_b200.uninstall()

The reference offers exactly two seams on this path and `install` uses both:

* `ResampleTest._register_subclass(key)` (plspy/core/bootstrap_permutation.py:44-50): re-registering a key replaces
  the class `ResampleTest._create` instantiates (:53-63), which is what the six method constructors call
  (plspy/core/pls_classes.py:268-282, 590-604, 868-884, 1145-1160, 1491-1509, 1858-1877).  `_create` publishes the
  method key by assigning `ResampleTest.pls_alg` on ITS OWN base class (:62); a class from another package never
  sees that attribute, so the six registered classes each pin their key as a class attribute.
* `split_half_resampling.split_half_test_train / split_half` are looked up on the module at call time
  (pls_classes.py:297, 306, 619, 628, 899, 908, 1175, 1184, 1524, 1536, 1892, 1904), so rebinding the two module
  attributes is enough.

X is uploaded once per analysis: the permutation / bootstrap object and the two split-half calls of one `PLS(...)`
share the `Engine` that holds it (keyed by the identity of the array the reference passes to all three).
"""
import weakref

from . import bootstrap_permutation as _bp
from . import split_half_resampling as _sh
from .engine import Engine

METHODS = ("mct", "rb", "cst", "csb", "mb", "cmb")

_state = None          # what install() replaced, for uninstall()
_options = {"precision": "fp64", "boot_algo": "auto", "x_storage": "fp64", "shard": "resamples"}
_shared = {"ref": None, "engine": None}


def _drop_engine(_ref=None):
    _shared["ref"] = None
    _shared["engine"] = None


def shared_engine(X):
    """The Engine holding `X` on the device; one entry, replaced when another matrix arrives and dropped when the
    matrix is garbage collected."""
    ref = _shared["ref"]
    if ref is not None and ref() is X and _shared["engine"] is not None:
        return _shared["engine"]
    eng = Engine(X, precision=_options["precision"], x_storage=_options["x_storage"], shard=_options["shard"])
    try:
        _shared["ref"] = weakref.ref(X, _drop_engine)
    except TypeError:           # not weak-referenceable (a torch tensor is; a list is not): do not cache
        return eng
    _shared["engine"] = eng
    return eng


class _InstalledResampleTest(_bp._ResampleTestPLS):
    """`_ResampleTestPLS` behind a foreign registry: same positional signature as the reference's class
    (bootstrap_permutation.py:139-159); the engine options come from `install(...)`."""

    def __init__(self, X, Y, U, s, V, cond_order, mctype, *args, **kwargs):
        nperm = kwargs.get("nperm", 1000)
        nboot = kwargs.get("nboot", 1000)
        for name, value in _options.items():
            kwargs.setdefault(name, value)
        _bp.resolve_options(self.pls_alg, kwargs.get("engine"), X, nboot, cond_order,       # before the engine uploads X
                            **{name: kwargs[name] for name in _options})
        if "engine" not in kwargs and (nperm > 0 or nboot > 0):
            kwargs["engine"] = shared_engine(X)
        super().__init__(X, Y, U, s, V, cond_order, mctype, *args, **kwargs)


def _pinned(key):
    return type(f"_ResampleTestPLS_{key}", (_InstalledResampleTest,), {"pls_alg": key, "__module__": __name__})


PINNED = {key: _pinned(key) for key in METHODS}


def _split_half_test_train(pls_alg, matrix, Y, cond_order, num_split, mctype=None, contrasts=None, bscan=None,
                           Xbscan=None, Ybscan=None):
    """split_half_resampling.py:23 -- the reference's signature; X is reused from the resampling step."""
    _bp.check_shard(_options["shard"], pls_alg)
    return _sh.split_half_test_train(pls_alg, matrix, Y, cond_order, num_split, mctype=mctype, contrasts=contrasts,
                                     bscan=bscan, Xbscan=Xbscan, Ybscan=Ybscan, engine=shared_engine(matrix))


def _split_half(pls_alg, matrix, Y, cond_order, num_split, mctype=None, contrasts=None, bscan=None, Xbscan=None,
                Ybscan=None, lv=1, CI=0.95):
    """split_half_resampling.py:404."""
    _bp.check_shard(_options["shard"], pls_alg)
    return _sh.split_half(pls_alg, matrix, Y, cond_order, num_split, mctype=mctype, contrasts=contrasts, bscan=bscan,
                          Xbscan=Xbscan, Ybscan=Ybscan, lv=lv, CI=CI, engine=shared_engine(matrix))


def install(plspy_module=None, precision="fp64", boot_algo="auto", x_storage="fp64", shard="resamples"):
    """Route the permutation / bootstrap / split-half loops of `plspy_module` (default: `import plspy`) through the
    GPU engine.  Idempotent; returns the module.  `precision`: "fp64" (exact) or "tf32x3" (fast bootstrap GEMM).
    `boot_algo`: "auto" (default), "direct" or "collapsed" (mct / cst in the exact mode; beyond 320 rows every group
    needs the same number of subjects in each condition and more bootstraps than subjects minus groups, checked per
    resampling test before X is uploaded: see `bootstrap_permutation.check_boot_algo`);
    a per-call option, applied to every resampling test while installed.  `x_storage`: "fp64" or "fp32" (mct / cst:
    the engine holds X as float32, see `bootstrap_permutation.check_x_storage`; the reference's own host analysis
    still sees X as passed, so the results are bit-identical to "fp64" when X holds float32 values).  Behaviour and
    multiblock analyses raise NotImplementedError with "fp32".  `shard`: "resamples" or "voxels" (mct / cst in a
    multi-process run: every rank holds only its columns of X, see `bootstrap_permutation.check_shard`); behaviour and
    multiblock analyses raise NotImplementedError with "voxels"."""
    global _state
    # the values themselves; what a method or design does not support is refused by each resampling test ("mct"
    # supports every value)
    _, _, x_storage, shard = _bp.resolve_options("mct", precision=precision, boot_algo=boot_algo, x_storage=x_storage,
                                                 shard=shard)
    if plspy_module is None:
        import plspy as plspy_module
    ref_bp = plspy_module.core.bootstrap_permutation
    ref_sh = plspy_module.core.split_half_resampling
    if _state is not None and _state["module"] is not plspy_module:
        uninstall()
    _options["precision"] = precision
    _options["boot_algo"] = boot_algo
    if _options["x_storage"] != x_storage or _options["shard"] != shard:
        _drop_engine()                                     # a cached engine holds X in the other storage or layout
    _options["x_storage"] = x_storage
    _options["shard"] = shard
    if _state is None:
        _state = {
            "module": plspy_module,
            "subclasses": dict(ref_bp.ResampleTest._subclasses),
            "tt": ref_sh.split_half_test_train,
            "sh": ref_sh.split_half,
        }
    for key in METHODS:
        ref_bp.ResampleTest._register_subclass(key)(PINNED[key])
        ref_bp.ResampleTest.register(PINNED[key])          # isinstance(result.resample_tests, plspy's ResampleTest)
    ref_sh.split_half_test_train = _split_half_test_train
    ref_sh.split_half = _split_half
    return plspy_module


def uninstall():
    """Put the reference's own implementations back and release the device copy of X."""
    global _state
    if _state is None:
        return
    mod = _state["module"]
    ref_bp = mod.core.bootstrap_permutation
    ref_sh = mod.core.split_half_resampling
    ref_bp.ResampleTest._subclasses.clear()
    ref_bp.ResampleTest._subclasses.update(_state["subclasses"])
    ref_sh.split_half_test_train = _state["tt"]
    ref_sh.split_half = _state["sh"]
    _state = None
    _drop_engine()


def installed():
    return _state is not None
