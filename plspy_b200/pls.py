"""`PLS(...)` driver with the reference's signature and argument validation (plspy/core/pls.py:21-93)."""
import inspect

import numpy as np

from . import bootstrap_permutation, pls_classes

methods = {
    "mct": pls_classes._MeanCentreTaskPLS,
    "rb": pls_classes._RegularBehaviourPLS,
    "cst": pls_classes._ContrastTaskPLS,
    "csb": pls_classes._ContrastBehaviourPLS,
    "mb": pls_classes._MultiblockPLS,
    "cmb": pls_classes._ContrastMultiblockPLS,
}


def _boot_layout(pls_method, args, kwargs):
    """(num_boot, cond_order) of a PLS(...) call as the method class will see them -- its defaults included, the
    cond_order derived from groups_sizes and num_conditions when not given -- or None where they cannot be read (the
    class reports malformed arguments itself)."""
    try:
        bound = inspect.signature(methods[pls_method]).bind(*args, **kwargs)
    except (KeyError, TypeError):
        return None, None
    bound.apply_defaults()
    a = bound.arguments
    cond_order = a.get("cond_order")
    if cond_order is None:
        try:
            cond_order = np.array([[int(n)] * int(a["num_conditions"]) for n in a["groups_sizes"]])
        except (KeyError, TypeError, ValueError):
            cond_order = None
    return a.get("num_boot"), cond_order


def PLS(*args, **kwargs):
    """PLS(X, groups_sizes, num_conditions, Y=None, cond_order=None, num_perm=..., num_boot=..., mctype=...,
    contrasts=..., bscan=..., num_split=..., lv=..., CI=0.95, pls_method="mct")

    Drop-in for `plspy.PLS`: same arguments, same result attributes; the permutation, bootstrap and
    split-half loops run on a B200 through libplsb200.  Extra optional keywords: `perm_indices`,
    `boot_indices` (pre-generated resampling index matrices), `engine` (an `Engine` already holding X),
    `precision` ("fp64" = exact mode, default; "tf32x3" = fast mode for the bootstrap moment GEMM),
    `rotate_method` (2 = derived, the reference's behaviour and the default; 1 = Procrustes; 0 = per-permutation SVD,
    mct only -- see `_ResampleTestPLS._permutation_test`), `analysis` ("host" = LAPACK on the cross-block matrix as
    in the reference, default; "device" = through the Gram matrix on the GPU, sign of each latent
    variable fixed by convention -- see device_analysis.py), `boot_algo` ("auto" = "collapsed" for mct / cst
    with precision="fp64", at most 320 rows and num_boot > N, else "direct", default; "direct" = the bootstrap moments of
    the B x p x K salience GEMM; "collapsed" = mct / cst with precision="fp64": the same exact standard errors from
    the covariance of the subjects' draw counts (a GEMM over ns - G pseudo-resamples, ns subjects in G groups) or, for
    draws without that structure and at most 320 rows, from K covariance matrices of N x N; beyond 320 rows it needs
    every group to have the same number of subjects in each condition and num_boot > ns - G -- see
    bootstrap_permutation.check_boot_algo; `resample_tests.boot_algo` reports the one that ran), `x_storage` ("fp64" =
    X held as float64 on the device, default; "fp32" = mct / cst: X.astype(float32) held as float32 -- half the device
    memory -- with every result bit-identical to the "fp64" run on the widened float32 matrix; the host-side steps see
    the same widened values -- see bootstrap_permutation.check_x_storage), `shard` ("resamples" = in a multi-process
    run every GPU holds the whole of X and takes a share of the resamples, default; "voxels" = mct / cst: every GPU
    holds only its share of the columns of X and runs every bootstrap on them, so an X larger than one GPU's memory
    can be analysed -- see bootstrap_permutation.check_shard).
    """
    pls_method = kwargs.pop("pls_method", "mct")
    kwargs["pls_alg"] = pls_method
    if "num_split" in kwargs:
        if kwargs["num_split"] < 0 or not isinstance(kwargs["num_split"], int):
            raise ValueError("Invalid number of splits provided. Value must be a positive integer.")
        if "CI" in kwargs:
            if kwargs["CI"] is None or kwargs["CI"] < 0 or kwargs["CI"] > 1:
                raise ValueError("CI should be within 0 and 1.")
        if "lv" in kwargs:
            if kwargs["lv"] <= 0 or not isinstance(kwargs["lv"], int):
                raise ValueError("lv must be a positive integer greater than 0.")
    if "num_boot" in kwargs:
        if kwargs["num_boot"] < 0 or not isinstance(kwargs["num_boot"], int):
            raise ValueError("Invalid number of bootstraps provided. Value must be a positive integer.")
    if "num_perm" in kwargs:
        if kwargs["num_perm"] < 0 or not isinstance(kwargs["num_perm"], int):
            raise ValueError("Invalid number of permutations provided. Value must be a positive integer.")
    # the engine options, before any GPU work (the engine's upload of X starts with the analysis)
    nboot, cond_order = _boot_layout(pls_method, args, kwargs)
    bootstrap_permutation.resolve_options(
        pls_method, kwargs.get("engine"), args[0] if args else kwargs.get("X"), nboot, cond_order,
        kwargs.get("precision", "fp64"), kwargs.get("boot_algo", "auto"), kwargs.get("x_storage"), kwargs.get("shard"))
    return pls_classes.PLSBase._create(pls_method, *args, **kwargs)
