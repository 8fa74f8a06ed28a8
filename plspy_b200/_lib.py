"""ctypes binding of libplsb200.so (the C ABI declared in include/plsb200.h).

The library is the product: there is no CPU fallback.  If the shared object is missing this module
raises at import time with the build command, and every call raises `PlsB200Error` with the library's
own message when a kernel or an argument check fails.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libplsb200.so")

c_double_p = ctypes.c_void_p   # device pointers are passed as integers
c_int32_p = ctypes.c_void_p
c_int64 = ctypes.c_int64
c_int = ctypes.c_int
c_size_t = ctypes.c_size_t
c_void_p = ctypes.c_void_p
c_double = ctypes.c_double


class PlsB200Error(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -m plspy_b200.build` "
        "(needs nvcc; cross-compiles for sm_100a without a GPU). plspy_b200 has no CPU fallback."
    )

lib = ctypes.CDLL(LIB_PATH)

# name -> (restype, argtypes); must list every symbol of include/plsb200.h (tests/test_abi.py checks)
SIGNATURES = {
    "plsb200_abi_version": (c_int, []),
    "plsb200_last_error": (ctypes.c_char_p, []),
    "plsb200_launch_count": (c_int64, []),
    "plsb200_copy2d_h2d": (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, c_size_t, c_size_t, c_void_p]),
    "plsb200_widen_f32_f64": (c_int, [c_void_p, c_double_p, c_int64, c_void_p]),
    "plsb200_gram_f64_workspace": (c_size_t, [c_int, c_int64]),
    "plsb200_gram_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_gram_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_gram_stacked_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_int64, c_double_p,
                                         c_void_p, c_size_t, c_void_p]),
    "plsb200_gram_stack_fuses": (c_int, [c_int, c_int]),
    "plsb200_gram_tf32_image_bytes": (c_size_t, [c_int, c_int64]),
    "plsb200_gram_tf32_split": (c_int, [c_double_p, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "plsb200_gram_tf32_split_x32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "plsb200_gram_tf32_workspace": (c_size_t, [c_int, c_int64]),
    "plsb200_gram_tf32": (c_int, [c_void_p, c_int, c_int64, c_double_p, c_int, c_void_p, c_size_t, c_void_p]),
    "plsb200_xv_f64_workspace": (c_size_t, [c_int, c_int64, c_int]),
    "plsb200_xv_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_double_p, c_void_p,
                               c_size_t, c_void_p]),
    "plsb200_xv_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_double_p, c_void_p,
                                   c_size_t, c_void_p]),
    "plsb200_nspace_f64": (c_int, [c_double_p, c_int, c_double_p, c_int, c_int32_p, c_int, c_double_p, c_int,
                                   c_double_p, c_double_p, c_void_p]),
    "plsb200_nspace_dmma_f64_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "plsb200_nspace_dmma_f64": (c_int, [c_double_p, c_int, c_double_p, c_int, c_double_p, c_int, c_int, c_double_p,
                                        c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_nspace_gram_f64": (c_int, [c_double_p, c_int, c_double_p, c_int, c_int32_p, c_int, c_double_p, c_double_p,
                                        c_void_p]),
    "plsb200_perm_count_f64": (c_int, [c_double_p, c_int, c_int, c_double_p, c_double_p, c_double, c_double_p,
                                       c_void_p, c_double_p, c_void_p]),
    "plsb200_uhat_f64": (c_int, [c_double_p, c_int64, c_int, c_int, c_double_p, c_int, c_int32_p, c_int, c_double_p,
                                 c_void_p]),
    "plsb200_scatter_coef_f64": (c_int, [c_double_p, c_int, c_int, c_int32_p, c_int, c_double_p, c_void_p]),
    "plsb200_coef_project_f64": (c_int, [c_double_p, c_int, c_int, c_double_p, c_double_p, c_int, c_int, c_double_p,
                                         c_void_p]),
    "plsb200_boot_coef_bytes": (c_size_t, [c_int, c_int, c_int]),
    "plsb200_boot_coef_pack_f64": (c_int, [c_double_p, c_int, c_int, c_int32_p, c_int, c_double_p, c_void_p]),
    "plsb200_boot_moments_f64_workspace": (c_size_t, [c_int, c_int64, c_int, c_int]),
    "plsb200_boot_moments_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int,
                                         c_double_p, c_double_p, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_boot_moments_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int,
                                             c_double_p, c_double_p, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_boot_factor_coef_bytes": (c_size_t, [c_int, c_int, c_int]),
    "plsb200_boot_factor_pack_f64": (c_int, [c_double_p, c_int, c_int, c_double_p, c_int, c_int32_p, c_double_p,
                                             c_void_p]),
    "plsb200_boot_quad_coef_bytes": (c_size_t, [c_int, c_int]),
    "plsb200_boot_quad_coef_pack_f64": (c_int, [c_double_p, c_int, c_int, c_double_p, c_void_p]),
    "plsb200_boot_quad_f64_workspace": (c_size_t, [c_int, c_int64, c_int]),
    "plsb200_boot_quad_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_double_p, c_void_p,
                                      c_size_t, c_void_p]),
    "plsb200_boot_quad_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_double_p, c_void_p,
                                          c_size_t, c_void_p]),
    "plsb200_boot_counts_f64": (c_int, [c_int32_p, c_int, c_int, c_int32_p, c_int, c_double_p, c_int64, c_int32_p,
                                        c_void_p]),
    "plsb200_boot_factor_f64_workspace": (c_size_t, [c_int, c_int]),
    "plsb200_boot_factor_f64": (c_int, [c_double_p, c_int, c_int64, c_int32_p, c_int, c_double_p, c_void_p, c_size_t,
                                        c_void_p]),
    "plsb200_tf32_ximage_bytes":(c_size_t, [c_int, c_int64]),
    "plsb200_tf32_split_x": (c_int, [c_double_p, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "plsb200_tf32_split_x32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "plsb200_boot_coef_bytes_tf32": (c_size_t, [c_int, c_int, c_int]),
    "plsb200_boot_coef_pack_tf32": (c_int, [c_double_p, c_int, c_int, c_int32_p, c_int, c_void_p, c_void_p]),
    "plsb200_boot_moments_tf32_workspace": (c_size_t, [c_int, c_int64, c_int, c_int]),
    "plsb200_boot_moments_tf32": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_int, c_double_p, c_double_p,
                                          c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_boot_finalize_f64": (c_int, [c_double_p, c_double_p, c_int64, c_int, c_int64, c_double_p,
                                          c_double_p, c_double_p, c_void_p]),
    "plsb200_colstd_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_void_p]),
    "plsb200_sym_eig_f64": (c_int, [c_double_p, c_int, c_int, c_double_p, c_double_p, c_void_p, c_void_p]),
    "plsb200_split_gram_f64": (c_int, [c_double_p, c_int, c_int32_p, c_int, c_int32_p, c_int, c_int, c_double_p,
                                       c_double_p, c_int, c_double_p, c_double_p, c_double_p, c_void_p]),
    "plsb200_split_svd_f64_workspace": (c_size_t, [c_int, c_int]),
    "plsb200_split_svd_f64": (c_int, [c_double_p, c_double_p, c_double_p, c_int, c_int, c_double_p, c_double_p,
                                      c_double_p, c_double_p, c_double_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_cell_standardize_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_int32_p, c_int, c_double_p,
                                             c_double_p, c_void_p]),
    "plsb200_nspace_coef_f64": (c_int, [c_double_p, c_int, c_double_p, c_int, c_int, c_double_p, c_int, c_double_p,
                                        c_double_p, c_void_p]),
    "plsb200_nspace_coef_gram_f64": (c_int, [c_double_p, c_int, c_double_p, c_int, c_int, c_double_p, c_double_p, c_void_p]),
    "plsb200_rb_coef_f64": (c_int, [c_double_p, c_int, c_int, c_int32_p, c_int, c_int32_p, c_int, c_double_p, c_int,
                                    c_int, c_double_p, c_double_p, c_double_p, c_void_p]),
    "plsb200_rb_boot_f64_workspace": (c_size_t, [c_int, c_int64, c_int, c_int]),
    "plsb200_rb_boot_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_double_p, c_double_p, c_int,
                                    c_int, c_int,
                                    c_int32_p, c_int, c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                    c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_rb_boot_vs_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_double_p, c_double_p,
                                       c_int, c_int, c_int,
                                       c_int32_p, c_int, c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                       c_double_p, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_rb_boot_dmma_f64_workspace": (c_size_t, [c_int, c_int64, c_int, c_int, c_void_p, c_int, c_int, c_int]),
    "plsb200_rb_boot_dmma_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_double_p, c_double_p,
                                         c_int, c_int, c_int,
                                         c_void_p, c_int, c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                         c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_rb_boot_dmma_vs_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_double_p,
                                            c_double_p, c_int, c_int, c_int,
                                            c_void_p, c_int, c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                            c_double_p, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_rb_salience_dmma_f64_workspace": (c_size_t, [c_int, c_int, c_int, c_void_p, c_int, c_int]),
    "plsb200_rb_salience_dmma_pack_f64": (c_int, [c_double_p, c_double_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                                  c_void_p, c_size_t, c_void_p]),
    "plsb200_rb_salience_dmma_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_int64, c_int64,
                                             c_int, c_int, c_void_p, c_int, c_int, c_double_p, c_void_p, c_size_t,
                                             c_void_p]),
    "plsb200_rb_salience_f64": (c_int, [c_double_p, c_int, c_int64, c_double_p, c_int, c_int64, c_int64, c_int64,
                                        c_double_p, c_double_p, c_int, c_int, c_int32_p, c_int, c_int, c_double_p,
                                        c_void_p]),
    "plsb200_rb_lvcorr_f64": (c_int, [c_double_p, c_double_p, c_double_p, c_int32_p, c_int, c_int, c_int, c_int,
                                      c_int32_p, c_int, c_double_p, c_void_p]),
    "plsb200_half_gram_f64_workspace": (c_size_t, [c_int64, c_int, c_int]),
    "plsb200_half_gram_f64": (c_int, [c_double_p, c_double_p, c_int64, c_int32_p, c_double_p, c_int32_p, c_int, c_int,
                                      c_int, c_int, c_int, c_int, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_half_gram_win_f64_workspace": (c_size_t, [c_int64, c_int, c_int]),
    "plsb200_half_gram_win_f64": (c_int, [c_double_p, c_double_p, c_int64, c_int32_p, c_double_p, c_int32_p, c_int, c_int,
                                          c_int, c_int, c_int, c_int, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_host_task_permutations": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                               c_void_p]),
    "plsb200_host_bootstrap_draws": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
                                             c_void_p, c_void_p]),
    "plsb200_host_row_permutations": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "plsb200_host_split_draws": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                         c_void_p]),
    "plsb200_percentile_f64_workspace": (c_size_t, [c_int]),
    "plsb200_percentile_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_int64, c_double, c_double, c_double_p,
                                       c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_percentile_bc_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_int64, c_double_p, c_double, c_double,
                                          c_double_p, c_double_p, c_double_p, c_void_p, c_size_t, c_void_p]),
    "plsb200_percentile_bca_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_int64, c_double_p, c_double_p,
                                           c_double, c_double, c_double_p, c_double_p, c_double_p, c_void_p, c_size_t,
                                           c_void_p]),
    "plsb200_jack_accel_f64": (c_int, [c_double_p, c_int64, c_int, c_int32_p, c_int, c_double_p, c_double_p,
                                       c_void_p]),
    "plsb200_salience_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int32_p, c_int,
                                     c_double_p, c_void_p]),
    "plsb200_salience_series_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int32_p, c_int,
                                     c_double_p, c_void_p]),
    "plsb200_salience_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int32_p, c_int,
                                         c_double_p, c_void_p]),
    "plsb200_salience_series_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int32_p,
                                                c_int, c_double_p, c_void_p]),
    "plsb200_salience_coef_series_f64": (c_int, [c_double_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int,
                                                 c_double_p, c_void_p]),
    "plsb200_salience_coef_series_x32_f64": (c_int, [c_void_p, c_int, c_int64, c_int64, c_double_p, c_int, c_int,
                                                     c_double_p, c_void_p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)
    _f.restype = _res
    _f.argtypes = _args

ABI_VERSION = 3
if lib.plsb200_abi_version() != ABI_VERSION:
    raise ImportError(f"{LIB_PATH}: ABI version {lib.plsb200_abi_version()} != {ABI_VERSION}; rebuild")


def check(rc, what):
    if rc != 0:
        msg = lib.plsb200_last_error()
        raise PlsB200Error(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def launch_count():
    return int(lib.plsb200_launch_count())
