"""Host-side parts of the voxel-chunk salience export (no GPU): the workspace query and argument checks of the new entry
points, and the method on every result class."""
import numpy as np


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    from plspy_b200 import _lib
    return _lib.lib


def test_workspace_query_covers_the_designs_of_the_dmma_kernel():
    lib = _lib()
    cells = np.arange(0, 121, 20, dtype=np.int32)                  # 6 cells of 20 rows (BASELINE cfg 2)
    n = lib.plsb200_rb_salience_dmma_f64_workspace(120, 24, 1000, cells.ctypes.data, 6, 0)
    # packed coefficients of every bootstrap: 32 k-steps x 3 column blocks x 32 lanes + 32 x 4 weights, plus the MD
    # weight fragments of 125 batches of 8
    assert n >= 1000 * (32 * 3 * 32 + 32 * 4) * 8 + 125 * 32 * 32 * 8
    assert lib.plsb200_rb_salience_dmma_f64_workspace(120, 24, 2000, cells.ctypes.data, 6, 0) > n
    c17 = np.arange(0, 18, dtype=np.int32)                          # 17 cells: outside the DMMA kernel's buckets
    assert lib.plsb200_rb_salience_dmma_f64_workspace(17, 4, 10, c17.ctypes.data, 17, 0) == 0
    assert lib.plsb200_rb_boot_dmma_f64_workspace(17, 100, 4, 10, c17.ctypes.data, 17, 0, 1) == 0
    assert lib.plsb200_rb_salience_dmma_f64_workspace(120, 24, 10, None, 6, 0) == 0


def test_argument_errors_are_reported_without_a_gpu():
    lib = _lib()
    cells = np.arange(0, 121, 20, dtype=np.int32)
    rc = lib.plsb200_rb_salience_dmma_f64(None, 120, 100, None, 0, 0, 0, 10, 24, 8, cells.ctypes.data, 6, 0, None,
                                          None, 0, None)
    assert rc == -1 and b"null pointer" in lib.plsb200_last_error()
    rc = lib.plsb200_rb_salience_dmma_f64(8, 120, 100, None, 0, 0, 10, 10, 24, 8, cells.ctypes.data, 6, 0, 8, 8, 0, None)
    assert rc == -1 and b"bad shape" in lib.plsb200_last_error()            # an empty window
    rc = lib.plsb200_rb_salience_dmma_f64(8, 120, 100, None, 0, 0, 0, 101, 24, 8, cells.ctypes.data, 6, 0, 8, 8, 0,
                                          None)
    assert rc == -1 and b"bad shape" in lib.plsb200_last_error()            # a window past the row stride
    rc = lib.plsb200_rb_salience_dmma_pack_f64(None, None, 120, 24, 8, cells.ctypes.data, 6, 0, None, 0, None)
    assert rc == -1 and b"null pointer" in lib.plsb200_last_error()
    rc = lib.plsb200_rb_salience_f64(8, 120, 100, None, 0, 0, 0, 10, 8, 8, 24, 8, 8, 6, 0, None, None)
    assert rc == -1 and b"null pointer" in lib.plsb200_last_error()


def test_every_result_class_has_the_method():
    from plspy_b200 import bootstrap_permutation as bp, plugin
    assert callable(bp._ResampleTestPLS.right_sv_sampled_chunks)
    for cls in plugin.PINNED.values():
        assert cls.right_sv_sampled_chunks is bp._ResampleTestPLS.right_sv_sampled_chunks
