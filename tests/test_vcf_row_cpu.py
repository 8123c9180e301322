"""CPU (-m "not gpu"): the entry points of the VCF row's batch path (compact results with the called-site kernels, lists on
sparse tiles) are exported and bound, and refuse bad arguments before anything touches a device."""
import ctypes as C

import numpy as np

from basevar_b200 import capi

NEW = ("bv_tile_wait_calls_compact", "bv_tile_submit_sparse_lists", "bv_tile_wait_lists_compact")


def test_new_symbols_are_exported_and_bound(built_lib):
    lib = C.CDLL(built_lib)
    for name in NEW:
        assert hasattr(lib, name) and name in capi.EXPORTED_SYMBOLS


def test_arguments_are_refused_before_any_device_work(built_lib):
    lib = capi.load_library()
    S, N = 4, 16
    cells = capi.cell_pack([0, 1, 2, 3], 0, 0, 30)
    st = np.array([0, 1, 2, 3, 4], np.uint32)
    ref = np.frombuffer(b"ACGT", np.uint8).copy()
    t = capi.BvSparseTile(cells.ctypes.data, None, st.ctypes.data, ref.ctypes.data, None, S, N, capi.CELLS_U32, capi.OUT_COMPACT)
    lists = np.full((S, 4), capi.LIST_END, np.uint8)
    pb, pf, nf, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0), C.c_uint32(0)
    # a tile with sites needs its lists
    assert lib.bv_tile_submit_sparse_lists(None, 0, C.byref(t), None) == -1
    assert b"null lists" in lib.bv_last_error(None)
    # no context: nothing to submit to, nothing to wait for
    assert lib.bv_tile_submit_sparse_lists(None, 0, C.byref(t), lists.ctypes.data) == -1
    assert b"null context" in lib.bv_last_error(None)
    assert lib.bv_tile_wait_calls_compact(None, 0, C.byref(pb), C.byref(pf), C.byref(nf), None, 0, C.byref(n), None) == -1
    assert lib.bv_tile_wait_lists_compact(None, 0, C.byref(pb), C.byref(pf), C.byref(nf), None, 0, C.byref(n)) == -1
    assert b"null context" in lib.bv_last_error(None)
