"""CPU: the library exports the entry points of device-resident tiles with results of every form, and the Python binding's
bv_device_out has the C struct's layout."""
import ctypes as C

from basevar_b200 import capi


def test_device_tile_entry_points_are_exported(built_lib):
    lib = C.CDLL(capi.LIB_PATH)
    for name in ("bv_tile_run_device_sparse", "bv_tile_run_device_ex"):
        assert hasattr(lib, name), name
        assert name in capi.EXPORTED_SYMBOLS
    capi.load_library()


def test_device_out_layout():
    # two int32, then eleven pointers (include/basevar_b200.h, struct bv_device_out)
    assert C.sizeof(capi.BvDeviceOut) == 8 + 11 * 8
    assert capi.BvDeviceOut.d_out.offset == 8 and capi.BvDeviceOut.d_status.offset == 8 + 10 * 8
    assert (capi.RUN_PLAIN, capi.RUN_CALLS, capi.RUN_LISTS) == (0, 1, 2)
