"""ctypes binding of include/basevar_b200.h (the C ABI of libbasevar_b200.so).

This is the only way Python reaches the CUDA path; there is no fallback.  Loading fails loudly when
the library has not been built (``python -m basevar_b200.build``), and ``Engine`` creation fails
loudly when no CUDA device is usable.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbasevar_b200.so")

BV_OK = 0
BV_LOC_HOST, BV_LOC_DEVICE = 0, 1
BV_EM_ABS_INT_TRUNC, BV_EM_ABS_DOUBLE = 0, 1

BASE_N, STRAND_NONE = 5, 2

FLAG_BAD_STRAND, FLAG_BAD_QUAL, FLAG_ZERO_SUBSET, FLAG_MONO_QUAL = 0x01, 0x02, 0x04, 0x08
FLAG_NEAR_LRT, FLAG_LRT_BOUND, FLAG_EM_MAXITER, FLAG_LRT_TIE = 0x10, 0x20, 0x40, 0x80

# struct bv_site_out, 128 bytes
SITE_OUT_DTYPE = np.dtype(
    [
        ("depth", "<u4", (4,)),
        ("depth_other", "<u4"),
        ("reserved0", "<u4"),
        ("fwd", "<u4", (4,)),
        ("rev", "<u4", (4,)),
        ("n_alt", "u1"),
        ("alt", "u1", (4,)),
        ("n_active", "u1"),
        ("flags", "u1"),
        ("em_calls", "u1"),
        ("af", "<f8", (4,)),
        ("qual", "<f8"),
        ("chi2", "<f8"),
        ("fs_cvg", "<f8"),
        ("fs_vcf", "<f8"),
    ]
)
assert SITE_OUT_DTYPE.itemsize == 128


# struct bv_call_out (16 bytes), struct bv_group_out (40 bytes)
CALL_OUT_DTYPE = np.dtype([("site", "<u4"), ("mq_rank_sum", "<i4"), ("read_pos_rank_sum", "<i4"), ("base_q_rank_sum", "<i4")])
GROUP_OUT_DTYPE = np.dtype([("n_alt", "u1"), ("alt", "u1", (4,)), ("flags", "u1"), ("reserved", "u1", (2,)), ("af", "<f8", (4,))])
assert CALL_OUT_DTYPE.itemsize == 16 and GROUP_OUT_DTYPE.itemsize == 40
GROUP_NONE = 255
# struct bv_lrt_out (64 bytes): BaseType::lrt(list) of one site; lists are uint8 [n_sites][4] ended early by LIST_END
LRT_OUT_DTYPE = np.dtype([("n_alt", "u1"), ("alt", "u1", (4,)), ("n_active", "u1"), ("flags", "u1"), ("em_calls", "u1"),
                          ("af", "<f8", (4,)), ("qual", "<f8"), ("chi2", "<f8"), ("fs", "<f8")])
assert LRT_OUT_DTYPE.itemsize == 64
LIST_END = 255


class BvParams(C.Structure):
    _fields_ = [
        ("min_af", C.c_float),
        ("lrt_threshold", C.c_int32),
        ("em_max_iter", C.c_int32),
        ("em_eps", C.c_float),
        ("em_abs_mode", C.c_int32),
        ("max_samples", C.c_uint32),
        ("max_sites", C.c_uint32),
        ("n_slots", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class BvTile(C.Structure):
    _fields_ = [
        ("base", C.c_void_p),
        ("qual", C.c_void_p),
        ("strand", C.c_void_p),
        ("ref_base", C.c_void_p),
        ("pitch", C.c_uint64),
        ("n_sites", C.c_uint32),
        ("n_samples", C.c_uint32),
        ("location", C.c_int32),
        ("out_mode", C.c_int32),
    ]


class BvTileAux(C.Structure):
    _fields_ = [("mapq", C.c_void_p), ("rpr", C.c_void_p), ("rpr_pitch", C.c_uint64)]


class BvSparseTile(C.Structure):
    _fields_ = [
        ("cells", C.c_void_p),
        ("cells_aux", C.c_void_p),
        ("site_start", C.c_void_p),
        ("ref_base", C.c_void_p),
        ("out", C.c_void_p),
        ("n_sites", C.c_uint32),
        ("n_samples", C.c_uint32),
        ("format", C.c_uint32),
        ("out_mode", C.c_uint32),
    ]


CELLS_U32, CELLS_U16 = 0, 1
OUT_RECORDS, OUT_COMPACT = 0, 1
SITE_BRIEF_DTYPE = np.dtype([("w0", "<u4"), ("w1", "<u4")])   # struct bv_site_brief
RUN_PLAIN, RUN_CALLS, RUN_LISTS = 0, 1, 2


class BvDeviceOut(C.Structure):
    """struct bv_device_out: the device buffers of a device-resident tile's results (bv_tile_run_device_ex / _sparse)."""
    _fields_ = [
        ("kind", C.c_int32),
        ("out_mode", C.c_int32),
        ("d_out", C.c_void_p),
        ("d_brief", C.c_void_p),
        ("d_full", C.c_void_p),
        ("d_n_full", C.c_void_p),
        ("d_calls", C.c_void_p),
        ("d_groups", C.c_void_p),
        ("d_n_calls", C.c_void_p),
        ("d_lists", C.c_void_p),
        ("d_lrt", C.c_void_p),
        ("d_n_lrt", C.c_void_p),
        ("d_status", C.c_void_p),
    ]


def cell_pack(sample, base, strand, phred):
    """BV_CELL_PACK of include/basevar_b200.h (numpy arrays or ints)."""
    return (np.asarray(sample, np.uint32) | (np.asarray(base, np.uint32) << 20) | (np.asarray(strand, np.uint32) << 23)
            | (np.asarray(phred, np.uint32) << 25)).astype(np.uint32)


def cell_aux_pack(mapq, rpr):
    return (np.asarray(mapq, np.uint32) | (np.asarray(rpr, np.uint32) << 8)).astype(np.uint32)


class BvSynthModel(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("cov_thr", C.c_uint32),
        ("var_thr", C.c_uint32),
        ("multi_thr", C.c_uint32),
        ("q_lo", C.c_uint32),
        ("q_span", C.c_uint32),
        ("reserved", C.c_uint32),
        ("err_thr", C.c_uint32 * 96),
        ("af_thr", C.c_uint32 * 1024),
        ("af_extra_thr", C.c_uint32 * 256),
    ]


# every symbol include/basevar_b200.h declares: (name, restype, argtypes)
_SIGNATURES = [
    ("bv_version", C.c_int, []),
    ("bv_create", C.c_int, [C.c_int, C.POINTER(BvParams), C.POINTER(C.c_void_p)]),
    ("bv_destroy", None, [C.c_void_p]),
    ("bv_last_error", C.c_char_p, [C.c_void_p]),
    ("bv_set_params", C.c_int, [C.c_void_p, C.POINTER(BvParams)]),
    ("bv_launch_count", C.c_uint64, [C.c_void_p]),
    ("bv_h2d_bytes", C.c_uint64, [C.c_void_p]),
    ("bv_set_profiling", C.c_int, [C.c_void_p, C.c_int]),
    ("bv_last_kernel_times", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_last_em_kernel_times", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_last_fisher_kernel_time", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_tile_submit", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvTile)]),
    ("bv_tile_wait", C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    ("bv_tile_wait_compact", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]),
    ("bv_site_expand", None, [C.c_void_p, C.c_uint8, C.c_float, C.c_void_p]),
    ("bv_tile_run_device", C.c_int, [C.c_void_p, C.POINTER(BvTile), C.c_void_p, C.c_void_p]),
    ("bv_last_call_kernel_times", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_set_groups", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    ("bv_tile_submit_calls", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvTile), C.POINTER(BvTileAux)]),
    ("bv_tile_wait_calls", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p]),
    ("bv_tile_wait_calls_compact", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint32),
                                             C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p]),
    ("bv_tile_run_device_calls", C.c_int, [C.c_void_p, C.POINTER(BvTile), C.POINTER(BvTileAux)] + [C.c_void_p] * 5),
    ("bv_last_list_kernel_time", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_tile_submit_lists", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvTile), C.c_void_p]),
    ("bv_tile_wait_lists", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    ("bv_tile_run_device_lists", C.c_int, [C.c_void_p, C.POINTER(BvTile)] + [C.c_void_p] * 4),
    ("bv_synth_fill_rpr_device", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]),
    ("bv_synth_fill_rpr_host", C.c_int, [C.POINTER(BvSynthModel), C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]),
    ("bv_synth_set_model", C.c_int, [C.c_void_p, C.POINTER(BvSynthModel)]),
    ("bv_synth_fill_device", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64] + [C.c_void_p] * 6),
    ("bv_synth_fill_host", C.c_int, [C.POINTER(BvSynthModel), C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64] + [C.c_void_p] * 5),
    ("bv_tile_submit_sparse", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvSparseTile)]),
    ("bv_tile_submit_sparse_calls", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvSparseTile)]),
    ("bv_tile_submit_sparse_lists", C.c_int, [C.c_void_p, C.c_int, C.POINTER(BvSparseTile), C.c_void_p]),
    ("bv_tile_wait_lists_compact", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint32),
                                             C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]),
    ("bv_tile_run_device_sparse", C.c_int, [C.c_void_p, C.POINTER(BvSparseTile), C.POINTER(BvDeviceOut), C.c_void_p]),
    ("bv_tile_run_device_ex", C.c_int, [C.c_void_p, C.POINTER(BvTile), C.POINTER(BvTileAux), C.POINTER(BvDeviceOut), C.c_void_p]),
    ("bv_sparse_encode16_bound", C.c_uint64, [C.c_uint64, C.c_uint32, C.c_uint32]),
    ("bv_sparse_encode16", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                     C.POINTER(C.c_uint64)]),
    ("bv_synth_fill_sparse_host", C.c_int, [C.POINTER(BvSynthModel), C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                            C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    ("bv_suggest_tile_sites", C.c_uint32, [C.c_void_p, C.c_uint32, C.c_uint64]),
    ("bv_fisher_fs", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    ("bv_ranksum_test", C.c_int, [C.c_void_p] * 6 + [C.c_uint32, C.c_void_p]),
    ("bv_last_ranksum_kernel_time", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("bv_host_alloc", C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    ("bv_host_free", C.c_int, [C.c_void_p]),
]
EXPORTED_SYMBOLS = [s[0] for s in _SIGNATURES]

_lib = None


def load_library():
    """dlopen libbasevar_b200.so (no CUDA call is made by loading)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OSError(
                f"{LIB_PATH} is missing: build it with `python -m basevar_b200.build` "
                "(there is no CPU fallback for the basetype core)")
        lib = C.CDLL(LIB_PATH)
        for name, res, args in _SIGNATURES:
            fn = getattr(lib, name)  # AttributeError if the header and the library drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class BvError(RuntimeError):
    pass


def make_params(min_af=0.01, abs_mode=BV_EM_ABS_INT_TRUNC, max_samples=1, max_sites=0, n_slots=0,
                lrt_threshold=24, em_max_iter=100, em_eps=0.001):
    return BvParams(float(np.float32(min_af)), lrt_threshold, em_max_iter, float(np.float32(em_eps)), abs_mode,
                    max_samples, max_sites, n_slots, 0)


def cli_min_af(min_af, n_samples):
    """The CLI's clamp: std::min(float(100)/n_bam, min_af) in float (src/basetype_caller.cpp:122)."""
    return float(min(np.float32(100.0) / np.float32(n_samples), np.float32(min_af)))
