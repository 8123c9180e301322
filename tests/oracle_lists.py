"""TEST INFRASTRUCTURE ONLY: the CPU oracle of BaseType::lrt(specific_bases) over ordered candidate lists (bvo_site_list,
tests/oracle_lists.c, compiled together with oracle/bv_oracle.c).

The library is built on first use with gcc into the system's temporary directory, under a name that carries a hash of its
sources, so the repository tree is never written to and a changed source is never served stale."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import loader as L

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "oracle_lists.c"), os.path.join(ROOT, "oracle", "bv_oracle.c"), os.path.join(ROOT, "oracle", "bv_oracle.h"),
           os.path.join(ROOT, "include", "basevar_b200.h")]

# struct bv_lrt_out (include/basevar_b200.h), 64 bytes
LRT_OUT_DTYPE = np.dtype([("n_alt", "u1"), ("alt", "u1", (4,)), ("n_active", "u1"), ("flags", "u1"), ("em_calls", "u1"),
                          ("af", "<f8", (4,)), ("qual", "<f8"), ("chi2", "<f8"), ("fs", "<f8")])
assert LRT_OUT_DTYPE.itemsize == 64
LIST_END = 255

_lib = None


def library_path():
    """Build (if needed) and return the path of the list oracle's shared library."""
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"bv_oracle_lists_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"libbvoracle_lists_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, SOURCES[0], "-lm"])
        os.replace(tmp, path)
    return path


def load():
    global _lib
    if _lib is None:
        lib = C.CDLL(library_path())
        lib.bvo_site_list.restype = C.c_int
        lib.bvo_site_list.argtypes = [C.POINTER(C.c_uint8)] * 3 + [C.c_uint32, C.c_uint8, C.POINTER(C.c_uint8), C.c_int,
                                                                 C.POINTER(L.BvParams), C.c_void_p]
        _lib = lib
    return _lib


def _u8p(a):
    assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def oracle_lists(base, qual, strand, ref_base, lists, n_samples, min_af=0.01, abs_mode=0):
    """BaseType(row, min_af) + lrt(list) per site.  lists: uint8 [S][4], ended early by LIST_END.
    Returns a LRT_OUT_DTYPE array; a site whose list is invalid raises AssertionError."""
    lib = load()
    S = base.shape[0]
    out = np.zeros(S, LRT_OUT_DTYPE)
    prm = L.make_params(min_af, abs_mode)
    for s in range(S):
        lst = np.ascontiguousarray(lists[s], np.uint8)
        n = int(np.argmax(lst == LIST_END)) if (lst == LIST_END).any() else 4
        row = lambda a: _u8p(np.ascontiguousarray(a[s]))
        rc = lib.bvo_site_list(row(base), row(qual), row(strand), n_samples, int(ref_base[s]), _u8p(lst), n, C.byref(prm),
                               out[s:s + 1].ctypes.data)
        assert rc == 0, f"site {s}: invalid list {lst}"
    return out
