"""TEST INFRASTRUCTURE ONLY: ctypes loaders for the CPU oracle (oracle/bv_oracle.c) and for the
compiled reference (oracle/_ref/libbvref*.so, built by oracle/build_ref.sh from /root/reference).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs may
import this module.  Nothing under basevar_b200/ imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# numpy view of struct bv_site_out (include/basevar_b200.h), 128 bytes
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
# struct bv_call_out (16 bytes) and struct bv_group_out (40 bytes)
CALL_OUT_DTYPE = np.dtype([("site", "<u4"), ("mq_rank_sum", "<i4"), ("read_pos_rank_sum", "<i4"), ("base_q_rank_sum", "<i4")])
GROUP_OUT_DTYPE = np.dtype([("n_alt", "u1"), ("alt", "u1", (4,)), ("flags", "u1"), ("reserved", "u1", (2,)), ("af", "<f8", (4,))])
assert CALL_OUT_DTYPE.itemsize == 16 and GROUP_OUT_DTYPE.itemsize == 40


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


def make_params(min_af=0.01, abs_mode=0, max_samples=0, max_sites=0, n_slots=1, lrt_threshold=24, em_max_iter=100, em_eps=0.001):
    return BvParams(float(np.float32(min_af)), lrt_threshold, em_max_iter, float(np.float32(em_eps)), abs_mode, max_samples,
                    max_sites, n_slots, 0)


def _u8p(a):
    assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def build_oracle():
    """Compile oracle/bv_oracle.c (gcc) and, when /root/reference exists, oracle/_ref."""
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    if os.path.isdir(os.environ.get("BV_REFERENCE_DIR", "/root/reference")):
        subprocess.check_call(["bash", os.path.join(HERE, "build_ref.sh")], stdout=subprocess.DEVNULL)


_oracle = None


def load_oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(HERE, "libbvoracle.so")
        if not os.path.exists(path):
            build_oracle()
        lib = C.CDLL(path)
        lib.bvo_tile.restype = C.c_int
        lib.bvo_tile.argtypes = [C.POINTER(C.c_uint8)] * 4 + [C.c_uint64, C.c_uint32, C.c_uint32,
                                                              C.POINTER(BvParams), C.c_void_p]
        lib.bvo_gammaq.restype = C.c_double
        lib.bvo_gammaq.argtypes = [C.c_double, C.c_double]
        lib.bvo_chi2_test.restype = C.c_double
        lib.bvo_chi2_test.argtypes = [C.c_double, C.c_double]
        lib.bvo_fisher_two_sided.restype = C.c_double
        lib.bvo_fisher_two_sided.argtypes = [C.c_int] * 4
        lib.bvo_fs_from_table.restype = C.c_double
        lib.bvo_fs_from_table.argtypes = [C.c_int] * 4
        lib.bvo_sor_from_table.restype = C.c_double
        lib.bvo_sor_from_table.argtypes = [C.c_int] * 4
        lib.bvo_erfc.restype = C.c_double
        lib.bvo_erfc.argtypes = [C.c_double]
        lib.bvo_wilcoxon.restype = C.c_double
        lib.bvo_wilcoxon.argtypes = [C.POINTER(C.c_double), C.c_size_t, C.POINTER(C.c_double), C.c_size_t]
        lib.bvo_ranksums.restype = C.c_int
        lib.bvo_ranksums.argtypes = [C.POINTER(C.c_uint8)] * 3 + [C.POINTER(C.c_uint16), C.c_uint32, C.c_uint8, C.c_uint32,
                                                                C.POINTER(C.c_int32)]
        lib.bvo_group_site.restype = C.c_int
        lib.bvo_group_site.argtypes = [C.POINTER(C.c_uint8)] * 2 + [C.c_uint32, C.POINTER(C.c_uint8), C.c_uint32, C.c_uint8,
                                                                  C.POINTER(C.c_uint8), C.c_int, C.POINTER(BvParams), C.c_void_p]
        _oracle = lib
    return _oracle


def oracle_tile(base, qual, strand, ref_base, n_samples, min_af=0.01, abs_mode=0, lrt_threshold=24, em_max_iter=100, em_eps=0.001):
    """Run the C restatement over planes [S][pitch] (uint8).  Returns a SITE_OUT_DTYPE array."""
    lib = load_oracle()
    S, pitch = base.shape
    out = np.zeros(S, dtype=SITE_OUT_DTYPE)
    prm = make_params(min_af, abs_mode, lrt_threshold=lrt_threshold, em_max_iter=em_max_iter, em_eps=em_eps)
    rc = lib.bvo_tile(_u8p(base), _u8p(qual), _u8p(strand), _u8p(ref_base), pitch, S, n_samples, C.byref(prm),
                      out.ctypes.data)
    assert rc == 0
    return out


def _alt_mask(rec):
    m = 0
    for k in range(int(rec["n_alt"])):
        m |= 1 << int(rec["alt"][k])
    return m


def _group_order(ref_char, rec):
    """[upper REF, ALT...] as base codes (src/basetype_caller.cpp:750-753); a REF that is not A/C/G/T is left out."""
    order = []
    rc = "ACGT".find(chr(ref_char).upper())
    if rc >= 0:
        order.append(rc)
    for k in range(int(rec["n_alt"])):
        if int(rec["alt"][k]) not in order:
            order.append(int(rec["alt"][k]))
    return np.array(order, np.uint8)


def oracle_calls(base, qual, mapq, rpr, ref_base, n_samples, recs, sample_group=None, n_groups=0, min_af=0.01, abs_mode=0,
                 use_ref=False, lrt_threshold=24, em_max_iter=100, em_eps=0.001):
    """Rank sums and population-group calls of the called sites (recs: SITE_OUT_DTYPE of the same planes), from the C
    restatement or (use_ref) from the compiled reference.  Returns (calls sorted by site, groups[n_calls][n_groups])."""
    lib = load_ref(bool(abs_mode)) if use_ref else load_oracle()
    assert lib is not None
    sites = np.nonzero(recs["n_alt"] > 0)[0]
    calls = np.zeros(len(sites), CALL_OUT_DTYPE)
    groups = np.zeros((len(sites), max(n_groups, 0)), GROUP_OUT_DTYPE)
    # (the compiled reference has its parameters built in: it runs at the defaults only)
    assert not use_ref or (lrt_threshold, em_max_iter, em_eps) == (24, 100, 0.001)
    prm = make_params(min_af, abs_mode, lrt_threshold=lrt_threshold, em_max_iter=em_max_iter, em_eps=em_eps)
    u16p = C.POINTER(C.c_uint16)
    rpr = np.ascontiguousarray(rpr, np.uint16)
    for k, s in enumerate(sites):
        out3 = (C.c_int32 * 3)()
        row = lambda a: _u8p(np.ascontiguousarray(a[s]))
        rr = np.ascontiguousarray(rpr[s])
        fn = lib.bvref_ranksums if use_ref else lib.bvo_ranksums
        rc = fn(row(base), row(qual), row(mapq), rr.ctypes.data_as(u16p), n_samples, int(ref_base[s]), _alt_mask(recs[s]), out3)
        assert rc == 0
        calls[k] = (s, out3[0], out3[1], out3[2])
        for g in range(n_groups):
            if use_ref:
                alts = np.ascontiguousarray(recs[s]["alt"][:int(recs[s]["n_alt"])], np.uint8)
                rc = lib.bvref_group_site(row(base), row(qual), n_samples, _u8p(sample_group), g, int(ref_base[s]), _u8p(alts),
                                          len(alts), float(np.float32(min_af)), groups[k, g:g + 1].ctypes.data)
            else:
                order = _group_order(int(ref_base[s]), recs[s])
                rc = lib.bvo_group_site(row(base), row(qual), n_samples, _u8p(sample_group), g, int(ref_base[s]), _u8p(order),
                                        len(order), C.byref(prm), groups[k, g:g + 1].ctypes.data)
            assert rc == 0
    return calls, groups


_ref = {}


def ref_available(dblabs=False):
    name = "libbvref_dblabs.so" if dblabs else "libbvref.so"
    return os.path.exists(os.path.join(HERE, "_ref", name))


def load_ref(dblabs=False):
    """The compiled UNMODIFIED reference (None if oracle/_ref was never built)."""
    if dblabs not in _ref:
        name = "libbvref_dblabs.so" if dblabs else "libbvref.so"
        path = os.path.join(HERE, "_ref", name)
        if not os.path.exists(path):
            _ref[dblabs] = None
        else:
            lib = C.CDLL(path)
            lib.bvref_tile.restype = C.c_int
            lib.bvref_tile.argtypes = [C.POINTER(C.c_uint8)] * 4 + [C.c_uint64, C.c_uint32, C.c_uint32, C.c_float,
                                                                    C.c_int, C.c_void_p, C.POINTER(C.c_double)]
            lib.bvref_fisher_fs.restype = C.c_double
            lib.bvref_fisher_fs.argtypes = [C.c_int] * 4
            lib.bvref_abs_mode.restype = C.c_int
            lib.bvref_ranksums.restype = C.c_int
            lib.bvref_ranksums.argtypes = [C.POINTER(C.c_uint8)] * 3 + [C.POINTER(C.c_uint16), C.c_uint32, C.c_uint8,
                                                                      C.c_uint32, C.POINTER(C.c_int32)]
            lib.bvref_group_site.restype = C.c_int
            lib.bvref_group_site.argtypes = [C.POINTER(C.c_uint8)] * 2 + [C.c_uint32, C.POINTER(C.c_uint8), C.c_uint32,
                                                                        C.c_uint8, C.POINTER(C.c_uint8), C.c_int, C.c_float,
                                                                        C.c_void_p]
            _ref[dblabs] = lib
    return _ref[dblabs]


def ref_tile(base, qual, strand, ref_base, n_samples, min_af=0.01, dblabs=False, n_threads=1):
    """Run the compiled reference over planes.  Returns (records, core_seconds)."""
    lib = load_ref(dblabs)
    assert lib is not None, "oracle/_ref not built"
    S, pitch = base.shape
    out = np.zeros(S, dtype=SITE_OUT_DTYPE)
    secs = C.c_double(0.0)
    rc = lib.bvref_tile(_u8p(base), _u8p(qual), _u8p(strand), _u8p(ref_base), pitch, S, n_samples,
                        float(np.float32(min_af)), n_threads, out.ctypes.data, C.byref(secs))
    assert rc == 0
    return out, secs.value


# ---- helpers to build planes from explicit read lists (golden vectors) ---------------------------
BASE_CODE = {"A": 0, "C": 1, "G": 2, "T": 3, "N": 5, "+": 6, "-": 7}


def planes_from_reads(sites, pitch=None):
    """sites: list of (ref_char, [(base_char, phred, strand_char), ...]).  Uncovered cells pad the row."""
    n = max(1, max(len(r) for _, r in sites))
    if pitch is None:
        pitch = (n + 15) // 16 * 16
    S = len(sites)
    base = np.full((S, pitch), 5, np.uint8)
    qual = np.zeros((S, pitch), np.uint8)
    strand = np.full((S, pitch), 2, np.uint8)
    ref = np.zeros(S, np.uint8)
    for s, (rc, reads) in enumerate(sites):
        ref[s] = ord(rc)
        for i, (b, q, st) in enumerate(reads):
            base[s, i] = BASE_CODE.get(b, 4)
            qual[s, i] = q
            strand[s, i] = 0 if st == "+" else 1 if st == "-" else 2
    return base, qual, strand, ref, n
