"""TEST INFRASTRUCTURE ONLY: the free-standing ref_vs_alt_ranksumtest (src/basetype.cpp:201-242) restated for the tests of
bv_ranksum_test (kernel K9): the reads are classified by the rules K5's call_class and the oracle's bvo_ranksums follow, the
two classes go to the oracle's own bvo_wilcoxon (oracle/bv_oracle.c), and the phred rule of src/basetype.cpp:224-236 gives the
function's double.  tests/test_oracle_ranksum.py pins it to the compiled reference's outputs in tests/golden/calls_*.npz."""
import ctypes as C
import math

import numpy as np

from oracle import loader as L


def classify(bases, ref_char, alt_mask):
    """0 REF, 1 ALT, 2 neither: a code above 3 is in neither class; a base equal to the upper-cased REF is a REF read (before
    the ALT mask is looked at); another A/C/G/T base is an ALT read when its bit of alt_mask is set."""
    b = np.asarray(bases).astype(np.int64)
    up = ref_char - 32 if ord("a") <= ref_char <= ord("z") else ref_char
    ref_code = "ACGT".find(chr(up))
    cls = np.full(b.shape, 2, np.int64)
    acgt = b <= 3
    cls[acgt & (((int(alt_mask) >> np.minimum(b, 3)) & 1) == 1)] = 1
    cls[acgt & (b == ref_code)] = 0
    return cls


def ranksum_test(bases, values, ref_char, alt_mask):
    """ref_vs_alt_ranksumtest as a double, not truncated (10000 when a class is empty or p == 0)."""
    cls = classify(bases, ref_char, alt_mask)
    v = np.asarray(values).astype(np.float64)
    r = np.ascontiguousarray(v[cls == 0])
    a = np.ascontiguousarray(v[cls == 1])
    if len(r) == 0 or len(a) == 0:
        return 10000.0
    dp = C.POINTER(C.c_double)
    p = L.load_oracle().bvo_wilcoxon(r.ctypes.data_as(dp), len(r), a.ctypes.data_as(dp), len(a))
    if p == 0.0:   # log10(0) = -inf, so -10 log10 p is +inf
        return 10000.0
    ph = -10 * math.log10(p)
    return 10000.0 if math.isinf(ph) else ph


def ranksum_batch(bases, values, start, ref_base, alt_mask):
    """ranksum_test of every problem p = entries start[p]:start[p+1], as bv_ranksum_test takes them.  float64 [n]."""
    return np.array([ranksum_test(bases[start[p]:start[p + 1]], values[start[p]:start[p + 1]], int(ref_base[p]), int(alt_mask[p]))
                     for p in range(len(ref_base))], np.float64)


def alt_mask_of(rec):
    """ALT mask of a record's called alleles (bit b = base code b)."""
    m = 0
    for k in range(int(rec["n_alt"])):
        m |= 1 << int(rec["alt"][k])
    return m


def called_site_problems(base, qual, mapq, rpr, ref_base, n_samples, recs):
    """The three problems of every called site of recs (n_alt > 0), in the order of the site's bv_call_out fields: mapq, read
    position rank, base quality + 33.  Returns (sites, bases, values, start, ref, mask) with problem 3 k + t = field t of
    site k."""
    sites = np.nonzero(recs["n_alt"] > 0)[0]
    N = n_samples
    bases, values, ref, mask = [], [], [], []
    for s in sites:
        b = np.ascontiguousarray(base[s, :N])
        for plane in (mapq[s, :N].astype(np.int32), rpr[s, :N].astype(np.int32), qual[s, :N].astype(np.int32) + 33):
            bases.append(b)
            values.append(plane)
            ref.append(int(ref_base[s]))
            mask.append(alt_mask_of(recs[s]))
    start = np.arange(len(ref) + 1, dtype=np.uint64) * np.uint64(N)
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    return sites, cat(bases, np.uint8), cat(values, np.int32), start, np.array(ref, np.uint8), np.array(mask, np.uint8)


def truncate(ph):
    """(int) of the caller (src/basetype_caller.cpp:1151-1157); the values here are in [-0.0, 10000]."""
    return np.trunc(np.asarray(ph)).astype(np.int32)
