"""-m gpu: the device's numerical primitives, one level below the records, each against the oracle's double-precision restatement
of the reference and against a high-precision value of the same function (mpmath), at their branch points and range limits.

The record tests hold AF / QUAL / FS to 1e-9 relative; these hold each primitive to what its comment claims (1e-16 .. 1e-13), so a
primitive made wrong at the 1e-12 level fails here even where the records would still pass.  The probe library
(tests/cuda/numerics_probe.cu) compiles the shipping source and calls the shipping device functions with the tables of a real
context.  Every test prints the worst case it saw (run with -s).

The last test sends phreds above 95 through the record, group and list paths: the kernels clamp them into slot 95, so the records
must equal the oracle's on the same planes with phred clamped to 95, and BV_FLAG_BAD_QUAL must mark exactly the quality-dependent
sites that hold a read with phred > 93."""
import ctypes as C
import math
import os
import subprocess
from fractions import Fraction

import mpmath
import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import build, capi
from oracle import loader as L
from tests import oracle_lists as OL
from tests import util

HERE = os.path.dirname(os.path.abspath(__file__))
PROBE_SRC = os.path.join(HERE, "cuda", "numerics_probe.cu")
MAX_SAMPLES = 100000                  # Fisher tables up to max_samples + 1 = 100,001 reads
DBL_MIN = 2.2250738585072014e-308     # smallest positive normal double
DENORM = 5e-324                       # one step of the denormal grid
LN2 = math.log(2.0)
FISHER_BOTH, FISHER_LEFT, FISHER_RIGHT = -1, 0, 1   # bv_fisher_fast.h
NARROW_SUPPORT = 24                   # kFisherNarrowSupport


def build_probe(out_dir):
    """Compile the probe library with the library's own nvcc flags (sm_100a, -fmad=false); needs no GPU.  Returns its path."""
    out = os.path.join(out_dir, "libnumerics_probe.so")
    subprocess.check_call([build.NVCC] + build.FLAGS + ["-o", out, PROBE_SRC, os.path.join(build.CSRC, "bv_encode16.cpp")])
    return out


@pytest.fixture(scope="session")
def probe_path(tmp_path_factory):
    return build_probe(str(tmp_path_factory.mktemp("numerics_probe")))


def test_probe_builds_without_a_gpu(probe_path):
    """The probe reaches into the context (d_lut, d_logfact) and the device functions by name: a rename breaks it here first."""
    lib = C.CDLL(probe_path)
    for name in ("probe_log_tab", "probe_log_ratio", "probe_rcp_fast", "probe_ff_div", "probe_gammaq", "probe_qual_from_chi",
                 "probe_fisher", "probe_fs_from_table", "probe_erfc", "probe_ranksum_phred", "probe_is_active", "probe_iabs_trunc",
                 "bv_create", "bv_destroy"):
        assert hasattr(lib, name), name


class Probe:
    """The probe's wrappers over numpy arrays, on a context of the probe's own copy of the library."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.ctx = C.c_void_p()
        prm = capi.make_params(max_samples=MAX_SAMPLES)
        rc = self.lib.bv_create(0, C.byref(prm), C.byref(self.ctx))
        assert rc == 0, f"bv_create failed ({rc})"

    def close(self):
        self.lib.bv_destroy(self.ctx)

    def unary(self, name, x, out_dtype=np.float64):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(len(x), out_dtype)
        getattr(self.lib, name).argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        assert getattr(self.lib, name)(x.ctypes.data, y.ctypes.data, len(x)) == 0, name
        return y

    def log_tab(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y, bad = np.zeros(len(x)), np.zeros(len(x), np.uint32)
        self.lib.probe_log_tab.argtypes = [C.c_void_p] * 4 + [C.c_size_t]
        assert self.lib.probe_log_tab(self.ctx, x.ctypes.data, y.ctypes.data, bad.ctypes.data, len(x)) == 0
        return y, bad

    def binary(self, name, a, b):
        a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
        y = np.zeros(len(a))
        getattr(self.lib, name).argtypes = [C.c_void_p] * 3 + [C.c_size_t]
        assert getattr(self.lib, name)(a.ctypes.data, b.ctypes.data, y.ctypes.data, len(a)) == 0, name
        return y

    def fisher(self, tables, side):
        t = np.ascontiguousarray(tables, np.int32)
        y, whole = np.zeros(len(t)), np.zeros(len(t), np.uint8)
        self.lib.probe_fisher.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t]
        assert self.lib.probe_fisher(self.ctx, t.ctypes.data, side, y.ctypes.data, whole.ctypes.data, len(t)) == 0
        return y, whole.astype(bool)

    def fs_from_table(self, tables):
        t = np.ascontiguousarray(tables, np.int32)
        y = np.zeros(len(t))
        self.lib.probe_fs_from_table.argtypes = [C.c_void_p] * 3 + [C.c_size_t]
        assert self.lib.probe_fs_from_table(self.ctx, t.ctypes.data, y.ctypes.data, len(t)) == 0
        return y

    def ranksum_phred(self, twice, n1, n2):
        a = [np.ascontiguousarray(v, np.uint64) for v in (twice, n1, n2)]
        y = np.zeros(len(a[0]), np.int32)
        self.lib.probe_ranksum_phred.argtypes = [C.c_void_p] * 4 + [C.c_size_t]
        assert self.lib.probe_ranksum_phred(*(v.ctypes.data for v in a), y.ctypes.data, len(y)) == 0
        return y

    def is_active(self, dep, total, min_af):
        d, t = np.ascontiguousarray(dep, np.uint32), np.ascontiguousarray(total, np.uint32)
        y = np.zeros(len(d), np.uint8)
        self.lib.probe_is_active.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_size_t]
        assert self.lib.probe_is_active(d.ctypes.data, t.ctypes.data, min_af, y.ctypes.data, len(d)) == 0
        return y.astype(bool)

    def iabs_trunc(self, diff):
        d = np.ascontiguousarray(diff, np.float64)
        y = np.zeros(len(d), np.int64)
        self.lib.probe_iabs_trunc.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        assert self.lib.probe_iabs_trunc(d.ctypes.data, y.ctypes.data, len(d)) == 0
        return y


@pytest.fixture(scope="module")
def probe(probe_path):
    p = Probe(probe_path)
    yield p
    p.close()


def ulp_distance(a, b):
    """Distance in units in the last place between doubles of the same sign (ordered bit patterns)."""
    ia, ib = np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64)
    return np.abs(ia - ib)


def around(x, k=1):
    """x and its k neighbours on either side, as doubles."""
    x = np.atleast_1d(np.asarray(x, np.float64))
    out, lo, hi = [x], x.copy(), x.copy()
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return np.concatenate(out)


def mp_hi_lo(values, fn, dps=40):
    """fn (an mpmath function) of every value at dps digits, as a double-double (hi, lo)."""
    hi, lo = np.empty(len(values)), np.empty(len(values))
    with mpmath.workdps(dps):
        for i, v in enumerate(values.tolist()):
            r = fn(mpmath.mpf(v))
            h = float(r)
            hi[i], lo[i] = h, float(r - h)
    return hi, lo


# ---- log_tab (bv_em_kernels.cuh) ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_log_tab(probe):
    """|error| <= 2.8e-16 * max(|log x|, ln 2) over the normal range up to 2^20, next to 1, at every bucket edge +- 1 ulp in nine
    binades and at every power of two +- 1 ulp; `bad` for exactly 0, denormals, negatives, inf and NaN."""
    rng = np.random.default_rng(7)
    edges = 1.0 + np.arange(129) / 128.0                      # bucket i covers mantissas [edges[i], edges[i + 1])
    binades = np.array([-1022, -1021, -700, -64, -1, 0, 1, 10, 19])
    x = np.concatenate([
        np.exp2(rng.uniform(-1022, 20, 2_000_000)),
        1.0 + rng.uniform(-1e-3, 1e-3, 200_000),
        around(np.ldexp(edges[None, :], binades[:, None]).ravel()),
        around(np.ldexp(1.0, np.arange(-1022, 21))),
        around(1.0, 8),
    ])
    x = x[(x >= DBL_MIN) & (x <= 2.0 ** 20)]
    y, bad = probe.log_tab(x)
    assert not bad.any(), f"bad raised for positive normal arguments {x[bad != 0][:5]}"
    hi, lo = mp_hi_lo(x, mpmath.log)
    err = np.abs((y - hi) - lo)
    rel = err / np.maximum(np.abs(hi), LN2)
    w = int(np.argmax(rel))
    print(f"\nlog_tab: {len(x)} arguments, worst error {rel[w]:.3e} * max(|log x|, ln 2) at x = {x[w]!r} (bound 2.8e-16)")
    assert rel[w] <= 2.8e-16, (x[w], y[w], hi[w])

    # the range check: exactly the arguments outside the positive normals
    denorm = np.array([DENORM, np.nextafter(DBL_MIN, 0), 1e-310, 2.5e-320])
    outside = np.concatenate([[0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], denorm, -denorm, [-DBL_MIN, -1.0, -1e300, -np.finfo(float).max]])
    inside = np.concatenate([[DBL_MIN, np.nextafter(DBL_MIN, 1), np.finfo(float).max, np.nextafter(np.inf, 0) / 2, 1.0],
                             np.exp2(rng.uniform(-1022, 1024, 100_000))])
    inside = inside[np.isfinite(inside)]
    _, bad_out = probe.log_tab(outside)
    _, bad_in = probe.log_tab(inside)
    assert bad_out.all(), outside[bad_out == 0]
    assert not bad_in.any(), inside[bad_in != 0]


# ---- log_ratio (bv_em_kernels.cuh) ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_log_ratio(probe):
    """r in [1 - 2^-8, 1 + 2^-8].  Series side (|t| < 2^-10): the four terms leave out t^5 / 5 - t^6 / 6 + ..., so the error is at
    most |t|^5 / 5 plus the rounding of the sum.  That rounding was measured at 2.219e-16 |t| (t = -4.5e-13: 1 ulp of t), above the
    2e-16 |t| once claimed, so the bound allows 2 ulp (2^-51 |t|).  Next to the switch |t|^5 / 5 dominates: 1.8e-16 absolute, 1.8e-13
    of t.  Library side: within 1 ulp of log r."""
    rng = np.random.default_rng(8)
    edge = 2.0 ** -10
    r = np.concatenate([1.0 + rng.uniform(-2.0 ** -8, 2.0 ** -8, 200_000), 1.0 + np.exp2(rng.uniform(-60, -8, 50_000)),
                        1.0 - np.exp2(rng.uniform(-60, -8, 50_000)), around([1.0 - edge, 1.0 + edge], 4), around(1.0, 4),
                        [1.0 - 2.0 ** -8, 1.0 + 2.0 ** -8]])
    y = probe.unary("probe_log_ratio", r)
    hi, lo = mp_hi_lo(r, mpmath.log)
    err = np.abs((y - hi) - lo)
    t = r - 1.0
    series = np.abs(t) < edge
    bound = np.abs(t) ** 5 / 5 + 2.0 ** -51 * np.abs(t)
    ratio = np.where(series, err / np.where(bound > 0, bound, 1.0), 0.0)
    ws = int(np.argmax(ratio))
    ulps = np.where(series, 0.0, err / np.spacing(np.abs(hi)))
    wl = int(np.argmax(ulps))
    near = series & (np.abs(t) > 2.0 ** -11)
    wn = int(np.argmax(np.where(near, err, 0.0)))
    print(f"\nlog_ratio: series side worst {err[ws]:.3e} absolute = {err[ws] / abs(t[ws]):.3e} |t| at t = {t[ws]!r} "
          f"({ratio[ws]:.3f} of |t|^5/5 + 2^-51 |t|); next to the switch {err[wn]:.3e} absolute = {err[wn] / abs(t[wn]):.3e} |t| "
          f"at t = {t[wn]!r}; library side worst {ulps[wl]:.3f} ulp at t = {t[wl]!r}")
    assert ratio[ws] <= 1.0, (t[ws], y[ws], hi[ws])
    assert ulps[wl] <= 1.0, (t[wl], y[wl], hi[wl])
    # both sides of the switch are taken
    assert series[np.abs(t) == np.nextafter(edge, 0)].all() and not series[np.abs(t) == edge].any()


# ---- rcp_fast / ff_div (bv_fisher_fast.h) ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rcp_fast_and_ff_div(probe):
    rng = np.random.default_rng(9)
    p2 = np.ldexp(1.0, np.arange(-1022, 1))
    m = np.concatenate([np.exp2(rng.uniform(-1022, 0, 100_000)), p2, np.nextafter(p2[1:], 0), np.nextafter(p2[:-1], 1), [1.0, DBL_MIN]])
    y = probe.unary("probe_rcp_fast", m)
    exact = np.array([float(1 / Fraction(v)) for v in m.tolist()])   # 1 / m correctly rounded
    d = ulp_distance(y, exact)
    w = int(np.argmax(d))
    print(f"\nrcp_fast: {len(m)} marginals in [2^-1022, 1], worst {d[w]} ulp from the correctly rounded 1/m at m = {m[w]!r}")
    assert d[w] <= 1, (m[w], y[w], exact[w])
    assert np.isnan(probe.unary("probe_rcp_fast", [0.0])[0]), "rcp_fast(0) must be NaN (the EM posteriors 0 * inf are NaN)"

    # ff_div: the Fisher steps' integer products below 2^53
    num = np.floor(np.exp2(rng.uniform(0, 53, 200_000)))
    den = np.floor(np.exp2(rng.uniform(0, 53, 200_000)))
    a, b, c, e = (rng.integers(1, MAX_SAMPLES + 2, 50_000).astype(np.float64) for _ in range(4))
    num, den = np.concatenate([num, a * b, [1.0, 3.0, 2.0 ** 53 - 1]]), np.concatenate([den, c * e, [3.0, 2.0 ** 53 - 1, 3.0]])
    assert (num < 2.0 ** 53).all() and (den < 2.0 ** 53).all()
    y = probe.binary("probe_ff_div", num, den)
    d = ulp_distance(y, num / den)                            # IEEE division of exact integers: correctly rounded
    w = int(np.argmax(d))
    print(f"ff_div: {len(num)} integer quotients, worst {d[w]} ulp at {num[w]:.17g} / {den[w]:.17g}")
    assert d[w] <= 2, (num[w], den[w], y[w])


# ---- gammaq / qual_from_chi (bv_math.cuh) ---------------------------------------------------------------------------------------
def _qual_of_p(p):   # bvo_site's QUAL rule (oracle/bv_oracle.c): NaN -> 1, p == 0 -> 10000, -0.0 scrubbed
    if math.isnan(p):
        p = 1.0
    q = -10 * math.log10(p) if p != 0.0 else 10000.0
    return 0.0 if q == 0.0 else q


def _check_p(name, x, got, want, rtol=1e-12):
    """got / want: survival probabilities.  Normal values within rtol; denormal ones within one grid step plus rtol; the same zeros."""
    zero_diff = (got == 0) != (want == 0)
    assert not zero_diff.any(), f"{name}: only one side underflows to 0 at {x[zero_diff][:5]} (got {got[zero_diff][:5]}, want {want[zero_diff][:5]})"
    normal = want >= DBL_MIN
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        rel = np.where(normal, np.abs(got - want) / np.where(want > 0, want, 1), 0.0)
        sub = ~normal & (want > 0)
        steps = np.where(sub, (np.abs(got - want) - rtol * want) / DENORM, 0.0)
    assert np.array_equal(np.isnan(got), np.isnan(want)), name
    rel, steps = np.nan_to_num(rel), np.nan_to_num(steps)
    w = int(np.argmax(rel))
    print(f"{name}: worst {rel[w]:.3e} relative at {x[w]!r}; {int(sub.sum())} denormal results, worst {max(0.0, steps.max()):.2f} grid steps")
    assert rel[w] <= rtol, (x[w], got[w], want[w])
    assert steps.max() <= 1.0


@pytest.mark.gpu
def test_gammaq_and_qual(probe, oracle_lib):
    """QUAL from chi2 (qual_from_chi) and kf_gammaq (s = 0.5, 1, 1.5, 2) against the oracle (libm vs libdevice rounding only) at the
    switch from series to continued fraction (z = 1, z < s), the QUAL threshold region, the underflow of p (denormal near
    chi2 = 1,409, 0 near 1,483), and against mpmath's erfc / regularized upper incomplete gamma."""
    rng = np.random.default_rng(10)
    chi = np.concatenate([[0.0, -0.0, -1e-12, 1e-300, 1e-310, DENORM], np.geomspace(1e-6, 1.0, 2001),
                          np.arange(1.9, 2.1, 1e-4), around(2.0, 3), np.arange(23.9, 24.1, 1e-4), around(24.0, 2),
                          np.arange(1400.0, 1500.0, 0.01), rng.uniform(0, 1500, 5000), [1e4, np.inf, np.nan]])
    qual = probe.unary("probe_qual_from_chi", chi)
    p = probe.binary("probe_gammaq", np.full(len(chi), 0.5), chi / 2.0)
    p_o = np.array([oracle_lib.bvo_chi2_test(c, 1.0) for c in chi.tolist()])
    qual_o = np.array([_qual_of_p(v) for v in p_o.tolist()])

    assert qual[0] == 0.0 and math.copysign(1.0, qual[0]) == 1.0 and math.copysign(1.0, qual[1]) == 1.0, qual[:2]
    assert not ((qual == 0) & np.signbit(qual)).any(), "QUAL -0.0"
    print()
    pn = np.where(np.isnan(p_o), 1.0, p_o)
    _check_p("p = gammaq(0.5, chi2 / 2)", chi, np.where(np.isnan(p), 1.0, p), pn)
    normal = pn >= DBL_MIN
    ok = util.close(qual, qual_o, rtol=1e-12, atol=0.0)
    rel = np.where(normal & (qual_o != 0), np.abs(qual - qual_o) / np.where(qual_o != 0, qual_o, 1), 0.0)
    w = int(np.argmax(rel))
    print(f"QUAL: worst {rel[w]:.3e} relative at chi2 = {chi[w]!r} (QUAL {qual_o[w]!r}); "
          f"p denormal on [{chi[(pn > 0) & ~normal].min():.2f}, {chi[(pn > 0) & ~normal].max():.2f}], 0 from {chi[pn == 0][chi[pn == 0] > 0].min():.2f}")
    assert (ok | ~normal).all(), chi[~ok & normal][:5]
    assert np.array_equal(qual == 10000.0, qual_o == 10000.0)

    # the right function: erfc(sqrt(chi2 / 2)) where p > 1e-300
    sel = np.nonzero((pn > 1e-300) & (chi > 0) & np.isfinite(chi))[0][::4]
    with mpmath.workdps(30):
        ref = np.array([float(mpmath.erfc(mpmath.sqrt(mpmath.mpf(c) / 2))) for c in chi[sel].tolist()])
    worst = max(np.max(np.abs(p[sel] - ref) / ref), np.max(np.abs(p_o[sel] - ref) / ref))
    print(f"p against mpmath erfc(sqrt(chi2 / 2)): worst {worst:.3e} relative over {len(sel)} values (device and oracle)")
    assert worst <= 1e-9

    # kf_gammaq itself on both sides of its switches, s = 0.5 .. 2
    for s in (0.5, 1.0, 1.5, 2.0):
        z = np.concatenate([np.geomspace(1e-6, 1.0, 1001), around(1.0, 2), around(s, 2), np.linspace(1.0, s + 1, 1001),
                            rng.uniform(0, 800, 3000), np.arange(700.0, 760.0, 0.005)])
        got = probe.binary("probe_gammaq", np.full(len(z), s), z)
        want = np.array([oracle_lib.bvo_gammaq(s, v) for v in z.tolist()])
        _check_p(f"gammaq(s = {s})", z, got, want)
        sel = np.nonzero(want > 1e-300)[0][::8]
        with mpmath.workdps(30):
            ref = np.array([float(mpmath.gammainc(s, mpmath.mpf(v), mpmath.inf, regularized=True)) for v in z[sel].tolist()])
        assert np.max(np.abs(got[sel] - ref) / ref) <= 1e-9, s


# ---- Fisher exact test (bv_math.cuh, bv_fisher_fast.h) ------------------------------------------------------------------------
def _support(t):
    n11, n12, n21, n22 = (int(v) for v in t)
    n1_, n_1, n = n11 + n12, n11 + n21, n11 + n12 + n21 + n22
    return max(0, n1_ + n_1 - n), min(n1_, n_1)


def _table(n11, n1_, n_1, n):
    return [n11, n1_ - n11, n_1 - n11, n - n1_ - n_1 + n11]


def _lpmf(i, n1_, n_1, n):   # log of the hypergeometric pmf with glibc's lgamma, as the device's table gives it
    lf = lambda k: math.lgamma(k + 1)
    lb = lambda a, b: 0.0 if b == 0 or a == b else lf(a) - lf(b) - lf(a - b)
    return lb(n1_, i) + lb(n - n1_, n_1 - i) - lb(n, n_1)


def fisher_tables(rng):
    """The tables of the Fisher test, by the edge each one aims at."""
    T = {"support 23..26": [], "q near 1e-250": [], "symmetric": [], "margin 1": [], "lo == hi": [], "q == 0": [], "total 100,001": [],
         "random": []}
    for w in (23, 24, 25, 26):   # every outcome of margins with support exactly w wide, lo == 0 and lo > 0
        for n1_, n_1, n in ((w, 60, 200), (w, w, 2 * w), (w, 5000, MAX_SAMPLES + 1), (500, 1000, 1000 + w), (40000, 60000, 60000 + w)):
            lo, hi = max(0, n1_ + n_1 - n), min(n1_, n_1)
            assert hi - lo == w
            T["support 23..26"] += [_table(i, n1_, n_1, n) for i in range(lo, hi + 1)]
    for n1_, n_1, n in ((2000, 2000, 4000), (30000, 50000, MAX_SAMPLES + 1), (700, 5000, 9000), (3000, 40, 60000)):
        lo, hi = max(0, n1_ + n_1 - n), min(n1_, n_1)
        lp = np.array([_lpmf(i, n1_, n_1, n) for i in range(lo, hi + 1)]) / math.log(10)
        for k in np.nonzero(np.diff(np.sign(lp + 250)))[0]:   # the crossings of q = 1e-250, both flanks
            T["q near 1e-250"] += [_table(lo + int(i), n1_, n_1, n) for i in range(k - 2, k + 4) if 0 <= i <= hi - lo]
    for h in (5, 12, 30, 200, 3000, 50000):   # n1_ == n / 2: pmf(i) == pmf(n_1 - i), exact ties
        for _ in range(12):
            n_1 = int(rng.integers(1, 2 * h))
            i = int(rng.integers(max(0, n_1 - h), min(h, n_1) + 1))
            T["symmetric"].append(_table(i, h, n_1, 2 * h))
    for x in (1, 2, 3, 7, 50, 999, 1000, 1001, 40000, MAX_SAMPLES - 1):
        for y in sorted({y for y in (0, 1, 5, 1000, MAX_SAMPLES - x) if x + y <= MAX_SAMPLES}):
            T["margin 1"] += [[1, 0, x, y], [0, 1, x, y], [x, y, 1, 0], [x, y, 0, 1], [1, x, 0, y], [x, 1, y, 0]]
    for x, y in ((0, 0), (5, 0), (0, 7), (3, 9), (50000, 50001)):
        T["lo == hi"] += [[0, 0, x, y], [x, y, 0, 0], [x, 0, y, 0], [0, x, 0, y]]
    T["q == 0"] += [[50000, 0, 0, 50000], [0, 50000, 50000, 0], [50000, 1, 0, 50000], [40000, 100, 200, 59700]]
    for _ in range(40):
        cut = np.sort(rng.integers(0, MAX_SAMPLES + 2, 3))
        T["total 100,001"].append([int(cut[0]), int(cut[1] - cut[0]), int(cut[2] - cut[1]), int(MAX_SAMPLES + 1 - cut[2])])
    for scale in (3, 12, 60, 400, 3000, 25000):
        T["random"] += rng.integers(0, scale, size=(60, 4)).tolist()
    for k, v in T.items():
        assert v, k
        assert all(sum(t) <= MAX_SAMPLES + 1 and min(t) >= 0 for t in v), k
    return T


def exact_two_sided(t):
    """kt_fisher_exact's value with exact arithmetic: the sum of pmf(i) over the outcomes with pmf(i) <= pmf(n11), mpmath at 50
    digits.  Returns (p, clean): clean is False when an outcome other than an exact tie lies within 1e-7 of pmf(n11), where the
    reference's 1e-8 slack decides."""
    n11, n12, n21, n22 = (int(v) for v in t)
    n1_, n_1, n = n11 + n12, n11 + n21, n11 + n12 + n21 + n22
    lo, hi = max(0, n1_ + n_1 - n), min(n1_, n_1)
    if lo == hi:
        return 1.0, True
    with mpmath.workdps(50):
        lg = mpmath.loggamma
        c = lg(n + 1) - lg(n_1 + 1) - lg(n - n_1 + 1)

        def lp(i):
            return lg(n1_ + 1) - lg(i + 1) - lg(n1_ - i + 1) + lg(n - n1_ + 1) - lg(n_1 - i + 1) - lg(n - n1_ - n_1 + i + 1) - c

        lq, tie = lp(n11), mpmath.mpf(10) ** -40
        above = lambda i: lp(i) > lq + tie
        mode = min(max((n1_ + 1) * (n_1 + 1) // (n + 2), lo), hi)
        if not above(mode):
            return 1.0, True                       # q is the largest value: every outcome counts
        a, b = lo, mode                            # first i in [lo, mode] above q (the pmf rises there)
        while a < b:
            mid = (a + b) // 2
            a, b = (a, mid) if above(mid) else (mid + 1, b)
        iL = a
        a, b = mode, hi                            # last i in [mode, hi] above q (it falls there)
        while a < b:
            mid = (a + b + 1) // 2
            a, b = (mid, b) if above(mid) else (a, mid - 1)
        iR = a
        clean = True
        for i in (iL - 1, iL, iR, iR + 1):
            if lo <= i <= hi:
                d = abs(lp(i) - lq)
                clean &= bool(d <= tie or d > mpmath.mpf("1e-7"))
        total = mpmath.mpf(0)
        if iL > lo:                                # left tail, outwards: pmf(i-1) = pmf(i) i n22(i) / ((n1_-i+1)(n_1-i+1))
            i, p = iL - 1, mpmath.exp(lp(iL - 1))
            s = mpmath.mpf(0)
            while True:
                s += p
                if i == lo or p < s * mpmath.mpf(10) ** -30:
                    break
                p *= mpmath.mpf(i * (i + n - n1_ - n_1)) / ((n1_ - i + 1) * (n_1 - i + 1))
                i -= 1
            total += s
        if iR < hi:                                # right tail: pmf(i+1) = pmf(i) (n1_-i)(n_1-i) / ((i+1) n22(i+1))
            i, p = iR + 1, mpmath.exp(lp(iR + 1))
            s = mpmath.mpf(0)
            while True:
                s += p
                if i == hi or p < s * mpmath.mpf(10) ** -30:
                    break
                p *= mpmath.mpf((n1_ - i) * (n_1 - i)) / ((i + 1) * (i + 1 + n - n1_ - n_1))
                i += 1
            total += s
        return float(min(total, 1)), clean


@pytest.mark.gpu
def test_fisher_two_sided(probe, oracle_lib):
    """fisher_two_sided, the reference's walk (support <= 24) and the fast path (wider, q > 1e-250), each tail on its own: the two
    tails add up to the whole test bit for bit; the whole test against bvo_fisher_two_sided (1e-13 walked, 1e-9 fast) and against
    the exact tail sum (1e-10 where p > 1e-250); FS (fisher_margin1, fs_from_p) against bvo_fs_from_table."""
    rng = np.random.default_rng(11)
    groups = fisher_tables(rng)
    tables = np.array([t for v in groups.values() for t in v], np.int32)
    label = np.concatenate([[k] * len(v) for k, v in groups.items()])
    both, whole = probe.fisher(tables, FISHER_BOTH)
    left, wl = probe.fisher(tables, FISHER_LEFT)
    right, wr = probe.fisher(tables, FISHER_RIGHT)
    assert np.array_equal(whole, wl) and np.array_equal(whole, wr)
    # a pair of lanes (one tail each) forms the value of one thread, bit for bit
    pair = np.where(whole, both, np.minimum(1.0, left + right))
    assert (pair.view(np.int64) == both.view(np.int64)).all(), tables[pair != both][:5]
    assert (left[whole] == both[whole]).all() and (right[whole] == both[whole]).all()

    width = np.array([_support(t)[1] - _support(t)[0] for t in tables])
    want = np.array([oracle_lib.bvo_fisher_two_sided(*map(int, t)) for t in tables])
    q = np.array([math.exp(_lpmf(int(t[0]), int(t[0] + t[1]), int(t[0] + t[2]), int(t.sum()))) for t in tables])
    fast = (width > NARROW_SUPPORT) & (q > 1e-250)
    print()
    # Narrow supports: at most 24 steps of ff_div from the reference's own terms, 1e-13 -- plus, where the reference's right walk
    # steps on from the left walk's last term and the device's starts again from a direct evaluation (bv_math.cuh), the rounding of
    # that direct evaluation, exp() of nine glibc lgamma values: up to ~12 ulp of lgamma(n + 1), measured 1.29e-10 at
    # [99999, 1, 0, 1] (n = 100,001; the device is 4e-11 from the exact 2 / 100001 there, the oracle 1.7e-10).  Wide supports: the
    # bound tests/cpp/test_fisher_fast.cpp holds the host build of the fast path to (below q = 1e-250 they are walked).
    lg_ulp = np.array([np.spacing(math.lgamma(int(t.sum()) + 1)) for t in tables])
    for name, sel, rtol in (("supports <= 24 wide", width <= NARROW_SUPPORT, 1e-13 + 12 * lg_ulp), ("wider supports", width > NARROW_SUPPORT, 1e-9)):
        normal = sel & (want >= DBL_MIN)
        rel = np.where(normal, np.abs(both - want) / np.where(want > 0, want, 1) / rtol, 0.0)
        w = int(np.argmax(rel))
        # below DBL_MIN every term of the walk is rounded to the denormal grid: one step per term of the sum
        sub = sel & ~normal
        with np.errstate(over="ignore"):
            steps = np.where(sub, np.abs(both - want) / DENORM / (width + 2), 0.0)
        print(f"fisher vs oracle, {name}: {int(sel.sum())} tables, worst {rel[w]:.3f} of the bound "
              f"({abs(both[w] - want[w]) / want[w]:.3e} relative) at {tables[w].tolist()} ({label[w]}); "
              f"{int(sub.sum())} with p < DBL_MIN, worst {steps.max():.3f} grid steps per term")
        assert rel[w] <= 1.0, (tables[w], both[w], want[w])
        assert steps.max() <= 1.0
    assert fast.sum() > 100 and (~fast & (width > NARROW_SUPPORT)).sum() > 0 and (both == 0).any()
    assert set(label[fast]) >= {"support 23..26", "q near 1e-250"} and set(label[~fast & (width > 0)]) >= {"support 23..26", "q near 1e-250"}

    # The exact tail sums.  Each pmf value is exp() of nine glibc lgamma(k + 1) values added up (the reference's lbinom, and the
    # device's table of the same values): half an ulp of lgamma(n + 1) each, and as much again from the additions, so the reference's
    # own p is only good to about 12 ulp of lgamma(n + 1) relative -- 1.4e-9 at n = 100,001 (measured: the oracle is 2.9e-10 from the
    # exact sum at [0, 26, 5000, 94975]).  The bound is 1e-10 plus that.
    n_clean, worst, at = 0, 0.0, None
    for i, t in enumerate(tables):
        if want[i] <= 1e-250:
            continue
        p, clean = exact_two_sided(t)
        if not clean:
            continue
        n_clean += 1
        r = abs(both[i] - p) / p / (1e-10 + 12 * np.spacing(math.lgamma(int(t.sum()) + 1)))
        if r > worst:
            worst, at = r, (t.tolist(), label[i], both[i], p, abs(both[i] - p) / p)
    print(f"fisher vs exact tail sums (50 digits): {n_clean} tables, worst {worst:.3f} of the bound at {at}")
    assert worst <= 1.0, at
    assert n_clean > len(tables) // 2

    # FS of the same tables: the margin-1 closed form and fs_from_p around the fisher test
    fs = probe.fs_from_table(tables)
    fs_o = np.array([oracle_lib.bvo_fs_from_table(*map(int, t)) for t in tables])
    sel = want >= DBL_MIN
    ok = util.close(fs, fs_o, util.RTOL, util.FS_ATOL)
    assert ok[sel].all(), (tables[sel & ~ok][:5], fs[sel & ~ok][:5], fs_o[sel & ~ok][:5])
    assert np.array_equal(fs == 10000.0, fs_o == 10000.0) and not np.signbit(fs[fs == 0]).any()


# ---- erfc_as66 / ranksum_phred (bv_call_kernels.cuh) ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_erfc_as66(probe, oracle_lib):
    """kf_erfc on both signs, dense in [0, 8], and next to its two switches: the rational form below z = 10 / sqrt 2 (x = 5), the
    continued fraction above, and the early return at z = 37 (x = 37 / sqrt 2)."""
    sw = [5.0, 37.0 / math.sqrt(2.0)]
    x = np.concatenate([np.linspace(0, 8, 80_001), around(sw, 6), np.linspace(4.9, 5.1, 2001), np.linspace(25.9, 26.5, 2001),
                        [0.0, 30.0, 1e300, np.inf]])
    x = np.concatenate([x, -x])
    got = probe.unary("probe_erfc", x)
    want = np.array([oracle_lib.bvo_erfc(v) for v in x.tolist()])
    assert np.array_equal(got == 0, want == 0) and np.array_equal(got == 2, want == 2)
    rel = np.abs(got - want) / np.where(want != 0, want, 1)
    w = int(np.argmax(rel))
    print(f"\nerfc_as66: {len(x)} arguments, worst {rel[w]:.3e} relative at x = {x[w]!r}")
    assert rel[w] <= 1e-13, (x[w], got[w], want[w])


@pytest.mark.gpu
def test_ranksum_phred(probe, oracle_lib):
    """The int INFO value of a Wilcoxon rank-sum test from (2 x REF rank sum, n1, n2), n1, n2 up to 2^20, over the whole range of
    the rank sum, all-ties included: bit for bit the oracle's formula (bvo_wilcoxon: the same e, z and kf_erfc, glibc log10)."""
    rng = np.random.default_rng(12)
    n = 200_000
    n1 = np.floor(np.exp2(rng.uniform(0, 20, n))).astype(np.uint64)
    n2 = np.floor(np.exp2(rng.uniform(0, 20, n))).astype(np.uint64)
    n1[:4], n2[:4] = [1, 1, 1 << 20, 1 << 20], [1, 1 << 20, 1, 1 << 20]
    lo = n1 * (n1 + np.uint64(1))                            # every REF read above every ALT read
    span = np.uint64(2) * n1 * n2
    u = rng.random(n)
    twice = lo + np.floor(u * span.astype(np.float64)).astype(np.uint64)
    ties = n1 * (n1 + n2 + np.uint64(1))                     # z == 0: every value ties
    k = n // 8
    twice[:k] = ties[:k]
    twice[k:2 * k] = ties[k:2 * k] + np.uint64(1)
    twice[2 * k:3 * k] = lo[2 * k:3 * k]
    twice[3 * k:4 * k] = (lo + span)[3 * k:4 * k]
    twice = np.minimum(np.maximum(twice, lo), lo + span)
    got = probe.ranksum_phred(twice, n1, n2)
    want = np.empty(n, np.int64)
    for i, (t, a, b) in enumerate(zip(twice.tolist(), n1.tolist(), n2.tolist())):
        e = float(a * (a + b + 1)) / 2.0
        z = (float(t) / 2.0 - e) / math.sqrt(float(a * b * (a + b + 1)) / 12.0)
        p = 2 * (oracle_lib.bvo_erfc(abs(z) / math.sqrt(2.0)) / 2.0)
        ph = -10 * math.log10(p) if p > 0 else math.inf
        want[i] = 10000 if math.isinf(ph) else int(ph)
    bad = np.nonzero(got != want)[0]
    print(f"\nranksum_phred: {n} tests, values {got.min()}..{got.max()}, {len(bad)} differ")
    assert len(bad) == 0, [(int(twice[i]), int(n1[i]), int(n2[i]), int(got[i]), int(want[i])) for i in bad[:5]]
    assert (got[:k] == 0).all() and (got == 10000).any()


# ---- is_active (bv_common.cuh) --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_is_active(probe):
    """Exhaustive over totals 1 .. 2^20 and the depths next to min_af * total: exactly `(double)d / T >= min_af` (the reference's
    compare, src/basetype.cpp:137), for the float min_af values the engine and the CLI use, the smallest positive float, and four
    doubles.  For a float min_af (24-bit mantissa) and T < 2^29 the product min_af * T is exact, so the short-cut alone already gives
    the reference's answer and the 1e-9 window decides nothing; the doubles nearest 1/75, 1/99, 1/300 and 1e-5 are values for which
    the rounded product and the rounded quotient disagree (thousands of pairs each, three for 1e-5), the case the window is for."""
    f32 = lambda v: float(np.float32(v))
    mafs = [f32(v) for v in (0.01, 0.05, 0.001, 0.5, 1.0)] + [bv.cli_min_af(0.01, n) for n in (101, 300, 1003, 3000, 10000, 99999, 100000)]
    mafs.append(float(np.nextafter(np.float32(0), np.float32(1))))
    mafs += [1 / 75, 1 / 99, 1 / 300, 1e-5]
    T = np.arange(1, (1 << 20) + 1, dtype=np.int64)
    n_checked, n_window, n_split = 0, 0, 0
    for maf in mafs:
        base = np.floor(maf * T.astype(np.float64)).astype(np.int64)
        d = (base[:, None] + np.arange(-2, 4)[None, :])          # floor - 2 .. ceil + 2
        t = np.broadcast_to(T[:, None], d.shape)
        keep = (d >= 0) & (d <= t)
        d, t = d[keep], t[keep]
        got = probe.is_active(d, t, maf)
        want = d.astype(np.float64) / t.astype(np.float64) >= maf
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, (maf, [(int(d[i]), int(t[i]), bool(got[i])) for i in bad[:5]])
        x, thr = d.astype(np.float64), maf * t.astype(np.float64)
        n_window += int(((x <= thr * 1.000000001) & (x >= thr * 0.999999999)).sum())
        n_split += int(((x >= thr) != want).sum())
        n_checked += len(d)
    print(f"\nis_active: {n_checked} (depth, total) pairs over {len(mafs)} min_af values, {n_window} inside the 1e-9 window, "
          f"{n_split} where the product alone would be wrong; none differ")
    assert n_split > 1000


# ---- iabs_trunc (bv_math.cuh) ---------------------------------------------------------------------------------------------------
def _x86_iabs_trunc(v):
    """(double)abs((int)v) on x86-64: cvttsd2si gives INT_MIN for NaN and out-of-range values; abs(INT_MIN) is INT_MIN."""
    if math.isnan(v) or not (-2147483649.0 < v < 2147483648.0):
        return -2147483648
    t = int(v)                                   # truncation toward zero
    return -2147483648 if t == -2147483648 else abs(t)


@pytest.mark.gpu
def test_iabs_trunc(probe):
    """Over the differences of two log marginals (|diff| <= 1,500: log of a positive double lies in [-745, 710]) and the values
    next to the truncation's steps, plus +-0, NaN, +-inf and values out of int range.  (diff in (-2^31 - 1, -2^31] is left out: the
    device gives +2^31 where x86 gives INT_MIN, and no log-marginal difference comes near it.)"""
    rng = np.random.default_rng(13)
    steps = np.arange(-1500, 1501, dtype=np.float64)
    diff = np.concatenate([rng.uniform(-1500, 1500, 200_000), around(steps, 2), around(steps + 0.5, 1), around([0.5, -0.5, 1.0, -1.0], 2),
                           [0.0, -0.0, np.nan, np.inf, -np.inf, 2147483647.5, 2147483648.0, -2147483649.0, 1e10, -1e10, 1e300, -1e300]])
    y = probe.iabs_trunc(diff)
    want = np.array([_x86_iabs_trunc(v) for v in diff.tolist()], np.int64)
    bad = np.nonzero(y != want)[0]
    print(f"\niabs_trunc: {len(diff)} values, {len(bad)} differ from the x86-64 rule")
    assert len(bad) == 0, [(float(diff[i]), int(y[i]), int(want[i])) for i in bad[:5]]


# ---- phreds above 95 on the record, group and list paths -----------------------------------------------------------------------
def _quality_dependent(recs, ref_base, maf):
    """Sites K2 hands on (state BOUND or EM): two or more active alleles, or one that is not REF (bv_finish_kernels.cuh scalar_site)."""
    depth = recs["depth"].astype(np.int64)
    total = depth.sum(axis=1) + recs["depth_other"]
    with np.errstate(invalid="ignore", divide="ignore"):
        act = (depth / np.maximum(total, 1)[:, None]) >= maf
    act &= (total > 0)[:, None]
    ref_code = np.array(["ACGT".find(chr(c).upper()) for c in ref_base])
    is_ref = np.zeros_like(act)
    is_ref[ref_code >= 0, ref_code[ref_code >= 0]] = True
    n_act = act.sum(axis=1)
    return (n_act >= 2) | ((n_act == 1) & (act & ~is_ref).any(axis=1))


@pytest.mark.gpu
def test_phreds_above_95(built_lib, oracle_lib):
    """A dense tile with phreds 94..255 and the same tile as sparse BV_CELLS_U32 cells (7-bit phreds 94..127): depths and strand
    tables exact, calls / AF / QUAL / chi2 those of the oracle on the planes with phred clamped to 95 (the histogram slot such reads
    share), BV_FLAG_BAD_QUAL at exactly the quality-dependent sites with a read of phred > 93; the same tile through K6 (groups)
    and K8 (lists), whose histograms are their own."""
    from tests.test_gpu_lists import compare_to_oracle, random_lists
    rng = np.random.default_rng(14)
    S, N, G = 900, 400, 3
    maf = bv.cli_min_af(0.01, N)
    b, q, s, r = util.random_tile(rng, S, N, 0.6, 2, 93, nalt_max=3, other=0.01, indel=0.01)
    counted = b[:, :N] < 5
    hot = rng.random(S) < 0.5                                    # half of the rows get reads of phred > 93
    pick = counted & hot[:, None] & (rng.random((S, N)) < 0.05)
    q_dense = q.copy()
    q_dense[:, :N][pick] = rng.integers(94, 256, int(pick.sum()))
    q_dense[:, :N][pick & (rng.random((S, N)) < 0.3)] = 255
    q_sparse = np.where(q_dense > 127, 94 + (q_dense - 94) % 34, q_dense).astype(np.uint8)   # 7-bit cells: 94..127
    mapq, rpr = util.random_aux(rng, b, N)
    grp = util.random_groups(rng, N, G)
    lists = random_lists(rng, S)

    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=512, n_slots=2, min_af=maf)
    try:
        for name, qq in (("dense 94..255", q_dense), ("sparse u32 94..127", q_sparse)):
            assert (qq[:, :N][pick] > 93).all() and qq.max() >= (255 if name.startswith("dense") else 127)
            clamped = np.minimum(qq, 95).astype(np.uint8)
            want = L.oracle_tile(b, clamped, s, r, N, maf)
            if name.startswith("dense"):
                got = eng.call_host(b, qq, s, r, N)
            else:
                cells, _, site_start = bv.dense_to_sparse(b, qq, s, N)
                got = eng.call_sparse(cells, site_start, r, N)
            for f in ("depth", "depth_other", "fwd", "rev"):
                assert np.array_equal(got[f], want[f]), (name, f)
            ie, fe, flips = util.compare_records(got, want)
            assert len(ie) == 0 and len(fe) == 0, f"{name}: records differ from the clamped oracle at {ie[:5]} / {fe[:5]}"
            high = ((qq[:, :N] > 93) & counted).any(axis=1)
            qdep = _quality_dependent(got, r, maf)
            want_bad = high & qdep
            got_bad = (got["flags"] & capi.FLAG_BAD_QUAL) != 0
            assert np.array_equal(got_bad, want_bad), f"{name}: BAD_QUAL at {np.nonzero(got_bad != want_bad)[0][:10]}"
            print(f"\n{name}: {int(high.sum())} rows with phred > 93, {int(want_bad.sum())} of them quality dependent (BAD_QUAL), "
                  f"{int((got['n_alt'] > 0).sum())} called sites, {len(flips)} listed flips")
            assert want_bad.sum() > 50 and (high & ~qdep).sum() > 20

        # K5 / K6: the called sites' rank sums and the population groups, on the dense tile
        eng.set_groups(grp, G)
        recs, calls, groups = eng.call_host_calls(b, q_dense, s, r, mapq, rpr, N)
        clamped = np.minimum(q_dense, 95).astype(np.uint8)
        ie, fe, _ = util.compare_records(recs, L.oracle_tile(b, clamped, s, r, N, maf))
        assert len(ie) == 0 and len(fe) == 0
        want_calls, want_groups = L.oracle_calls(b, clamped, mapq, rpr, r, N, recs, grp, G, maf)
        # base_q_rank_sum ranks the raw phreds (qual + 33): only the other two fields and the groups are clamped values
        want_calls["base_q_rank_sum"] = L.oracle_calls(b, q_dense, mapq, rpr, r, N, recs, None, 0, maf)[0]["base_q_rank_sum"]
        bad = util.compare_calls(calls, groups, want_calls, want_groups)
        assert not bad, bad[:5]
        assert np.array_equal(groups["flags"] & capi.FLAG_BAD_QUAL, want_groups["flags"] & capi.FLAG_BAD_QUAL)
        assert ((groups["flags"] & capi.FLAG_BAD_QUAL) != 0).sum() > 20

        # K8: lrt(list) per site
        recs, lrt = eng.call_host_lists(b, q_dense, s, r, lists, N)
        want = OL.oracle_lists(b, clamped, s, r, lists, N, maf)
        depth = recs["depth"].sum(axis=1).astype(np.float64) + recs["depth_other"]
        compare_to_oracle(lrt, want, depth, "lists, phred > 95")
        assert ((lrt["flags"] & capi.FLAG_BAD_QUAL) != 0).sum() > 50
    finally:
        eng.close()
