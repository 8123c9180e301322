"""-m gpu: bv_ranksum_test (kernel K9, ref_vs_alt_ranksumtest of free-standing problems) through the C ABI and the Python engine,
against the rank-sum helper of the tests (tests/oracle_ranksum.py, pinned to the compiled reference by test_oracle_ranksum.py),
against the committed reference outputs of tests/golden/calls_*.npz and against K5's records of the same tiles."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import oracle_ranksum as R
from tests import util

pytestmark = pytest.mark.gpu
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAX_SAMPLES = 20000
I32_MIN, I32_MAX = -(2 ** 31), 2 ** 31 - 1
BV_ERR_ARG = -1   # include/basevar_b200.h
FIELDS = ("mq_rank_sum", "read_pos_rank_sum", "base_q_rank_sum")


@pytest.fixture(scope="module")
def engine(built_lib, oracle_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=MAX_SAMPLES, max_sites=2048, n_slots=2, min_af=0.01)
    yield eng
    eng.close()


def assert_same_as_helper(got, b, v, start, ref, mask, label):
    want = R.ranksum_batch(b, v, start, ref, mask)
    ok = util.close(got, want) & (np.signbit(got) == np.signbit(want))
    bad = np.nonzero(~ok)[0]
    assert len(bad) == 0, f"{label}: {len(bad)} problems differ, first {bad[:5]}: got {got[bad[:5]]} want {want[bad[:5]]}"


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN_DIR, "calls_*.npz"))), ids=os.path.basename)
@pytest.mark.parametrize("abs_mode", [0, 1])
def test_ranksum_called_sites_match_fixture_and_k5(engine, path, abs_mode):
    z = np.load(path)
    N, maf = int(z["n_samples"]), float(z["min_af"])
    key = "int" if abs_mode == 0 else "dbl"
    # the compiled reference's call set and rank sums
    want_recs = z["recs_" + key].view(L.SITE_OUT_DTYPE)
    want = z["calls_" + key].view(L.CALL_OUT_DTYPE)
    sites, b, v, start, ref, mask = R.called_site_problems(z["base"], z["qual"], z["mapq"], z["rpr"], z["ref_base"], N, want_recs)
    got = engine.ranksum_test(b, v, start, ref, mask)
    assert_same_as_helper(got, b, v, start, ref, mask, os.path.basename(path))
    got = R.truncate(got).reshape(-1, 3)
    for t, f in enumerate(FIELDS):
        assert np.array_equal(got[:, t], want[f]), f"{f} differs from the reference"
    # K5 on the same tile, for its own call set
    engine.set_params(min_af=maf, abs_mode=abs_mode)
    engine.set_groups(None, 0)
    recs, calls, _ = engine.call_host_calls(z["base"], z["qual"], z["strand"], z["ref_base"], z["mapq"], z["rpr"], N)
    sites, b, v, start, ref, mask = R.called_site_problems(z["base"], z["qual"], z["mapq"], z["rpr"], z["ref_base"], N, recs)
    assert np.array_equal(sites, calls["site"])
    got = R.truncate(engine.ranksum_test(b, v, start, ref, mask)).reshape(-1, 3)
    for t, f in enumerate(FIELDS):
        assert np.array_equal(got[:, t], calls[f]), f"{f} differs from K5's bv_call_out"


def _path(n, n1, n2, lo, hi):
    """The path K9 takes (csrc/bv_call_kernels.cuh): 'hist' (one window), 'windows' or 'pairwise'."""
    wins = ((hi - lo + 1) + 8191) // 8192
    sweeps = (min(n1, n2) + 2047) // 2048
    if wins == 1:
        return "hist"
    return "windows" if wins * ((n + 255) // 256 + 256) <= sweeps * n else "pairwise"


def _random_problems(rng):
    refs = [ord(c) for c in "ACGTNacgtn"]
    probs = []   # (bases, values, ref, mask)

    def add(n, values, mask=None, ref=None, bases=None):
        if bases is None:
            bases = rng.choice(8, n, p=[0.3, 0.25, 0.15, 0.15, 0.05, 0.04, 0.03, 0.03]).astype(np.uint8)
        probs.append((bases, np.asarray(values, np.int32), int(rng.choice(refs)) if ref is None else ref,
                      int(rng.integers(0, 16)) if mask is None else mask))

    for mask in range(16):   # every ALT mask, REF among the A/C/G/T/N upper and lower case
        for ref in refs:
            n = int(rng.integers(1, 300))
            add(n, rng.integers(0, 256, n), mask, ref)
    for n in (1, 2, 3, 31, 257, 1000, 4097, MAX_SAMPLES):   # lengths up to max_samples, three value ranges
        add(n, rng.integers(0, 256, n))
        add(n, rng.integers(0, 65536, n))
        add(n, rng.integers(I32_MIN, I32_MAX, n, endpoint=True))
    ext = np.array([I32_MIN, I32_MAX, I32_MIN, I32_MAX, 0, -1], np.int32)
    add(600, np.concatenate([ext, rng.integers(I32_MIN, I32_MAX, 594, endpoint=True)]), 0b0110, ord("A"),
        np.concatenate([np.array([0, 1, 2, 0, 1, 2], np.uint8), rng.choice(4, 594).astype(np.uint8)]))
    add(20000, rng.integers(0, 65536, 20000), 0b0010, ord("A"), rng.choice(2, 20000).astype(np.uint8))   # wide range, windows
    add(900, rng.integers(-3, 3, 900) * 1000000, 0b1000, ord("G"))                                      # few distinct, wide
    add(500, np.full(500, 42), 0b0100, ord("T"), rng.choice([2, 3], 500).astype(np.uint8))               # all tied: -0.0
    add(500, rng.integers(0, 50, 500), 0b0100, ord("T"), np.full(500, 3, np.uint8))                      # no ALT read: 10000
    add(500, rng.integers(0, 50, 500), 0b0100, ord("T"), np.full(500, 2, np.uint8))                      # no REF read: 10000
    return probs


def _pack(probs):
    start = np.zeros(len(probs) + 1, np.uint64)
    start[1:] = np.cumsum([len(p[0]) for p in probs])
    b = np.concatenate([p[0] for p in probs]).astype(np.uint8)
    v = np.concatenate([p[1] for p in probs]).astype(np.int32)
    return b, v, start, np.array([p[2] for p in probs], np.uint8), np.array([p[3] for p in probs], np.uint8)


def test_ranksum_random_problems(engine):
    rng = np.random.default_rng(2026)
    probs = _random_problems(rng)
    b, v, start, ref, mask = _pack(probs)
    got = engine.ranksum_test(b, v, start, ref, mask)
    assert_same_as_helper(got, b, v, start, ref, mask, "random")
    # every path of the kernel is taken, by the shapes of the inputs
    paths = set()
    for (pb, pv, pr, pm), g in zip(probs, got):
        cls = R.classify(pb, pr, pm)
        n1, n2 = int((cls == 0).sum()), int((cls == 1).sum())
        if n1 and n2:
            sel = pv[cls < 2].astype(np.int64)
            paths.add(_path(len(pb), n1, n2, int(sel.min()), int(sel.max())))
        else:
            assert g == 10000.0
    assert paths == {"hist", "windows", "pairwise"}, paths
    assert got[-3] == 0.0 and np.signbit(got[-3]) and got[-2] == 10000.0 and got[-1] == 10000.0
    # one call per problem gives the same values
    for p in (0, 17, len(probs) - 4, len(probs) - 3):
        s0, s1 = int(start[p]), int(start[p + 1])
        one = engine.ranksum_test(b[s0:s1], v[s0:s1], np.array([0, s1 - s0], np.uint64), ref[p:p + 1], mask[p:p + 1])
        assert one.tobytes() == got[p:p + 1].tobytes()


def test_ranksum_complete_separation_100k(built_lib, oracle_lib):
    """One problem of 100,000 reads whose ALT values all lie below the REF values: p underflows to 0, so 10000."""
    n = 100000
    eng = bv.BaseTypeEngine(device=0, max_samples=n, min_af=0.01)
    try:
        bases = np.repeat(np.array([0, 3], np.uint8), n // 2)
        values = np.concatenate([np.arange(n // 2, n), np.arange(0, n // 2)]).astype(np.int32)
        start = np.array([0, n], np.uint64)
        got = eng.ranksum_test(bases, values, start, np.array([ord("A")], np.uint8), np.array([1 << 3], np.uint8))
        assert got[0] == 10000.0 and R.ranksum_test(bases, values, ord("A"), 1 << 3) == 10000.0
        # the same reads, interleaved values: a finite answer, through the full-range path too
        rng = np.random.default_rng(9)
        for vals in (rng.integers(0, 60, n), rng.integers(0, 20000, n), rng.integers(I32_MIN, I32_MAX, n, endpoint=True)):
            vals = vals.astype(np.int32)
            got = eng.ranksum_test(bases, vals, start, np.array([ord("A")], np.uint8), np.array([1 << 3], np.uint8))
            assert_same_as_helper(got, bases, vals, start, np.array([ord("A")], np.uint8), np.array([1 << 3], np.uint8), "100k")
    finally:
        eng.close()


def test_ranksum_refusals_launches_and_profiling(built_lib, oracle_lib):
    lib = capi.load_library()
    eng = bv.BaseTypeEngine(device=0, max_samples=1000, max_sites=2048, n_slots=2, min_af=0.01)
    ref_eng = bv.BaseTypeEngine(device=0, max_samples=1000, max_sites=2048, n_slots=2, min_af=0.01)
    try:
        ctx = eng._ctx
        b = np.array([0, 1, 0, 1, 2, 3], np.uint8)
        v = np.arange(6, dtype=np.int32)
        ref, mask = np.array([ord("A"), ord("C")], np.uint8), np.array([2, 1], np.uint8)
        out = np.zeros(2, np.float64)
        P = lambda a: a.ctypes.data

        def call(bb=b, vv=v, st=np.array([0, 3, 6], np.uint64), rr=ref, mm=mask, n=2, oo=out, ptr=None):
            args = [P(bb), P(vv), P(st), P(rr), P(mm), n, P(oo)]
            if ptr is not None:
                args[ptr] = None
            return lib.bv_ranksum_test(ctx, *args)

        l0 = eng.launch_count
        assert lib.bv_ranksum_test(ctx, None, None, None, None, None, 0, None) == capi.BV_OK   # n == 0: nothing launched
        assert eng.launch_count == l0
        for k in (0, 1, 2, 3, 4, 6):
            assert call(ptr=k) == BV_ERR_ARG
        assert call(st=np.array([1, 3, 6], np.uint64)) == BV_ERR_ARG             # start[0] != 0
        assert call(st=np.array([0, 4, 3], np.uint64)) == BV_ERR_ARG             # not ascending
        assert call(mm=np.array([2, 16], np.uint8)) == BV_ERR_ARG                # alt_mask > 15
        long_b, long_v = np.zeros(1002, np.uint8), np.zeros(1002, np.int32)
        assert call(bb=long_b, vv=long_v, st=np.array([0, 1, 1002], np.uint64)) == BV_ERR_ARG   # 1,001 > max_samples
        assert eng.launch_count == l0
        assert call() == capi.BV_OK and eng.launch_count == l0 + 1                    # the context is still usable
        assert out.tobytes() == R.ranksum_batch(b, v, np.array([0, 3, 6], np.uint64), ref, mask).tobytes()
        # the existing entry points launch what they launched before, on a context that used K9 and on one that did not
        rng = np.random.default_rng(4)
        S, N = 300, 500
        tb, tq, ts, tr = util.random_tile(rng, S, N, 0.3, 5, 40)
        mapq, rpr = util.random_aux(rng, tb, N, 150)
        lists = np.tile(np.array([0, 1, 2, 3], np.uint8), (S, 1))
        counts = []
        for e in (eng, ref_eng):
            c0 = e.launch_count
            e.call_host(tb, tq, ts, tr, N)
            c1 = e.launch_count
            e.call_host_calls(tb, tq, ts, tr, mapq, rpr, N)
            c2 = e.launch_count
            e.call_host_lists(tb, tq, ts, tr, lists, N)
            counts.append((c1 - c0, c2 - c1, e.launch_count - c2))
        assert counts[0] == counts[1] == (7, 8, 8), counts
        # K9's profiling event
        eng.set_profiling(True)
        eng.ranksum_test(b, v, np.array([0, 3, 6], np.uint64), ref, mask)
        assert eng.last_ranksum_kernel_time() > 0
    finally:
        eng.close()
        ref_eng.close()
