"""-m gpu: every route that decides a record, held to the oracle at non-default LRT / EM parameters (bv_params::lrt_threshold,
em_max_iter, em_eps), and the parameter values the library refuses.

Each point of the grid runs one tile through the called-site kernels with groups (records, K5 rank sums, K6 groups), the same
tile with A,C,G,T lists and with [REF, ALT...] lists (K8), and as a sparse BV_CELLS_U16 tile with compact results, which must
give the dense tile's bytes.  The tile is built so that every route is taken, and the test checks that it was:
  * K1: sites whose reads all agree (one active allele, the EM's closed form);
  * K3: REF with 22-40 reads plus a minor allele of 1-4 reads at phred 2-40, so 2G falls on both sides of 23.9 -- the bound
    settles sites only at lrt_threshold >= 24, where its proof holds, and none below;
  * K4a: a single non-REF active allele (closed form), and the last elimination round with the single-allele models;
  * K4b: EM tasks of 2-4 active alleles (int mode through bv_em_task_kernel, fabs through bv_em_iter_kernel); a second tile
    of more than kG4MaxTasks tasks gives the int mode one lane per task instead of four.
Besides util.compare_records, BV_FLAG_EM_MAXITER and em_calls must be the oracle's at every site the bound did not settle and
whose call is the same (the fields em_max_iter changes).  No tile has a phred-0 read of an active allele: the loop count of an
EM whose marginals are NaN is not modelled by the closed forms."""
import ctypes as C

import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import oracle_lists as OL
from tests import util
from tests.test_gpu_lists import compare_to_oracle

pytestmark = pytest.mark.gpu
N, MIN_AF, G = 300, 0.01, 3
G4_MAX_TASKS = 12288   # bv_em_kernels.cuh kG4MaxTasks
BV_ERR_ARG = -1        # include/basevar_b200.h
DEFAULTS = dict(lrt_threshold=24, em_max_iter=100, em_eps=0.001)

# one parameter at a time over its range (the defaults are the controls), then a few combinations
POINTS = ([dict(lrt_threshold=v) for v in (0, 1, 5, 10, 23, 24, 25, 40, 1000)] +
          [dict(em_max_iter=v) for v in (0, 1, 2, 3, 100, 500)] +
          [dict(em_eps=v) for v in (0.0, 1e-7, 0.001, 0.5, 1.0, 1.0001, 2.5, 7.0, 1e30)] +
          [dict(lrt_threshold=5, em_max_iter=1), dict(lrt_threshold=40, em_eps=0.0), dict(em_max_iter=2, em_eps=2.5),
           dict(lrt_threshold=10, em_eps=1e30), dict(lrt_threshold=1000, em_max_iter=0), dict(em_max_iter=3, em_eps=1.0001)])


def pid(p):
    names = {"lrt_threshold": "lrt", "em_max_iter": "iter", "em_eps": "eps"}
    return "-".join(f"{names[k]}{v:g}" for k, v in p.items())


def full(p):
    return {**DEFAULTS, **p}


def param_tile(seed=5):
    """Random multi-allelic rows (K1 / K4 sites), planted bound rows and planted single non-REF rows; phred >= 1."""
    rng = np.random.default_rng(seed)
    b, q, s, r = util.random_tile(rng, 500, N, 0.9, 1, 40, nalt_max=3)
    extra_b, extra_q = [], []
    refs = []
    for kind in ["bound"] * 200 + ["alt"] * 60:
        ref = int(rng.integers(0, 4))
        rb = np.full(b.shape[1], 5, np.uint8)
        rq = np.zeros(b.shape[1], np.uint8)
        if kind == "bound":   # REF x 22-40 at phred 20-40, a minor allele of 1-4 reads at phred 2-40
            o = (ref + int(rng.integers(1, 4))) % 4
            nr, no = int(rng.integers(22, 41)), int(rng.integers(1, 5))
            cells = rng.choice(N, nr + no, replace=False)
            rb[cells[:nr]], rq[cells[:nr]] = ref, rng.integers(20, 41, nr)
            rb[cells[nr:]], rq[cells[nr:]] = o, rng.integers(2, 41, no)
        else:                 # every read one non-REF base
            a = (ref + int(rng.integers(1, 4))) % 4
            cells = rng.choice(N, int(rng.integers(5, 60)), replace=False)
            rb[cells], rq[cells] = a, rng.integers(1, 41, len(cells))
        extra_b.append(rb)
        extra_q.append(rq)
        refs.append(ord("ACGT"[ref]))
    b = np.vstack([b, np.array(extra_b)])
    q = np.vstack([q, np.array(extra_q)])
    s = np.vstack([s, np.where(np.array(extra_b) < 5, rng.integers(0, 2, (len(extra_b), b.shape[1])), 2).astype(np.uint8)])
    r = np.concatenate([r, np.array(refs, np.uint8)])
    order = rng.permutation(len(r))
    return b[order], q[order], s[order], r[order], order >= 500   # (the planted rows)


@pytest.fixture(scope="module")
def engine(built_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=2000, max_sites=2048, n_slots=2, min_af=MIN_AF)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def tile():
    b, q, s, r, planted = param_tile()
    rng = np.random.default_rng(6)
    mapq, rpr = util.random_aux(rng, b, N)
    return dict(b=b, q=q, s=s, r=r, planted=planted, mapq=mapq, rpr=rpr, grp=util.random_groups(rng, N, G))


def check_em_fields(got, want, label, bound=None):
    """BV_FLAG_EM_MAXITER and em_calls: the oracle's, at sites with the same call that the bound did not settle."""
    same = (got["n_alt"] == want["n_alt"]) & (got["alt"] == want["alt"]).all(axis=1) & (got["n_active"] == want["n_active"])
    if bound is not None:
        same &= ~bound
    mi = capi.FLAG_EM_MAXITER
    bad = np.nonzero(same & (((got["flags"] & mi) != (want["flags"] & mi)) | (got["em_calls"] != want["em_calls"])))[0]
    assert len(bad) == 0, (f"{label}: EM_MAXITER / em_calls differ at {len(bad)} sites, first {bad[:5].tolist()}:\n"
                           f" got  {util.describe(got[bad[0]])}\n want {util.describe(want[bad[0]])}")


def qual_within_chi2_noise(got, want, depth):
    """got with the oracle's QUAL where the two differ by no more than chi2's own noise explains.  QUAL is a function of chi2,
    which carries an absolute noise of 1e-9 + 1e-12 * depth (the slack the comparisons give it): at chi2 near 0 -- a call kept at
    lrt_threshold 0 -- that is a relative error of QUAL far above 1e-9.  It is relayed as a relative error (QUAL ~ chi2^k,
    k <= 2 for up to three ALTs); elsewhere this is tighter than the comparisons' own 1e-9."""
    chi_tol = 1e-9 + 1e-12 * depth
    with np.errstate(divide="ignore"):
        q_rtol = 2 * chi_tol / np.abs(want["chi2"])
    near = util.close(got["qual"], want["qual"], rtol=q_rtol) & util.close(got["chi2"], want["chi2"], atol=chi_tol)
    got = got.copy()
    got["qual"][near] = want["qual"][near]
    return got


def check_records(got, want, label):
    got = qual_within_chi2_noise(got, want, got["depth"].sum(axis=1).astype(np.float64) + got["depth_other"])
    ie, fe, flips = util.compare_records(got, want)
    assert len(ie) == 0 and len(fe) == 0, (
        f"{label}: {len(ie)} exact / {len(fe)} float mismatches, first {ie[:5].tolist()} / {fe[:5].tolist()}:\n"
        f" got  {util.describe(got[(list(ie) + list(fe))[0]])}\n want {util.describe(want[(list(ie) + list(fe))[0]])}")
    assert len(flips) <= 3, f"{label}: {len(flips)} threshold / tie flips"
    util.report_flips(label, got, want, flips)
    check_em_fields(got, want, label, bound=(got["flags"] & capi.FLAG_LRT_BOUND) != 0)


def ref_alt_lists(recs, r):
    lists = np.full((len(r), 4), capi.LIST_END, np.uint8)
    for i in range(len(r)):
        lst = ["ACGT".index(chr(r[i]))] + [int(a) for a in recs["alt"][i][:int(recs["n_alt"][i])]]
        lists[i, :len(lst)] = lst
    return lists


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("point", POINTS, ids=pid)
def test_routes_vs_oracle(engine, tile, point, abs_mode):
    if point.get("em_max_iter") == 500 and abs_mode == 0:
        pytest.skip("em_max_iter 500: a fabs-mode point (EMs of more than 100 iterations)")
    prm = full(point)
    label = f"params {pid(point)} abs={abs_mode}"
    b, q, s, r = tile["b"], tile["q"], tile["s"], tile["r"]
    if prm["em_max_iter"] == 500:   # the tile has EMs that need more than 100 iterations (and fewer than 500)
        n100 = (L.oracle_tile(b, q, s, r, N, MIN_AF, abs_mode)["flags"] & capi.FLAG_EM_MAXITER != 0).sum()
        n500 = (L.oracle_tile(b, q, s, r, N, MIN_AF, abs_mode, **prm)["flags"] & capi.FLAG_EM_MAXITER != 0).sum()
        assert n100 > 0 and n500 < n100, (n100, n500)
    engine.set_params(min_af=MIN_AF, abs_mode=abs_mode, **prm)
    engine.set_groups(tile["grp"], G)
    recs, calls, groups = engine.call_host_calls(b, q, s, r, tile["mapq"], tile["rpr"], N)
    want = L.oracle_tile(b, q, s, r, N, MIN_AF, abs_mode, **prm)
    check_records(recs, want, label)

    # every route was taken
    bound = (recs["flags"] & capi.FLAG_LRT_BOUND) != 0
    ref_code = np.array(["ACGT".find(chr(c)) for c in r])
    if prm["lrt_threshold"] >= 24:   # K3 settles sites, and sends the others of its list to the EM
        assert bound.sum() >= 20 and (tile["planted"] & ~bound & (recs["em_calls"] >= 2) & (recs["n_active"] >= 1)).sum() >= 20, label
    else:
        assert bound.sum() == 0, f"{label}: K3 settled {bound.sum()} sites below lrt_threshold 24"
    one = (recs["n_active"] == 1) & (recs["em_calls"] == 1)
    assert (one & (recs["n_alt"] == 0)).sum() >= 20, label                                    # K1 / K2 closed form
    assert (one & (recs["n_alt"] == 1) & (recs["alt"][:, 0] != ref_code)).sum() >= 20, label   # K4a closed form
    assert (recs["em_calls"] >= 2).sum() >= 50, label                                         # K4b
    if prm["lrt_threshold"] >= 24:   # the last elimination round (single-allele models) was reached
        assert ((want["em_calls"] >= 3) & (want["n_active"] == 1)).sum() >= 5, label

    # K5 / K6 at the same parameters (for our call set, so that a listed flip does not cascade)
    want_calls, want_groups = L.oracle_calls(b, q, tile["mapq"], tile["rpr"], r, N, recs, tile["grp"], G, MIN_AF, abs_mode, **prm)
    bad = util.compare_calls(calls, groups, want_calls, want_groups)
    soft = set(np.nonzero((recs["flags"] & (capi.FLAG_NEAR_LRT | capi.FLAG_LRT_TIE)) != 0)[0].tolist())
    bad = [x for x in bad if not (x[0].startswith("group") and int(calls["site"][x[1][0]]) in soft)]
    assert not bad, f"{label}: {len(bad)} called-site mismatches, first {bad[:5]}"

    # K8 over A,C,G,T and over [REF, ALT...]
    depth = recs["depth"].sum(axis=1).astype(np.float64) + recs["depth_other"]
    for name, lists in (("ACGT", np.tile(np.arange(4, dtype=np.uint8), (len(r), 1))), ("REF-ALT", ref_alt_lists(recs, r))):
        _, lrt = engine.call_host_lists(b, q, s, r, lists, N)
        want_l = OL.oracle_lists(b, q, s, r, lists, N, MIN_AF, abs_mode, **prm)
        lrt = qual_within_chi2_noise(lrt, want_l, depth)
        flips = compare_to_oracle(lrt, want_l, depth, f"{label} lists {name}")
        util.report_flips(f"{label} lists {name}", lrt, want_l, flips)
        check_em_fields(lrt, want_l, f"{label} lists {name}")

    # a sparse BV_CELLS_U16 tile with compact results: the dense tile's bytes
    cells, _, st = bv.dense_to_sparse(b, q, s, N)
    words, _, st16 = bv.sparse_encode16(cells, st)
    out = np.zeros(len(r), L.SITE_OUT_DTYPE)
    engine.run_sparse_tiles(engine.sparse_tiles(words, st16, r, N, compact=True),
                            compact=lambda s0, ns, briefs, fl: engine.expand_compact(briefs, fl, r[s0:s0 + ns], out[s0:s0 + ns]))
    assert out.tobytes() == recs.tobytes(), f"{label}: the compact BV_CELLS_U16 tile differs from the dense tile"


# int mode with more than kG4MaxTasks EM tasks: one lane per task (the tile above has a few hundred tasks: four lanes)
G1_POINTS = [dict(), dict(em_max_iter=0), dict(em_max_iter=1), dict(em_eps=0.0), dict(em_eps=2.5), dict(em_eps=1e30),
             dict(lrt_threshold=5, em_max_iter=1)]


@pytest.mark.parametrize("point", G1_POINTS, ids=lambda p: pid(p) or "defaults")
def test_one_lane_per_task_vs_oracle(engine, point):
    rng = np.random.default_rng(11)
    n, maf = 64, 0.05
    shape = [(int(x), 4) for x in rng.integers(4, 21, G4_MAX_TASKS // 11 + 100)]
    b, q, s, r = util.binned_tile(rng, shape, n, maf)
    assert (util.active_counts(b, n, maf) == 4).all() and 11 * len(shape) > G4_MAX_TASKS
    prm = full(point)
    engine.set_params(min_af=maf, abs_mode=0, **prm)
    got = engine.call_host(b, q, s, r, n)
    want = L.oracle_tile(b, q, s, r, n, maf, 0, **prm)
    label = f"params g1 {pid(point) or 'defaults'}"
    ie, fe, flips = util.compare_records(got, want)
    assert len(ie) == 0 and len(fe) == 0, (f"{label}: {len(ie)} exact / {len(fe)} float mismatches, first {ie[:5].tolist()} / {fe[:5].tolist()}:"
                                           f"\n got  {util.describe(got[(list(ie) + list(fe))[0]])}\n want {util.describe(want[(list(ie) + list(fe))[0]])}")
    assert len(flips) <= 3, f"{label}: {len(flips)} flips"
    util.report_flips(label, got, want, flips)
    phred0 = ((q[:, :n] == 0) & (b[:, :n] < 4)).any(axis=1)   # (NaN marginals: see the module docstring)
    check_em_fields(got[~phred0], want[~phred0], label)
    assert (got["em_calls"] >= 4).sum() > len(shape) // 2


# ---- values the library refuses ----------------------------------------------------------------------------------------------
REFUSED = [("em_max_iter", -1), ("em_max_iter", -2147483648), ("em_abs_mode", 2), ("em_abs_mode", -1), ("min_af", 0.0),
           ("min_af", -0.01), ("min_af", float("inf")), ("min_af", float("nan")), ("em_eps", float("nan"))]


@pytest.mark.parametrize("field,value", REFUSED, ids=lambda v: str(v))
def test_refused_parameters_change_nothing(engine, tile, field, value):
    engine.set_params(min_af=MIN_AF, abs_mode=0, lrt_threshold=10, em_max_iter=7, em_eps=0.5)
    b, q, s, r = tile["b"], tile["q"], tile["s"], tile["r"]
    before = engine.call_host(b, q, s, r, N)
    kept = bytes(engine.params)
    p = capi.BvParams.from_buffer_copy(engine.params)
    setattr(p, field, value)
    lib = engine.lib
    assert lib.bv_set_params(engine._ctx, C.byref(p)) == BV_ERR_ARG
    assert field.encode() in lib.bv_last_error(engine._ctx)
    with pytest.raises(bv.BvError):
        engine.set_params(**{"abs_mode" if field == "em_abs_mode" else field: value})
    assert bytes(engine.params) == kept
    assert engine.call_host(b, q, s, r, N).tobytes() == before.tobytes(), f"{field}={value}: the refused call changed the records"
    # bv_create refuses the same values
    ctx = C.c_void_p()
    assert lib.bv_create(0, C.byref(p), C.byref(ctx)) == BV_ERR_ARG and not ctx.value
    assert field.encode() in lib.bv_last_error(None)
