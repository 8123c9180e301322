"""-m gpu: BaseType::lrt(specific_bases) over per-site ordered candidate lists (K8 bv_list_kernel) through the C ABI.
  1. every order of every non-empty subset of A,C,G,T, dealt at random over the sites, against the oracle (bvo_site_list, tests/oracle_lists.c);
  2. the list A,C,G,T at every site against the site's own record, bit for bit;
  3. [REF, ALT...] lists with one group that holds every sample against K6's bv_group_out, bit for bit;
  4. records of a lists submit, empty lists, refused lists, the device-resident variant, launch counts.
Call differences against the oracle are allowed only where the ORACLE's flags mark a tie or threshold case."""
import ctypes as C
import itertools

import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import oracle_lists as OL
from tests import util

pytestmark = pytest.mark.gpu
SOFT = capi.FLAG_NEAR_LRT | capi.FLAG_LRT_TIE
ALL_LISTS = [p for k in range(1, 5) for c in itertools.combinations(range(4), k) for p in itertools.permutations(c)]   # 64


@pytest.fixture(scope="module")
def engine(built_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=20000, max_sites=2048, n_slots=3, min_af=0.01)
    yield eng
    eng.close()


def random_lists(rng, S):
    lists = np.full((S, 4), capi.LIST_END, np.uint8)
    for s, k in enumerate(rng.integers(0, len(ALL_LISTS), S)):
        lists[s, :len(ALL_LISTS[k])] = ALL_LISTS[k]
    return lists


def same_f64(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def compare_to_oracle(got, want, depth, label):
    """Exact: ALT list, n_active, em_calls, the BAD_* / ZERO_SUBSET / MONO_QUAL flags; floats under util's tolerances.  A
    different call is accepted only at a site the oracle flags NEAR_LRT / LRT_TIE."""
    soft = (want["flags"] & SOFT) != 0
    call_diff = (got["n_alt"] != want["n_alt"]) | (got["alt"] != want["alt"]).any(axis=1) | (got["n_active"] != want["n_active"])
    bad = call_diff & ~soft
    same = ~call_diff
    hard = capi.FLAG_BAD_STRAND | capi.FLAG_BAD_QUAL | capi.FLAG_ZERO_SUBSET
    bad |= (got["flags"] & hard) != (want["flags"] & hard)
    bad |= same & ~soft & ((got["flags"] & capi.FLAG_MONO_QUAL) != (want["flags"] & capi.FLAG_MONO_QUAL))
    bad |= same & ~soft & (got["em_calls"] != want["em_calls"])
    for k in range(4):
        bad |= same & (got["n_alt"] > k) & ~util.close(got["af"][:, k], want["af"][:, k])
    bad |= same & ~soft & (got["n_alt"] > 0) & ~util.close(got["qual"], want["qual"])
    badst = (want["flags"] & capi.FLAG_BAD_STRAND) != 0
    bad |= same & (got["n_alt"] > 0) & ~badst & ~util.close(got["fs"], want["fs"], atol=util.FS_ATOL)
    bad |= same & ~soft & ~util.close(got["chi2"], want["chi2"], atol=1e-9 + 1e-12 * depth)
    idx = np.nonzero(bad)[0]
    assert len(idx) == 0, f"{label}: {len(idx)} sites differ from the oracle, first {idx[:5].tolist()}: {got[idx[:2]]} vs {want[idx[:2]]}"
    return np.nonzero(call_diff & soft)[0]


def run_and_check(engine, b, q, s, r, lists, N, maf, abs_mode, label, pin_flips=False):
    """pin_flips: the listed flips are held to tests/golden/flips_r02.json under `label` (util.report_flips)."""
    engine.set_params(min_af=maf, abs_mode=abs_mode)
    recs, lrt = engine.call_host_lists(b, q, s, r, lists, N)
    want = OL.oracle_lists(b, q, s, r, lists, N, maf, abs_mode)
    depth = recs["depth"].sum(axis=1).astype(np.float64) + recs["depth_other"]
    flips = compare_to_oracle(lrt, want, depth, label)
    if pin_flips:
        util.report_flips(label, lrt, want, flips)
    return recs, lrt, flips


MIN_AFS = [0.01, 0.05, "cli"]


def maf_of(m, N):
    return bv.cli_min_af(0.01, N) if m == "cli" else m


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("min_af", MIN_AFS)
@pytest.mark.parametrize(
    "name,S,N,kw",
    [
        ("C2-like", 6000, 1000, dict(coverage=0.1, variant_frac=0.1)),
        ("C1-like-N100", 4000, 100, dict(coverage=0.065, variant_frac=0.2)),
        ("C3-like", 300, 10000, dict(coverage=0.1, variant_frac=0.2)),
        ("C5-like", 300, 2000, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
        ("odd-N", 1500, 1003, dict(coverage=0.3, variant_frac=0.3, multi_frac=0.5)),
        ("tiny-N", 1500, 7, dict(coverage=0.8, variant_frac=0.5)),
        ("long-row", 40, 5003, dict(coverage=0.5, variant_frac=0.5, multi_frac=0.5)),
    ],
)
def test_lists_synthetic_vs_oracle(engine, name, S, N, kw, min_af, abs_mode):
    model = bv.synth.make_model(seed=777 + N, **kw)
    b, q, s, _, r = bv.synth_fill_host(model, 0, S, N)
    lists = random_lists(np.random.default_rng(N + abs_mode), S)
    run_and_check(engine, b, q, s, r, lists, N, maf_of(min_af, N), abs_mode, f"{name} maf={min_af} mode={abs_mode}")


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("min_af", MIN_AFS)
def test_lists_fuzz_vs_oracle(engine, min_af, abs_mode):
    rng = np.random.default_rng(99 + abs_mode)
    for (S, N, cov, qlo, qhi, other, indel, bad) in [(400, 40, 0.9, 0, 40, 0.05, 0.05, 0.0), (300, 300, 0.3, 2, 60, 0.01, 0.02, 0.01),
                                                      (100, 64, 0.8, 0, 93, 0.02, 0.0, 0.0), (30, 4500, 0.4, 0, 60, 0.01, 0.01, 0.0)]:
        b, q, s, r = util.random_tile(rng, S, N, cov, qlo, qhi, other=other, indel=indel, bad_strand=bad)
        r[rng.random(S) < 0.05] = ord("N")
        r[rng.random(S) < 0.05] = ord("g")
        run_and_check(engine, b, q, s, r, random_lists(rng, S), N, maf_of(min_af, N), abs_mode, f"fuzz N={N} maf={min_af}")
    # deep rows with every phred 0..95: more than kSmemBins = 160 bins per row, so lrt_on_bins works through the spill rows
    N = 3000
    maf = maf_of(min_af, N)
    b, q, s, r = util.binned_tile(rng, util.deep_shape(rng, 80, N, maf), N, maf)
    assert (util.bin_counts(b, q, N) > 160).all()
    _, lrt, _ = run_and_check(engine, b, q, s, r, random_lists(rng, len(r)), N, maf, abs_mode, f"lists deep-wide-phred maf={min_af} mode={abs_mode}",
                              pin_flips=True)
    assert (lrt["em_calls"] >= 3).sum() > 10


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("min_af", MIN_AFS)
def test_acgt_lists_equal_the_records(engine, min_af, abs_mode):
    """lrt(A,C,G,T) against the site's own record.  Bit for bit: n_alt / alt / n_active / fs, em_calls except where the bound
    of K3 decided the site without an EM (BV_FLAG_LRT_BOUND), and af / qual / chi2 wherever the record took at most one EM.
    Where it took the EMs of several subsets the record comes from K4b's thread-per-task EM, whose sums are associated
    differently from those of lrt_on_bins (K8, K6): there af / qual / chi2 agree to util's tolerance and the sites are printed.
    Every EM site of a record is decided by K4b whatever the context's max_sites (tests/test_gpu_em_scratch.py)."""
    for (S, N, kw) in [(6000, 1000, dict(coverage=0.1, variant_frac=0.1)), (500, 2000, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
                       (300, 10000, dict(coverage=0.1, variant_frac=0.2)), (2000, 7, dict(coverage=0.8, variant_frac=0.5))]:
        model = bv.synth.make_model(seed=31 + N, **kw)
        b, q, s, _, r = bv.synth_fill_host(model, 0, S, N)
        engine.set_params(min_af=maf_of(min_af, N), abs_mode=abs_mode)
        lists = np.tile(np.arange(4, dtype=np.uint8), (S, 1))
        recs, lrt = engine.call_host_lists(b, q, s, r, lists, N)
        label = f"N={N} maf={min_af} mode={abs_mode}"
        for f in ("n_alt", "n_active"):
            assert (lrt[f] == recs[f]).all(), f"{label}: {f} differs at {np.nonzero(lrt[f] != recs[f])[0][:10]}"
        assert (lrt["alt"] == recs["alt"]).all(), label
        assert same_f64(lrt["fs"], recs["fs_vcf"]).all(), f"{label}: fs differs at {np.nonzero(~same_f64(lrt['fs'], recs['fs_vcf']))[0][:10]}"
        bound = (recs["flags"] & capi.FLAG_LRT_BOUND) != 0
        d_em = np.nonzero(~bound & (lrt["em_calls"] != recs["em_calls"]))[0]
        assert len(d_em) == 0, f"{label}: em_calls differs at {d_em[:10]}"
        live = np.arange(4)[None, :] < recs["n_alt"][:, None]
        same = (same_f64(lrt["af"], recs["af"]) | ~live).all(axis=1) & same_f64(lrt["qual"], recs["qual"])
        same &= bound | same_f64(lrt["chi2"], recs["chi2"])
        diff = np.nonzero(~same)[0]
        one_em = recs["em_calls"] <= 1
        assert not one_em[diff].any(), f"{label}: a site decided by at most one EM differs: {diff[one_em[diff]][:10]}"
        close = (util.close(lrt["af"], recs["af"]) | ~live).all(axis=1) & util.close(lrt["qual"], recs["qual"])
        close &= bound | util.close(lrt["chi2"], recs["chi2"], atol=1e-9)
        assert close[diff].all(), f"{label}: beyond tolerance at {diff[~close[diff]][:10]}"
        if len(diff):
            rel = np.abs(lrt["chi2"][diff] - recs["chi2"][diff]) / np.maximum(np.abs(recs["chi2"][diff]), 1e-300)
            print(f"acgt-vs-record {label}: {len(diff)} of {int((recs['em_calls'] > 1).sum())} multi-EM sites not bit-identical "
                  f"(max rel chi2 diff {rel.max():.2e}), sites {diff[:20].tolist()}")


@pytest.mark.parametrize("abs_mode", [0, 1])
def test_ref_alt_lists_equal_the_group_kernel(engine, abs_mode):
    """[REF, ALT...] at the called sites with one group of every sample: K6's bv_group_out, bit for bit."""
    for (S, N, kw) in [(4000, 1000, dict(coverage=0.1, variant_frac=0.2, multi_frac=0.3)),
                       (400, 2000, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
                       (150, 3000, None)]:   # util.binned_tile: rows of more than 160 bins (K6's and K8's spill rows)
        if kw is None:
            rng = np.random.default_rng(abs_mode)
            b, q, s, r = util.binned_tile(rng, util.deep_shape(rng, S, N, 0.01), N, 0.01)
            mapq, rpr = util.random_aux(rng, b, N)
        else:
            model = bv.synth.make_model(seed=5 + N, **kw)
            b, q, s, mapq, r = bv.synth_fill_host(model, 0, S, N, with_mapq=True)
            rpr = bv.synth_fill_rpr_host(model, 0, S, N)
        engine.set_params(min_af=0.01, abs_mode=abs_mode)
        engine.set_groups(np.zeros(N, np.uint8), 1)
        recs, calls, groups = engine.call_host_calls(b, q, s, r, mapq, rpr, N)
        engine.set_groups(None, 0)
        lists = np.full((S, 4), capi.LIST_END, np.uint8)
        for k, site in enumerate(calls["site"]):
            order = L._group_order(int(r[site]), recs[site])
            lists[site, :len(order)] = order
        recs2, lrt = engine.call_host_lists(b, q, s, r, lists, N)
        assert recs2.tobytes() == recs.tobytes()
        got = lrt[calls["site"]]
        g = groups[:, 0]
        assert len(g) > 50
        assert (got["n_alt"] == g["n_alt"]).all() and (got["alt"] == g["alt"]).all()
        assert same_f64(got["af"], g["af"]).all()
        lrt_flags = capi.FLAG_ZERO_SUBSET | capi.FLAG_NEAR_LRT | capi.FLAG_LRT_TIE | capi.FLAG_EM_MAXITER | capi.FLAG_BAD_QUAL
        assert ((got["flags"] & lrt_flags) == (g["flags"] & lrt_flags)).all()
        if kw is None:
            assert (util.bin_counts(b, q, N)[calls["site"]] > 160).all()
        uncalled = np.setdiff1d(np.arange(S), calls["site"])
        assert lrt[uncalled].tobytes() == bytes(64 * len(uncalled))


def test_lists_records_skips_refusals_and_launches(engine):
    rng = np.random.default_rng(5)
    S, N = 3000, 500
    b, q, s, r = util.random_tile(rng, S, N, 0.3, 5, 40)
    engine.set_params(min_af=0.01, abs_mode=0)
    lists = random_lists(rng, S)
    lists[rng.random(S) < 0.3] = capi.LIST_END
    l0 = engine.launch_count
    plain = engine.call_host(b, q, s, r, N)
    l1 = engine.launch_count
    recs, lrt = engine.call_host_lists(b, q, s, r, lists, N)
    l2 = engine.launch_count
    assert recs.tobytes() == plain.tobytes()
    tiles = (S + 2047) // 2048
    assert l1 - l0 == 7 * tiles and l2 - l1 == 8 * tiles, (l1 - l0, l2 - l1)
    empty = np.all(lists == capi.LIST_END, axis=1)
    assert lrt[empty].tobytes() == bytes(64 * int(empty.sum())) and empty.sum() > 100
    uncovered = recs["depth"].sum(axis=1) + recs["depth_other"] == 0
    assert lrt[uncovered].tobytes() == bytes(64 * int(uncovered.sum()))
    # refused: repeated base, code > 3 -- BV_ERR_ARG at submit, the slot stays usable
    lib, ctx = engine.lib, engine._ctx
    t = capi.BvTile(b.ctypes.data, q.ctypes.data, s.ctypes.data, r.ctypes.data, b.shape[1], 100, N, capi.BV_LOC_HOST, 0)
    for bad in ([1, 1, 255, 255], [0, 4, 255, 255], [2, 9, 255, 255], [3, 0, 1, 0]):
        bl = lists[:100].copy()
        bl[37] = bad
        l3 = engine.launch_count
        assert lib.bv_tile_submit_lists(ctx, 0, C.byref(t), bl.ctypes.data) == -1
        assert engine.launch_count == l3
    out = np.zeros(100, capi.SITE_OUT_DTYPE)
    lo = np.zeros(100, capi.LRT_OUT_DTYPE)
    assert lib.bv_tile_submit_lists(ctx, 0, C.byref(t), lists[:100].ctypes.data) == 0
    assert lib.bv_tile_wait_lists(ctx, 0, out.ctypes.data, lo.ctypes.data) == 0
    assert out.tobytes() == plain[:100].tobytes() and lo.tobytes() == lrt[:100].tobytes()
    # profiling event of K8
    engine.set_profiling(True)
    engine.call_host_lists(b, q, s, r, lists, N)
    assert engine.last_list_kernel_time() > 0
    engine.set_profiling(False)


def test_lists_device_resident_equals_host_path(engine):
    import torch
    N, S, pitch = 1000, 2000, 1008
    model = bv.synth.make_model(seed=8, coverage=0.1, variant_frac=0.3, multi_frac=0.3)
    engine.synth_set_model(model)
    engine.set_params(min_af=0.01, abs_mode=0)
    dev = torch.device("cuda:0")
    planes = [torch.empty((S, pitch), dtype=torch.uint8, device=dev) for _ in range(3)]
    ref = torch.empty(S, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    engine.synth_fill_device(0, S, N, pitch, planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), None, ref.data_ptr(), st)
    hb, hq, hs, _, hr = bv.synth_fill_host(model, 0, S, N, pitch)
    lists = random_lists(np.random.default_rng(3), S)
    d_lists = torch.from_numpy(lists).to(dev)
    d_out = torch.zeros(S * 128, dtype=torch.uint8, device=dev)
    d_lrt = torch.zeros(S * 64, dtype=torch.uint8, device=dev)
    l0 = engine.launch_count
    engine.call_device_lists(planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), ref.data_ptr(), d_lists.data_ptr(),
                             S, N, pitch, d_out.data_ptr(), d_lrt.data_ptr(), st)
    torch.cuda.synchronize()
    assert engine.launch_count - l0 == 8
    recs_h, lrt_h = engine.call_host_lists(hb, hq, hs, hr, lists, N)
    assert d_out.cpu().numpy().tobytes() == recs_h.tobytes()
    assert d_lrt.cpu().numpy().tobytes() == lrt_h.tobytes()
    assert (lrt_h["n_alt"] > 0).sum() > 100
