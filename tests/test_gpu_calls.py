"""-m gpu: the called-site kernels (K5 rank sums, K6 population groups) through the C ABI against the CPU oracle and
against the committed outputs of the compiled reference (tests/golden/calls_*.npz).
Rank sums are integers and must be bit-exact; group ALT lists exact, group AFs within util.RTOL."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import util

pytestmark = pytest.mark.gpu
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def engine(built_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=20000, max_sites=2048, n_slots=3, min_af=0.01)
    yield eng
    eng.close()


def _soft_sites(recs):
    return set(np.nonzero((recs["flags"] & (capi.FLAG_NEAR_LRT | capi.FLAG_LRT_TIE)) != 0)[0].tolist())


def _run_and_check(engine, b, q, s, r, mapq, rpr, N, grp, G, maf, abs_mode, label, pin_flips=False):
    """pin_flips: the records' listed flips are held to tests/golden/flips_r02.json under `label` (util.report_flips)."""
    engine.set_params(min_af=maf, abs_mode=abs_mode)
    engine.set_groups(grp, G)
    recs, calls, groups = engine.call_host_calls(b, q, s, r, mapq, rpr, N)
    want_recs = L.oracle_tile(b, q, s, r, N, maf, abs_mode)
    ie, fe, flips = util.compare_records(recs, want_recs)
    assert len(ie) == 0 and len(fe) == 0, f"{label}: records differ at {ie[:5]} / {fe[:5]}"
    if pin_flips:
        util.report_flips(label, recs, want_recs, flips)
    # every called site is listed exactly once
    assert np.array_equal(calls["site"], np.nonzero(recs["n_alt"] > 0)[0]), label
    # the oracle's called-site outputs for OUR call set (so that a listed tie flip does not cascade)
    want_calls, want_groups = L.oracle_calls(b, q, mapq, rpr, r, N, recs, grp, G, maf, abs_mode)
    bad = util.compare_calls(calls, groups, want_calls, want_groups)
    soft = _soft_sites(recs)
    bad = [x for x in bad if not (x[0].startswith("group") and int(calls["site"][x[1][0]]) in soft)]
    assert not bad, f"{label}: {len(bad)} mismatches, first {bad[:5]}"
    return recs, calls, groups


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN_DIR, "calls_*.npz"))), ids=os.path.basename)
@pytest.mark.parametrize("abs_mode", [0, 1])
def test_calls_match_reference_fixture(engine, path, abs_mode):
    z = np.load(path)
    N, G, maf = int(z["n_samples"]), int(z["n_groups"]), float(z["min_af"])
    key = "int" if abs_mode == 0 else "dbl"
    recs, calls, groups = _run_and_check(engine, z["base"], z["qual"], z["strand"], z["ref_base"], z["mapq"], z["rpr"], N,
                                         z["sample_group"], G, maf, abs_mode, os.path.basename(path))
    # and against what the compiled reference itself produced
    want_calls = z["calls_" + key].view(L.CALL_OUT_DTYPE)
    want_groups = z["groups_" + key].view(L.GROUP_OUT_DTYPE).reshape(len(want_calls), G)
    want_recs = z["recs_" + key].view(L.SITE_OUT_DTYPE)
    same_set = np.array_equal(recs["n_alt"], want_recs["n_alt"]) and np.array_equal(recs["alt"], want_recs["alt"])
    if same_set:
        bad = util.compare_calls(calls, groups, want_calls, want_groups)
        soft = _soft_sites(recs)
        bad = [x for x in bad if not (x[0].startswith("group") and int(calls["site"][x[1][0]]) in soft)]
        assert not bad, bad[:5]
    else:   # only listed threshold / tie flips may change the call set
        diff = np.nonzero((recs["n_alt"] != want_recs["n_alt"]) | (recs["alt"] != want_recs["alt"]).any(axis=1))[0]
        assert set(diff.tolist()) <= _soft_sites(recs), diff


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize(
    "name,S,N,G,kw",
    [
        ("C2-like", 12000, 1000, 4, dict(coverage=0.1, variant_frac=0.1)),
        ("C1-like-N100", 6000, 100, 2, dict(coverage=0.065, variant_frac=0.2)),
        ("C3-like", 800, 10000, 30, dict(coverage=0.1, variant_frac=0.2)),
        ("C5-like", 600, 2000, 3, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
        ("odd-N", 2000, 1003, 5, dict(coverage=0.3, variant_frac=0.3, multi_frac=0.5)),
        ("tiny-N", 2000, 7, 2, dict(coverage=0.8, variant_frac=0.5)),
        ("deep-wide-phred", 120, 3000, 1, None),   # util.binned_tile: rows of more than 160 bins (K6's spill rows)
    ],
)
def test_calls_synthetic(engine, name, S, N, G, kw, abs_mode):
    maf = bv.cli_min_af(0.01, N)
    if kw is None:
        rng = np.random.default_rng(S + abs_mode)
        b, q, s, r = util.binned_tile(rng, util.deep_shape(rng, S, N, maf), N, maf)
        mapq, rpr = util.random_aux(rng, b, N)
    else:
        model = bv.synth.make_model(seed=4321 + N, **kw)
        b, q, s, mapq, r = bv.synth_fill_host(model, 0, S, N, with_mapq=True)
        rpr = bv.synth_fill_rpr_host(model, 0, S, N)
    rng = np.random.default_rng(N)
    grp = util.random_groups(rng, N, G)
    recs, calls, groups = _run_and_check(engine, b, q, s, r, mapq, rpr, N, grp, G, maf, abs_mode, f"calls {name} abs={abs_mode}",
                                         pin_flips=kw is None)
    assert len(calls) > 0
    if kw is None:   # the one group's rows (90 % of the samples) still pass kSmemBins at most called sites
        g0 = np.nonzero(grp == 0)[0]
        deep = util.bin_counts(b[:, g0], q[:, g0], len(g0))[calls["site"]] > 160
        assert deep.sum() > len(calls) // 2 and len(calls) > 50


def test_calls_pinned_planes_zero_copy_and_no_groups(engine):
    """Pinned aux planes are read in place (no upload); results equal the pageable path.  No groups: K6 is off."""
    import torch
    rng = np.random.default_rng(11)
    S, N = 3000, 500
    b, q, s, r = util.random_tile(rng, S, N, 0.3, 5, 40)
    mapq, rpr = util.random_aux(rng, b, N, 150)
    engine.set_params(min_af=0.01, abs_mode=0)
    engine.set_groups(None, 0)
    before = engine.h2d_bytes
    recs0, calls0, groups0 = engine.call_host_calls(b, q, s, r, mapq, rpr, N)
    pageable_bytes = engine.h2d_bytes - before
    assert groups0.shape == (len(calls0), 0)
    pinned = [torch.from_numpy(a).pin_memory() for a in (b, q, s, mapq)] + [torch.from_numpy(rpr.view(np.int16)).pin_memory()]
    pb, pq, ps, pm = (t.numpy() for t in pinned[:4])
    pr = pinned[4].numpy().view(np.uint16)
    before = engine.h2d_bytes
    recs1, calls1, _ = engine.call_host_calls(pb, pq, ps, r, pm, pr, N)
    pinned_bytes = engine.h2d_bytes - before
    assert recs0.tobytes() == recs1.tobytes() and calls0.tobytes() == calls1.tobytes()
    assert pinned_bytes < pageable_bytes / 2, (pinned_bytes, pageable_bytes)
    launches = engine.launch_count
    engine.call_host_calls(pb[:100], pq[:100], ps[:100], r[:100], pm[:100], pr[:100], N)
    assert engine.launch_count - launches == 8   # K1..K3, K4a, K4b (two builds, one of them works), Fisher tests + K5


def test_calls_device_resident_equals_host_path(engine):
    import torch
    N, S, pitch = 1000, 2000, 1008
    model = bv.synth.make_model(seed=5, coverage=0.1, variant_frac=0.3, multi_frac=0.3)
    engine.synth_set_model(model)
    engine.set_params(min_af=0.01, abs_mode=0)
    G = 3
    grp = util.random_groups(np.random.default_rng(1), N, G)
    engine.set_groups(grp, G)
    dev = torch.device("cuda:0")
    planes = [torch.empty((S, pitch), dtype=torch.uint8, device=dev) for _ in range(4)]
    d_rpr = torch.empty((S, pitch), dtype=torch.int16, device=dev)
    ref = torch.empty(S, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    lib, ctx = engine.lib, engine._ctx
    engine.synth_fill_device(0, S, N, pitch, planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), planes[3].data_ptr(),
                             ref.data_ptr(), st)
    rc = lib.bv_synth_fill_rpr_device(ctx, 0, S, N, pitch, d_rpr.data_ptr(), C.c_void_p(st))
    assert rc == 0
    torch.cuda.synchronize()
    hb, hq, hs, hm, hr = bv.synth_fill_host(model, 0, S, N, pitch, with_mapq=True)
    hrpr = bv.synth_fill_rpr_host(model, 0, S, N)
    assert np.array_equal(d_rpr.cpu().numpy().view(np.uint16)[:, :hrpr.shape[1]], hrpr)
    d_out = torch.zeros(S * 128, dtype=torch.uint8, device=dev)
    d_calls = torch.zeros(S * 16, dtype=torch.uint8, device=dev)
    d_groups = torch.zeros(S * G * 40, dtype=torch.uint8, device=dev)
    d_n = torch.zeros(1, dtype=torch.int32, device=dev)
    t = capi.BvTile(planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), ref.data_ptr(), pitch, S, N, capi.BV_LOC_DEVICE, 0)
    a = capi.BvTileAux(planes[3].data_ptr(), d_rpr.data_ptr(), pitch)
    rc = lib.bv_tile_run_device_calls(ctx, C.byref(t), C.byref(a), d_out.data_ptr(), d_calls.data_ptr(), d_groups.data_ptr(),
                                      d_n.data_ptr(), C.c_void_p(st))
    assert rc == 0, lib.bv_last_error(ctx)
    torch.cuda.synchronize()
    n = int(d_n.item())
    calls = d_calls.cpu().numpy().view(capi.CALL_OUT_DTYPE)[:n]
    groups = d_groups.cpu().numpy().view(capi.GROUP_OUT_DTYPE)[:n * G].reshape(n, G)
    order = np.argsort(calls["site"])
    recs_h, calls_h, groups_h = engine.call_host_calls(hb, hq, hs, hr, hm, hrpr, N)
    assert d_out.cpu().numpy().view(capi.SITE_OUT_DTYPE).tobytes() == recs_h.tobytes()
    assert calls[order].tobytes() == calls_h.tobytes()
    assert groups[order].tobytes() == groups_h.tobytes()
    assert n == int((recs_h["n_alt"] > 0).sum()) and n > 100
