"""-m gpu: the VCF row's batch outputs on the transport meant for production -- sparse cells in, compact records out.
  1. compact results with the called-site kernels (bv_tile_wait_calls_compact), dense host and sparse tiles in both cell
     formats, both em_abs_modes, with and without groups: the same records, calls and groups as records mode, byte for byte;
  2. lrt(list) on sparse tiles (bv_tile_submit_sparse_lists): records and bv_lrt_out equal to the dense bv_tile_submit_lists,
     and the packed compact output (bv_tile_wait_lists_compact) equal to the full output at the listed sites;
  3. empty tiles, tiles without lists, malformed cells, refusals, launch counts of every entry point, kernel timing."""
import ctypes as C

import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import util

pytestmark = pytest.mark.gpu
SHAPES = {
    "C2-like": (6000, 1000, dict(coverage=0.1, variant_frac=0.1)),
    "C5-like": (600, 2000, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
}


@pytest.fixture(scope="module")
def engine(built_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=4000, max_sites=2048, n_slots=3, min_af=0.01)
    yield eng
    eng.close()


def synth(name, seed=0):
    S, N, kw = SHAPES[name]
    model = bv.synth.make_model(seed=9000 + N + seed, **kw)
    b, q, s, mapq, r = bv.synth_fill_host(model, 0, S, N, with_mapq=True)
    rpr = bv.synth_fill_rpr_host(model, 0, S, N)
    cells, aux, st, ref = bv.synth_fill_sparse_host(model, 0, S, N, with_aux=True)
    assert np.array_equal(ref, r)
    return dict(S=S, N=N, b=b, q=q, s=s, mapq=mapq, rpr=rpr, r=r, cells=cells, aux=aux, st=st)


def cells_of(d, fmt):
    if fmt == "u32":
        return d["cells"], d["aux"], d["st"]
    return bv.sparse_encode16(d["cells"], d["st"], d["aux"])


def run_calls(engine, d, transport, compact):
    if transport == "dense":
        return engine.call_host_calls(d["b"], d["q"], d["s"], d["r"], d["mapq"], d["rpr"], d["N"], compact=compact)
    cells, aux, st = cells_of(d, transport)
    return engine.call_sparse_calls(cells, aux, st, d["r"], d["N"], compact=compact)


@pytest.mark.parametrize("groups", [0, 3])
@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("transport", ["dense", "u32", "u16"])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_compact_calls_equal_records_mode(engine, name, transport, abs_mode, groups):
    d = synth(name)
    engine.set_params(min_af=bv.cli_min_af(0.01, d["N"]), abs_mode=abs_mode)
    engine.set_groups(util.random_groups(np.random.default_rng(d["N"]), d["N"], groups) if groups else None, groups)
    recs0, calls0, groups0 = run_calls(engine, d, transport, False)
    recs1, calls1, groups1 = run_calls(engine, d, transport, True)
    engine.set_groups(None, 0)
    assert recs1.tobytes() == recs0.tobytes()
    assert len(calls1) == len(calls0) > 10
    assert calls1.tobytes() == calls0.tobytes() and groups1.tobytes() == groups0.tobytes()
    assert groups1.shape == (len(calls1), groups)
    assert np.array_equal(calls1["site"], np.nonzero(recs1["n_alt"] > 0)[0])
    tiles = engine.compact_tiles
    assert len(tiles) == (d["S"] + 2047) // 2048
    assert all(n_full == n_bit31 for n_full, n_bit31 in tiles), tiles
    assert len(calls1) <= sum(t[0] for t in tiles) < d["S"]   # a called site always travels as a full record


def ref_alt_lists(recs, r):
    """[REF, ALT...] at the called sites (the -G path's lists), empty elsewhere."""
    lists = np.full((len(recs), 4), capi.LIST_END, np.uint8)
    for site in np.nonzero(recs["n_alt"] > 0)[0]:
        order = L._group_order(int(r[site]), recs[site])
        lists[site, :len(order)] = order
    return lists


def mixed_lists(rng, S):
    """Random orders of random subsets, a third of them empty, some ended after one or two entries."""
    lists = np.full((S, 4), capi.LIST_END, np.uint8)
    for s in range(S):
        k = int(rng.integers(0, 5))
        lists[s, :k] = rng.permutation(4)[:k]
    return lists


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("fmt", ["u32", "u16"])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_sparse_lists_equal_the_dense_lists(engine, name, fmt, abs_mode):
    d = synth(name, seed=1)
    S, N = d["S"], d["N"]
    engine.set_params(min_af=bv.cli_min_af(0.01, N), abs_mode=abs_mode)
    plain = engine.call_host(d["b"], d["q"], d["s"], d["r"], N)
    cells, _, st = cells_of(d, fmt)
    for label, lists in [("ACGT", np.tile(np.arange(4, dtype=np.uint8), (S, 1))), ("REF+ALT", ref_alt_lists(plain, d["r"])),
                         ("mixed", mixed_lists(np.random.default_rng(S + abs_mode), S))]:
        recs_d, lrt_d = engine.call_host_lists(d["b"], d["q"], d["s"], d["r"], lists, N)
        recs_s, lrt_s = engine.call_sparse_lists(cells, st, d["r"], lists, N)
        assert recs_s.tobytes() == recs_d.tobytes() == plain.tobytes(), label
        assert lrt_s.tobytes() == lrt_d.tobytes(), label
        recs_c, lrt_c = engine.call_sparse_lists(cells, st, d["r"], lists, N, compact=True)
        listed = lists[:, 0] != capi.LIST_END
        assert recs_c.tobytes() == plain.tobytes(), label
        assert len(lrt_c) == int(listed.sum()) and lrt_c.tobytes() == lrt_d[listed].tobytes(), label
        assert all(n_full == n_bit31 for n_full, n_bit31 in engine.compact_tiles)
        if label == "REF+ALT":
            assert (lrt_c["n_alt"] > 0).sum() > 10


def sparse_tile(cells, st, ref, n_sites, n_samples, out_mode, fmt=capi.CELLS_U32):
    return capi.BvSparseTile(cells.ctypes.data, None, st.ctypes.data, ref.ctypes.data, None, n_sites, n_samples, fmt, out_mode)


def test_sparse_lists_empty_tiles_no_lists_and_malformed_cells(engine):
    d = synth("C2-like", seed=2)
    N = d["N"]
    engine.set_params(min_af=0.01, abs_mode=0)
    lib, ctx = engine.lib, engine._ctx
    # empty tile: nothing comes back, as for bv_tile_submit_lists
    for compact in (False, True):
        recs, lrt = engine.call_sparse_lists(d["cells"][:0], np.zeros(1, np.uint32), d["r"][:0], np.zeros((0, 4), np.uint8), N,
                                             compact=compact)
        assert len(recs) == 0 and len(lrt) == 0
    # a tile without lists: all-zero entries (records mode) / none at all (compact), and no K8 launch
    S = 1500
    cells, st = d["cells"][:int(d["st"][S])], d["st"][:S + 1].copy()
    none = np.full((S, 4), capi.LIST_END, np.uint8)
    plain = engine.call_sparse(cells, st, d["r"][:S], N)
    l0 = engine.launch_count
    recs, lrt = engine.call_sparse_lists(cells, st, d["r"][:S], none, N)
    assert engine.launch_count - l0 == 9   # K0, the seven of a tile, K8
    assert recs.tobytes() == plain.tobytes() and lrt.tobytes() == bytes(64 * S)
    l0 = engine.launch_count
    recs, lrt = engine.call_sparse_lists(cells, st, d["r"][:S], none, N, compact=True)
    assert engine.launch_count - l0 == 9   # K0, the seven, K7 (nothing listed: no K8)
    assert recs.tobytes() == plain.tobytes() and len(lrt) == 0
    # malformed cells (a sample >= n_samples): BV_ERR_ARG at the wait, in both result forms; the slot then runs a normal tile
    bad = cells.copy()
    bad[17] = capi.cell_pack(N + 3, 0, 0, 30)
    lists = mixed_lists(np.random.default_rng(1), S)
    lo = np.zeros(S, capi.LRT_OUT_DTYPE)
    for mode in (capi.OUT_RECORDS, capi.OUT_COMPACT):
        t = sparse_tile(bad, st, d["r"], S, N, mode)
        assert lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), lists.ctypes.data) == 0
        if mode == capi.OUT_RECORDS:
            rc = lib.bv_tile_wait_lists(ctx, 0, None, lo.ctypes.data)
        else:
            pb, pf, nf, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0), C.c_uint32(0)
            rc = lib.bv_tile_wait_lists_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), lo.ctypes.data, S, C.byref(n))
        assert rc == -1 and b"sparse tile" in lib.bv_last_error(ctx)
    recs, lrt = engine.call_sparse_lists(cells, st, d["r"][:S], lists, N)
    recs_d, lrt_d = engine.call_host_lists(d["b"][:S], d["q"][:S], d["s"][:S], d["r"][:S], lists, N)
    assert recs.tobytes() == recs_d.tobytes() and lrt.tobytes() == lrt_d.tobytes()


def test_refusals_leave_the_slot_usable(engine):
    d = synth("C2-like", seed=3)
    N, S = d["N"], 800
    engine.set_params(min_af=0.01, abs_mode=0)
    lib, ctx = engine.lib, engine._ctx
    cells, st, r = d["cells"][:int(d["st"][S])], d["st"][:S + 1].copy(), d["r"][:S].copy()
    lists = mixed_lists(np.random.default_rng(4), S)
    want_recs, want_lrt = engine.call_sparse_lists(cells, st, r, lists, N)
    # a repeated base, a code above 3: refused at submit, nothing launched, in both result forms
    for mode in (capi.OUT_RECORDS, capi.OUT_COMPACT):
        t = sparse_tile(cells, st, r, S, N, mode)
        for bad in ([1, 1, 255, 255], [0, 4, 255, 255], [3, 0, 1, 0]):
            bl = lists.copy()
            bl[37] = bad
            l0 = engine.launch_count
            assert lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), bl.ctypes.data) == -1
            assert engine.launch_count == l0
    # lists and the called-site outputs do not come from one submit: the calls waits refuse a lists slot
    t = sparse_tile(cells, st, r, S, N, capi.OUT_RECORDS)
    assert lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), lists.ctypes.data) == 0
    n = C.c_uint32(0)
    assert lib.bv_tile_wait_calls(ctx, 0, None, None, 0, C.byref(n), None) == -3
    pb, pf, nf = C.c_void_p(), C.c_void_p(), C.c_uint32(0)
    assert lib.bv_tile_wait_calls_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), None, 0, C.byref(n), None) == -3
    assert lib.bv_tile_wait_lists_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), None, 0, C.byref(n)) == -3
    out = np.zeros(S, capi.SITE_OUT_DTYPE)
    lo = np.zeros(S, capi.LRT_OUT_DTYPE)
    assert lib.bv_tile_wait_lists(ctx, 0, out.ctypes.data, lo.ctypes.data) == 0
    assert out.tobytes() == want_recs.tobytes() and lo.tobytes() == want_lrt.tobytes()
    # a compact lists slot is collected by its own wait
    t = sparse_tile(cells, st, r, S, N, capi.OUT_COMPACT)
    assert lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), lists.ctypes.data) == 0
    assert lib.bv_tile_wait_lists(ctx, 0, None, lo.ctypes.data) == -3
    assert lib.bv_tile_wait_lists_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), lo.ctypes.data, 3, C.byref(n)) == -1
    assert n.value == int((lists[:, 0] != capi.LIST_END).sum()) > 3   # max_lrt too small: BV_ERR_ARG, nothing copied
    # device-resident tiles have no compact form
    t = capi.BvTile(1 << 20, 1 << 20, 1 << 20, 1 << 20, 1008, 10, N, capi.BV_LOC_DEVICE, capi.OUT_COMPACT)
    a = capi.BvTileAux(1 << 20, 1 << 20, 1008)
    l0 = engine.launch_count
    assert lib.bv_tile_run_device_calls(ctx, C.byref(t), C.byref(a), C.c_void_p(1 << 20), C.c_void_p(1 << 20), None,
                                        C.c_void_p(1 << 20), None) == -1
    assert lib.bv_tile_run_device_lists(ctx, C.byref(t), C.c_void_p(1 << 20), C.c_void_p(1 << 20), C.c_void_p(1 << 20), None) == -1
    assert lib.bv_tile_submit_calls(ctx, 0, C.byref(t), C.byref(a)) == -1
    assert engine.launch_count == l0
    # and the same slot then runs a normal tile to the same records
    recs, lrt = engine.call_sparse_lists(cells, st, r, lists, N)
    assert recs.tobytes() == want_recs.tobytes() and lrt.tobytes() == want_lrt.tobytes()


def test_launch_counts_and_timing(engine):
    """Launches per tile of every entry point (abs mode 0, one tile with reads): the existing ones as before, the new forms
    one kernel more per added stage (K7 for compact results, K8 for lists)."""
    d = synth("C2-like", seed=4)
    N, S = d["N"], 1000
    engine.set_params(min_af=0.01, abs_mode=0)
    b, q, s, mq, rp, r = (d[k][:S] for k in ("b", "q", "s", "mapq", "rpr", "r"))
    cells, aux, st = d["cells"][:int(d["st"][S])], d["aux"][:int(d["st"][S])], d["st"][:S + 1].copy()
    lists = ref_alt_lists(engine.call_host(b, q, s, r, N), r)

    def count(fn):
        l0 = engine.launch_count
        fn()
        return engine.launch_count - l0

    grp = util.random_groups(np.random.default_rng(2), N, 2)
    assert count(lambda: engine.call_host(b, q, s, r, N)) == 7
    assert count(lambda: engine.call_sparse(cells, st, r, N)) == 8
    assert count(lambda: engine.call_host_lists(b, q, s, r, lists, N)) == 8
    assert count(lambda: engine.call_host_calls(b, q, s, r, mq, rp, N)) == 8
    assert count(lambda: engine.call_sparse_calls(cells, aux, st, r, N)) == 9
    tiles = engine.sparse_tiles(cells, st, r, N, compact=True)
    assert count(lambda: engine.run_sparse_tiles(tiles, compact=None)) == 9
    assert count(lambda: engine.call_host_calls(b, q, s, r, mq, rp, N, compact=True)) == 9
    assert count(lambda: engine.call_sparse_calls(cells, aux, st, r, N, compact=True)) == 10
    assert count(lambda: engine.call_sparse_lists(cells, st, r, lists, N)) == 9
    assert count(lambda: engine.call_sparse_lists(cells, st, r, lists, N, compact=True)) == 10
    engine.set_groups(grp, 2)
    assert count(lambda: engine.call_host_calls(b, q, s, r, mq, rp, N)) == 9
    assert count(lambda: engine.call_sparse_calls(cells, aux, st, r, N)) == 10
    assert count(lambda: engine.call_sparse_calls(cells, aux, st, r, N, compact=True)) == 11
    # kernel timing covers the new paths
    engine.set_profiling(True)
    engine.call_sparse_calls(cells, aux, st, r, N, compact=True)
    t = engine.last_call_kernel_times()
    assert t["bv_ranksum_kernel"] > 0 and t["bv_group_kernel"] > 0
    engine.call_sparse_lists(cells, st, r, lists, N, compact=True)
    assert engine.last_list_kernel_time() > 0
    engine.set_profiling(False)
    engine.set_groups(None, 0)
