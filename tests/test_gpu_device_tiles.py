"""-m gpu: pileups held in device memory, every result form (bv_tile_run_device_sparse / bv_tile_run_device_ex with a
bv_device_out), held byte for byte to the host route of the same cells (bv_tile_submit_sparse* + bv_tile_wait*).

The host route is the yardstick: records, called sites and lists of a device tile must be the bytes the host entry points give.
Two things are free by design and are put in a canonical order before the comparison: the order of the full records of a
compact tile (K7 appends them with atomics; the briefs point into the list, so the records they stand for are compared), and
the order of the called sites (bv_call_out::site names the row)."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import basevar_b200 as bv
from basevar_b200 import capi

pytestmark = pytest.mark.gpu

MAX_SITES = 3000
MAX_SAMPLES = 100000
SHAPES = {7: 3000, 1000: 3000, 10000: 600, 100000: 148}   # sites per tile; 148 x 100,000: one tile of the C4 shard shape


@pytest.fixture(scope="module")
def engine(built_lib):
    eng = bv.BaseTypeEngine(device=0, max_samples=MAX_SAMPLES, max_sites=MAX_SITES, n_slots=1,
                            min_af=bv.cli_min_af(0.01, 1000))
    yield eng
    eng.close()


@functools.lru_cache(maxsize=8)
def _tile(N, coverage, S=None):
    S = SHAPES[N] if S is None else S
    model = bv.synth.make_model(seed=1000 + N + int(coverage * 1000), coverage=coverage, variant_frac=0.1, multi_frac=0.2)
    cells, aux, st, ref = bv.synth_fill_sparse_host(model, 0, S, N, with_aux=True)
    words, aux16, st16 = bv.sparse_encode16(cells, st, aux)
    return {capi.CELLS_U32: (cells, aux, st), capi.CELLS_U16: (words, aux16, st16)}, ref


def _lists(S, seed, refused=True):
    """Per-site candidate lists: empty, valid (1..4 distinct bases in random order) and, with `refused`, a few the host entry
    points refuse (a repeated base, a code above 3).  Returns (lists as given, lists with the refused ones emptied)."""
    rng = np.random.default_rng(seed)
    lists = np.full((S, 4), capi.LIST_END, np.uint8)
    for i in range(S):
        k = int(rng.integers(0, 5))
        lists[i, :k] = rng.permutation(4)[:k]
    host = lists.copy()
    if refused and S >= 8:
        bad = rng.choice(S, size=max(2, S // 50), replace=False)
        for j, i in enumerate(bad):
            lists[i] = (1, 1, capi.LIST_END, capi.LIST_END) if j % 2 else (0, 7, capi.LIST_END, capi.LIST_END)
            host[i] = capi.LIST_END
    return lists, host


def _check(eng, rc, what):
    assert rc == capi.BV_OK, f"{what} failed ({rc}): {eng.lib.bv_last_error(eng._ctx).decode()}"


def _views(pb, pf, nf, S):
    briefs = np.ctypeslib.as_array(C.cast(pb, C.POINTER(C.c_uint32)), shape=(S * 2,)).view(capi.SITE_BRIEF_DTYPE).copy() if S else \
        np.zeros(0, capi.SITE_BRIEF_DTYPE)
    full = (np.ctypeslib.as_array(C.cast(pf, C.POINTER(C.c_uint8)), shape=(nf * 128,)).view(capi.SITE_OUT_DTYPE).copy()
            if nf else np.zeros(0, capi.SITE_OUT_DTYPE))
    return briefs, full


def host_route(eng, cells, aux, st, ref, N, fmt, kind, compact, lists=None):
    """The same cells through the slot of a host tile; the results in the form DeviceResult.to_numpy gives them."""
    lib, ctx = eng.lib, eng._ctx
    S = len(ref)
    t = capi.BvSparseTile(cells.ctypes.data, aux.ctypes.data if kind == "calls" else None, st.ctypes.data, ref.ctypes.data, None, S, N,
                          fmt, capi.OUT_COMPACT if compact else capi.OUT_RECORDS)
    if kind == "calls":
        _check(eng, lib.bv_tile_submit_sparse_calls(ctx, 0, C.byref(t)), "bv_tile_submit_sparse_calls")
    elif kind == "lists":
        _check(eng, lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), lists.ctypes.data), "bv_tile_submit_sparse_lists")
    else:
        _check(eng, lib.bv_tile_submit_sparse(ctx, 0, C.byref(t)), "bv_tile_submit_sparse")
    r = {"status": 0}
    pb, pf, nf, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0), C.c_uint32(0)
    out = np.zeros(S, capi.SITE_OUT_DTYPE)
    ng = getattr(eng, "n_groups", 0)
    if kind == "calls":
        calls = np.zeros(max(S, 1), capi.CALL_OUT_DTYPE)
        groups = np.zeros(max(S * ng, 1), capi.GROUP_OUT_DTYPE)
        if compact:
            _check(eng, lib.bv_tile_wait_calls_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), calls.ctypes.data, S, C.byref(n),
                                                       groups.ctypes.data if ng else None), "bv_tile_wait_calls_compact")
        else:
            _check(eng, lib.bv_tile_wait_calls(ctx, 0, out.ctypes.data, calls.ctypes.data, S, C.byref(n),
                                               groups.ctypes.data if ng else None), "bv_tile_wait_calls")
        r["calls"] = calls[:n.value]
        r["groups"] = groups[:n.value * ng] if ng else None
    elif kind == "lists":
        lrt = np.zeros(max(S, 1), capi.LRT_OUT_DTYPE)
        if compact:
            _check(eng, lib.bv_tile_wait_lists_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), lrt.ctypes.data, S, C.byref(n)),
                   "bv_tile_wait_lists_compact")
            r["lrt"] = lrt[:n.value]
        else:
            _check(eng, lib.bv_tile_wait_lists(ctx, 0, out.ctypes.data, lrt.ctypes.data), "bv_tile_wait_lists")
            r["lrt"] = lrt[:S]
    elif compact:
        _check(eng, lib.bv_tile_wait_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf)), "bv_tile_wait_compact")
    else:
        _check(eng, lib.bv_tile_wait(ctx, 0, out.ctypes.data), "bv_tile_wait")
    if compact:
        r["brief"], r["full"] = _views(pb, pf, nf.value, S)
    else:
        r["records"] = out
    return r


def canonical(eng, r, ref):
    """Records (compact results expanded through their briefs), called sites sorted by row, everything as bytes."""
    c = {"status": r["status"]}
    if "brief" in r:
        b, full = r["brief"], r["full"]
        is_full = (b["w0"] & 0x80000000) != 0
        assert int(is_full.sum()) == len(full), "every full record is pointed at by one brief"
        assert sorted((b["w0"][is_full] & 0x7fffffff).tolist()) == list(range(len(full)))
        rec = np.zeros(len(b), capi.SITE_OUT_DTYPE)
        eng.expand_compact(b, full, ref, rec)
        c["records"] = rec.tobytes()
        c["is_full"] = is_full.tobytes()
        c["brief_words"] = b[~is_full].tobytes()
    else:
        c["records"] = r["records"].tobytes()
    if r.get("calls") is not None:
        order = np.argsort(r["calls"]["site"], kind="stable")
        c["calls"] = r["calls"][order].tobytes()
        if r.get("groups") is not None:
            ng = len(r["groups"]) // max(len(r["calls"]), 1)
            c["groups"] = r["groups"].reshape(-1, ng)[order].tobytes() if len(r["calls"]) else b""
    if "lrt" in r:
        c["lrt"] = r["lrt"].tobytes()
    return c


def _dev(a):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if t.dtype == torch.uint32:
        t = t.view(torch.int32)
    elif t.dtype == torch.uint16:
        t = t.view(torch.int16)
    return t.cuda()


def poisoned(eng, S, kind, compact):
    """Result tensors filled with 0xee, counts and status included: an entry the device route does not write cannot match the
    host's bytes by chance."""
    out = eng.device_result(S, calls=kind == "calls", lists=kind == "lists", compact=compact)
    for v in vars(out).values():
        if isinstance(v, torch.Tensor) and v.dtype == torch.uint8:
            v.fill_(0xee)
        elif isinstance(v, torch.Tensor):
            v.fill_(-0x11111112)   # 0xeeeeeeee
    return out


def device_route(eng, cells, aux, st, ref, N, kind, compact, lists=None):
    res = eng.call_device_sparse(_dev(cells), _dev(st), _dev(ref), N, cells_aux=_dev(aux) if kind == "calls" else None,
                                 lists=_dev(lists) if kind == "lists" else None, calls=kind == "calls", compact=compact,
                                 out=poisoned(eng, len(ref), kind, compact))
    return res.to_numpy()


def _set_groups(eng, n_groups, N):
    if n_groups:
        eng.set_groups((np.arange(N) % n_groups).astype(np.uint8), n_groups)
    else:
        eng.set_groups(None, 0)


@pytest.mark.parametrize("kind", ["plain", "calls0", "calls3", "lists"])
@pytest.mark.parametrize("compact", [False, True], ids=["records", "compact"])
@pytest.mark.parametrize("fmt", [capi.CELLS_U32, capi.CELLS_U16], ids=["u32", "u16"])
@pytest.mark.parametrize("coverage", [0.1, 0.993])
@pytest.mark.parametrize("N", sorted(SHAPES))
def test_device_sparse_equals_host_route(engine, N, coverage, fmt, compact, kind):
    forms, ref = _tile(N, coverage)
    cells, aux, st = forms[fmt]
    base_kind = "calls" if kind.startswith("calls") else kind
    _set_groups(engine, 3 if kind == "calls3" else 0, N)
    lists = host_lists = None
    if kind == "lists":
        lists, host_lists = _lists(len(ref), seed=N)
    want = canonical(engine, host_route(engine, cells, aux, st, ref, N, fmt, base_kind, compact, host_lists), ref)
    got = canonical(engine, device_route(engine, cells, aux, st, ref, N, base_kind, compact, lists), ref)
    assert got.keys() == want.keys()
    for k in want:
        assert got[k] == want[k], f"N={N} coverage={coverage} {kind} compact={compact}: {k} differs from the host route"
    if kind == "lists" and compact:
        assert len(got["lrt"]) // 64 == int((host_lists[:, 0] != capi.LIST_END).sum())


def _dense_host(eng, b, q, s, r, N, compact, kind="plain", mapq=None, rpr=None, lists=None):
    """Dense host tile through slot 0 (bv_tile_submit / _calls / _lists)."""
    lib, ctx = eng.lib, eng._ctx
    S, pitch = b.shape
    t = capi.BvTile(b.ctypes.data, q.ctypes.data, s.ctypes.data, r.ctypes.data, pitch, S, N, capi.BV_LOC_HOST,
                    capi.OUT_COMPACT if compact else capi.OUT_RECORDS)
    out = np.zeros(S, capi.SITE_OUT_DTYPE)
    res = {"status": 0}
    pb, pf, nf, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0), C.c_uint32(0)
    if kind == "calls":
        aux = capi.BvTileAux(mapq.ctypes.data, rpr.ctypes.data, rpr.shape[1])
        _check(eng, lib.bv_tile_submit_calls(ctx, 0, C.byref(t), C.byref(aux)), "bv_tile_submit_calls")
        calls = np.zeros(max(S, 1), capi.CALL_OUT_DTYPE)
        if compact:
            _check(eng, lib.bv_tile_wait_calls_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), calls.ctypes.data, S, C.byref(n), None),
                   "bv_tile_wait_calls_compact")
        else:
            _check(eng, lib.bv_tile_wait_calls(ctx, 0, out.ctypes.data, calls.ctypes.data, S, C.byref(n), None), "bv_tile_wait_calls")
        res["calls"], res["groups"] = calls[:n.value], None
    elif kind == "lists":
        _check(eng, lib.bv_tile_submit_lists(ctx, 0, C.byref(t), lists.ctypes.data), "bv_tile_submit_lists")
        lrt = np.zeros(S, capi.LRT_OUT_DTYPE)
        _check(eng, lib.bv_tile_wait_lists(ctx, 0, out.ctypes.data, lrt.ctypes.data), "bv_tile_wait_lists")
        res["lrt"] = lrt
    else:
        _check(eng, lib.bv_tile_submit(ctx, 0, C.byref(t)), "bv_tile_submit")
        if compact:
            _check(eng, lib.bv_tile_wait_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf)), "bv_tile_wait_compact")
        else:
            _check(eng, lib.bv_tile_wait(ctx, 0, out.ctypes.data), "bv_tile_wait")
    if compact:
        res["brief"], res["full"] = _views(pb, pf, nf.value, S)
    else:
        res["records"] = out
    return res


@pytest.mark.parametrize("kind", ["plain", "calls", "lists"])
@pytest.mark.parametrize("compact", [False, True], ids=["records", "compact"])
def test_device_dense_ex_equals_host_dense(engine, compact, kind):
    N, S = 1000, 2000
    _set_groups(engine, 0, N)
    model = bv.synth.make_model(seed=77, coverage=0.1, variant_frac=0.2, multi_frac=0.2)
    b, q, s, m, r = bv.synth_fill_host(model, 0, S, N, with_mapq=True)
    rpr = bv.synth_fill_rpr_host(model, 0, S, N)
    lists = host_lists = None
    if kind == "lists":
        lists, host_lists = _lists(S, seed=5)
    if kind == "lists" and compact:
        # the host's compact lists are those of sparse tiles: the same pileup in sparse form
        cells, _, st = bv.dense_to_sparse(b, q, s, N)
        want = host_route(engine, cells, None, st, r, N, capi.CELLS_U32, "lists", True, host_lists)
    else:
        want = _dense_host(engine, b, q, s, r, N, compact, kind, m, rpr, host_lists)
    res = engine.call_device_dense(_dev(b), _dev(q), _dev(s), _dev(r), N, mapq=_dev(m), rpr=_dev(rpr),
                                   lists=_dev(lists) if lists is not None else None, calls=kind == "calls", compact=compact,
                                   out=poisoned(engine, S, kind, compact))
    assert canonical(engine, res.to_numpy(), r) == canonical(engine, want, r)


def test_existing_device_entry_points_still_refuse_compact(engine):
    N, S = 100, 64
    d = torch.zeros((S, 112), dtype=torch.uint8, device="cuda")
    ref = torch.full((S,), ord("A"), dtype=torch.uint8, device="cuda")
    t = capi.BvTile(d.data_ptr(), d.data_ptr(), d.data_ptr(), ref.data_ptr(), 112, S, N, capi.BV_LOC_DEVICE, capi.OUT_COMPACT)
    lists = torch.full((S, 4), capi.LIST_END, dtype=torch.uint8, device="cuda")
    out = torch.empty((S, 128), dtype=torch.uint8, device="cuda")
    lrt = torch.empty((S, 64), dtype=torch.uint8, device="cuda")
    rc = engine.lib.bv_tile_run_device_lists(engine._ctx, C.byref(t), lists.data_ptr(), out.data_ptr(), lrt.data_ptr(), None)
    assert rc == -1


def test_empty_tile_and_empty_sites(engine):
    _set_groups(engine, 0, 10)
    N = 1000
    dev = torch.device("cuda")
    for compact in (False, True):
        for kind in ("plain", "calls", "lists"):
            e32 = torch.zeros(0, dtype=torch.int32, device=dev)
            res = engine.call_device_sparse(e32, torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.uint8, device=dev),
                                            N, cells_aux=e32 if kind == "calls" else None,
                                            lists=torch.zeros((0, 4), dtype=torch.uint8, device=dev) if kind == "lists" else None,
                                            calls=kind == "calls", compact=compact)
            got = res.to_numpy()
            assert got["status"] == 0
            assert len(got.get("records", got.get("brief"))) == 0
            for k in ("calls", "lrt"):
                if k in got:
                    assert len(got[k]) == 0
    # sites without cells among covered ones, and a tile without a single cell
    model = bv.synth.make_model(seed=3, coverage=0.0005, variant_frac=0.1)
    cells, aux, st, ref = bv.synth_fill_sparse_host(model, 0, 500, N, with_aux=True)
    assert (np.diff(st) == 0).sum() > 100
    lists, _ = _lists(500, seed=9, refused=False)
    for compact in (False, True):
        for kind in ("plain", "calls", "lists"):
            want = canonical(engine, host_route(engine, cells, aux, st, ref, N, capi.CELLS_U32, kind, compact, lists), ref)
            got = canonical(engine, device_route(engine, cells, aux, st, ref, N, kind, compact, lists), ref)
            assert got == want, (kind, compact)
    none = np.zeros(0, np.uint32)
    st0 = np.zeros(301, np.uint32)
    ref0 = np.full(300, ord("C"), np.uint8)
    for compact in (False, True):
        want = canonical(engine, host_route(engine, none, None, st0, ref0, N, capi.CELLS_U32, "plain", compact), ref0)
        got = canonical(engine, device_route(engine, none, None, st0, ref0, N, "plain", compact), ref0)
        assert got == want


def test_tile_of_max_sites(engine):
    _set_groups(engine, 0, 10)
    forms, ref = _tile(1000, 0.1)
    assert len(ref) == MAX_SITES
    cells, aux, st = forms[capi.CELLS_U16]
    for compact in (False, True):
        want = canonical(engine, host_route(engine, cells, aux, st, ref, 1000, capi.CELLS_U16, "plain", compact), ref)
        got = canonical(engine, device_route(engine, cells, aux, st, ref, 1000, "plain", compact), ref)
        assert got == want
    # one site more is refused before anything is queued
    more = np.concatenate([st, st[-1:]])
    with pytest.raises(bv.BvError, match="max_sites"):
        engine.call_device_sparse(_dev(cells), _dev(more), _dev(np.concatenate([ref, ref[:1]])), 1000)


def test_malformed_cells_report_status_and_leave_the_context_usable(engine):
    _set_groups(engine, 0, 10)
    N = 1000
    model = bv.synth.make_model(seed=11, coverage=0.1, variant_frac=0.1)
    cells, aux, st, ref = bv.synth_fill_sparse_host(model, 0, 400, N, with_aux=True)
    words, aux16, st16 = bv.sparse_encode16(cells, st, aux)
    # a cell whose sample is >= N
    bad = cells.copy()
    bad[st[10]] = capi.cell_pack(N + 3, 0, 0, 30)
    # offsets that descend (within the cell array)
    desc = st.copy()
    desc[20], desc[21] = st[21] + 2, st[20]
    desc16 = st16.copy()
    desc16[30], desc16[31] = st16[31] + 1, st16[30]
    for compact in (False, True):
        for c, s_, kind in ((bad, st, "plain"), (cells, desc, "calls"), (words, desc16, "lists")):
            lists = _lists(400, seed=1, refused=False)[0] if kind == "lists" else None
            a = aux if c is not words else aux16
            got = device_route(engine, c, a, s_, ref, N, kind, compact, lists)
            assert got["status"] != 0, (kind, compact)
        # the next, well-formed tile is right
        want = canonical(engine, host_route(engine, words, aux16, st16, ref, N, capi.CELLS_U16, "calls", compact), ref)
        got = canonical(engine, device_route(engine, words, aux16, st16, ref, N, "calls", compact), ref)
        assert got == want and got["status"] == 0
    # the host route reports the same tiles as malformed
    t = capi.BvSparseTile(bad.ctypes.data, None, st.ctypes.data, ref.ctypes.data, None, 400, N, capi.CELLS_U32, 0)
    _check(engine, engine.lib.bv_tile_submit_sparse(engine._ctx, 0, C.byref(t)), "bv_tile_submit_sparse")
    assert engine.lib.bv_tile_wait(engine._ctx, 0, None) == -1


def test_host_pointers_are_refused(engine):
    N = 100
    model = bv.synth.make_model(seed=5, coverage=0.1, variant_frac=0.1)
    cells, aux, st, ref = bv.synth_fill_sparse_host(model, 0, 50, N)
    d_cells, d_st, d_ref = _dev(cells), _dev(st), _dev(ref)
    out = torch.empty((50, 128), dtype=torch.uint8, device="cuda")
    launches = engine.launch_count

    def run(c, s, r, o):
        t = capi.BvSparseTile(c, None, s, r, None, 50, N, capi.CELLS_U32, 0)
        d = capi.BvDeviceOut()
        d.kind, d.out_mode, d.d_out = capi.RUN_PLAIN, capi.OUT_RECORDS, o
        return engine.lib.bv_tile_run_device_sparse(engine._ctx, C.byref(t), C.byref(d), None)

    pinned = torch.empty(50 * 128, dtype=torch.uint8, pin_memory=True)
    for args in ((cells.ctypes.data, d_st.data_ptr(), d_ref.data_ptr(), out.data_ptr()),
                 (d_cells.data_ptr(), st.ctypes.data, d_ref.data_ptr(), out.data_ptr()),
                 (d_cells.data_ptr(), d_st.data_ptr(), ref.ctypes.data, out.data_ptr()),
                 (d_cells.data_ptr(), d_st.data_ptr(), d_ref.data_ptr(), pinned.data_ptr()),
                 (d_cells.data_ptr(), d_st.data_ptr(), d_ref.data_ptr(), None),
                 (d_cells.data_ptr() + 1, d_st.data_ptr(), d_ref.data_ptr(), out.data_ptr())):
        assert run(*args) == -1
        assert b"device" in engine.lib.bv_last_error(engine._ctx) or b"aligned" in engine.lib.bv_last_error(engine._ctx) \
            or b"null" in engine.lib.bv_last_error(engine._ctx)
    assert engine.launch_count == launches   # nothing was queued
    # a dense tile of host planes is refused too
    b, q, s, _, r = bv.synth_fill_host(model, 0, 50, N)
    t = capi.BvTile(b.ctypes.data, q.ctypes.data, s.ctypes.data, r.ctypes.data, b.shape[1], 50, N, capi.BV_LOC_DEVICE, 0)
    d = capi.BvDeviceOut()
    d.kind, d.out_mode, d.d_out = capi.RUN_PLAIN, capi.OUT_RECORDS, out.data_ptr()
    assert engine.lib.bv_tile_run_device_ex(engine._ctx, C.byref(t), None, C.byref(d), None) == -1
    t.location = capi.BV_LOC_HOST
    assert engine.lib.bv_tile_run_device_ex(engine._ctx, C.byref(t), None, C.byref(d), None) == -1


def test_two_streams_with_an_event_between(engine):
    _set_groups(engine, 0, 10)
    N = 1000
    (f1, ref1), (f2, ref2) = _tile(1000, 0.1), _tile(10000, 0.1)
    c1, a1, s1 = f1[capi.CELLS_U16]
    c2, a2, s2 = f2[capi.CELLS_U32]
    alone1 = canonical(engine, device_route(engine, c1, a1, s1, ref1, N, "plain", True), ref1)
    alone2 = canonical(engine, device_route(engine, c2, a2, s2, ref2, 10000, "plain", False), ref2)
    args1 = (_dev(c1), _dev(s1), _dev(ref1))
    args2 = (_dev(c2), _dev(s2), _dev(ref2))
    torch.cuda.synchronize()
    st1, st2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(st1):
        r1 = engine.call_device_sparse(*args1, N, compact=True)
        ev = torch.cuda.Event()
        ev.record(st1)
    st2.wait_event(ev)
    with torch.cuda.stream(st2):
        r2 = engine.call_device_sparse(*args2, 10000, compact=False)
    torch.cuda.synchronize()
    assert canonical(engine, r1.to_numpy(), ref1) == alone1
    assert canonical(engine, r2.to_numpy(), ref2) == alone2


@pytest.fixture(scope="module")
def wide_engine(built_lib):
    """Tiles of several 4,096-site chunks of bv_list_pairs_kernel."""
    eng = bv.BaseTypeEngine(device=0, max_samples=400, max_sites=5 * 4096, n_slots=1, min_af=bv.cli_min_af(0.01, 400))
    yield eng
    eng.close()


def test_compact_lists_of_several_chunks(wide_engine):
    """bv_list_pairs_kernel over tiles of several chunks (one CTA each: published counts, the prefix over the chunks in front,
    the pair count from the last chunk), site counts that are and are not a multiple of a chunk, lists kept densely and
    sparsely, repeated calls on one context (the chunk counts' epoch tags) and a tile larger than any before it (the buffers
    grow, the tags start again): the bytes of bv_tile_submit_sparse_lists + bv_tile_wait_lists_compact."""
    eng = wide_engine
    N = 400
    model = bv.synth.make_model(seed=31, coverage=0.1, variant_frac=0.1, multi_frac=0.2)
    cells, _, st, ref = bv.synth_fill_sparse_host(model, 0, 5 * 4096, N)
    words, _, st16 = bv.sparse_encode16(cells, st)
    checked = 0
    for S, seed, keep in ((4096 + 1, 1, 1.0), (3 * 4096 + 17, 2, 0.5), (3 * 4096 + 17, 3, 0.02), (2 * 4096, 4, 0.7),
                          (5 * 4096, 5, 0.3), (5 * 4096, 6, 0.0), (3 * 4096 + 17, 7, 0.9)):
        rng = np.random.default_rng(seed)
        lists, host = _lists(S, seed)
        drop = rng.random(S) >= keep   # make the kept lists dense or sparse
        lists[drop] = capi.LIST_END
        host[drop] = capi.LIST_END
        c16, s16 = words[:int(st16[S])], st16[:S + 1]
        for fmt, (c, s_) in ((capi.CELLS_U16, (c16, s16)), (capi.CELLS_U32, (cells[:int(st[S])], st[:S + 1]))):
            want = canonical(eng, host_route(eng, c, None, s_, ref[:S], N, fmt, "lists", True, host), ref[:S])
            got = canonical(eng, device_route(eng, c, None, s_, ref[:S], N, "lists", True, lists), ref[:S])
            assert got == want, (S, seed, fmt)
            assert len(got["lrt"]) // 64 == int((host[:, 0] != capi.LIST_END).sum())
            checked += 1
    assert checked == 14
