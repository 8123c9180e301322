"""Host-side driver of the CUDA basetype core, a thin layer over the C ABI (include/basevar_b200.h).

``BaseTypeEngine`` plays the role of the reference's per-site loop in ``_variant_calling_unit`` /
``_basevar_caller`` (src/basetype_caller.cpp:586-611, 738-743): it is handed the pileup of many sites
(as packed SoA planes instead of one BatchInfo per site) and returns one record per site holding
what ``BaseType`` + ``strand_bias`` would have produced.  Tiles are pipelined over ``n_slots`` CUDA
streams (H2D copy, kernel, D2H copy per slot).
"""
import collections
import ctypes as C

import numpy as np

from . import capi
from .capi import BvError, BvSparseTile, BvTile, BvTileAux, CALL_OUT_DTYPE, GROUP_OUT_DTYPE, LRT_OUT_DTYPE, SITE_OUT_DTYPE


def _ptr(a):
    return a.ctypes.data if isinstance(a, np.ndarray) else int(a)


class BaseTypeEngine:
    def __init__(self, device=0, max_samples=1, max_sites=0, n_slots=0, min_af=0.01,
                 abs_mode=capi.BV_EM_ABS_INT_TRUNC):
        self.lib = capi.load_library()
        self.params = capi.make_params(min_af, abs_mode, max_samples, max_sites, n_slots)
        self._ctx = C.c_void_p()
        rc = self.lib.bv_create(device, C.byref(self.params), C.byref(self._ctx))
        if rc != capi.BV_OK:
            raise BvError(f"bv_create failed ({rc}): {self.lib.bv_last_error(None).decode()}")
        self.device = device

    # -- lifecycle ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None):
            self.lib.bv_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != capi.BV_OK:
            raise BvError(f"{what} failed ({rc}): {self.lib.bv_last_error(self._ctx).decode()}")

    def set_params(self, min_af=None, abs_mode=None):
        if min_af is not None:
            self.params.min_af = float(np.float32(min_af))
        if abs_mode is not None:
            self.params.em_abs_mode = abs_mode
        self._check(self.lib.bv_set_params(self._ctx, C.byref(self.params)), "bv_set_params")

    def suggest_tile_sites(self, n_samples, max_bytes):
        """Largest tile (sites) that fits max_bytes of planes and that the count kernel's persistent warps split evenly."""
        return int(self.lib.bv_suggest_tile_sites(self._ctx, n_samples, max_bytes))

    @property
    def launch_count(self):
        return int(self.lib.bv_launch_count(self._ctx))

    @property
    def h2d_bytes(self):
        """Bytes uploaded by the bv_tile_submit* calls so far (planes or cells of host tiles, lists of lists tiles)."""
        return int(self.lib.bv_h2d_bytes(self._ctx))

    KERNEL_NAMES = ("bv_count_kernel", "bv_scalar_kernel", "bv_bound_kernel", "bv_em_kernel")

    def set_profiling(self, on=True):
        self._check(self.lib.bv_set_profiling(self._ctx, int(on)), "bv_set_profiling")

    def last_kernel_times(self):
        """Durations (ms) of the four kernels of the most recent tile (profiling must be on); waits for it."""
        ms = (C.c_float * 4)()
        self._check(self.lib.bv_last_kernel_times(self._ctx, ms), "bv_last_kernel_times")
        return dict(zip(self.KERNEL_NAMES, (float(x) for x in ms)))

    EM_KERNEL_NAMES = ("bv_hist_kernel", "bv_em_task_kernel", "bv_fisher_kernel")

    def last_em_kernel_times(self):
        """Durations (ms) of the two kernels K4 consists of (row histograms, EM tasks + decisions) and of the kernel that runs the
        Fisher tests K2 and K4b listed, for the same tile."""
        ms = (C.c_float * 3)()
        self._check(self.lib.bv_last_em_kernel_times(self._ctx, ms), "bv_last_em_kernel_times")
        self._check(self.lib.bv_last_fisher_kernel_time(self._ctx, C.cast(C.byref(ms, 8), C.POINTER(C.c_float))), "bv_last_fisher_kernel_time")
        return dict(zip(self.EM_KERNEL_NAMES, (float(x) for x in ms)))

    # -- the slot pipeline -------------------------------------------------------------------------
    def _site_ranges(self, S):
        """(site0, n_sites) of the tiles of S sites, max_sites each; no sites is one empty tile."""
        step = self.params.max_sites
        assert step >= 1, "engine was created without slots"
        return [(s0, min(step, S - s0)) for s0 in range(0, max(S, 1), step)]

    def _pipeline(self, tiles, submit, wait):
        """submit(slot, tile) each tile on the slots in turn, at most n_slots in flight, and wait(slot, tile) for each in submit
        order: the oldest before its slot takes the next tile, the rest at the end.  A tile stays referenced until its wait, and
        with it the arrays its descriptor points into."""
        n_slots = self.params.n_slots
        assert n_slots >= 1, "engine was created without slots"
        pending, slot = collections.deque(), 0
        for tile in tiles:
            if len(pending) == n_slots:
                wait(*pending.popleft())
            submit(slot, tile)
            pending.append((slot, tile))
            slot = (slot + 1) % n_slots
        for p in pending:
            wait(*p)

    def _dense_tiles(self, base, qual, strand, ref_base, n_samples, out_mode=capi.OUT_RECORDS):
        """(BvTile, site0, None) of each tile of host planes [S][pitch]."""
        S, pitch = base.shape
        return ((BvTile(base[s0:].ctypes.data, qual[s0:].ctypes.data, strand[s0:].ctypes.data, ref_base[s0:].ctypes.data, pitch, ns,
                        n_samples, capi.BV_LOC_HOST, out_mode), s0, None) for s0, ns in self._site_ranges(S))

    def _sparse_tiles(self, cells, cells_aux, site_start, ref_base, n_samples, fmt=None, out_mode=capi.OUT_RECORDS, out=None,
                      pinned=False):
        """(BvSparseTile, site0, its site_start) of each tile: the per-tile offsets start at 0, rebased from the whole-run array (a
        packer writes them so), and must live until the tile's wait.  out: records array the D2H copy writes in place.  pinned:
        the rebased offsets are pinned (a pageable source makes cudaMemcpyAsync wait for the uploads queued in front of it)."""
        if fmt is None:
            fmt = capi.CELLS_U16 if cells.dtype == np.uint16 else capi.CELLS_U32   # uint16: the delta-coded compact form
        for s0, ns in self._site_ranges(ref_base.shape[0]):
            c0 = int(site_start[s0])
            st = site_start[s0:s0 + ns + 1]
            if c0 or pinned:
                st = _alloc(ns + 1, np.uint32, pinned)
                st[:] = site_start[s0:s0 + ns + 1] - np.uint32(c0)
            # (cells[c0:] of a tile without cells is the end of the array, which the tile never reads)
            t = BvSparseTile(cells[c0:].ctypes.data, cells_aux[c0:].ctypes.data if cells_aux is not None else None, st.ctypes.data,
                             ref_base[s0:].ctypes.data, out[s0:].ctypes.data if out is not None else None, ns, n_samples, fmt, out_mode)
            yield t, s0, st

    # -- tiles from host memory --------------------------------------------------------------------
    def call_host(self, base, qual, strand, ref_base, n_samples, out=None):
        """Run planes [S][pitch] (numpy uint8, ideally pinned) through the slot pipeline.

        Returns a numpy record array (capi.SITE_OUT_DTYPE) with one record per site."""
        S, pitch = base.shape
        assert qual.shape == base.shape and strand.shape == base.shape and ref_base.shape[0] == S
        for a in (base, qual, strand, ref_base):
            assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
        if out is None:
            out = np.zeros(S, dtype=SITE_OUT_DTYPE)

        def submit(slot, tile):
            self._check(self.lib.bv_tile_submit(self._ctx, slot, C.byref(tile[0])), "bv_tile_submit")

        def wait(slot, tile):
            self._check(self.lib.bv_tile_wait(self._ctx, slot, out[tile[1]:].ctypes.data), "bv_tile_wait")

        self._pipeline(self._dense_tiles(base, qual, strand, ref_base, n_samples), submit, wait)
        return out

    # -- sparse tiles from host memory: only the covered cells cross PCIe ---------------------------------
    def call_sparse(self, cells, site_start, ref_base, n_samples, out=None, out_pinned=False):
        """cells: uint32 BV_CELL_PACK words grouped by site; site_start: uint32 [S + 1] offsets into cells.

        Tiles of max_sites sites go through the slot pipeline (upload of the cells, K0 expand, K1..K4, D2H of the
        records).  With out_pinned=True `out` is pinned host memory and the D2H DMA writes the records in place."""
        S = ref_base.shape[0]
        assert cells.dtype in (np.uint32, np.uint16) and site_start.dtype == np.uint32 and site_start.shape[0] == S + 1
        if out is None:
            out = np.zeros(S, dtype=SITE_OUT_DTYPE)
        tiles = self._sparse_tiles(cells, None, site_start, ref_base, n_samples, out=out if out_pinned else None)
        self.run_sparse_tiles(tiles, out=None if out_pinned else out)
        return out

    def sparse_tiles(self, cells, site_start, ref_base, n_samples, out_pinned=None, compact=False):
        """The tile descriptors call_sparse would submit, built once (list of ctypes structs + the arrays they point into).
        out_pinned: pinned SITE_OUT_DTYPE array [S] the records are DMA'd into.  compact: BV_OUT_COMPACT tiles (8 bytes per
        site + the full records of the sites that need one; collect with run_sparse_tiles(..., compact=...))."""
        S = ref_base.shape[0]
        assert cells.dtype in (np.uint32, np.uint16) and site_start.dtype == np.uint32 and site_start.shape[0] == S + 1
        return list(self._sparse_tiles(cells, None, site_start, ref_base, n_samples, out_mode=capi.OUT_COMPACT if compact else capi.OUT_RECORDS,
                                       out=out_pinned if not compact else None, pinned=out_pinned is not None))

    def run_sparse_tiles(self, tiles, repeats=1, out=None, compact=None):
        """Submit the tiles `repeats` times over the slots without draining the pipeline in between (the steps of a
        benchmark run, or the tiles of a long region); every slot is waited for before its next submit and at the end.
        compact: for BV_OUT_COMPACT tiles a callable (site0, n_sites, briefs, full_records) that consumes a tile's compact
        result (numpy views of the slot's pinned staging, valid during the call only); None drops them (timing runs)."""
        def submit(slot, tile):
            self._check(self.lib.bv_tile_submit_sparse(self._ctx, slot, C.byref(tile[0])), "bv_tile_submit_sparse")

        def wait(slot, tile):
            t, s0, _ = tile
            if t.out_mode != capi.OUT_COMPACT:
                self._check(self.lib.bv_tile_wait(self._ctx, slot, out[s0:].ctypes.data if out is not None else None), "bv_tile_wait")
                return
            pb, pf, nf = C.c_void_p(), C.c_void_p(), C.c_uint32(0)
            self._check(self.lib.bv_tile_wait_compact(self._ctx, slot, C.byref(pb), C.byref(pf), C.byref(nf)), "bv_tile_wait_compact")
            ns = int(t.n_sites)
            if compact is not None and ns:
                compact(s0, ns, *self._compact_views(pb, pf, nf.value, ns))

        self._pipeline((tile for _ in range(repeats) for tile in tiles), submit, wait)

    def _compact_views(self, pb, pf, nf, ns):
        """numpy views of a compact tile's briefs and full records (the slot's pinned staging)."""
        briefs = np.ctypeslib.as_array(C.cast(pb, C.POINTER(C.c_uint32)), shape=(ns * 2,)).view(capi.SITE_BRIEF_DTYPE) if ns else \
            np.zeros(0, capi.SITE_BRIEF_DTYPE)
        full = (np.ctypeslib.as_array(C.cast(pf, C.POINTER(C.c_uint8)), shape=(nf * 128,)).view(SITE_OUT_DTYPE)
                if nf else np.zeros(0, SITE_OUT_DTYPE))
        return briefs, full

    def _collect_compact(self, pb, pf, nf, ref_base, out):
        """Expand a compact tile into `out` (n_sites records) and note (n_full, briefs that point at a full record)."""
        ns = len(out)
        briefs, full = self._compact_views(pb, pf, nf.value, ns)
        if ns:
            self.expand_compact(briefs, full, ref_base, out)
        self.compact_tiles.append((int(nf.value), int(((briefs["w0"] & 0x80000000) != 0).sum())))

    def expand_compact(self, briefs, full, ref_base, out):
        """Records of one compact tile into out[:n] (host helper bv_site_expand for the brief-only sites)."""
        is_full = (briefs["w0"] & 0x80000000) != 0
        idx = np.nonzero(is_full)[0]
        out[idx] = full[briefs["w0"][idx] & 0x7fffffff]
        tmp = np.zeros(1, SITE_OUT_DTYPE)
        b = np.ascontiguousarray(briefs)
        for i in np.nonzero(~is_full)[0]:
            self.lib.bv_site_expand(b[i:].ctypes.data, int(ref_base[i]), self.params.min_af, tmp.ctypes.data)
            out[i] = tmp[0]
        return out

    def _run_calls(self, S, tiles, submit, ref_base, compact):
        """The slot pipeline of tiles with the called-site kernels.  Returns (records, calls sorted by GLOBAL site index,
        groups[n_calls][n_groups]); with compact=True the records are expanded from the compact form and self.compact_tiles
        receives (n_full, briefs pointing at a full record) per tile."""
        G = getattr(self, "n_groups", 0)
        step = self.params.max_sites
        out = np.zeros(S, dtype=SITE_OUT_DTYPE)
        calls, groups = [], []
        tmp_calls = np.zeros(step, CALL_OUT_DTYPE)
        tmp_groups = np.zeros((step, max(G, 1)), GROUP_OUT_DTYPE)
        gp = tmp_groups.ctypes.data if G else None
        self.compact_tiles = []

        def wait(slot, tile):
            t, s0, _ = tile
            ns, n = int(t.n_sites), C.c_uint32(0)
            if compact:
                pb, pf, nf = C.c_void_p(), C.c_void_p(), C.c_uint32(0)
                self._check(self.lib.bv_tile_wait_calls_compact(self._ctx, slot, C.byref(pb), C.byref(pf), C.byref(nf), tmp_calls.ctypes.data,
                                                                step, C.byref(n), gp), "bv_tile_wait_calls_compact")
                self._collect_compact(pb, pf, nf, ref_base[s0:s0 + ns], out[s0:s0 + ns])
            else:
                self._check(self.lib.bv_tile_wait_calls(self._ctx, slot, out[s0:].ctypes.data, tmp_calls.ctypes.data, step, C.byref(n), gp),
                            "bv_tile_wait_calls")
            c = tmp_calls[:n.value].copy()
            c["site"] += s0
            calls.append(c)
            groups.append(tmp_groups.reshape(-1)[:n.value * G].reshape(n.value, G).copy() if G else np.zeros((n.value, 0), GROUP_OUT_DTYPE))

        self._pipeline(tiles, submit, wait)
        calls = np.concatenate(calls) if calls else np.zeros(0, CALL_OUT_DTYPE)
        groups = np.concatenate(groups) if groups else np.zeros((0, G), GROUP_OUT_DTYPE)
        order = np.argsort(calls["site"], kind="stable")
        return out, calls[order], groups[order]

    def call_sparse_calls(self, cells, cells_aux, site_start, ref_base, n_samples, compact=False):
        """call_sparse plus the called-site outputs; returns what call_host_calls returns.  compact=True: the tiles ask for
        BV_OUT_COMPACT (briefs + the full records of the sites that need one), expanded here; self.compact_tiles receives
        (n_full, briefs pointing at a full record) per tile."""
        S = ref_base.shape[0]
        assert cells.dtype in (np.uint32, np.uint16) and cells_aux.dtype == np.uint32 and site_start.dtype == np.uint32

        def submit(slot, tile):
            self._check(self.lib.bv_tile_submit_sparse_calls(self._ctx, slot, C.byref(tile[0])), "bv_tile_submit_sparse_calls")

        tiles = self._sparse_tiles(cells, cells_aux, site_start, ref_base, n_samples, out_mode=capi.OUT_COMPACT if compact else capi.OUT_RECORDS)
        return self._run_calls(S, tiles, submit, ref_base, compact)

    # -- called sites: rank sums + population groups ---------------------------------------------------
    CALL_KERNEL_NAMES = ("bv_ranksum_kernel", "bv_group_kernel")

    def last_call_kernel_times(self):
        ms = (C.c_float * 2)()
        self._check(self.lib.bv_last_call_kernel_times(self._ctx, ms), "bv_last_call_kernel_times")
        return dict(zip(self.CALL_KERNEL_NAMES, (float(x) for x in ms)))

    def set_groups(self, sample_group, n_groups):
        """sample_group: uint8 [n_samples], group index or capi.GROUP_NONE; groups numbered in ascending-name order."""
        self.n_groups = int(n_groups)
        if n_groups:
            sample_group = np.ascontiguousarray(sample_group, np.uint8)
            self._check(self.lib.bv_set_groups(self._ctx, sample_group.ctypes.data, len(sample_group), n_groups), "bv_set_groups")
        else:
            self._check(self.lib.bv_set_groups(self._ctx, None, 0, 0), "bv_set_groups")

    def call_host_calls(self, base, qual, strand, ref_base, mapq, rpr, n_samples, compact=False):
        """Like call_host, plus the called-site outputs.  mapq: uint8 [S][pitch]; rpr: uint16 [S][rpr_pitch].
        Returns (records, calls sorted by GLOBAL site index, groups[n_calls][n_groups]).  compact: as in call_sparse_calls."""
        S, pitch = base.shape
        assert mapq.shape == base.shape and mapq.dtype == np.uint8 and rpr.dtype == np.uint16 and rpr.shape[0] == S
        rpr_pitch = rpr.shape[1]

        def submit(slot, tile):
            t, s0, _ = tile
            a = BvTileAux(mapq[s0:].ctypes.data, rpr[s0:].ctypes.data, rpr_pitch)
            self._check(self.lib.bv_tile_submit_calls(self._ctx, slot, C.byref(t), C.byref(a)), "bv_tile_submit_calls")

        tiles = self._dense_tiles(base, qual, strand, ref_base, n_samples, capi.OUT_COMPACT if compact else capi.OUT_RECORDS)
        return self._run_calls(S, tiles, submit, ref_base, compact)

    # -- lrt(specific_bases): per-site ordered candidate lists -------------------------------------------
    def call_host_lists(self, base, qual, strand, ref_base, lists, n_samples):
        """Like call_host, plus BaseType::lrt(list) of every site.  lists: uint8 [S][4], 1..4 distinct base codes per site
        in caller order, ended early by capi.LIST_END (a row of LIST_END skips the site).
        Returns (records, lrt_out: capi.LRT_OUT_DTYPE [S])."""
        S, pitch = base.shape
        lists = np.ascontiguousarray(lists, np.uint8)
        assert lists.shape == (S, 4)
        out = np.zeros(S, dtype=SITE_OUT_DTYPE)
        lrt = np.zeros(S, dtype=LRT_OUT_DTYPE)

        def submit(slot, tile):
            self._check(self.lib.bv_tile_submit_lists(self._ctx, slot, C.byref(tile[0]), lists[tile[1]:].ctypes.data), "bv_tile_submit_lists")

        def wait(slot, tile):
            s0 = tile[1]
            self._check(self.lib.bv_tile_wait_lists(self._ctx, slot, out[s0:].ctypes.data, lrt[s0:].ctypes.data), "bv_tile_wait_lists")

        self._pipeline(self._dense_tiles(base, qual, strand, ref_base, n_samples), submit, wait)
        return out, lrt

    def call_sparse_lists(self, cells, site_start, ref_base, lists, n_samples, fmt=None, compact=False):
        """call_sparse plus BaseType::lrt(list) per site (bv_tile_submit_sparse_lists).  lists as in call_host_lists; fmt:
        capi.CELLS_U32 / CELLS_U16, or None to take it from cells.dtype.  Returns (records, lrt): lrt is LRT_OUT_DTYPE [S]
        (compact=False), or with compact=True one entry per site whose list is non-empty, in site order (the records are then
        expanded from the compact form; self.compact_tiles as in call_sparse_calls)."""
        S = ref_base.shape[0]
        assert cells.dtype in (np.uint32, np.uint16) and site_start.dtype == np.uint32 and site_start.shape[0] == S + 1
        lists = np.ascontiguousarray(lists, np.uint8)
        assert lists.shape == (S, 4)
        out = np.zeros(S, dtype=SITE_OUT_DTYPE)
        lrt = np.zeros(S, dtype=LRT_OUT_DTYPE)
        step = self.params.max_sites
        packed, tmp = [], np.zeros(step, LRT_OUT_DTYPE)
        self.compact_tiles = []

        def submit(slot, tile):
            self._check(self.lib.bv_tile_submit_sparse_lists(self._ctx, slot, C.byref(tile[0]), lists[tile[1]:].ctypes.data),
                        "bv_tile_submit_sparse_lists")

        def wait(slot, tile):
            t, s0, _ = tile
            if not compact:
                self._check(self.lib.bv_tile_wait_lists(self._ctx, slot, out[s0:].ctypes.data, lrt[s0:].ctypes.data), "bv_tile_wait_lists")
                return
            ns = int(t.n_sites)
            pb, pf, nf, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0), C.c_uint32(0)
            self._check(self.lib.bv_tile_wait_lists_compact(self._ctx, slot, C.byref(pb), C.byref(pf), C.byref(nf), tmp.ctypes.data, step,
                                                            C.byref(n)), "bv_tile_wait_lists_compact")
            self._collect_compact(pb, pf, nf, ref_base[s0:s0 + ns], out[s0:s0 + ns])
            packed.append(tmp[:n.value].copy())

        tiles = self._sparse_tiles(cells, None, site_start, ref_base, n_samples, fmt, capi.OUT_COMPACT if compact else capi.OUT_RECORDS)
        self._pipeline(tiles, submit, wait)
        if compact:
            lrt = np.concatenate(packed) if packed else np.zeros(0, LRT_OUT_DTYPE)
        return out, lrt

    def call_device_lists(self, d_base, d_qual, d_strand, d_ref, d_lists, n_sites, n_samples, pitch, d_out, d_lrt_out, stream=0):
        """Device-resident call_host_lists: every argument a device pointer (int); d_lists uint8 [n_sites][4], d_lrt_out
        n_sites LRT_OUT_DTYPE entries.  Asynchronous on `stream` (a cudaStream_t handle)."""
        t = BvTile(int(d_base), int(d_qual), int(d_strand), int(d_ref), pitch, n_sites, n_samples, capi.BV_LOC_DEVICE, 0)
        self._check(self.lib.bv_tile_run_device_lists(self._ctx, C.byref(t), C.c_void_p(int(d_lists)), C.c_void_p(int(d_out)),
                                                      C.c_void_p(int(d_lrt_out)), C.c_void_p(int(stream))), "bv_tile_run_device_lists")

    def last_list_kernel_time(self):
        """Duration (ms) of K8 (bv_list_kernel, or bv_list_packed_kernel for compact sparse lists) of the most recent lists tile
        (profiling must be on); waits for it."""
        ms = C.c_float(0.0)
        self._check(self.lib.bv_last_list_kernel_time(self._ctx, C.byref(ms)), "bv_last_list_kernel_time")
        return float(ms.value)

    # -- ref_vs_alt_ranksumtest of free-standing problems ------------------------------------------------
    def ranksum_test(self, bases, values, start, ref_base, alt_mask):
        """ref_vs_alt_ranksumtest (src/basetype.cpp:201-242) of n problems on the device (bv_ranksum_test).  Problem p is
        entries start[p]:start[p+1] of bases (uint8 BV_BASE_* codes) and values (int32), ref_base[p] its REF character
        (ASCII code) and alt_mask[p] its ALT bases (bit b = base code b).  Returns float64 [n], not truncated."""
        bases = np.ascontiguousarray(bases, np.uint8)
        values = np.ascontiguousarray(values, np.int32)
        start = np.ascontiguousarray(start, np.uint64)
        ref_base = np.ascontiguousarray(ref_base, np.uint8)
        alt_mask = np.ascontiguousarray(alt_mask, np.uint8)
        n = len(ref_base)
        assert start.shape == (n + 1,) and alt_mask.shape == (n,) and bases.shape == values.shape
        assert int(start[-1]) <= len(bases)
        out = np.zeros(n, np.float64)
        self._check(self.lib.bv_ranksum_test(self._ctx, _ptr(bases), _ptr(values), _ptr(start), _ptr(ref_base), _ptr(alt_mask), n,
                                             _ptr(out)), "bv_ranksum_test")
        return out

    def last_ranksum_kernel_time(self):
        """Duration (ms) of K9 bv_ranksum_test_kernel of the most recent ranksum_test (profiling must be on); waits for it."""
        ms = C.c_float(0.0)
        self._check(self.lib.bv_last_ranksum_kernel_time(self._ctx, C.byref(ms)), "bv_last_ranksum_kernel_time")
        return float(ms.value)

    # -- device-resident tiles ---------------------------------------------------------------------
    def call_device(self, d_base, d_qual, d_strand, d_ref, n_sites, n_samples, pitch, d_out, stream=0):
        """All arguments are device pointers (ints); stream is a cudaStream_t handle (int).  Asynchronous."""
        t = BvTile(int(d_base), int(d_qual), int(d_strand), int(d_ref), pitch, n_sites, n_samples,
                   capi.BV_LOC_DEVICE, 0)
        self._check(self.lib.bv_tile_run_device(self._ctx, C.byref(t), C.c_void_p(int(d_out)),
                                                C.c_void_p(int(stream))), "bv_tile_run_device")

    # -- synthetic pileups -------------------------------------------------------------------------
    def synth_set_model(self, model):
        self._model = model
        self._check(self.lib.bv_synth_set_model(self._ctx, C.byref(model)), "bv_synth_set_model")

    def synth_fill_device(self, site0, n_sites, n_samples, pitch, d_base, d_qual, d_strand, d_mapq, d_ref, stream=0):
        self._check(self.lib.bv_synth_fill_device(self._ctx, site0, n_sites, n_samples, pitch, int(d_base), int(d_qual),
                                                  int(d_strand), int(d_mapq) if d_mapq else None, int(d_ref),
                                                  C.c_void_p(int(stream))), "bv_synth_fill_device")


def synth_fill_rpr_host(model, site0, n_sites, n_samples):
    """Read-position-rank plane (uint16 [n_sites][round8(n_samples)]) of the synthetic genome, host twin."""
    lib = capi.load_library()
    rp = (n_samples + 7) // 8 * 8
    rpr = np.empty((n_sites, rp), np.uint16)
    rc = lib.bv_synth_fill_rpr_host(C.byref(model), site0, n_sites, n_samples, rp, rpr.ctypes.data)
    if rc != capi.BV_OK:
        raise BvError(f"bv_synth_fill_rpr_host failed ({rc}): {lib.bv_last_error(None).decode()}")
    return rpr


def synth_fill_host(model, site0, n_sites, n_samples, pitch=None, with_mapq=False):
    """Host twin of the device generator (no CUDA needed).  Returns (base, qual, strand, mapq|None, ref_base)."""
    lib = capi.load_library()
    if pitch is None:
        pitch = (n_samples + 15) // 16 * 16
    base = np.empty((n_sites, pitch), np.uint8)
    qual = np.empty((n_sites, pitch), np.uint8)
    strand = np.empty((n_sites, pitch), np.uint8)
    mapq = np.empty((n_sites, pitch), np.uint8) if with_mapq else None
    ref = np.empty(n_sites, np.uint8)
    rc = lib.bv_synth_fill_host(C.byref(model), site0, n_sites, n_samples, pitch, base.ctypes.data, qual.ctypes.data,
                                strand.ctypes.data, mapq.ctypes.data if with_mapq else None, ref.ctypes.data)
    if rc != capi.BV_OK:
        raise BvError(f"bv_synth_fill_host failed ({rc}): {lib.bv_last_error(None).decode()}")
    return base, qual, strand, mapq, ref


def dense_to_sparse(base, qual, strand, n_samples, mapq=None, rpr=None):
    """Sparse form (cells, cells_aux | None, site_start) of dense planes: every cell that is not the uncovered triple
    (BV_BASE_N, phred 0, BV_STRAND_NONE), in sample order within a site."""
    b, q, s = base[:, :n_samples], qual[:, :n_samples], strand[:, :n_samples]
    cov = (b != capi.BASE_N) | (q != 0) | (s != capi.STRAND_NONE)
    if mapq is not None:
        cov |= (mapq[:, :n_samples] != 0) | (rpr[:, :n_samples] != 0)
    site, samp = np.nonzero(cov)
    cells = capi.cell_pack(samp, b[site, samp], s[site, samp], q[site, samp])
    aux = capi.cell_aux_pack(mapq[site, samp], rpr[site, samp]) if mapq is not None else None
    site_start = np.zeros(base.shape[0] + 1, np.uint32)
    np.cumsum(cov.sum(axis=1), out=site_start[1:])
    return cells, aux, site_start


def _alloc(k, dt, pinned):
    if pinned:
        import torch
        tdt = {np.uint32: torch.int32, np.uint16: torch.int16, np.uint8: torch.uint8}[dt]
        return torch.empty(max(k, 1), dtype=tdt, pin_memory=True).numpy().view(dt)[:k]
    return np.empty(k, dt)


def sparse_encode16(cells, site_start, aux=None, pinned=False):
    """BV_CELLS_U32 -> BV_CELLS_U16 (2 bytes per cell, samples delta-coded; cells must ascend by sample within a site).
    Returns (words uint16, aux uint32 | None, start uint32).  Raises BvError for cells the compact form cannot carry."""
    lib = capi.load_library()
    S = site_start.shape[0] - 1
    cells = np.ascontiguousarray(cells, np.uint32)
    site_start = np.ascontiguousarray(site_start, np.uint32)
    n = C.c_uint64(0)
    rc = lib.bv_sparse_encode16(cells.ctypes.data, None, site_start.ctypes.data, S, None, None, 0, None, C.byref(n))
    if rc != capi.BV_OK:
        raise BvError(f"bv_sparse_encode16 failed ({rc}): {lib.bv_last_error(None).decode()}")
    words = _alloc(n.value, np.uint16, pinned)
    aux16 = _alloc(n.value, np.uint32, pinned) if aux is not None else None
    start = _alloc(S + 1, np.uint32, pinned)
    rc = lib.bv_sparse_encode16(cells.ctypes.data, aux.ctypes.data if aux is not None else None, site_start.ctypes.data, S,
                                words.ctypes.data, aux16.ctypes.data if aux is not None else None, n.value, start.ctypes.data, C.byref(n))
    if rc != capi.BV_OK:
        raise BvError(f"bv_sparse_encode16 failed ({rc}): {lib.bv_last_error(None).decode()}")
    return words, aux16, start


def synth_fill_sparse_host(model, site0, n_sites, n_samples, with_aux=False, pinned=False):
    """Host twin of the generator in sparse form.  Returns (cells, cells_aux | None, site_start, ref_base)."""
    lib = capi.load_library()
    site_start = _alloc(n_sites + 1, np.uint32, pinned)
    ref = _alloc(n_sites, np.uint8, pinned)
    total = n_sites * n_samples
    # one pass with room for the expected number of cells + 6 sigma; a second, exact one if that was too small
    exp = total * (model.cov_thr / 2.0 ** 32)
    cap = int(min(total, exp + 6.0 * np.sqrt(exp + 1.0) + 64))
    n = C.c_uint64(0)
    for attempt in range(2):
        cells = _alloc(cap, np.uint32, pinned)
        aux = _alloc(cap, np.uint32, pinned) if with_aux else None
        rc = lib.bv_synth_fill_sparse_host(C.byref(model), site0, n_sites, n_samples, cells.ctypes.data,
                                           aux.ctypes.data if with_aux else None, cap, site_start.ctypes.data, ref.ctypes.data, C.byref(n))
        if rc == capi.BV_OK:
            return cells[:n.value], (aux[:n.value] if with_aux else None), site_start, ref
        if attempt == 0:
            rc2 = lib.bv_synth_fill_sparse_host(C.byref(model), site0, n_sites, n_samples, None, None, 0, None, None, C.byref(n))
            if rc2 != capi.BV_OK:
                break
            cap = int(n.value)
    raise BvError(f"bv_synth_fill_sparse_host failed ({rc}): {lib.bv_last_error(None).decode()}")
