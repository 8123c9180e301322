"""Measure the VCF row's batch path on a C2-shaped sparse tile: compact results with the called-site kernels, lists on sparse
tiles, and the gain over the per-site route an integrator would otherwise take.

    python tools/vcf_row_bench.py [--sites 262144] [--samples 1000] [--tiles 20] [--groups 4] [--per-site 300] [--out FILE]

The tile is the synthetic C2 genome (0.1x, 1,000 samples, 1.9 % variant sites) in BV_CELLS_U16 form, in pinned host memory.
  calls      bv_tile_submit_sparse_calls with BV_OUT_RECORDS (records copied to a caller buffer by bv_tile_wait_calls) vs
             BV_OUT_COMPACT (bv_tile_wait_calls_compact, views of the pinned staging); D2H bytes per tile from the formats and the
             tile's counts, and the median of --tiles blocking submit + wait pairs (host clock, slot 0).
  lists      [REF, ALT...] at the called sites: the dense full-output path (bv_tile_submit_lists: 4 bytes up and 64 down per site)
             vs the packed sparse path (bv_tile_submit_sparse_lists with BV_OUT_COMPACT: 8 up and 64 down per listed site); K8
             time by CUDA events (bv_last_list_kernel_time), median over --tiles runs.
  per_site   the first --per-site called sites: the documented per-site route (3 x bv_ranksum_test + one one-row lrt(list) tile
             per group, as bvhost::ref_vs_alt_ranksumtest and BaseType(&group_bi, min_af).lrt([REF, ALT...]) issue them) vs one
             batch submit + wait of a sparse tile of those sites with compact results, calls and groups.  Host clock; the
             per-site calls go through ctypes, the same C entry points the C++ mirror calls.
The card's name and power limit are read in the same run and written with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # the numbers below still stand, without the card's description
        return {"gpu": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=262144)
    ap.add_argument("--samples", type=int, default=1000)
    ap.add_argument("--tiles", type=int, default=20)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--per-site", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import basevar_b200 as bv
    from basevar_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("vcf_row_bench: no CUDA device (there is nothing to time on the CPU)")
    S, N, G = args.sites, args.samples, args.groups
    maf = bv.cli_min_af(0.01, N)
    model = bv.synth.make_model(seed=2024, coverage=0.1, variant_frac=0.019)
    cells32, aux32, st32, ref = bv.synth_fill_sparse_host(model, 0, S, N, with_aux=True, pinned=True)
    words, aux16, st16 = bv.sparse_encode16(cells32, st32, aux32, pinned=True)
    grp = np.random.default_rng(1).integers(0, G, N).astype(np.uint8)
    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=S, n_slots=1, min_af=maf)
    eng.set_groups(grp, G)
    lib, ctx = eng.lib, eng._ctx

    def check(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {lib.bv_last_error(ctx).decode()}")

    recs_buf = torch.empty(S * 128, dtype=torch.uint8, pin_memory=True).numpy().view(capi.SITE_OUT_DTYPE)
    calls_buf = np.zeros(S, capi.CALL_OUT_DTYPE)
    groups_buf = np.zeros(S * G, capi.GROUP_OUT_DTYPE)
    n, nf = C.c_uint32(0), C.c_uint32(0)
    pb, pf = C.c_void_p(), C.c_void_p()

    def calls_tile(mode):
        t = capi.BvSparseTile(words.ctypes.data, aux16.ctypes.data, st16.ctypes.data, ref.ctypes.data, None, S, N, capi.CELLS_U16, mode)
        t0 = time.perf_counter()
        check(lib.bv_tile_submit_sparse_calls(ctx, 0, C.byref(t)), "submit")
        if mode == capi.OUT_RECORDS:
            check(lib.bv_tile_wait_calls(ctx, 0, recs_buf.ctypes.data, calls_buf.ctypes.data, S, C.byref(n), groups_buf.ctypes.data), "wait")
        else:
            check(lib.bv_tile_wait_calls_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), calls_buf.ctypes.data, S, C.byref(n),
                                                 groups_buf.ctypes.data), "wait")
        return 1e3 * (time.perf_counter() - t0)

    result = dict(gpu_info(), sites=S, samples=N, groups=G, min_af=maf, tiles=args.tiles, cells=int(len(cells32)),
                  u16_words=int(len(words)))
    calls = {}
    for label, mode in (("records", capi.OUT_RECORDS), ("compact", capi.OUT_COMPACT)):
        for _ in range(3):
            calls_tile(mode)
        ms = [calls_tile(mode) for _ in range(args.tiles)]
        n_calls = int(n.value)
        side = n_calls * (16 + 40 * G) + 24 * 4   # calls, groups, counters
        d2h = S * 128 + side if mode == capi.OUT_RECORDS else S * 8 + int(nf.value) * 128 + side
        calls[label] = {"submit_wait_ms_median": float(np.median(ms)), "submit_wait_ms_min": float(np.min(ms)),
                        "submit_wait_ms_max": float(np.max(ms)), "d2h_bytes": d2h, "n_calls": n_calls}
        if mode == capi.OUT_COMPACT:
            calls[label]["n_full"] = int(nf.value)
    result["calls"] = calls
    plain = recs_buf.copy()

    # [REF, ALT...] at the called sites: dense full-output path vs packed sparse path
    from oracle import loader as L
    called = np.nonzero(plain["n_alt"] > 0)[0]
    lists = np.full((S, 4), capi.LIST_END, np.uint8)
    for site in called:
        order = L._group_order(int(ref[site]), plain[site])
        lists[site, :len(order)] = order
    b, q, s, mq_plane, r = bv.synth_fill_host(model, 0, S, N, with_mapq=True)
    pitch = b.shape[1]
    lrt_full = np.zeros(S, capi.LRT_OUT_DTYPE)
    lrt_packed = np.zeros(S, capi.LRT_OUT_DTYPE)
    eng.set_profiling(True)

    def dense_lists():
        t = capi.BvTile(b.ctypes.data, q.ctypes.data, s.ctypes.data, r.ctypes.data, pitch, S, N, capi.BV_LOC_HOST, 0)
        check(lib.bv_tile_submit_lists(ctx, 0, C.byref(t), lists.ctypes.data), "submit_lists")
        check(lib.bv_tile_wait_lists(ctx, 0, None, lrt_full.ctypes.data), "wait_lists")
        return eng.last_list_kernel_time()

    def sparse_lists():
        t = capi.BvSparseTile(words.ctypes.data, None, st16.ctypes.data, ref.ctypes.data, None, S, N, capi.CELLS_U16, capi.OUT_COMPACT)
        check(lib.bv_tile_submit_sparse_lists(ctx, 0, C.byref(t), lists.ctypes.data), "submit_sparse_lists")
        check(lib.bv_tile_wait_lists_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), lrt_packed.ctypes.data, S, C.byref(n)),
              "wait_lists_compact")
        return eng.last_list_kernel_time()

    out = {}
    for label, fn in (("dense_full", dense_lists), ("sparse_packed", sparse_lists)):
        for _ in range(3):
            fn()
        ms = [fn() for _ in range(args.tiles)]
        out[label] = {"k8_ms_median": float(np.median(ms)), "k8_ms_min": float(np.min(ms)), "k8_ms_max": float(np.max(ms))}
    eng.set_profiling(False)
    n_listed = int(n.value)
    assert n_listed == len(called) and lrt_packed[:n_listed].tobytes() == lrt_full[called].tobytes()
    out["dense_full"].update(h2d_list_bytes=4 * S, d2h_lrt_bytes=64 * S)
    out["sparse_packed"].update(h2d_list_bytes=8 * n_listed, d2h_lrt_bytes=64 * n_listed)
    result["lists"] = dict(out, listed_sites=n_listed)

    # the per-site route vs one batch submit, for the first K called sites
    K = min(args.per_site, len(called))
    sites = called[:K]
    rpr_plane = bv.synth_fill_rpr_host(model, 0, S, N)
    one = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=1, n_slots=1, min_af=maf)
    members = [np.nonzero(grp == g)[0] for g in range(G)]
    starts = np.array([0, N], np.uint64)

    def per_site():
        t0 = time.perf_counter()
        for site in sites:
            rec = plain[site]
            mask = np.uint8(sum(1 << int(a) for a in rec["alt"][:rec["n_alt"]]))
            row = np.ascontiguousarray(b[site, :N])
            for vals in (mq_plane[site, :N], rpr_plane[site, :N], q[site, :N]):
                one.ranksum_test(row, vals.astype(np.int32), starts, ref[site:site + 1], np.array([mask], np.uint8))
            for m in members:
                gp = (len(m) + 15) // 16 * 16
                gb = np.full((1, gp), capi.BASE_N, np.uint8)
                gq = np.zeros((1, gp), np.uint8)
                gs = np.full((1, gp), capi.STRAND_NONE, np.uint8)
                gb[0, :len(m)] = b[site, m]; gq[0, :len(m)] = q[site, m]; gs[0, :len(m)] = s[site, m]
                one.call_host_lists(gb, gq, gs, ref[site:site + 1], lists[site:site + 1], len(m))
        return 1e3 * (time.perf_counter() - t0)

    c0 = st32[sites].astype(np.int64)
    c1 = st32[sites + 1].astype(np.int64)
    idx = np.concatenate([np.arange(x, y) for x, y in zip(c0, c1)])
    sub_cells = torch.from_numpy(cells32[idx].view(np.int32)).pin_memory().numpy().view(np.uint32)
    sub_aux = torch.from_numpy(aux32[idx].view(np.int32)).pin_memory().numpy().view(np.uint32)
    sub_st = np.zeros(K + 1, np.uint32)
    sub_st[1:] = np.cumsum(c1 - c0)
    sub_ref = np.ascontiguousarray(ref[sites])

    def batch():
        t = capi.BvSparseTile(sub_cells.ctypes.data, sub_aux.ctypes.data, sub_st.ctypes.data, sub_ref.ctypes.data, None, K, N,
                              capi.CELLS_U32, capi.OUT_COMPACT)
        t0 = time.perf_counter()
        check(lib.bv_tile_submit_sparse_calls(ctx, 0, C.byref(t)), "submit")
        check(lib.bv_tile_wait_calls_compact(ctx, 0, C.byref(pb), C.byref(pf), C.byref(nf), calls_buf.ctypes.data, S, C.byref(n),
                                             groups_buf.ctypes.data), "wait")
        return 1e3 * (time.perf_counter() - t0)

    per_site()
    batch()
    ps = [per_site() for _ in range(3)]
    bt = [batch() for _ in range(args.tiles)]
    assert int(n.value) == K
    result["per_site"] = {"called_sites": K, "device_round_trips_per_site": 3 + G, "per_site_ms_median": float(np.median(ps)),
                          "batch_ms_median": float(np.median(bt)), "speedup": float(np.median(ps) / np.median(bt))}
    one.close()
    eng.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
