"""Time a C2-shaped pileup that is already in device memory, in each of its forms, next to the host route of the same cells.

    python tools/device_tiles_bench.py [--sites 262144] [--samples 1000] [--reps 20] [--out FILE]

The tile is the synthetic C2 genome (0.1x, 1,000 samples, 262,144 sites) in BV_CELLS_U16 form.  Medians of --reps calls after
--warmup, each call timed on its own:
  device_sparse_records   bv_tile_run_device_sparse, BV_OUT_RECORDS (CUDA events around the call on its stream; the result
                          tensors are allocated once, before the timed calls)
  device_sparse_compact   bv_tile_run_device_sparse, BV_OUT_COMPACT (CUDA events)
  host_sparse_pinned      bv_tile_submit_sparse + bv_tile_wait of the same cells from pinned host memory (host clock around
                          the submit and the wait, which ends in a device synchronise)
  device_dense            bv_tile_run_device on the dense planes of the same pileup (CUDA events)
The records of every route are compared with those of the dense route, byte for byte.  HBM bytes written per site are counted
from the shapes and the tile's number of full records (what the code writes, not a measurement).  The card's name and power
limit are read in the same run and written with the numbers.
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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import basevar_b200 as bv
    from basevar_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("device_tiles_bench: no CUDA device (there is nothing to time on the CPU)")
    info = gpu_info()
    S, N = args.sites, args.samples
    pitch = (N + 15) // 16 * 16
    model = bv.synth.make_model(seed=2024, coverage=0.1, variant_frac=0.01, multi_frac=0.1)
    cells, _, st, ref = bv.synth_fill_sparse_host(model, 0, S, N)
    words, _, st16 = bv.sparse_encode16(cells, st, pinned=True)
    ref_p = torch.from_numpy(ref).pin_memory().numpy()
    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=S, n_slots=1, min_af=bv.cli_min_af(0.01, N))
    dev = torch.device("cuda")
    d_words = torch.from_numpy(np.ascontiguousarray(words)).view(torch.int16).to(dev)
    d_st = torch.from_numpy(np.ascontiguousarray(st16)).view(torch.int32).to(dev)
    d_ref = torch.from_numpy(ref).to(dev)
    # the dense planes of the same pileup, generated on the device
    eng.synth_set_model(model)
    planes = torch.empty((3, S, pitch), dtype=torch.uint8, device=dev)
    d_ref_dense = torch.empty(S, dtype=torch.uint8, device=dev)
    eng.synth_fill_device(0, S, N, pitch, planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), None, d_ref_dense.data_ptr(),
                          torch.cuda.current_stream().cuda_stream)
    d_dense_out = torch.empty((S, 128), dtype=torch.uint8, device=dev)
    host_out = np.zeros(S, capi.SITE_OUT_DTYPE)
    tile = capi.BvSparseTile(words.ctypes.data, None, st16.ctypes.data, ref_p.ctypes.data, None, S, N, capi.CELLS_U16, 0)
    stream = torch.cuda.current_stream()

    # the result tensors of each form, allocated once outside the timed calls
    outs = {c: eng.device_result(S, compact=c) for c in (False, True)}

    def dev_sparse(compact):
        return lambda: eng.call_device_sparse(d_words, d_st, d_ref, N, compact=compact, out=outs[compact])

    def dense():
        eng.call_device(planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), d_ref_dense.data_ptr(), S, N, pitch,
                        d_dense_out.data_ptr(), stream.cuda_stream)

    def host_call():
        eng._check(eng.lib.bv_tile_submit_sparse(eng._ctx, 0, C.byref(tile)), "bv_tile_submit_sparse")
        eng._check(eng.lib.bv_tile_wait(eng._ctx, 0, host_out.ctypes.data), "bv_tile_wait")

    def time_events(fn):
        ts = []
        for i in range(args.warmup + args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            if i >= args.warmup:
                ts.append(e0.elapsed_time(e1))
        return ts

    def time_host(fn):
        ts = []
        for i in range(args.warmup + args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            t1 = time.perf_counter()
            if i >= args.warmup:
                ts.append(1e3 * (t1 - t0))
        return ts

    res = {}
    res["device_sparse_records"] = time_events(dev_sparse(False))
    res["device_sparse_compact"] = time_events(dev_sparse(True))
    res["host_sparse_pinned"] = time_host(host_call)
    res["device_dense"] = time_events(dense)
    # the records of every route are the bytes of the dense route
    torch.cuda.synchronize()
    want = bv.device_to_numpy(d_dense_out, capi.SITE_OUT_DTYPE)
    rec = eng.call_device_sparse(d_words, d_st, d_ref, N).to_numpy()
    cmp = eng.call_device_sparse(d_words, d_st, d_ref, N, compact=True).to_numpy()
    expanded = np.zeros(S, capi.SITE_OUT_DTYPE)
    eng.expand_compact(cmp["brief"], cmp["full"], ref, expanded)
    same = {"device_sparse_records": rec["records"].tobytes() == want.tobytes(),
            "device_sparse_compact": expanded.tobytes() == want.tobytes(),
            "host_sparse_pinned": host_out.tobytes() == want.tobytes()}
    n_full = len(cmp["full"])
    planes_b = 3 * pitch
    written = {   # bytes the kernels write to device memory per site (K0 planes, K1..KF records, K1 briefs, K7 full records)
        "device_sparse_records": {"planes": planes_b, "records": 128},
        "device_sparse_compact": {"planes": planes_b, "records_scratch": 128, "briefs": 8, "full_records": round(128 * n_full / S, 2)},
        "host_sparse_pinned": {"planes": planes_b, "records": 128},
        "device_dense": {"records": 128},
    }
    for k, v in written.items():
        v["total"] = round(sum(v.values()), 2)
    out = {"card": info, "shape": {"sites": S, "samples": N, "format": "BV_CELLS_U16", "cells": int(st16[-1]),
                                   "full_records": n_full, "full_fraction": round(n_full / S, 4)},
           "median_ms": {k: round(float(np.median(v)), 4) for k, v in res.items()},
           "min_ms": {k: round(float(np.min(v)), 4) for k, v in res.items()},
           "reps": args.reps, "records_equal_dense": same, "hbm_bytes_written_per_site_counted": written}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    eng.close()
    if not all(same.values()):
        raise SystemExit(f"device_tiles_bench: records differ from the dense route: {same}")


if __name__ == "__main__":
    main()
