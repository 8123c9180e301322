"""Time K8 bv_list_kernel (BaseType::lrt(list) per site) on a C2-shaped device-resident tile beside the standard step.

    python tools/lists_bench.py [--sites 262144] [--samples 1000] [--reps 20] [--out FILE]

The tile is the synthetic C2 genome (0.1x, 1,000 samples) generated on the device.  Two list inputs:
  acgt      the list A,C,G,T at every site (every covered site costs one pass over its row);
  ref_alt2  [REF, one ALT] at 2 % of the sites (the ALT is the site's most frequent non-REF base), the others empty.
For each: K8 alone (CUDA events around the kernel, bv_last_list_kernel_time) and the whole lists step
(bv_tile_run_device_lists: standard kernels + K8), next to the standard step (bv_tile_run_device), all CUDA events over
--reps launches after a warm-up.  The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

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
        raise SystemExit("lists_bench: no CUDA device (there is nothing to time on the CPU)")
    S, N = args.sites, args.samples
    pitch = (N + 15) // 16 * 16
    maf = bv.cli_min_af(0.01, N)
    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=0, n_slots=0, min_af=maf)
    eng.synth_set_model(bv.synth.make_model(seed=2024, coverage=0.1, variant_frac=0.019))
    dev = torch.device("cuda:0")
    planes = [torch.empty((S, pitch), dtype=torch.uint8, device=dev) for _ in range(3)]
    ref = torch.empty(S, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    eng.synth_fill_device(0, S, N, pitch, planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), None, ref.data_ptr(), st)
    d_out = torch.zeros(S * 128, dtype=torch.uint8, device=dev)
    d_lrt = torch.zeros(S * 64, dtype=torch.uint8, device=dev)
    ptrs = (planes[0].data_ptr(), planes[1].data_ptr(), planes[2].data_ptr(), ref.data_ptr())

    def standard():
        eng.call_device(*ptrs, S, N, pitch, d_out.data_ptr(), st)

    def lists_step(d_lists):
        eng.call_device_lists(*ptrs, d_lists.data_ptr(), S, N, pitch, d_out.data_ptr(), d_lrt.data_ptr(), st)

    def time_step(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.reps

    def time_k8(d_lists):
        eng.set_profiling(True)
        ms = []
        for i in range(args.warmup + args.reps):
            lists_step(d_lists)
            t = eng.last_list_kernel_time()
            if i >= args.warmup:
                ms.append(t)
        eng.set_profiling(False)
        return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

    standard()
    torch.cuda.synchronize()
    recs = d_out.cpu().numpy().view(capi.SITE_OUT_DTYPE)
    ref_h = ref.cpu().numpy()
    acgt = np.tile(np.arange(4, dtype=np.uint8), (S, 1))
    rng = np.random.default_rng(7)
    ref_alt = np.full((S, 4), capi.LIST_END, np.uint8)
    pick = np.nonzero(rng.random(S) < 0.02)[0]
    rc = np.array(["ACGT".find(chr(c).upper()) for c in ref_h[pick]])
    dep = recs["depth"][pick].astype(np.int64)
    dep[np.arange(len(pick)), np.maximum(rc, 0)] = -1
    ref_alt[pick, 0] = np.maximum(rc, 0)
    ref_alt[pick, 1] = np.argmax(dep, axis=1)
    result = dict(gpu_info(), sites=S, samples=N, min_af=maf, reps=args.reps,
                  covered_sites=int(((recs["depth"].sum(axis=1) + recs["depth_other"]) > 0).sum()),
                  standard_step_ms=time_step(standard))
    for name, lists in (("acgt", acgt), ("ref_alt2", ref_alt)):
        d_lists = torch.from_numpy(lists).to(dev)
        med, lo, hi = time_k8(d_lists)
        result[name] = {"sites_with_list": int((lists[:, 0] != capi.LIST_END).sum()), "k8_ms_median": med, "k8_ms_min": lo,
                        "k8_ms_max": hi, "lists_step_ms": time_step(lambda: lists_step(d_lists))}
    eng.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
