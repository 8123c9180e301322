"""Time bv_ranksum_test (kernel K9, ref_vs_alt_ranksumtest of free-standing problems) on three shapes, plus the bound case.

    python tools/ranksum_bench.py [--reps 20] [--warmup 3] [--out FILE]

Shapes (REF A; ALT C and G; bases drawn A 60 %, C 20 %, G 10 %, T / N / indel the rest):
  mapq_10k_x_1k    10,000 problems x 1,000 reads, mapq-like values (0, 20, 37, 60): the histogram path;
  one_100k         one problem of 100,000 reads, mapq-like values: the largest call the C++ mirror makes for one site;
  wide_2k_x_1k     2,000 problems x 1,000 reads, values over the whole int32 range: the pairwise path;
  wide16_100_x_20k 100 problems x 20,000 reads, values 0..65535: the window path;
  one_100k_int32   one problem of 100,000 reads over the whole int32 range: the costliest kind of problem (pairwise).
For each: K9 alone (CUDA events around the kernel, bv_last_ranksum_kernel_time) and the whole blocking call on a host clock
(checks, copies in, K9, copy out), medians over --reps calls after --warmup.  The card's name and power limit are read in the
same run and printed with the numbers.
"""
import argparse
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


def problems(rng, n_problems, n_reads, kind):
    total = n_problems * n_reads
    bases = rng.choice(8, total, p=[0.6, 0.2, 0.1, 0.04, 0.0, 0.04, 0.01, 0.01]).astype(np.uint8)
    if kind == "mapq":
        values = rng.choice(np.array([60, 60, 60, 37, 20, 0], np.int32), total)
    elif kind == "u16":
        values = rng.integers(0, 65536, total).astype(np.int32)
    else:
        values = rng.integers(-(2 ** 31), 2 ** 31 - 1, total, endpoint=True).astype(np.int32)
    start = np.arange(n_problems + 1, dtype=np.uint64) * np.uint64(n_reads)
    ref = np.full(n_problems, ord("A"), np.uint8)
    mask = np.full(n_problems, 0b0110, np.uint8)
    return bases, values, start, ref, mask


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import basevar_b200 as bv

    if not torch.cuda.is_available():
        raise SystemExit("ranksum_bench: no CUDA device (there is nothing to time on the CPU)")
    eng = bv.BaseTypeEngine(device=0, max_samples=100000, max_sites=0, n_slots=0)
    rng = np.random.default_rng(2026)
    result = dict(gpu_info(), reps=args.reps)
    for name, n_problems, n_reads, kind in (("mapq_10k_x_1k", 10000, 1000, "mapq"), ("one_100k", 1, 100000, "mapq"),
                                            ("wide_2k_x_1k", 2000, 1000, "int32"), ("wide16_100_x_20k", 100, 20000, "u16"),
                                            ("one_100k_int32", 1, 100000, "int32")):
        p = problems(rng, n_problems, n_reads, kind)
        reps = args.reps if name != "one_100k_int32" else max(3, args.reps // 4)
        k9, call = [], []
        eng.set_profiling(True)
        for i in range(args.warmup + reps):
            t0 = time.perf_counter()
            eng.ranksum_test(*p)
            t1 = time.perf_counter()
            if i >= args.warmup:
                call.append((t1 - t0) * 1e3)
                k9.append(eng.last_ranksum_kernel_time())
        eng.set_profiling(False)
        result[name] = {"problems": n_problems, "reads_per_problem": n_reads, "values": kind, "reps": reps,
                        "k9_ms_median": float(np.median(k9)), "k9_ms_min": float(np.min(k9)), "k9_ms_max": float(np.max(k9)),
                        "call_ms_median": float(np.median(call)), "call_ms_min": float(np.min(call))}
    eng.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
