#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native basetype core (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2|C3|C4|C5] [--impl ours|reference] [--dump-outputs DIR]

metric  : sample-sites/s of the BaseType core (likelihoods, EM, LRT, QUAL, strand-bias Fisher)
workload: N = 1: BASELINE.json configs[1] = synthetic 1,000 samples x 1 Mb at 0.1x ("C2", SURVEY.md 8d).
          N > 1: BASELINE.json configs[3] = synthetic 100,000 samples x 64 Mb at 0.1x ("C4"), the region cut into one
          contiguous shard per GPU at 100-kb task boundaries; every rank times the first `sites_per_gpu` sites of ITS shard
          (the whole shard is 19 TB / N of planes and cannot be resident).  --config overrides either.
step    : one pass of the basetype core (kernels K1 count, K2 scalar, K3 bound, K4a histograms, K4b EM tasks + decisions)
          over the whole per-GPU workload (S sites x N samples).
value   : whole-job sample-sites/s with the planes resident in HBM (kernels only, CUDA events, max over ranks).
e2e     : the same metric through the C ABI with HOST buffers, copies inside the timed region, tiles pipelined over the
          slots' streams and over the steps: sparse tiles (pinned u16 words of the covered reads -> bv_tile_submit_sparse: H2D, K0
          expand, K1..K4, D2H of the 128-byte records -> bv_tile_wait).  e2e_from_cells: from one u32 per covered cell (what a
          packer holds), nothing prepared outside the clock: shipped as is (BV_CELLS_U32) or re-coded to u16 words by the host
          encoder on worker threads; both listed, the faster one reported.  e2e_dense: dense pinned planes (bv_tile_submit).  fabric: bare pinned copies of the e2e leg's bytes, all ranks at once.
roofline: algorithmic bytes S*(3N+128) per step / average step time (all kernels), against MEASURED_PEAKS.json hbm_gbs; the
          per-kernel durations are measured live with CUDA events between the kernels (bv_set_profiling).
configs : N = 1 only: the other BASELINE.json shapes (C3, C4 shard shape, C5 in both EM abs modes), each with value, roofline,
          per-kernel times and the reference CPU baseline on a sub-range of >= 1e9 sample-sites of the same planes.
cpu_baseline: the UNMODIFIED reference (oracle/_ref/libbvref.so: BaseType ctor + lrt() + strand_bias) on the host cores.
dump    : --dump-outputs DIR writes the records of the last timed step (rank 0's) as DIR/<field>.npy, so that two builds can be
          compared output for output on the same seeded inputs.
Multi-GPU: sites are sharded by contiguous region, one process per GPU, no collective on the data path
          (weak scaling: every GPU gets its own S sites); torch.distributed only for the barrier / max-time.
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sample-sites/sec, BaseType EM+LRT"
UNIT = "sample-sites/s"
C4_REGION = 64_000_000

# sites per GPU of the resident (kernel-only) leg of each workload; whole rounds of the count kernel's persistent warps
RESIDENT_SITES = {"C2": 1_000_000, "C3": 303_104, "C4": 37_888, "C5": 1_000_000}
BASELINE_CONFIG = {"C2": "BASELINE.json configs[1]", "C3": "BASELINE.json configs[2]",
                   "C4": "BASELINE.json configs[3], one region shard per GPU", "C5": "BASELINE.json configs[4]"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(config, n_samples, sites):
    """DRAM bytes (read + write) of one step from the committed `ncu --set full` capture of this workload, or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    e = t.get(config)
    if not e or e.get("n_samples") != n_samples or e.get("sites") != sites:
        return None
    return e["dram_bytes_per_step"]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank's host threads -- and, by first touch, its pinned staging buffers -- on the CPUs next to its GPU (one
    host worker per GPU, as in the C++ runner).  Returns the CPU list, or None when the topology cannot be read."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        if cpus and len(cpus) < ncpu:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


def workload_of(args, world):
    """(name, config dict, sites per GPU, site0 of `rank`) of the main workload."""
    import basevar_b200 as bv
    from basevar_b200 import shard
    name = args.config or ("C2" if world == 1 else "C4")
    cfg = dict(bv.synth.CONFIGS[name])
    S = int(args.sites or RESIDENT_SITES[name])

    def site0(rank):
        if name == "C4":   # contiguous region shards cut at 100-kb task boundaries (src/basetype_caller.cpp:474-510)
            return shard.shard_region(0, C4_REGION, world)[rank][0]
        return shard.rank_site_range(rank, world, S)[0]
    return name, cfg, S, site0


def config_block(name, cfg, S, maf, abs_mode, world):
    """The `config` object: identical in both arms (the driver compares them)."""
    n = cfg["n_samples"]
    pitch = (n + 15) // 16 * 16
    return {"workload": f"{name}: synthetic {n} samples x {S} sites per GPU at coverage {cfg['coverage']} ({BASELINE_CONFIG[name]})",
            "n_samples": n, "sites_per_gpu": S, "min_af": maf, "em_abs_mode": abs_mode,
            "l2": "inputs (3 planes, %.2f GB per GPU) larger than L2; no flush needed" % (3 * S * pitch / 1e9),
            "parallelism": f"region-sharded x{world}, no collective"}


def host_threads(world):
    return max(1, (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)) // max(world, 1))


def fill_sparse_parallel(model, site0, S, n_samples, n_threads):
    """Host twin of the generator in sparse form, over `n_threads` threads (ctypes calls release the GIL)."""
    import basevar_b200 as bv
    n_threads = max(1, min(n_threads, S // 256 or 1))
    cuts = [S * i // n_threads for i in range(n_threads + 1)]
    with cf.ThreadPoolExecutor(n_threads) as ex:
        parts = list(ex.map(lambda i: bv.synth_fill_sparse_host(model, site0 + cuts[i], cuts[i + 1] - cuts[i], n_samples), range(n_threads)))
    cells = np.concatenate([p[0] for p in parts])
    site_start = np.zeros(S + 1, np.uint32)
    off = 0
    for i, p in enumerate(parts):
        site_start[cuts[i]:cuts[i + 1] + 1] = p[2] + np.uint32(off)
        off += p[0].shape[0]
    ref = np.concatenate([p[3] for p in parts])
    return cells, site_start, ref


def pinned(arr):
    import torch
    tdt = {np.dtype(np.uint32): torch.int32, np.dtype(np.uint16): torch.int16, np.dtype(np.uint8): torch.uint8}[arr.dtype]
    t = torch.empty(max(arr.shape[0], 1), dtype=tdt, pin_memory=True).numpy().view(arr.dtype)[:arr.shape[0]]
    t[:] = arr
    return t


def reference_tile(planes, n_samples, maf, abs_mode, cores):
    """The unmodified reference over dense host planes: (sample-sites/s, seconds of the slowest thread in reference code)."""
    from oracle import loader as L
    b, q, s, r = planes
    _, core_s = L.ref_tile(b, q, s, r, n_samples, maf, dblabs=bool(abs_mode), n_threads=cores)
    return b.shape[0] * n_samples / core_s, core_s


def reference_arm(args, rank, world):
    """--impl reference: the unmodified reference on the host cores, bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import loader as L
    import basevar_b200 as bv
    cores = os.cpu_count() or 1
    if L.load_ref(bool(args.abs_mode)) is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libbvref.so was not built (needs /root/reference at build time)"}))
        return
    name, cfg, S, site0 = workload_of(args, world)
    n_samples = cfg["n_samples"]
    maf = bv.cli_min_af(0.01, n_samples)
    model = bv.synth.make_model(cfg["seed"], cfg["coverage"], cfg["variant_frac"], cfg["multi_frac"])
    # every site of the workload when that is about a second of reference time per step, else a prefix of >= 1e9 sample-sites
    sites = int(min(S, max(args.ref_min_sample_sites // n_samples, 2000)))
    nt = max(1, min(cores, sites // 512))
    cuts = [sites * i // nt for i in range(nt + 1)]
    with cf.ThreadPoolExecutor(nt) as ex:   # host twin of the generator (plain C loop of libbasevar_b200.so; no GPU involved)
        parts = list(ex.map(lambda i: bv.synth_fill_host(model, site0(0) + cuts[i], cuts[i + 1] - cuts[i], n_samples), range(nt)))
    planes = tuple(np.concatenate([p[k] for p in parts]) for k in (0, 1, 2, 4))
    times, cores_t = [], []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        _, core_s = reference_tile(planes, n_samples, maf, args.abs_mode, cores)
        wall = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(wall); cores_t.append(core_s)
    # the slowest thread's time inside BaseType/lrt/strand_bias (the shim's BatchInfo fill is not charged)
    t = float(np.mean(cores_t))
    value = sites * n_samples / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": config_block(name, cfg, S, maf, args.abs_mode, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": f"first {sites} of the {S} sites x {n_samples} samples ({sites * n_samples:.3g} sample-sites per step); "
                                   f"reference BaseType ctor+lrt()+strand_bias per site, {cores} threads over contiguous site ranges; "
                                   f"time = slowest thread inside the reference code (wall incl. BatchInfo fill {1e3 * float(np.mean(times)):.1f} ms)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "libraries": "compute: oracle/_ref/libbvref.so (unmodified reference sources); libbasevar_b200.so is mapped for the host "
                     "twin of the synthetic generator only (no CUDA call, no kernel)",
    }
    print(json.dumps(line))


class Resident:
    """Device-resident planes of one workload on this rank, and the kernel-only timing over them."""

    def __init__(self, bv, torch, dev, local_rank, name, cfg, S, site0, abs_mode, n_slots=0, tile_sites=0):
        self.torch, self.name, self.cfg, self.S = torch, name, cfg, S
        self.N = cfg["n_samples"]
        self.pitch = (self.N + 15) // 16 * 16
        self.maf = bv.cli_min_af(0.01, self.N)
        self.abs_mode = abs_mode
        self.eng = bv.BaseTypeEngine(device=local_rank, max_samples=self.N, max_sites=tile_sites, n_slots=n_slots, min_af=self.maf, abs_mode=abs_mode)
        self.model = bv.synth.make_model(cfg["seed"], cfg["coverage"], cfg["variant_frac"], cfg["multi_frac"])
        self.eng.synth_set_model(self.model)
        self.base, self.qual, self.strand = (torch.empty((S, self.pitch), dtype=torch.uint8, device=dev) for _ in range(3))
        self.ref = torch.empty(S, dtype=torch.uint8, device=dev)
        self.out = torch.empty(S * 128, dtype=torch.uint8, device=dev)
        self.stream = torch.cuda.current_stream().cuda_stream
        self.eng.synth_fill_device(site0, S, self.N, self.pitch, self.base.data_ptr(), self.qual.data_ptr(), self.strand.data_ptr(), 0,
                                   self.ref.data_ptr(), self.stream)
        torch.cuda.synchronize()

    def step(self):
        self.eng.call_device(self.base.data_ptr(), self.qual.data_ptr(), self.strand.data_ptr(), self.ref.data_ptr(), self.S, self.N, self.pitch,
                             self.out.data_ptr(), self.stream)

    def timed(self, steps, warmup, barrier):
        """(total ms, per-step ms list, launches) of `steps` steps after `warmup`."""
        torch = self.torch
        for _ in range(max(warmup, 3)):
            self.step()
        barrier()
        l0 = self.eng.launch_count
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            self.step()
            ev[i + 1].record()
        barrier()
        return ev[0].elapsed_time(ev[-1]), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], self.eng.launch_count - l0

    def kernel_ms(self, steps):
        """Live per-kernel durations (CUDA events between the kernels, recorded by the library), averaged."""
        self.eng.set_profiling(True)
        ks, es = None, None
        for _ in range(steps):
            self.step()
            k, e = self.eng.last_kernel_times(), self.eng.last_em_kernel_times()
            ks = k if ks is None else {n: ks[n] + v for n, v in k.items()}
            es = e if es is None else {n: es[n] + v for n, v in e.items()}
        self.eng.set_profiling(False)
        out = {n: v / steps for n, v in ks.items()}
        out.update({n: v / steps for n, v in es.items()})
        out["bv_em_kernel"] = out.pop("bv_em_kernel")   # = bv_hist_kernel + bv_em_task_kernel (bv_fisher_kernel follows them)
        return out

    def records(self):
        import basevar_b200 as bv
        return self.out.cpu().numpy().view(bv.SITE_OUT_DTYPE)

    def host_planes(self, ns):
        """The first ns rows of the planes as host arrays (the same bytes the host twin of the generator writes)."""
        return tuple(t[:ns].cpu().numpy() for t in (self.base, self.qual, self.strand, self.ref))

    def roofline(self, avg_ms, kernel_ms, peak, peak_src):
        algo = self.S * (3 * self.N + 128)
        ach = algo / (avg_ms * 1e-3) / 1e9
        k1b = self.S * (2 * self.N + 128)
        k1 = k1b / (kernel_ms["bv_count_kernel"] * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": load_traffic(self.name, self.N, self.S), "peak_source": peak_src, "algorithmic_bytes_per_launch": algo,
                "kernel": "the step's kernels together (K1 bv_count_kernel, K2 bv_scalar_kernel, K3 bv_bound_kernel, K4a bv_hist_kernel, "
                          "K4b bv_em_task_kernel, bv_fisher_kernel; bv_em_kernel = K4a + K4b)",
                "avg_launch_ms": avg_ms, "kernel_ms": kernel_ms,
                # K1 alone moves 2 of the 3 planes (base + strand; the qual plane is read only where the result depends on it)
                "k1_bytes": k1b, "k1_achieved": k1, "k1_frac": k1 / peak}

    def close(self):
        self.eng.close()
        del self.base, self.qual, self.strand, self.ref, self.out
        self.torch.cuda.empty_cache()


def cpu_baseline(res, ns, cores):
    from oracle import loader as L
    if L.load_ref(bool(res.abs_mode)) is None:
        return {"value": None, "unit": UNIT, "cores": cores, "kind": "reference", "sample": "oracle/_ref not built"}
    v, core_s = reference_tile(res.host_planes(ns), res.N, res.maf, res.abs_mode, cores)
    return {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "seconds": core_s,
            "sample": f"first {ns} sites x {res.N} samples of the same planes ({ns * res.N:.3g} sample-sites); unmodified reference "
                      f"BaseType ctor+lrt()+strand_bias, {cores} threads, slowest thread's time in reference code"}


DUMP_SITES = 1 << 18   # sites per dump: 156 bytes of .npy each, about 41 MB in all


def dump_outputs(path, rec):
    """One DIR/<field>.npy per field of struct bv_site_out: counts, codes and flags as float32 (exact, all are below 2^24), the
    floating-point fields as float64, and site.npy with the site indices.  More than DUMP_SITES sites: the same seeded sample of
    sites every run."""
    os.makedirs(path, exist_ok=True)
    S = rec.shape[0]
    site = np.arange(S) if S <= DUMP_SITES else np.sort(np.random.default_rng(0).choice(S, DUMP_SITES, replace=False))
    rec = rec[site]
    np.save(os.path.join(path, "site.npy"), site.astype(np.float64))
    for f in rec.dtype.names:
        if not f.startswith("reserved"):
            np.save(os.path.join(path, f + ".npy"), rec[f].astype(np.float64 if rec[f].dtype.kind == "f" else np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the kernel-only leg (the headline value)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=["C2", "C3", "C4", "C5"], help="main workload (default: C2 on one GPU, C4 shards on several)")
    ap.add_argument("--sites", type=int, default=0, help="sites per GPU of the main workload (default: RESIDENT_SITES)")
    ap.add_argument("--abs-mode", type=int, default=0, help="0 = as-built int abs() in EM, 1 = fabs")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--slots", type=int, default=4, help="in-flight tiles of the e2e legs (each slot: a stream, device planes, pinned staging)")
    ap.add_argument("--tile-sites", type=int, default=0, help="sites per host tile of the e2e legs (default 262144: ~40 us of copy set-up per tile; one K1 round, 9472, for long rows)")
    ap.add_argument("--e2e-sites", type=int, default=0, help="sites per GPU of the e2e legs (default: the workload's, 2 tiles for C4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the `configs` block (C3, C4 shape, C5 x 2 abs modes)")
    ap.add_argument("--no-e2e-extra", action="store_true", help="skip the e2e_sparse_u32 / e2e_dense / fabric legs")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not bind the rank to the CPUs next to its GPU")
    ap.add_argument("--ref-min-sample-sites", type=int, default=1_000_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step as DIR/<field>.npy (a fixed sample of %d sites when there are more); "
                         "with several GPUs, rank 0's shard only" % DUMP_SITES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the records of the device path: not with --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import basevar_b200 as bv
    from basevar_b200 import capi, shard
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the basetype core has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 and not args.no_numa_bind else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = capi.load_library()
    peak, peak_src = load_peaks()
    cores = os.cpu_count() or 1
    n_host = host_threads(world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    name, cfg, S, site0_of = workload_of(args, world)
    site0 = site0_of(rank)
    n_samples = cfg["n_samples"]
    pitch = (n_samples + 15) // 16 * 16
    long_rows = n_samples > 4096
    tile_sites = int(args.tile_sites or (9472 if long_rows else 262144))
    tile_sites = min(tile_sites, S)
    main_res = Resident(bv, torch, dev, local_rank, name, cfg, S, site0, args.abs_mode, n_slots=args.slots, tile_sites=tile_sites)
    eng, model, maf = main_res.eng, main_res.model, main_res.maf

    # ---- kernel-only leg: the planes are resident in HBM ---------------------------------------------------------
    clocks = ClockSampler(local_rank)
    clocks.start()
    total_ms, per_step_ms, launches = main_res.timed(args.steps, args.warmup, barrier)
    total_ms_max = shard.max_over_ranks(total_ms, dev)
    value = world * S * n_samples * args.steps / (total_ms_max * 1e-3)
    dev_rec = main_res.records()
    kernel_ms = main_res.kernel_ms(args.steps)

    # ---- end to end through the C ABI with host buffers --------------------------------------------------------
    # sparse tiles: pinned host arrays of the covered cells -> bv_tile_submit_sparse (H2D of the cells, K0 expand, K1..K4, D2H of
    # the 128-byte records straight into a pinned buffer) -> bv_tile_wait; tiles and steps pipelined over 3 slots
    Se = int(args.e2e_sites or (2 * tile_sites if long_rows else S))
    Se = min(Se, S)
    t_prep = time.perf_counter()
    cells32, start32, s_ref = fill_sparse_parallel(model, site0, Se, n_samples, n_host)
    cells32, start32, s_ref = pinned(cells32), pinned(start32), pinned(s_ref)
    t_prep = time.perf_counter() - t_prep
    t1 = time.perf_counter()
    words16, _, start16 = bv.sparse_encode16(cells32, start32, pinned=True)   # 2 bytes per cell, samples delta-coded
    t_prep16 = time.perf_counter() - t1
    rec_sp = torch.empty(Se * 128, dtype=torch.uint8, pin_memory=True).numpy().view(bv.SITE_OUT_DTYPE)
    e2e_launches = 0

    def sparse_leg(cell_words, starts, steps, compact=False):
        """Tiles of the given cell words through the slots, `steps` passes back to back.  compact: BV_OUT_COMPACT tiles (8 bytes
        per site + a full record for the sites that need one, written by the device into the slot's pinned staging)."""
        nonlocal e2e_launches
        rec_sp[:] = 0
        tiles = eng.sparse_tiles(cell_words, starts, s_ref, n_samples, out_pinned=rec_sp, compact=compact)
        d2h = [0]

        def expand(s0, ns, briefs, full):   # verification pass only (not timed): rebuild the records from the compact form
            d2h[0] += 8 * ns + 128 * len(full)
            eng.expand_compact(briefs, full, s_ref[s0:s0 + ns], rec_sp[s0:s0 + ns])

        eng.run_sparse_tiles(tiles, 1, compact=expand if compact else None)   # warm-up; fills rec_sp
        records = rec_sp.tobytes()
        # every slot sizes its cell buffer at its first tile (cudaMalloc synchronises the device): a pass that reaches all slots
        eng.run_sparse_tiles(tiles, -(-args.slots // len(tiles)))
        barrier()
        l0, up0 = eng.launch_count, eng.h2d_bytes
        t0 = time.perf_counter()
        eng.run_sparse_tiles(tiles, steps)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        dt_max = shard.max_over_ranks(dt, dev)
        e2e_launches += eng.launch_count - l0
        return {"value": world * Se * n_samples / dt_max, "ms": 1e3 * dt_max, "uploaded": (eng.h2d_bytes - up0) // steps,
                "records": records if compact else rec_sp.tobytes(), "tiles": len(tiles), "d2h": d2h[0] if compact else Se * 128}

    # results in compact form when the records are a sizeable part of the traffic (short rows: 128 bytes per site against 2 bytes
    # per covered read); for 100,000-sample rows they are under 1 % of it and travel whole
    use_compact = Se * 128 > 0.05 * words16.shape[0] * 2
    leg16 = sparse_leg(words16, start16, args.e2e_steps, compact=use_compact)
    same_sp = bool(dev_rec[:Se].tobytes() == leg16["records"])
    leg16_full = sparse_leg(words16, start16, max(3, args.e2e_steps // 2), compact=not use_compact)

    # the same with the host encoder inside the clock: u32 cells (what a packer has per covered read) -> u16 words by worker
    # threads, one tile each, into a ring of pinned buffers; the main thread submits in order
    def from_cells_leg(steps):
        nonlocal e2e_launches
        n_slots = args.slots
        workers = max(1, min(n_host - 1, 12))
        ring = n_slots + workers
        tiles = []
        for s0 in range(0, Se, tile_sites):
            ns = min(tile_sites, Se - s0)
            c0, c1 = int(start32[s0]), int(start32[s0 + ns])
            tiles.append((s0, ns, c0, c1, np.ascontiguousarray(start32[s0:s0 + ns + 1] - np.uint32(c0))))
        max_cells = max(t[3] - t[2] for t in tiles)
        cap = int(lib.bv_sparse_encode16_bound(max_cells, tile_sites, n_samples)) + (1 << 20) // 31 + 64
        bufs = [(torch.empty(cap, dtype=torch.int16, pin_memory=True).numpy().view(np.uint16),
                 torch.empty(tile_sites + 1, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)) for _ in range(ring)]

        def encode(k):
            s0, ns, c0, c1, st = tiles[k % len(tiles)]
            w, so = bufs[k % ring]
            n = C.c_uint64(0)
            rc = lib.bv_sparse_encode16(cells32[c0:].ctypes.data if c1 > c0 else cells32.ctypes.data, None, st.ctypes.data, ns, w.ctypes.data, None, cap,
                                        so.ctypes.data, C.byref(n))
            if rc != capi.BV_OK:
                raise bv.BvError(lib.bv_last_error(None).decode())
            return capi.BvSparseTile(w.ctypes.data, None, so.ctypes.data, s_ref[s0:].ctypes.data, rec_sp[s0:].ctypes.data, ns, n_samples, capi.CELLS_U16, 0)

        def run(n_steps):
            total = n_steps * len(tiles)
            with cf.ThreadPoolExecutor(workers) as ex:
                futs, pending, slot, nxt = {}, [], 0, 0
                for k in range(total):
                    while nxt < total and nxt < k + workers:   # tile nxt's buffer was last used by tile nxt - ring, waited for below
                        futs[nxt] = ex.submit(encode, nxt)
                        nxt += 1
                    if len(pending) == n_slots:
                        eng._check(lib.bv_tile_wait(eng._ctx, pending.pop(0), None), "bv_tile_wait")
                    t = futs.pop(k).result()
                    eng._check(lib.bv_tile_submit_sparse(eng._ctx, slot, C.byref(t)), "bv_tile_submit_sparse")
                    pending.append(slot)
                    slot = (slot + 1) % n_slots
                for ps in pending:
                    eng._check(lib.bv_tile_wait(eng._ctx, ps, None), "bv_tile_wait")

        rec_sp[:] = 0
        run(-(-n_slots // len(tiles)))   # warm-up that reaches every slot
        barrier()
        l0 = eng.launch_count
        t0 = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        dt_max = shard.max_over_ranks((time.perf_counter() - t0) / steps, dev)
        e2e_launches += eng.launch_count - l0
        return {"value": world * Se * n_samples / dt_max, "unit": UNIT, "ms_per_step": 1e3 * dt_max, "encoder_threads": workers,
                "steps": steps, "records_match_device_path": bool(dev_rec[:Se].tobytes() == rec_sp.tobytes()),
                "what": "bv_sparse_encode16 (u32 cell per covered read -> delta-coded u16 words) runs inside the timed region, one tile per "
                        "worker thread, ahead of the submitting thread"}

    # What a packer holds per covered read is one u32 cell.  Two ways from there, both with everything inside the clock:
    # ship the u32 cells as they are (BV_CELLS_U32: twice the bytes, no host work), or re-code them to u16 words on the host
    # first (bv_sparse_encode16 on worker threads).  e2e_from_cells reports the faster of the two, both are listed.
    leg32 = sparse_leg(cells32, start32, args.e2e_steps, compact=use_compact)
    leg_enc = from_cells_leg(max(3, args.e2e_steps // 2))
    leg_cells = {"value": max(leg32["value"], leg_enc["value"]), "unit": UNIT,
                 "ms_per_step": min(leg32["ms"], leg_enc["ms_per_step"]),
                 "via": "BV_CELLS_U32 as is" if leg32["value"] >= leg_enc["value"] else "host encoder -> BV_CELLS_U16",
                 "u32_as_is": {"value": leg32["value"], "ms_per_step": leg32["ms"], "h2d_bytes_per_step": int(leg32["uploaded"]),
                               "d2h_bytes_per_step": int(leg32["d2h"]), "steps": args.e2e_steps,
                               "result_transport": "BV_OUT_COMPACT" if use_compact else "BV_OUT_RECORDS",
                               "records_match_device_path": bool(dev_rec[:Se].tobytes() == leg32["records"])},
                 "host_encode16": leg_enc}

    extra = {}
    if not args.no_e2e_extra:
        # bare copies of the headline leg's bytes (pinned, both directions at once, all ranks at once): what the host fabric gives
        h_up = torch.empty(int(leg16["uploaded"]), dtype=torch.uint8, pin_memory=True)
        d_up = torch.empty_like(h_up, device=dev)
        d_dn = torch.empty(int(leg16["d2h"]), dtype=torch.uint8, device=dev)
        h_dn = torch.empty(int(leg16["d2h"]), dtype=torch.uint8, pin_memory=True)
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
        for reps in (1, args.e2e_steps):
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                with torch.cuda.stream(s_up):
                    d_up.copy_(h_up, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    h_dn.copy_(d_dn, non_blocking=True)
            torch.cuda.synchronize()
            fab = shard.max_over_ranks((time.perf_counter() - t0) / reps, dev)
        extra["fabric"] = {"ms_per_step": 1e3 * fab, "h2d_gbs_per_gpu": leg16["uploaded"] / fab / 1e9, "d2h_gbs_per_gpu": leg16["d2h"] / fab / 1e9,
                           "aggregate_gbs": world * (leg16["uploaded"] + leg16["d2h"]) / fab / 1e9,
                           "e2e_fraction_of_fabric": fab / (leg16["ms"] * 1e-3),
                           "what": "cudaMemcpyAsync of the e2e leg's H2D and D2H bytes per step from / to pinned memory on two streams, every rank "
                                   "at the same time, no kernels: the floor the host memory / PCIe fabric sets for the e2e step"}
        del h_up, d_up, d_dn, h_dn
        if world == 1 and name == "C2":
            # dense tiles: pinned planes -> bv_tile_submit (H2D of base + strand, qual rows read in place) -> bv_tile_wait
            h_planes = [torch.empty((S, pitch), dtype=torch.uint8, pin_memory=True) for _ in range(3)]
            h_ref = torch.empty(S, dtype=torch.uint8, pin_memory=True)
            for h, d in zip(h_planes, (main_res.base, main_res.qual, main_res.strand)):
                h.copy_(d)
            h_ref.copy_(main_res.ref)
            torch.cuda.synchronize()
            hb, hq, hs = (h.numpy() for h in h_planes)
            rec = np.zeros(S, dtype=bv.SITE_OUT_DTYPE)
            eng.call_host(hb, hq, hs, h_ref.numpy(), n_samples, out=rec)  # warm-up (also first touch of `rec`)
            barrier()
            l0, up0, t0 = eng.launch_count, eng.h2d_bytes, time.perf_counter()
            for _ in range(2):
                eng.call_host(hb, hq, hs, h_ref.numpy(), n_samples, out=rec)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / 2
            e2e_launches += eng.launch_count - l0
            uploaded = (eng.h2d_bytes - up0) // 2
            qual_rows = int((((dev_rec["flags"] & 0x20) != 0) | (dev_rec["em_calls"] >= 3) | ((dev_rec["n_alt"] > 0) & (dev_rec["em_calls"] == 1))).sum())
            extra["e2e_dense"] = {"value": S * n_samples / dt, "unit": UNIT, "h2d_bytes_per_step": int(uploaded + pitch * qual_rows),
                                  "uploaded_bytes_per_step": int(uploaded), "d2h_bytes_per_step": int(S * 128), "ms_per_step": 1e3 * dt,
                                  "records_match_device_path": bool(dev_rec.tobytes() == rec.tobytes())}
            del h_planes, h_ref
    clk = clocks.stop()

    line = None
    if rank == 0:
        avg_ms = float(np.mean(per_step_ms))
        conf = config_block(name, cfg, S, maf, args.abs_mode, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": conf,
            "workload_stats": {"variant_sites": int((dev_rec["n_alt"] > 0).sum()), "mean_em_calls": float(dev_rec["em_calls"].mean()),
                               "n_active_hist": np.bincount(dev_rec["n_active"], minlength=5).tolist(),
                               "flagged_near_lrt_or_tie": int(((dev_rec["flags"] & 0x90) != 0).sum()),
                               "site0_of_rank0": int(site0),
                               "host_binding": (f"rank 0 on the {len(numa_cpus)} CPUs next to its GPU" if numa_cpus else "none")},
            "roofline": main_res.roofline(avg_ms, kernel_ms, peak, peak_src),
            # e2e (headline): sparse host tiles in the compact form.  h2d = 2 bytes per covered cell (+ 4 % "skip" words) + the
            # site offsets + REF bases
            "e2e": {"value": leg16["value"], "unit": UNIT, "h2d_bytes_per_step": int(leg16["uploaded"]), "d2h_bytes_per_step": int(leg16["d2h"]),
                    "ms_per_step": leg16["ms"], "steps": args.e2e_steps, "sites_per_gpu": Se,
                    "transport": "sparse tiles, BV_CELLS_U16 (bv_tile_submit_sparse): pinned u16 words of the covered reads, sample indices "
                                 "delta-coded; expanded into the dense planes on the device (K0); results as named in result_transport (BV_OUT_COMPACT: 8 "
                                 "bytes per site + the 128-byte record of every site that is not all-REF, written by the device into pinned "
                                 "staging; bv_site_expand rebuilds the rest); tiles and steps pipelined over the slots (no drain between steps)",
                    "result_transport": "BV_OUT_COMPACT" if use_compact else "BV_OUT_RECORDS",
                    "other_result_transport": {"value": leg16_full["value"], "ms_per_step": leg16_full["ms"], "d2h_bytes_per_step": int(leg16_full["d2h"]),
                                               "records_match_device_path": bool(dev_rec[:Se].tobytes() == leg16_full["records"]),
                                               "what": "the same with " + ("BV_OUT_RECORDS: a 128-byte record for every site" if use_compact else
                                                                            "BV_OUT_COMPACT: 8 bytes per site + the full records of the sites that need one")},
                    "cells_per_step": int(cells32.shape[0]), "words_per_step": int(words16.shape[0]),
                    "tile_sites": tile_sites, "slots": args.slots, "records_match_device_path": same_sp,
                    "host_prep_s_untimed": t_prep + t_prep16},
            "e2e_from_cells": leg_cells,
            "gpu_launches": int(launches + e2e_launches),
            "clocks": clk,
        }
        line.update(extra)
        if world > 1:
            line["scaling_note"] = ("N > 1 runs the C4 region shards (BASELINE.json configs[3]); the N = 1 line of the same command is C2 "
                                    "(configs[1]) with the C4 shard shape under configs.C4: compare this value with N x that one")
    if world == 1 and not args.no_cpu_baseline:
        ns = int(min(S, max(args.ref_min_sample_sites // n_samples, 2000)))
        line["cpu_baseline"] = cpu_baseline(main_res, ns, cores)
    main_res.close()

    # ---- the other BASELINE.json shapes (one GPU): kernel-only value, roofline, per-kernel times, reference beside each --------
    if world == 1 and not args.no_configs and args.config is None:
        configs = {}
        steps = max(5, args.steps // 2)
        for key, cname, mode in (("C3", "C3", 0), ("C4", "C4", 0), ("C5", "C5", 0), ("C5_dblabs", "C5", 1)):
            ccfg = dict(bv.synth.CONFIGS[cname])
            cS = RESIDENT_SITES[cname]
            c0 = shard.shard_region(0, C4_REGION, 8)[3][0] if cname == "C4" else 0   # C4: the shard GPU 3 of 8 takes
            r = Resident(bv, torch, dev, local_rank, cname, ccfg, cS, c0, mode)
            tot, per, _ = r.timed(steps, 3, barrier)
            km = r.kernel_ms(steps)
            rec = r.records()
            entry = {"config": config_block(cname, ccfg, cS, r.maf, mode, 1), "value": cS * r.N * steps / (tot * 1e-3), "unit": UNIT,
                     "ms_per_step": tot / steps, "steps": steps, "roofline": r.roofline(float(np.mean(per)), km, peak, peak_src),
                     "workload_stats": {"variant_sites": int((rec["n_alt"] > 0).sum()), "mean_em_calls": float(rec["em_calls"].mean()),
                                        "n_active_hist": np.bincount(rec["n_active"], minlength=5).tolist(),
                                        "flagged_near_lrt_or_tie": int(((rec["flags"] & 0x90) != 0).sum()), "site0": int(c0)}}
            if not args.no_cpu_baseline:
                entry["cpu_baseline"] = cpu_baseline(r, int(min(cS, max(args.ref_min_sample_sites // r.N, 2000))), cores)
            configs[key] = entry
            r.close()
        line["configs"] = configs
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dev_rec)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
