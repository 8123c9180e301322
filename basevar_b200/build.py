"""Build the CUDA library in-tree: basevar_b200/libbasevar_b200.so (sm_100a only).

    python -m basevar_b200.build            # rebuild if sources are newer than the .so
    python -m basevar_b200.build --force

-fmad=false: the x86-64 reference build contracts nothing, so the device code must not either
(see csrc/bv_math.cuh).  -lineinfo keeps ncu's source page usable.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbasevar_b200.so")
SOURCES = [os.path.join(CSRC, "bv_api.cu"), os.path.join(CSRC, "bv_encode16.cpp")]   # the .cpp goes to the host compiler as is
DEPS = SOURCES + [os.path.join(CSRC, f) for f in ("bv_common.cuh", "bv_count_kernel.cuh", "bv_finish_kernels.cuh", "bv_em_kernels.cuh", "bv_call_kernels.cuh", "bv_list_kernel.cuh", "bv_expand_kernel.cuh", "bv_math.cuh",
                                                  "bv_fisher_fast.h", "bv_synth.cuh")] + [
    os.path.join(HERE, "..", "include", "basevar_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUDA_HOME = os.path.dirname(os.path.dirname(os.path.realpath(NVCC)))
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    subprocess.check_call(cmd)
    return LIB


HOST_LIB = os.path.join(HERE, "libbasevar_b200_host.so")
HOST_SRC = [os.path.join(HERE, "host", f) for f in ("bv_host.cpp", "bv_caller.cpp", "bv_bam.cpp", "bv_pileup.cpp")]
HOST_DEPS = HOST_SRC + [os.path.join(HERE, "host", f) for f in ("bv_host.hpp", "bv_caller.hpp", "bv_bam.hpp", "bv_pileup.hpp")] + [
    os.path.join(HERE, "..", "include", "basevar_b200.h")]
CLI = os.path.join(HERE, "bin", "basevar")   # `basevar basetype ...` over BAM files (host/bv_main.cpp)
ROOT = os.path.dirname(HERE)
CPP_TESTS = {"test_host_cpu": [], "test_host_gpu": ["-ldl"], "test_fisher_fast": ["-ldl", "-lm"], "test_caller_cpu": [],
             "test_caller_gpu": ["-lz"], "pileup_dump": ["-lz"], "test_lists_gpu": ["-ldl", "-lm"],
             "test_ranksum_gpu": ["-ldl", "-lm"], "test_vcf_row_gpu": ["-ldl", "-lm"],
             # (allocates the device buffers of Context::run_device with the CUDA runtime; the host layer itself has no CUDA)
             "test_device_gpu": ["-I" + os.path.join(CUDA_HOME, "include"), "-L" + os.path.join(CUDA_HOME, "lib64"), "-lcudart",
                                 "-Wl,-rpath," + os.path.join(CUDA_HOME, "lib64")]}


# What the programs linked against the host layer compile in: they are linked again when their source or one of these changes.
# A library rebuilt behind an unchanged interface is picked up at load time (both libraries are shared), without a relink.
PROGRAM_HEADERS = [h for h in HOST_DEPS if h.endswith((".hpp", ".h"))] + [os.path.join(CSRC, "bv_fisher_fast.h")]


def _stale(target, sources):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in sources)


def build_host(force=False):
    """The C++ host layer (g++) over the C ABI, and its test programs under tests/cpp/bin/."""
    build(force=False)
    cxx = os.environ.get("CXX", "g++")
    if force or not os.path.exists(HOST_LIB) or any(os.path.getmtime(d) > os.path.getmtime(HOST_LIB) for d in HOST_DEPS + [LIB]):
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-Wall", "-fPIC", "-shared", "-o", HOST_LIB] + HOST_SRC +
                              ["-L" + HERE, "-lbasevar_b200", "-Wl,-rpath,$ORIGIN", "-lpthread", "-lz"])
    bindir = os.path.join(ROOT, "tests", "cpp", "bin")
    os.makedirs(bindir, exist_ok=True)
    for name, extra in CPP_TESTS.items():
        src = os.path.join(ROOT, "tests", "cpp", name + ".cpp")
        exe = os.path.join(bindir, name)
        if force or _stale(exe, [src] + PROGRAM_HEADERS):
            subprocess.check_call([cxx, "-std=c++17", "-O2", "-Wall", "-o", exe, src, "-L" + HERE, "-lbasevar_b200_host",
                                   "-lbasevar_b200", "-Wl,-rpath," + HERE, "-lpthread"] + extra)
    main_src = os.path.join(HERE, "host", "bv_main.cpp")
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    if force or _stale(CLI, [main_src] + PROGRAM_HEADERS):
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-Wall", "-o", CLI, main_src, "-L" + HERE, "-lbasevar_b200_host",
                               "-lbasevar_b200", "-Wl,-rpath," + HERE, "-Wl,-rpath,$ORIGIN/..", "-lpthread", "-lz"])
    return HOST_LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_host(force="--force" in sys.argv)
    print(LIB)
