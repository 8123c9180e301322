"""-m gpu: the VCF row's batch path of the C++ host mirror (tests/cpp/test_vcf_row_gpu.cpp) -- SparsePacker with compact
results, the called-site kernels and population groups, TilePacker's rpr plane, sparse lists -- against the per-site drop-in
route and the oracle's bvo_group_site."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")


@pytest.mark.gpu
def test_host_vcf_row_gpu(built_lib, oracle_lib):
    from basevar_b200 import build
    build.build_host()
    p = subprocess.run([os.path.join(BIN, "test_vcf_row_gpu"), oracle_lib._name], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "ALL OK" in p.stdout, p.stdout[-4000:] + p.stderr[-2000:]
    assert "checked against the drop-in route" in p.stdout
