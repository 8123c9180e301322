"""-m gpu: ref_vs_alt_ranksumtest of the C++ host mirror (tests/cpp/test_ranksum_gpu.cpp), both overloads, against the oracle's
bvo_wilcoxon and against the batch path's bv_call_out of a called site."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")


@pytest.mark.gpu
def test_host_ranksum_gpu(built_lib, oracle_lib):
    from basevar_b200 import build
    build.build_host()
    p = subprocess.run([os.path.join(BIN, "test_ranksum_gpu"), oracle_lib._name], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "ALL OK" in p.stdout, p.stdout[-4000:] + p.stderr[-2000:]
    assert "called site ALT" in p.stdout
