"""-m gpu: Context::run_device of the C++ host mirror (tests/cpp/test_device_gpu.cpp): pileups in device memory, sparse and
dense, every result form, against Context::submit / wait of the same host tiles on the SURVEY.md 8c vectors and a synthetic
tile."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")


@pytest.mark.gpu
def test_host_run_device_gpu(built_lib):
    from basevar_b200 import build
    build.build_host()
    p = subprocess.run([os.path.join(BIN, "test_device_gpu")], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "ALL OK" in p.stdout, p.stdout[-4000:] + p.stderr[-2000:]
    assert "device-resident results checked" in p.stdout
