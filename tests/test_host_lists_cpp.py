"""-m gpu: BaseType(&bi, min_af).lrt(list) of the C++ host mirror (tests/cpp/test_lists_gpu.cpp) against the oracle's
bvo_site_list (tests/oracle_lists.c) on the known-answer vectors of SURVEY.md 8c with reordered and shortened lists."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")


@pytest.mark.gpu
def test_host_lrt_lists_gpu(built_lib, oracle_lib):
    from basevar_b200 import build
    from tests import oracle_lists
    build.build_host()
    p = subprocess.run([os.path.join(BIN, "test_lists_gpu"), oracle_lists.library_path()], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "ALL OK" in p.stdout, p.stdout[-4000:] + p.stderr[-2000:]
    assert "through the mono-allelic rule" in p.stdout
