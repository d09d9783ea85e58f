"""include/ff/ff.hpp -- the FastFlow-API-compatible runtime the builder API runs over -- on the CPU: nested pipeline / all-to-all graphs,
combined nodes, channel ids, end-of-stream notification order, ff_poll, the MPMC queue (tests/cpp/test_ff_runtime.cpp)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INC = os.path.join(ROOT, "include")


@pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")
def test_ff_runtime_unit():
    exe = os.path.join(ROOT, "tests", "cpp", "test_ff_runtime.bin")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-I" + INC, os.path.join(ROOT, "tests", "cpp", "test_ff_runtime.cpp"), "-o", exe])
    for _ in range(3):  # threads: repeat
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0 and "ff runtime OK" in out.stdout, out.stdout + out.stderr
