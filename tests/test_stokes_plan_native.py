"""The library's own C++ of the rectangular exchange plans and the local divergence matrices (csrc/exchange_plan.h),
checked without a GPU: tests/native/exchange_plan_check.cu plays all ranks of a partition in one process and compares
the partitioned products with the global ones bitwise."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_exchange_plan_native_check(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = str(tmp_path / "exchange_plan_check")
    subprocess.check_call([nvcc, "-std=c++17", "-O2", "-x", "cu", "-w", "-I", os.path.join(ROOT, "control_b200", "csrc"),
                           "-o", exe, os.path.join(ROOT, "tests", "native", "exchange_plan_check.cu")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "exchange plan check: 0 failures" in out.stdout
