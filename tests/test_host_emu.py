"""CPU runs of the device index logic: the register FFTs and the per-lane pipeline of the fused kernels are
__host__ __device__ code; tests/host_emu/*.cu emulate the lanes sequentially and compare against a
double-precision naive DFT (and check the shared-memory exchange addressing for bank conflicts)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.mark.parametrize("name", ["test_fft_regs", "test_warp_core", "test_mixed_radix"])
def test_host_emulation(name, tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    exe = tmp_path / name
    src = os.path.join(ROOT, "tests", "host_emu", name + ".cu")
    r = subprocess.run([NVCC, "-O1", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets",
                        "-I", os.path.join(ROOT, "include"), "-o", str(exe), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
