"""CPU side of the streamed-frame generic kernel (csrc/specinv_generic_stream.cu).

1. The capacity rules of the three tile launchers (launch_mr in specinv_generic_mr.cu, launch_tile and
   launch_dft_tile in specinv_generic.cu) restated at the B200's 227 KB opt-in limit: the shapes the streamed kernel
   exists for are refused by every tile kernel, and the tile kernels' own shapes are not.
2. specinv_plan_bytes accepts n_fft up to 32768.
3. Host emulation of the mixed-radix plan and passes at M = 6000, 8192 and 16384 against a float64 DFT."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
OPTIN = 227 * 1024          # cudaDevAttrMaxSharedMemoryPerBlockOptin of the B200


def mr_fits(n, hop, es):
    """launch_mr: two CTAs per SM, or one fat CTA when the owned / halo ratio is poor; M <= 4096."""
    M = n // 2
    if M > 4096 or n % 2:
        return False
    frame = (M + (M >> 4) + 1) * 2 * es
    perm = (M * 2 + 15) // 16 * 16
    halo = (n - 1) // hop
    big = OPTIN - 1024 - perm
    cap = min(228 * 1024 // 2 - 1024 - 256 - perm, big) // frame
    if cap - halo < (2 * halo if halo > 1 else 2):
        cap = big // frame
    return cap - halo >= 1


def _tile_rule(frame, halo):
    big = OPTIN - 1024
    cap = min(big, 100 * 1024) // frame
    if cap - halo < (2 * halo if halo > 1 else 2):
        cap = big // frame
    owned = cap - halo
    return owned >= 1 and (owned + halo) * frame <= big


def tile_fits(n, hop, es):
    """launch_tile (radix-2^2, powers of two)."""
    M = n // 2
    return n & (n - 1) == 0 and _tile_rule((M + (M >> 4)) * 2 * es, (n - 1) // hop)


def dft_fits(n, hop, es):
    """launch_dft_tile (direct DFT): N time samples and N/2 + 1 bins per frame."""
    return _tile_rule((n + 2 * (n // 2 + 1)) * es, (n - 1) // hop)


def tile_kernel_for(n, hop, es):
    """The tile kernel launch_tile picks (None: none holds the shape; n_fft > 8192 never reaches them)."""
    if n > 8192:
        return None
    if mr_fits(n, hop, es):
        return "mr"
    if n & (n - 1) == 0:
        return "tile" if tile_fits(n, hop, es) else None
    return "dft" if dft_fits(n, hop, es) else None


REFUSED = [(8192, 2048, 8), (4096, 512, 8), (2048, 128, 8), (6000, 750, 8),
           (8192, 1024, 4), (4096, 256, 4), (6000, 375, 4)]
HELD = [(8192, 2048, 4), (4096, 1024, 8), (400, 100, 4), (400, 100, 8), (1024, 256, 4)]


@pytest.mark.parametrize("n,hop,es", REFUSED, ids=[f"{n}-{h}-fp{8 * e}" for n, h, e in REFUSED])
def test_no_tile_kernel_holds_these_shapes(n, hop, es):
    assert not mr_fits(n, hop, es) and not tile_fits(n, hop, es) and not dft_fits(n, hop, es)
    assert tile_kernel_for(n, hop, es) is None


@pytest.mark.parametrize("n,hop,es", HELD, ids=[f"{n}-{h}-fp{8 * e}" for n, h, e in HELD])
def test_tile_kernels_keep_their_shapes(n, hop, es):
    assert tile_kernel_for(n, hop, es) == "mr"


def test_plan_bytes_up_to_32768():
    from spectrogram_inversion_b200 import _lib
    handle = _lib.lib()
    nbytes = C.c_size_t()
    for n, dt in ((16384, _lib.F32), (16384, _lib.F64), (32768, _lib.F32), (32768, _lib.F64)):
        d = _lib.make_desc(n, n // 4, 10, 1, True, 0, False, True, dt)
        assert handle.specinv_plan_bytes(C.byref(d), C.byref(nbytes)) == 0
        assert nbytes.value >= 2 * n * (8 if dt == _lib.F64 else 4)
    d = _lib.make_desc(32769, 8192, 10, 1, True, 0, False, False, _lib.F32)
    assert handle.specinv_plan_bytes(C.byref(d), C.byref(nbytes)) == -1      # SPECINV_ERR_INVALID


def test_mixed_radix_passes_at_large_sizes(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    exe = tmp_path / "test_mixed_radix_large"
    src = os.path.join(ROOT, "tests", "host_emu", "test_mixed_radix_large.cu")
    r = subprocess.run([NVCC, "-O1", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets",
                        "-I", os.path.join(ROOT, "include"), "-o", str(exe), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
