"""ctypes binding of libspecinv_b200.so (include/specinv_b200.h).

There is deliberately no fallback: if the CUDA library is missing or a call fails, a
RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_PKG = os.path.dirname(os.path.abspath(__file__))
# SPECINV_B200_LIB: load another build of the same ABI (kernel A/B experiments)
LIB_PATH = os.environ.get("SPECINV_B200_LIB") or os.path.join(_PKG, "lib", "libspecinv_b200.so")

F32, F64 = 0, 1
PAD_MODES = {"reflect": 0, "constant": 1, "replicate": 2, "circular": 3}
ERR_UNSUPPORTED = -2

EXPORTS = (
    "specinv_abi_version", "specinv_error_string", "specinv_signal_length",
    "specinv_plan_bytes", "specinv_plan_init", "specinv_plan_envelope",
    "specinv_pack_complex", "specinv_pack_real", "specinv_unpack_complex",
    "specinv_stft", "specinv_istft", "specinv_gl_iter", "specinv_admm_iter",
    "specinv_metric_sums", "specinv_phase_init", "specinv_spec_abs", "specinv_rtisi_la", "specinv_plan_init_ranged",
    "specinv_phase_init_ex", "specinv_halo_sum", "specinv_fill_padding", "specinv_plan_unit_envelope",
    "specinv_halo_area_bytes", "specinv_ipc_alloc", "specinv_ipc_open", "specinv_ipc_close", "specinv_ipc_free",
    "specinv_halo_exchange", "specinv_halo_status",
    "specinv_gl_run_workspace_bytes", "specinv_gl_run", "specinv_gl_run_status",
    "specinv_rtisi_state_bytes", "specinv_rtisi_la_steps", "specinv_rtisi_la_stream", "specinv_plan_inv_env_window",
    "specinv_gl_rebuilt_iter", "specinv_mel_inverse", "specinv_pghi_workspace_bytes", "specinv_pghi",
    "specinv_pghi_stream_state_bytes", "specinv_pghi_stream",
)


class Desc(C.Structure):
    """struct specinv_desc"""
    _fields_ = [("n_fft", C.c_int32), ("hop", C.c_int32), ("n_frames", C.c_int32), ("batch", C.c_int32),
                ("center", C.c_int32), ("pad_mode", C.c_int32), ("normalized", C.c_int32),
                ("onesided", C.c_int32), ("dtype", C.c_int32), ("reserved", C.c_int32 * 7)]


_lib: Optional[C.CDLL] = None


def _declare(lib: C.CDLL) -> None:
    vp, i64, dbl = C.c_void_p, C.c_int64, C.c_double
    dp = C.POINTER(Desc)
    lib.specinv_abi_version.restype = C.c_int
    lib.specinv_abi_version.argtypes = []
    lib.specinv_error_string.restype = C.c_char_p
    lib.specinv_error_string.argtypes = [C.c_int]
    sigs = {
        "specinv_signal_length": [dp, C.POINTER(i64)],
        "specinv_plan_bytes": [dp, C.POINTER(C.c_size_t)],
        "specinv_plan_init": [dp, vp, vp, vp],
        "specinv_plan_unit_envelope": [dp, vp, vp],
        "specinv_ipc_alloc": [C.c_size_t, C.POINTER(vp), vp],
        "specinv_ipc_open": [vp, C.POINTER(vp)],
        "specinv_ipc_close": [vp],
        "specinv_ipc_free": [vp],
        "specinv_halo_exchange": [C.c_int, vp, i64, C.c_int, i64, i64, vp, vp, vp, C.c_uint32, vp],
        "specinv_gl_run_workspace_bytes": [dp, C.POINTER(C.c_size_t)],
        "specinv_gl_run": [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl, C.c_int, C.c_int, C.c_int, vp, vp, vp],
        "specinv_gl_run_status": [dp, vp, C.POINTER(C.c_uint32), vp],
        "specinv_halo_status": [C.c_int, vp, C.c_int, i64, C.POINTER(C.c_uint32), vp],
        "specinv_plan_envelope": [dp, vp, vp, vp],
        "specinv_plan_init_ranged": [dp, vp, vp, i64, i64, vp],
        "specinv_phase_init_ex": [dp, vp, vp, vp, vp, vp, vp, vp],
        "specinv_halo_sum": [C.c_int, vp, i64, vp, i64, vp, i64, C.c_int, i64, vp],
        "specinv_fill_padding": [C.c_int, vp, i64, C.c_int, i64, i64, C.c_int, i64, C.c_int, vp],
        "specinv_pack_complex": [dp, vp, i64, i64, i64, vp, vp, vp],
        "specinv_pack_real": [dp, vp, i64, i64, i64, vp, vp, vp],
        "specinv_unpack_complex": [dp, vp, vp, vp, i64, i64, i64, vp],
        "specinv_phase_init": [dp, vp, vp, vp, vp, vp],
        "specinv_spec_abs": [dp, vp, vp, vp, vp, vp],
        "specinv_rtisi_la": [dp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, dbl, dbl, vp],
        "specinv_rtisi_state_bytes": [dp, C.c_int, C.POINTER(C.c_size_t)],
        "specinv_rtisi_la_steps": [dp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, dbl, dbl, C.c_int, C.c_int, vp, vp],
        "specinv_rtisi_la_stream": [dp, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp, i64, i64, vp, C.c_int, C.c_int, C.c_int,
                                    dbl, dbl, C.c_int, C.c_int, C.c_int, vp, vp],
        "specinv_plan_inv_env_window": [dp, vp, i64, i64, i64, vp, vp],
        "specinv_stft": [dp, vp, vp, vp, vp, vp],
        "specinv_istft": [dp, vp, vp, vp, vp, vp],
        "specinv_gl_iter": [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl, vp, vp],
        "specinv_gl_rebuilt_iter": [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl, vp, vp],
        "specinv_admm_iter": [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl, vp, vp],
        "specinv_metric_sums": [C.c_int, vp, vp, i64, vp, vp],
        "specinv_mel_inverse": [C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, i64, vp],
        "specinv_pghi_workspace_bytes": [C.c_int, C.c_int, C.c_int, i64, C.POINTER(C.c_size_t)],
        "specinv_pghi": [C.c_int, vp, i64, i64, i64, vp, C.c_int, C.c_int, i64, C.c_int, C.c_int, C.c_int, dbl, dbl, vp,
                         C.c_size_t, vp],
        "specinv_pghi_stream_state_bytes": [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)],
        "specinv_pghi_stream": [C.c_int, vp, i64, i64, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, vp,
                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, dbl, dbl, vp],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    lib.specinv_halo_area_bytes.restype = C.c_size_t
    lib.specinv_halo_area_bytes.argtypes = [C.c_int, C.c_int, i64]


def lib() -> C.CDLL:
    """Load (once) and return the CUDA library; raise loudly when it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m spectrogram_inversion_b200.build` "
                "(there is no CPU / PyTorch fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        _declare(handle)
        if handle.specinv_abi_version() != 1:
            raise RuntimeError("libspecinv_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().specinv_error_string(code).decode()
        exc = NotImplementedError if code == ERR_UNSUPPORTED else RuntimeError
        raise exc(f"specinv_b200 {what} failed: {msg} (code {code})")


def make_desc(n_fft: int, hop: int, n_frames: int, batch: int, center: bool, pad_mode: int,
              normalized: bool, onesided: bool, dtype: int) -> Desc:
    d = Desc()
    d.n_fft, d.hop, d.n_frames, d.batch = int(n_fft), int(hop), int(n_frames), int(batch)
    d.center, d.pad_mode, d.normalized, d.onesided = int(bool(center)), int(pad_mode), int(bool(normalized)), int(bool(onesided))
    d.dtype = int(dtype)
    return d
