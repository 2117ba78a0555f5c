"""torch.library custom ops and direct calls: thin wrappers that hand raw device pointers and the current CUDA
stream to the C ABI of libspecinv_b200.so.  No computation happens in Python/PyTorch here.  This module is the only
caller of the library: streamed entries go through `_call`, size queries through `_size`."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib

# number of CUDA kernels of libspecinv_b200.so launched through this module (bench.py reports it)
LAUNCHES = [0]

_DT = {torch.float32: _lib.F32, torch.float64: _lib.F64, torch.complex64: _lib.F32, torch.complex128: _lib.F64}
# the complex dtype of each real dtype the kernels take
CDT = {torch.float32: torch.complex64, torch.float64: torch.complex128}


class _Entries(dict):
    def __missing__(self, entry: str):
        fn = self[entry] = getattr(_lib.lib(), "specinv_" + entry)
        return fn


_FNS = _Entries()      # entry name -> ctypes function of specinv_<name>, looked up on first use


def _call(entry, device: torch.device, args: tuple, kernels: int, what: Optional[str] = None) -> None:
    """specinv_<entry>(*args, stream) (``entry``: a name or a ctypes function) on ``device``'s current stream, entered
    only when not current: a failure raises (``what`` names it, the entry by default), success adds ``kernels``."""
    fn = _FNS[entry] if isinstance(entry, str) else entry
    stream = torch.cuda.current_stream(device).cuda_stream
    if torch.cuda.current_device() == device.index:
        code = fn(*args, stream)
    else:
        with torch.cuda.device(device):
            code = fn(*args, stream)
    if code:
        _lib.check(code, what or entry)
    LAUNCHES[0] += kernels


def _size(entry: str, *args) -> int:
    """The size_t that specinv_<entry>(*args, size_t* bytes) computes on the host (no stream, no launch)."""
    fn = _FNS[entry]
    if fn.restype is C.c_size_t:        # specinv_halo_area_bytes returns it instead
        return fn(*args)
    n = C.c_size_t(0)
    _lib.check(fn(*args, C.byref(n)), entry)
    return n.value


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError("spectrogram_inversion_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _lib.lib()


def _p(t: Optional[Tensor]):
    """Device pointer of t; NULL for None or an empty tensor."""
    return t.data_ptr() if t is not None and t.numel() else None


def desc(dtype: torch.dtype, n_fft: int, hop: int, n_frames: int, batch: int, center: bool, pad_mode: int,
         normalized: bool, onesided: bool):
    """A struct specinv_desc as the entries take it: by reference (which keeps the struct alive)."""
    return C.byref(_lib.make_desc(n_fft, hop, n_frames, batch, center, pad_mode, normalized, onesided, _DT[dtype]))


def _need_cuda(*ts: Tensor) -> None:
    for t in ts:
        if t.numel() and not t.is_cuda:
            raise RuntimeError("specinv_b200 ops only run on CUDA tensors (no CPU fallback)")
        if t.numel() and not t.is_contiguous():
            raise RuntimeError("specinv_b200 ops need contiguous buffers")


def pointers(tensors):
    """Device pointers for `iter_direct` (None / empty tensor = NULL)."""
    return [_p(t) for t in tensors]


def iter_direct(entry, what: str, device: torch.device, desc_ref, ptrs, coef: float, sums_ptr) -> None:
    """The per-iteration launch of ``entry`` (gl_iter, admm_iter, gl_rebuilt_iter) without the custom ops' dispatch,
    which costs ~40 us per call: more than a whole iteration of a small problem (24 us at BASELINE cfg1).  ``ptrs``:
    the pointers between the descriptor and the coefficient (`pointers`)."""
    _call(entry, device, (desc_ref, *ptrs, coef, sums_ptr), 1, what)


# ---- the calls of engine.py and sharding.py ----------------------------------------------------------------------
def plan_bytes(desc_ref) -> int:
    return _size("plan_bytes", desc_ref)


def plan_envelope(plan: Tensor, desc_ref, env: Tensor) -> None:
    _call("plan_envelope", plan.device, (desc_ref, _p(plan), _p(env)), kernels=0)


def plan_unit_envelope(plan: Tensor, desc_ref) -> None:
    _call("plan_unit_envelope", plan.device, (desc_ref, _p(plan)), kernels=0)


def gl_run_workspace_bytes(desc_ref) -> Optional[int]:
    """Workspace of the persistent kernel, or None when the problem does not fit it (SPECINV_ERR_UNSUPPORTED)."""
    try:
        return _size("gl_run_workspace_bytes", desc_ref)
    except NotImplementedError:
        return None


def gl_run(desc_ref, tensors, lr: float, n_iters: int, iter0: int, eva_iter: int, sums: Optional[Tensor],
           workspace: Tensor) -> None:
    """Iterations iter0 .. iter0 + n_iters - 1 in one persistent kernel (specinv_gl_run); ``tensors``: plan, x_in,
    x_out, q_in main / nyq, q_out main / nyq, mag main / nyq."""
    _call("gl_run", workspace.device, (desc_ref, *pointers(tensors), float(lr), int(n_iters), int(iter0), int(eva_iter),
          _p(sums), _p(workspace)), kernels=1)


def gl_run_status(desc_ref, workspace: Tensor) -> int:
    """0, or the iteration at which a CTA of the last persistent run timed out (synchronises the current stream)."""
    status = C.c_uint32(0)
    _call("gl_run_status", workspace.device, (desc_ref, _p(workspace), C.byref(status)), kernels=0)
    return status.value


def ipc_alloc_halo_area(dtype: torch.dtype, rows: int, ov: int) -> Tuple[int, bytes]:
    """(pointer, 64-byte IPC handle) of a zeroed halo area on the current device (specinv_ipc_alloc)."""
    area, handle = C.c_void_p(), C.create_string_buffer(64)
    nbytes = _size("halo_area_bytes", _DT[dtype], int(rows), int(ov))
    _lib.check(_FNS["ipc_alloc"](nbytes, C.byref(area), handle), "ipc_alloc")
    return area.value, handle.raw


def ipc_open(handle: bytes) -> int:
    """Map another process's area from its IPC handle on the current device (specinv_ipc_open)."""
    peer = C.c_void_p()
    _lib.check(_FNS["ipc_open"](C.create_string_buffer(handle, 64), C.byref(peer)), "ipc_open")
    return peer.value


def ipc_release(peers, area: Optional[int]) -> None:
    """Unmap the neighbours' areas, free this rank's; return codes are not raised, so that all of them are released."""
    for p in peers:
        if p:
            _FNS["ipc_close"](p)
    if area is not None:
        _FNS["ipc_free"](area)


def halo_exchange(x: Tensor, rows: int, ov: int, area: int, left: Optional[int], right: Optional[int], seq: int):
    """Exchange number ``seq`` of x's partial sums with the left / right neighbour's area (None: no neighbour)."""
    _call("halo_exchange", x.device, (_DT[x.dtype], _p(x), x.stride(0), int(rows), x.shape[1], int(ov), area, left,
          right, int(seq)), kernels=0)


def halo_status(device: torch.device, dtype: torch.dtype, area: int, rows: int, ov: int) -> int:
    """0, or the number of the exchange that timed out waiting for a neighbour (synchronises the current stream)."""
    status = C.c_uint32(0)
    _call("halo_status", device, (_DT[dtype], area, int(rows), int(ov), C.byref(status)), kernels=0)
    return status.value


@torch.library.custom_op("specinv_b200::plan_init", mutates_args=("plan",), device_types="cuda")
def plan_init(plan: Tensor, window: Tensor, n_fft: int, hop: int, n_frames: int, batch: int, center: bool,
              pad_mode: int, normalized: bool, onesided: bool) -> None:
    _need_cuda(plan, window)
    d = desc(window.dtype, n_fft, hop, n_frames, batch, center, pad_mode, normalized, onesided)
    _call("plan_init", plan.device, (d, _p(window), _p(plan)), kernels=2)


@torch.library.custom_op("specinv_b200::stft", mutates_args=("out_main", "out_nyq"), device_types="cuda")
def stft(plan: Tensor, x: Tensor, out_main: Tensor, out_nyq: Tensor, n_fft: int, hop: int, center: bool,
         pad_mode: int, normalized: bool, onesided: bool) -> None:
    _need_cuda(plan, x, out_main, out_nyq)
    d = desc(x.dtype, n_fft, hop, out_main.shape[1], out_main.shape[0], center, pad_mode, normalized, onesided)
    _call("stft", x.device, (d, _p(plan), _p(x), _p(out_main), _p(out_nyq)), kernels=1)


@torch.library.custom_op("specinv_b200::istft", mutates_args=("x_out",), device_types="cuda")
def istft(plan: Tensor, in_main: Tensor, in_nyq: Tensor, x_out: Tensor, n_fft: int, hop: int, center: bool,
          pad_mode: int, normalized: bool, onesided: bool) -> None:
    _need_cuda(plan, in_main, in_nyq, x_out)
    d = desc(x_out.dtype, n_fft, hop, in_main.shape[1], in_main.shape[0], center, pad_mode, normalized, onesided)
    _call("istft", x_out.device, (d, _p(plan), _p(in_main), _p(in_nyq), _p(x_out)), kernels=1)


@torch.library.custom_op("specinv_b200::gl_iter",
                         mutates_args=("x_out", "q_out_main", "q_out_nyq", "sums"), device_types="cuda")
def gl_iter(plan: Tensor, x_in: Tensor, x_out: Tensor, q_in_main: Tensor, q_in_nyq: Tensor, q_out_main: Tensor,
            q_out_nyq: Tensor, mag_main: Tensor, mag_nyq: Tensor, sums: Tensor, lr: float, n_fft: int, hop: int,
            center: bool, pad_mode: int, normalized: bool, onesided: bool) -> None:
    _need_cuda(plan, x_in, x_out, q_in_main, q_in_nyq, q_out_main, q_out_nyq, mag_main, mag_nyq, sums)
    d = desc(x_in.dtype, n_fft, hop, q_in_main.shape[1], q_in_main.shape[0], center, pad_mode, normalized, onesided)
    _call("gl_iter", x_in.device, (d, _p(plan), _p(x_in), _p(x_out), _p(q_in_main), _p(q_in_nyq), _p(q_out_main),
          _p(q_out_nyq), _p(mag_main), _p(mag_nyq), float(lr), _p(sums)), kernels=1)


@torch.library.custom_op("specinv_b200::admm_iter",
                         mutates_args=("x_out", "X_out_main", "X_out_nyq", "U_out_main", "U_out_nyq", "sums"),
                         device_types="cuda")
def admm_iter(plan: Tensor, x_in: Tensor, x_out: Tensor, X_in_main: Tensor, X_in_nyq: Tensor, U_in_main: Tensor,
              U_in_nyq: Tensor, X_out_main: Tensor, X_out_nyq: Tensor, U_out_main: Tensor, U_out_nyq: Tensor,
              mag_main: Tensor, mag_nyq: Tensor, sums: Tensor, rho: float, n_fft: int, hop: int, center: bool,
              pad_mode: int, normalized: bool, onesided: bool) -> None:
    _need_cuda(plan, x_in, x_out, X_in_main, X_in_nyq, U_in_main, U_in_nyq, X_out_main, X_out_nyq, U_out_main,
               U_out_nyq, mag_main, mag_nyq, sums)
    d = desc(x_in.dtype, n_fft, hop, X_in_main.shape[1], X_in_main.shape[0], center, pad_mode, normalized, onesided)
    _call("admm_iter", x_in.device, (d, _p(plan), _p(x_in), _p(x_out), _p(X_in_main), _p(X_in_nyq), _p(U_in_main),
          _p(U_in_nyq), _p(X_out_main), _p(X_out_nyq), _p(U_out_main), _p(U_out_nyq), _p(mag_main), _p(mag_nyq),
          float(rho), _p(sums)), kernels=1)


@torch.library.custom_op("specinv_b200::pack", mutates_args=("out_main", "out_nyq"), device_types="cuda")
def pack(spec: Tensor, out_main: Tensor, out_nyq: Tensor, n_fft: int, onesided: bool) -> None:
    """(B, F, T) strided real or complex tensor -> split frame-major layout."""
    if not spec.is_cuda:
        raise RuntimeError("specinv_b200 ops only run on CUDA tensors (no CPU fallback)")
    B, Fb, T = spec.shape
    d = desc(spec.dtype, n_fft, 1, T, B, False, 0, False, onesided)
    sb, sf, st = spec.stride()
    _call("pack_complex" if spec.is_complex() else "pack_real", spec.device, (d, _p(spec), sb, sf, st, _p(out_main),
          _p(out_nyq)), kernels=1, what="pack")


@torch.library.custom_op("specinv_b200::unpack", mutates_args=("spec_out",), device_types="cuda")
def unpack(in_main: Tensor, in_nyq: Tensor, spec_out: Tensor, n_fft: int, onesided: bool) -> None:
    B, Fb, T = spec_out.shape
    d = desc(spec_out.dtype, n_fft, 1, T, B, False, 0, False, onesided)
    sb, sf, st = spec_out.stride()
    _call("unpack_complex", spec_out.device, (d, _p(in_main), _p(in_nyq), _p(spec_out), sb, sf, st), kernels=1,
          what="unpack")


@torch.library.custom_op("specinv_b200::metric_sums", mutates_args=("out3",), device_types="cuda")
def metric_sums(a: Tensor, b: Tensor, out3: Tensor) -> None:
    """out3[0] += sum (a-b)^2, out3[1] += sum a^2, out3[2] += sum b^2."""
    _need_cuda(a, b, out3)
    if a.numel() != b.numel() or a.dtype != b.dtype:
        raise RuntimeError("metric_sums: shape/dtype mismatch")
    _call("metric_sums", a.device, (_DT[a.dtype], _p(a), _p(b), a.numel(), _p(out3)), kernels=1)


@torch.library.custom_op("specinv_b200::phase_init", mutates_args=("c_main", "c_nyq"), device_types="cuda")
def phase_init(mag_main: Tensor, mag_nyq: Tensor, c_main: Tensor, c_nyq: Tensor, n_fft: int, hop: int,
               onesided: bool) -> None:
    """split real magnitude -> split complex start (methods.py:572-615), one fused kernel."""
    _need_cuda(mag_main, mag_nyq, c_main, c_nyq)
    d = desc(mag_main.dtype, n_fft, hop, mag_main.shape[1], mag_main.shape[0], False, 0, False, onesided)
    _call("phase_init", mag_main.device, (d, _p(mag_main), _p(mag_nyq), _p(c_main), _p(c_nyq)), kernels=1)


@torch.library.custom_op("specinv_b200::spec_abs", mutates_args=("mag_main", "mag_nyq"), device_types="cuda")
def spec_abs(c_main: Tensor, c_nyq: Tensor, mag_main: Tensor, mag_nyq: Tensor, n_fft: int, onesided: bool) -> None:
    _need_cuda(c_main, c_nyq, mag_main, mag_nyq)
    d = desc(mag_main.dtype, n_fft, 1, mag_main.shape[1], mag_main.shape[0], False, 0, False, onesided)
    _call("spec_abs", mag_main.device, (d, _p(c_main), _p(c_nyq), _p(mag_main), _p(mag_nyq)),
          kernels=2 if onesided else 1)


@torch.library.custom_op("specinv_b200::rtisi_la", mutates_args=("x_out", "scratch"), device_types="cuda")
def rtisi_la(plan: Tensor, window: Tensor, mag_main: Tensor, mag_nyq: Tensor, x_out: Tensor, scratch: Tensor,
             look_ahead: int, asymmetric: bool, max_iter: int, alpha: float, synth_coeff: float, n_fft: int, hop: int,
             center: bool, pad_mode: int, normalized: bool, onesided: bool) -> None:
    """RTISI_LA's loops + final overlap-add (methods.py:353-408) as one persistent kernel."""
    _need_cuda(plan, window, mag_main, mag_nyq, x_out, scratch)
    d = desc(x_out.dtype, n_fft, hop, mag_main.shape[1], mag_main.shape[0], center, pad_mode, normalized, onesided)
    _call("rtisi_la", x_out.device, (d, _p(plan), _p(window), _p(mag_main), _p(mag_nyq), _p(x_out), _p(scratch),
          int(look_ahead), int(bool(asymmetric)), int(max_iter), float(alpha), float(synth_coeff)), kernels=2)


@torch.library.custom_op("specinv_b200::rtisi_la_steps", mutates_args=("x_out", "scratch", "state"), device_types="cuda")
def rtisi_la_steps(plan: Tensor, window: Tensor, mag_main: Tensor, mag_nyq: Tensor, x_out: Tensor, scratch: Tensor,
                   state: Tensor, look_ahead: int, asymmetric: bool, max_iter: int, alpha: float, synth_coeff: float,
                   step_begin: int, step_end: int, n_fft: int, hop: int, center: bool, pad_mode: int, normalized: bool,
                   onesided: bool) -> None:
    """Outer steps [step_begin, step_end) of RTISI_LA (methods.py:363-404) with the sliding state in `state`
    (`rtisi_state_bytes` bytes; read when step_begin > 0, written when step_end < T + look_ahead)."""
    _need_cuda(plan, window, mag_main, mag_nyq, x_out, scratch, state)
    d = desc(x_out.dtype, n_fft, hop, mag_main.shape[1], mag_main.shape[0], center, pad_mode, normalized, onesided)
    _call("rtisi_la_steps", x_out.device, (d, _p(plan), _p(window), _p(mag_main), _p(mag_nyq), _p(x_out), _p(scratch),
          int(look_ahead), int(bool(asymmetric)), int(max_iter), float(alpha), float(synth_coeff), int(step_begin),
          int(step_end), _p(state)), kernels=2)


@torch.library.custom_op("specinv_b200::rtisi_la_stream", mutates_args=("x_out", "scratch", "state"), device_types="cuda")
def rtisi_la_stream(plan: Tensor, window: Tensor, mag_main: Tensor, mag_nyq: Tensor, x_out: Tensor, inv_env: Tensor,
                    scratch: Tensor, state: Tensor, n_frames: int, frame0: int, x0: int, look_ahead: int,
                    asymmetric: bool, max_iter: int, alpha: float, synth_coeff: float, step_begin: int, step_end: int,
                    final: bool, n_fft: int, hop: int, center: bool, normalized: bool, onesided: bool) -> None:
    """Outer steps [step_begin, step_end) of a stream of `n_frames` frames so far: magnitude rows (B, n_rows, .) are
    frames frame0 + r, x_out (B, x_len) and inv_env (x_len,) are samples x0 + c (include/specinv_b200.h)."""
    _need_cuda(plan, window, mag_main, mag_nyq, x_out, inv_env, scratch, state)
    d = desc(x_out.dtype, n_fft, hop, n_frames, x_out.shape[0], center, 1, normalized, onesided)
    _call("rtisi_la_stream", x_out.device, (d, _p(plan), _p(window), _p(mag_main), _p(mag_nyq), int(frame0),
          mag_main.shape[1], _p(x_out), _p(inv_env), int(x0), x_out.shape[1], _p(scratch), int(look_ahead),
          int(bool(asymmetric)), int(max_iter), float(alpha), float(synth_coeff), int(step_begin), int(step_end),
          int(bool(final)), _p(state)), kernels=2)


def plan_inv_env_window(plan: Tensor, out: Tensor, x0: int, total_frames: int, n_fft: int, hop: int, n_frames: int,
                        center: bool, normalized: bool, onesided: bool) -> None:
    """out[j] = 1/envelope of sample x0 + j of a signal of total_frames frames (-1: not known yet), from a plan of
    n_frames frames (specinv_plan_inv_env_window)."""
    _need_cuda(plan, out)
    d = desc(out.dtype, n_fft, hop, n_frames, 1, center, 1, normalized, onesided)
    _call("plan_inv_env_window", plan.device, (d, _p(plan), int(x0), out.numel(), int(total_frames), _p(out)),
          kernels=1)


def rtisi_state_bytes(ref: Tensor, n_fft: int, hop: int, n_frames: int, batch: int, normalized: bool, onesided: bool,
                      look_ahead: int) -> int:
    d = desc(ref.dtype, n_fft, hop, n_frames, batch, False, 0, normalized, onesided)
    return _size("rtisi_state_bytes", d, int(look_ahead))


@torch.library.custom_op("specinv_b200::plan_init_ranged", mutates_args=("plan",), device_types="cuda")
def plan_init_ranged(plan: Tensor, window: Tensor, n_fft: int, hop: int, n_frames: int, batch: int, normalized: bool,
                     onesided: bool, frame_offset: int, total_frames: int) -> None:
    """plan for frames [frame_offset, frame_offset + n_frames) of a longer signal (frame-range sharding)."""
    _need_cuda(plan, window)
    d = desc(window.dtype, n_fft, hop, n_frames, batch, False, 0, normalized, onesided)
    _call("plan_init_ranged", plan.device, (d, _p(window), _p(plan), int(frame_offset), int(total_frames)), kernels=2)


@torch.library.custom_op("specinv_b200::phase_init_ex", mutates_args=("c_main", "c_nyq", "phase_out"),
                         device_types="cuda")
def phase_init_ex(mag_main: Tensor, mag_nyq: Tensor, c_main: Tensor, c_nyq: Tensor, phase_in: Tensor,
                  phase_out: Tensor, n_fft: int, hop: int, onesided: bool) -> None:
    """phase_init over a frame range: phase_in / phase_out are (B, F) float64 running phases (may be empty)."""
    _need_cuda(mag_main, mag_nyq, c_main, c_nyq, phase_in, phase_out)
    d = desc(mag_main.dtype, n_fft, hop, mag_main.shape[1], mag_main.shape[0], False, 0, False, onesided)
    _call("phase_init_ex", mag_main.device, (d, _p(mag_main), _p(mag_nyq), _p(c_main), _p(c_nyq), _p(phase_in),
          _p(phase_out)), kernels=1)


@torch.library.custom_op("specinv_b200::halo_sum", mutates_args=("out",), device_types="cuda")
def halo_sum(left: Tensor, right: Tensor, out: Tensor) -> None:
    """out = left + right for (rows, n) views with unit inner stride (out may alias left or right)."""
    for t in (left, right, out):
        if not t.is_cuda or t.dim() != 2 or t.stride(1) != 1:
            raise RuntimeError("halo_sum needs 2-D CUDA views with unit inner stride")
    rows, n = out.shape
    _call("halo_sum", out.device, (_DT[out.dtype], _p(left), left.stride(0), _p(right), right.stride(0), _p(out),
          out.stride(0), rows, n), kernels=1)


def fill_padding_direct(x: Tensor, padded_offset: int, pad: int, signal_len: int, pad_mode: int) -> None:
    """The `fill_padding` op without its dispatch, like `iter_direct`: it runs after every iteration."""
    _call("fill_padding", x.device, (_DT[x.dtype], _p(x), x.stride(0), x.shape[0], int(padded_offset), x.shape[1],
          int(pad), int(signal_len), int(pad_mode)), kernels=1)


@torch.library.custom_op("specinv_b200::fill_padding", mutates_args=("x",), device_types="cuda")
def fill_padding(x: Tensor, padded_offset: int, pad: int, signal_len: int, pad_mode: int) -> None:
    """re-create the global centre padding inside the rank-local padded buffer x (rows, local_len)."""
    _need_cuda(x)
    fill_padding_direct(x, padded_offset, pad, signal_len, pad_mode)


# ---- fake (meta) kernels --------------------------------------------------------------------------------------
# Every op writes into caller-owned buffers and returns nothing, so its FakeTensor / meta implementation is "check
# the arguments, do nothing": torch.compile, FakeTensorMode and torch.export can trace through code that calls them
# (SURVEY.md section 8b).  The checks are the ones that do not need data: shapes that the C entry point derives
# sizes from.
def _fake_nothing(*args, **kwargs) -> None:
    return None


def _fake_iter(plan, x_in, x_out, *rest) -> None:
    if x_in.shape != x_out.shape:
        raise RuntimeError("specinv_b200: x_in / x_out shape mismatch")
    return None


ALL_OPS = (plan_init, stft, istft, gl_iter, admm_iter, pack, unpack, metric_sums, phase_init, spec_abs, rtisi_la,
           rtisi_la_steps, plan_init_ranged, phase_init_ex, halo_sum, fill_padding)
for _op in ALL_OPS:
    _op.register_fake(_fake_iter if _op in (gl_iter, admm_iter) else _fake_nothing)
del _op


def _fake_rtisi_la_stream(plan, window, mag_main, mag_nyq, x_out, inv_env, *rest) -> None:
    if x_out.dim() != 2 or inv_env.shape != (x_out.shape[1],) or mag_main.shape[0] != x_out.shape[0]:
        raise RuntimeError("specinv_b200: rtisi_la_stream window shapes disagree")
    return None


# the streaming entry (spectrogram_inversion_b200.streaming)
STREAM_OPS = (rtisi_la_stream,)
rtisi_la_stream.register_fake(_fake_rtisi_la_stream)


def _check_mel_inverse(P: Tensor, mel: Tensor, out: Tensor, f_lo: int, f_hi: int) -> None:
    if P.dim() != 2 or mel.dim() != 3 or out.dim() != 3:
        raise RuntimeError("specinv_b200: mel_inverse needs P (n_stft, n_mels), mel (B, n_mels, T), out (B, n_stft, T)")
    F, M = P.shape
    if tuple(mel.shape[:2]) != (out.shape[0], M) or tuple(out.shape[1:]) != (F, mel.shape[2]):
        raise RuntimeError(f"specinv_b200: mel_inverse shapes disagree: P {list(P.shape)}, mel {list(mel.shape)}, "
                           f"out {list(out.shape)}")
    if not P.dtype == mel.dtype == out.dtype or P.dtype not in (torch.float32, torch.float64):
        raise RuntimeError("specinv_b200: mel_inverse needs P, mel and out of one dtype, float32 or float64")
    if not 0 <= f_lo <= f_hi <= F:
        raise RuntimeError(f"specinv_b200: mel_inverse row range [{f_lo}, {f_hi}) outside [0, {F})")


def mel_inverse_direct(P: Tensor, mel: Tensor, out: Tensor, f_lo: int, f_hi: int) -> None:
    """out[b, f, t] = relu(sum_j P[f, j] mel[b, j, t]) for rows f in [f_lo, f_hi), 0 elsewhere (specinv_mel_inverse),
    called straight through ctypes: the module's one launch per call skips the custom op's dispatch (see
    `iter_direct`)."""
    _need_cuda(P, mel, out)
    _check_mel_inverse(P, mel, out, f_lo, f_hi)
    B, F, T = out.shape
    _call("mel_inverse", out.device, (_DT[out.dtype], _p(P), F, P.shape[1], int(f_lo), int(f_hi), _p(mel), _p(out), B,
          T), kernels=1)


@torch.library.custom_op("specinv_b200::mel_inverse", mutates_args=("out",), device_types="cuda")
def mel_inverse(P: Tensor, mel: Tensor, out: Tensor, f_lo: int, f_hi: int) -> None:
    """torchaudio's InverseMelScale as one GEMM: out (B, n_stft, T) = relu(P @ mel), P = pinv(fb.T) (n_stft, n_mels),
    mel (B, n_mels, T); rows of P outside [f_lo, f_hi) are zero and their outputs are written as zeros."""
    mel_inverse_direct(P, mel, out, f_lo, f_hi)


def _fake_mel_inverse(P, mel, out, f_lo, f_hi) -> None:
    _check_mel_inverse(P, mel, out, f_lo, f_hi)
    return None


# torchaudio_compat.InverseMelScale
MEL_OPS = (mel_inverse,)
mel_inverse.register_fake(_fake_mel_inverse)


def pghi_direct(mag: Tensor, out: Tensor, n_fft: int, hop: int, win_length: int, gamma: float, tol: float) -> None:
    """out (B, T, F) complex, contiguous = mag (B, F, T) real, any strides, times e^{i phi} of PGHI (specinv_pghi),
    called straight through ctypes like `mel_inverse_direct`; the workspace comes from torch's allocator."""
    _need_cuda(out)
    if not mag.is_cuda:
        raise RuntimeError("specinv_b200 ops only run on CUDA tensors (no CPU fallback)")
    B, F, T = mag.shape
    if tuple(out.shape) != (B, T, F) or out.dtype != CDT.get(mag.dtype):
        raise RuntimeError(f"specinv_b200: pghi shapes / dtypes disagree: mag {list(mag.shape)} {mag.dtype}, "
                           f"out {list(out.shape)} {out.dtype}")
    dt = _DT[mag.dtype]
    sb, sf, st = mag.stride()
    with torch.cuda.device(out.device):         # the workspace's size depends on the device's shared memory
        ws = torch.empty(_size("pghi_workspace_bytes", dt, B, F, T), dtype=torch.uint8, device=out.device)
        _call("pghi", out.device, (dt, _p(mag), sb, sf, st, _p(out), B, F, T, int(n_fft), int(hop), int(win_length),
              float(gamma), float(tol), _p(ws), ws.numel()), kernels=1)


def pghi_stream_state_bytes(dtype: torch.dtype, batch: int, n_bins: int) -> int:
    return _size("pghi_stream_state_bytes", _DT[dtype], int(batch), int(n_bins))


def pghi_stream_direct(mag: Tensor, frame0: int, n_final: int, final: bool, state: Tensor, out: Tensor, n_fft: int,
                       hop: int, win_length: int, gamma: float, tol: float) -> None:
    """Finalise n_final frames of a PGHI stream (specinv_pghi_stream): mag (B, F, n_rows) real, any strides, row r is
    frame frame0 + r; out (B, n_final, F) complex, contiguous; state from `pghi_stream_state_bytes`.  Straight
    through ctypes like `pghi_direct`."""
    _need_cuda(state, out)
    if not mag.is_cuda:
        raise RuntimeError("specinv_b200 ops only run on CUDA tensors (no CPU fallback)")
    B, F, R = mag.shape
    if tuple(out.shape) != (B, n_final, F) or out.dtype != CDT.get(mag.dtype):
        raise RuntimeError(f"specinv_b200: pghi_stream shapes / dtypes disagree: mag {list(mag.shape)} {mag.dtype}, "
                           f"out {list(out.shape)} {out.dtype}")
    sb, sf, st = mag.stride()
    _call("pghi_stream", out.device, (_DT[mag.dtype], _p(mag), sb, sf, st, int(frame0), R, int(n_final),
          int(bool(final)), _p(state), state.numel(), _p(out), B, F, int(n_fft), int(hop), int(win_length),
          float(gamma), float(tol)), kernels=1 if n_final else 0)
