"""CPU-side checks of streaming RTISI-LA: the fake kernel of its custom op, the host-side argument checks of
specinv_rtisi_la_stream / specinv_plan_inv_env_window (they return SPECINV_ERR_INVALID before any launch, so no
device is needed) and the emitted-count rule E(n) against the reference's output-length rule."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import specinv_oracle as O


@pytest.fixture(scope="module")
def lib():
    from spectrogram_inversion_b200.build import build_library
    build_library()
    from spectrogram_inversion_b200 import _lib
    return _lib


def test_stream_op_has_a_fake_kernel():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from spectrogram_inversion_b200 import _ops
    assert _ops.rtisi_la_stream not in _ops.ALL_OPS and _ops.rtisi_la_stream in _ops.STREAM_OPS
    with FakeTensorMode():
        f = lambda *shape, dt=torch.float32: torch.empty(*shape, dtype=dt, device="cuda")
        B, M = 2, 64
        plan, state = torch.empty(4096, dtype=torch.uint8, device="cuda"), torch.empty(8192, dtype=torch.uint8, device="cuda")
        k = (128, 32, True, False, True)
        args = (f(128), f(B, 5, M), f(B, 5))
        assert _ops.rtisi_la_stream(plan, *args, f(B, 96), f(96), f(256), state, 9, 4, 160, 3, False, 25, 0.99, 0.1,
                                    7, 9, False, *k) is None
        with pytest.raises(RuntimeError):      # the 1/envelope window must match the output window
            _ops.rtisi_la_stream(plan, *args, f(B, 96), f(95), f(256), state, 9, 4, 160, 3, False, 25, 0.99, 0.1,
                                 7, 9, False, *k)
        with pytest.raises(RuntimeError):      # one magnitude window per signal
            _ops.rtisi_la_stream(plan, f(128), f(B + 1, 5, M), f(B + 1, 5), f(B, 96), f(96), f(256), state, 9, 4, 160,
                                 3, False, 25, 0.99, 0.1, 7, 9, False, *k)


def _call(lib, **over):
    """specinv_rtisi_la_stream with n_fft 1024 / hop 256, centred, look_ahead 3 (P = 512): 20 frames so far, steps
    [10, 20) on rows of frames 7 .. 19, samples [(10-3)*256 - 512, (20-3)*256 - 512) = [1280, 3840)."""
    p = dict(n_fft=1024, hop=256, n_frames=20, B=2, center=True, frame0=7, n_rows=13, x0=1280, x_len=2560, la=3,
             max_iter=25, alpha=0.99, sb=10, se=20, final=0, dtype=lib.F32)
    p.update(over)
    d = lib.make_desc(p["n_fft"], p["hop"], p["n_frames"], p["B"], p["center"], 0, False, True, p["dtype"])
    ptr = lambda name: None if over.get(name, 1) is None else C.c_void_p(0x1000)
    return lib.lib().specinv_rtisi_la_stream(
        C.byref(d), ptr("plan"), ptr("window"), ptr("mag_main"), ptr("mag_nyq"), p["frame0"], p["n_rows"], ptr("x_out"),
        ptr("inv_env"), p["x0"], p["x_len"], ptr("scratch"), p["la"], 0, p["max_iter"], p["alpha"], 0.25, p["sb"],
        p["se"], p["final"], ptr("state"), None)


BAD_STREAM_ARGS = [
    dict(plan=None), dict(window=None), dict(mag_main=None), dict(mag_nyq=None), dict(x_out=None), dict(inv_env=None),
    dict(scratch=None), dict(state=None),
    dict(n_frames=0), dict(max_iter=0), dict(alpha=-0.5), dict(final=2),
    dict(se=21),                                   # a step past the frames pushed so far, not final
    dict(se=24, final=1, x_len=(19 * 256 + 1024 - 1024) - 1280),   # past n_frames + LA even when final
    dict(sb=11, se=10), dict(sb=20, se=20),        # empty range: only the final launch at n_frames + LA
    dict(sb=-1),
    dict(frame0=8, n_rows=12),                     # the resume re-reads frame 10 - 3 = 7
    dict(n_rows=12),                               # does not reach frame 19
    dict(n_rows=14),                               # past the frames pushed
    dict(frame0=-1, n_rows=14), dict(n_rows=-1),
    dict(x0=1024, x_len=2816),                     # x window starts before the first sample these steps finish
    dict(x_len=2559), dict(x_len=2816),            # ... ends short of / past the last one
    dict(final=1, se=23),                          # the last final step's window runs to L = 19 * 256 = 4864
    dict(n_fft=1000, hop=0), dict(dtype=7),
]


@pytest.mark.parametrize("bad", BAD_STREAM_ARGS, ids=lambda b: ",".join(f"{k}={v}" for k, v in b.items()))
def test_stream_entry_rejects_bad_arguments_before_any_launch(lib, bad):
    assert _call(lib, **bad) == -1


def test_inv_env_window_rejects_bad_arguments(lib):
    h = lib.lib()
    short = lib.make_desc(1024, 256, 5, 1, True, 0, False, True, lib.F32)        # T0 = 5: (5 - 1) * 256 >= 1024
    tiny = lib.make_desc(1024, 256, 4, 1, True, 0, False, True, lib.F32)         # (4 - 1) * 256 < 1024
    p, out = C.c_void_p(0x1000), C.c_void_p(0x2000)
    assert h.specinv_plan_inv_env_window(C.byref(short), None, 0, 16, -1, out, None) == -1
    assert h.specinv_plan_inv_env_window(C.byref(short), p, 0, 16, -1, None, None) == -1
    assert h.specinv_plan_inv_env_window(C.byref(short), p, -1, 16, -1, out, None) == -1
    assert h.specinv_plan_inv_env_window(C.byref(short), p, 0, 16, 4, out, None) == -1      # a plan of 4 frames reads it
    assert h.specinv_plan_inv_env_window(C.byref(tiny), p, 0, 16, 40, out, None) == -1      # head and tail overlap
    assert h.specinv_plan_inv_env_window(C.byref(short), p, 0, 10 * 256 + 1, 11, out, None) == -1   # past L(11)
    assert h.specinv_plan_inv_env_window(C.byref(short), p, 0, 4 * 256 + 1, 5, out, None) == -1     # past L(5)
    assert h.specinv_plan_inv_env_window(C.byref(short), p, 0, 0, -1, None, None) == 0      # nothing to gather


def _emitted_by_restatement(n, n_fft, hop, look_ahead, center):
    """Samples of [0, L(n)) finished by the commits of steps 0 .. n-1 (methods.py:401-408): step i commits frame
    i - LA, whose overlap-add block [(i-LA)*hop - P, (i-LA+1)*hop - P) of the trimmed signal is complete then."""
    a = O.args_helper(n_fft // 2 + 1, np.float32, hop_length=hop, center=center)
    LA = (n_fft - 1) // hop if look_ahead < 0 else look_ahead
    L = a.signal_length(n) if n else 0
    done = 0
    for i in range(n):
        if i >= LA:
            done = max(done, min((i - LA + 1) * hop - a.pad, L))
    return max(done, 0)


@pytest.mark.parametrize("n_fft,hop", [(1024, 256), (256, 160), (250, 62), (512, 512), (64, 7)])
@pytest.mark.parametrize("look_ahead", [-1, 0, 1, 3, 9])
@pytest.mark.parametrize("center", [True, False])
def test_emitted_count_rule(n_fft, hop, look_ahead, center):
    from spectrogram_inversion_b200.streaming import emitted_samples
    for n in range(0, 40):
        assert emitted_samples(n, n_fft, hop, look_ahead, center) == _emitted_by_restatement(n, n_fft, hop, look_ahead,
                                                                                            center), n


def test_stream_options_are_checked_like_rtisi_la():
    from spectrogram_inversion_b200 import RTISIStream
    with pytest.raises(AssertionError):
        RTISIStream(max_iter=0)
    with pytest.raises(AssertionError):
        RTISIStream(alpha=-0.1)
    with pytest.raises(TypeError, match="unexpected keyword argument 'foo'"):
        RTISIStream(foo=1)
    RTISIStream(asymmetric_window=True, foo=1)          # the asymmetric path ignores unknown keys, as RTISI_LA does
    s = RTISIStream(max_iter=1)
    with pytest.raises(RuntimeError, match="no frame"):
        s.flush()
    with pytest.raises(AssertionError):
        s.push(torch.rand(65, 3).to(torch.complex64))
    with pytest.raises(NotImplementedError):
        s.push(torch.rand(65, 3, requires_grad=True))
