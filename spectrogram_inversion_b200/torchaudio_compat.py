"""``torchaudio.functional.griffinlim`` and ``torchaudio.transforms.GriffinLim`` on the fused sm_100a kernels.

Same signatures, defaults, argument checks and recurrence as torchaudio, so a TTS or vocoder pipeline that ends in
torchaudio's Griffin-Lim can switch by changing the import.  torchaudio's fast Griffin-Lim takes the momentum on the
previous REBUILT spectrum (``a_k = S_k - m S_{k-1}``), not on the previous momentum spectrum like ``griffin_lim``
(``q_k = S_k - m q_{k-1}``); every iteration is one launch of ``specinv_gl_rebuilt_iter``.

The one-shot preprocessing runs on torch ops on the input's device, exactly as torchaudio runs it:
``specgram.pow(1 / power)``, the random (``torch.rand`` of the complex dtype) or all-ones start phases and their
product.  The same seed therefore gives the same start as torchaudio, for host and CUDA inputs alike.

These names are not exported at the package's top level: ``griffinlim`` next to ``griffin_lim`` would invite mistakes.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch
from torch import Tensor

from . import _lib, _ops
from .engine import SplitSpec, StftPlan, compute_device
from .stft_args import StftArgs

__all__ = ["griffinlim", "GriffinLim"]

_CPLX = {torch.float32: torch.complex64, torch.float64: torch.complex128}


def _check(shape, window: Optional[Tensor], n_fft: int, hop_length: int, win_length: int, n_iter: int,
           length: Optional[int]) -> None:
    """What torch.istft / torch.stft would reject inside torchaudio's loop, raised before any launch."""
    F, T = shape[-2], shape[-1]
    if F != n_fft // 2 + 1:
        raise RuntimeError("griffinlim: expected the frequency dimension (2nd to the last) of the spectrogram to match "
                           f"n_fft / 2 + 1 = {n_fft // 2 + 1}, but got {F}")
    if not 0 < win_length <= n_fft:
        raise RuntimeError(f"griffinlim: expected 0 < win_length <= n_fft, but got win_length={win_length}")
    if not 0 < hop_length <= win_length:
        raise RuntimeError(f"griffinlim: expected 0 < hop_length <= win_length, but got hop_length={hop_length}")
    if window is not None and tuple(window.shape) != (win_length,):
        raise RuntimeError(f"griffinlim: expected a 1D window tensor of size equal to win_length={win_length}, but got "
                           f"window with size {list(window.shape)}")
    if T < 1:
        raise RuntimeError("griffinlim: the spectrogram has no frames")
    if n_iter < 0:
        raise ValueError(f"griffinlim: n_iter must be >= 0, got {n_iter}")
    if n_iter == 0:
        if length is not None and length < 0:
            raise RuntimeError(f"griffinlim: length must be >= 0, got {length}")
        return
    # the loop's torch.stft of the length-`length` signal must give T frames again (torchaudio's a_k = S_k - m S_{k-1}
    # broadcasts them), and its reflect padding needs n_fft // 2 < length
    n = (T - 1) * hop_length if length is None else length
    if length is not None and 1 + length // hop_length != T:
        raise RuntimeError(f"griffinlim: length={length} gives {1 + length // hop_length} STFT frames, the spectrogram "
                           f"has {T}: with n_iter > 0 the length must lie in [{(T - 1) * hop_length}, "
                           f"{T * hop_length - 1}]")
    if n <= n_fft // 2:
        raise RuntimeError(f"griffinlim: reflect padding of {n_fft // 2} samples needs a longer signal than {n} samples")


class _Runner:
    """Buffers and launches of one call: the centred plan (``length`` None), or one un-centred frame range that holds
    the whole reflect-padded signal (``sharding.CudaRangeEngine`` with frame_offset 0, total_frames T) whose padding
    is re-created from ``length`` before every STFT."""

    def __init__(self, args: StftArgs, B: int, T: int, dtype: torch.dtype, dev: torch.device, length: Optional[int]):
        self.args, self.length, self.device = args, length, dev
        if length is None:
            self.engine = None
            self.plan = StftPlan(args, T, B, dtype, dev)
        else:
            from .sharding import CudaRangeEngine
            self.engine = CudaRangeEngine(args, T, B, dtype, dev, 0, T)
            self.engine.signal_len = length        # fill_padding mirrors around the caller's length
            self.plan = self.engine.plan
        self.P = 0 if length is None else args.pad      # buffer position of output sample 0
        # output samples [0, n_valid) come from the overlap-add; torch.istft zero-pads the rest (length > L0 + n_fft/2)
        L = self.plan.length
        self.out_len = L if length is None else length
        self.n_valid = min(self.out_len, L - self.P)
        self._fn = _lib.lib().specinv_gl_rebuilt_iter

    def check_envelope(self) -> None:
        """torch.istft's check: the window envelope over the output must not fall below 1e-11 (one host sync)."""
        if self.n_valid <= 0:
            return
        p = self.plan
        env = torch.empty(p.length, dtype=p.dtype, device=self.device)
        with torch.cuda.device(self.device):
            _ops._ok(_lib.lib().specinv_plan_envelope(p.desc_ref, _lib.C.c_void_p(p.buf.data_ptr()),
                                                      _lib.C.c_void_p(env.data_ptr()),
                                                      _lib.C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                     "plan_envelope", 0)
        low = float(env[self.P:self.P + self.n_valid].abs().min())
        if low < 1e-11:
            raise RuntimeError(f"istft(...): window overlap add min: {low:g} (below 1e-11): the window and hop leave "
                               "output samples that no frame covers")

    def istft(self, c: SplitSpec, x: Tensor) -> None:
        self.plan.istft(c, x)

    def iterate(self, x_in: Tensor, x_out: Tensor, s_in: Optional[SplitSpec], s_out: Optional[SplitSpec],
                mag: SplitSpec, m: float, sums: Optional[Tensor] = None) -> None:
        """One fused pass: s = STFT(x_in); s_out = s; x_out = ISTFT(mag * a / (|a| + 1e-16)), a = s - m s_in.
        ``s_in`` / ``s_out`` None (m == 0): plain Griffin-Lim, no state."""
        st = (None,) * 4 if s_in is None else (s_in.main, s_in.nyq, s_out.main, s_out.nyq)
        ptrs = _ops.pointers((self.plan.buf, x_in, x_out, *st, mag.main, mag.nyq))
        _ops.iter_direct(self._fn, "gl_rebuilt_iter", self.device, self.plan.desc_ref, ptrs, float(m),
                         sums.data_ptr() if sums is not None else None)

    def restore_padding(self, x: Tensor) -> None:
        if self.engine is not None:
            self.engine.fill_padding(x)

    def output(self, x: Tensor) -> Tensor:
        if self.engine is None:
            return x
        out = torch.zeros(x.shape[0], self.out_len, dtype=x.dtype, device=x.device)
        if self.n_valid > 0:
            out[:, :self.n_valid] = x[:, self.P:self.P + self.n_valid]
        return out


def _padded_window(window: Optional[Tensor], n_fft: int, win_length: int, dtype: torch.dtype,
                   dev: torch.device) -> Tensor:
    """The window as torch.stft / torch.istft apply it: centred in n_fft samples (ones when None)."""
    w = torch.ones(win_length, dtype=dtype) if window is None else window.detach()
    w = w.to(device=dev, dtype=dtype)
    left = (n_fft - win_length) // 2
    return torch.nn.functional.pad(w, [left, n_fft - win_length - left]).contiguous()


def griffinlim(specgram: Tensor, window: Tensor, n_fft: int, hop_length: int, win_length: int, power: float,
               n_iter: int, momentum: float, length: Optional[int], rand_init: bool) -> Tensor:
    r"""Waveform from a linear magnitude spectrogram by (fast) Griffin-Lim: ``torchaudio.functional.griffinlim``.

    Args:
        specgram (Tensor): magnitude spectrogram ``(..., freq, frames)``, freq = ``n_fft // 2 + 1``, raised to
            ``power``; float32 or float64, on the GPU or the host.
        window (Tensor): window of ``win_length`` samples (centred in ``n_fft``), or None for a rectangular one.
        n_fft, hop_length, win_length (int): the STFT of the spectrogram (always centred, reflect padding,
            unnormalised, onesided, as torchaudio fixes it).
        power (float): exponent of the spectrogram (1 for magnitude, 2 for power).
        n_iter (int): iterations; 0 returns the inverse STFT of the start.
        momentum (float): fast Griffin-Lim momentum in [0, 1); 0 is plain Griffin-Lim.
        length (int or None): output length.  With ``n_iter > 0`` it must give back the spectrogram's frame count,
            ``1 + length // hop_length == frames``; samples past ``(frames - 1) * hop_length + n_fft // 2`` are zeros.
        rand_init (bool): random start phases (``torch.rand`` of the complex dtype, drawn on specgram's device) if
            True, all ones otherwise.

    Returns:
        Tensor: ``(..., time)`` on specgram's device.

    Raises ``ValueError`` for a momentum outside [0, 1) (torchaudio's message), ``RuntimeError`` where torch.stft /
    torch.istft would fail inside torchaudio's loop (also when the window envelope falls below 1e-11), and
    ``NotImplementedError`` for an input that requires grad (there is no gradient path).
    """
    if not 0 <= momentum < 1:
        raise ValueError("momentum must be in range [0, 1). Found: {}".format(momentum))
    if specgram.requires_grad:
        raise NotImplementedError("torchaudio_compat.griffinlim has no gradient path: the input must not require grad")
    _check(specgram.shape, window, n_fft, hop_length, win_length, n_iter, length)
    m = momentum / (1 + momentum)

    # pack batch, then torchaudio's preprocessing, op for op on the input's device
    shape = specgram.size()
    specgram = specgram.reshape([-1] + list(shape[-2:]))
    specgram = specgram.pow(1 / power)
    cdt = _CPLX.get(specgram.dtype)
    if cdt is None:
        raise NotImplementedError(f"dtype {specgram.dtype} is not supported (float32 / float64 only)")
    if rand_init:
        angles = torch.rand(specgram.size(), dtype=cdt, device=specgram.device)
    else:
        angles = torch.full(specgram.size(), 1, dtype=cdt, device=specgram.device)
    start = specgram * angles

    B, _, T = specgram.shape
    dev = compute_device(specgram)
    dtype = specgram.dtype
    args = StftArgs(n_fft=int(n_fft), hop_length=int(hop_length), win_length=int(n_fft),
                    window=_padded_window(window, n_fft, win_length, dtype, dev), center=True, pad_mode="reflect",
                    normalized=False, onesided=True)
    run = _Runner(args, B, T, dtype, dev, None if length is None else int(length))
    run.check_envelope()
    mag = run.plan.pack(specgram)
    c = run.plan.pack(start)
    x = [run.plan.empty_signal(), run.plan.empty_signal()]
    run.istft(c, x[0])                                      # x_0 = ISTFT(mag * angles_0)
    del c
    if m == 0:
        s = [None, None]                                    # plain Griffin-Lim keeps no state
    else:
        s = [run.plan.empty_spec(), run.plan.empty_spec()]  # S_0 = 0: S_1 - m * 0 == S_1 exactly
        s[0].main.zero_()
        s[0].nyq.zero_()
    cur = 0
    for _ in range(n_iter):
        run.restore_padding(x[cur])
        run.iterate(x[cur], x[cur ^ 1], s[cur], s[cur ^ 1], mag, m)
        cur ^= 1
    y = run.output(x[cur])
    y = y.reshape(shape[:-2] + y.shape[-1:])
    if y.device == specgram.device:
        return y
    out = torch.empty(y.shape, dtype=y.dtype, pin_memory=specgram.is_pinned())
    out.copy_(y, non_blocking=True)
    torch.cuda.current_stream(y.device).synchronize()
    return out


class GriffinLim(torch.nn.Module):
    r"""``torchaudio.transforms.GriffinLim`` on the fused kernels: same constructor, defaults and buffer.

    Args:
        n_fft (int): default 400.  n_iter (int): default 32.  win_length (int or None): default ``n_fft``.
        hop_length (int or None): default ``win_length // 2``.  window_fn: default ``torch.hann_window``.
        power (float): default 2.  wkwargs (dict or None): arguments of ``window_fn``.  momentum (float): default
        0.99.  length (int or None): default None.  rand_init (bool): default True.

    The window is a registered buffer: ``.to()`` moves it and ``state_dict()`` holds it, as in torchaudio.
    """
    __constants__ = ["n_fft", "n_iter", "win_length", "hop_length", "power", "length", "momentum", "rand_init"]

    def __init__(self, n_fft: int = 400, n_iter: int = 32, win_length: Optional[int] = None,
                 hop_length: Optional[int] = None, window_fn: Callable[..., Tensor] = torch.hann_window,
                 power: float = 2.0, wkwargs: Optional[dict] = None, momentum: float = 0.99,
                 length: Optional[int] = None, rand_init: bool = True) -> None:
        super().__init__()
        if not (0 <= momentum < 1):
            raise ValueError("momentum must be in the range [0, 1). Found: {}".format(momentum))
        self.n_fft = n_fft
        self.n_iter = n_iter
        self.win_length = win_length if win_length is not None else n_fft
        self.hop_length = hop_length if hop_length is not None else self.win_length // 2
        window = window_fn(self.win_length) if wkwargs is None else window_fn(self.win_length, **wkwargs)
        self.register_buffer("window", window)
        self.length = length
        self.power = power
        self.momentum = momentum
        self.rand_init = rand_init

    def forward(self, specgram: Tensor) -> Tensor:
        return griffinlim(specgram, self.window, self.n_fft, self.hop_length, self.win_length, self.power, self.n_iter,
                          self.momentum, self.length, self.rand_init)
