"""``torchaudio.functional.griffinlim`` and ``torchaudio.transforms.GriffinLim`` on the fused sm_100a kernels.

Same signatures, defaults, argument checks and recurrence as torchaudio, so a TTS or vocoder pipeline that ends in
torchaudio's Griffin-Lim can switch by changing the import.  torchaudio's fast Griffin-Lim takes the momentum on the
previous REBUILT spectrum (``a_k = S_k - m S_{k-1}``), not on the previous momentum spectrum like ``griffin_lim``
(``q_k = S_k - m q_{k-1}``); every iteration is one launch of ``specinv_gl_rebuilt_iter``.

The one-shot preprocessing runs on torch ops on the input's device, exactly as torchaudio runs it:
``specgram.pow(1 / power)``, the random (``torch.rand`` of the complex dtype) or all-ones start phases and their
product.  The same seed therefore gives the same start as torchaudio, for host and CUDA inputs alike.

``InverseMelScale`` is ``torchaudio.transforms.InverseMelScale`` with the same filterbank, bit for bit, so that
``InverseMelScale`` -> ``GriffinLim`` takes a mel spectrogram to a waveform as torchaudio's Tacotron2 Griffin-Lim
vocoder does.  torchaudio's ``relu(lstsq(fb.T, mel).solution)`` is ``relu(P @ mel)`` per frame with
``P = pinv(fb.T)``; ``P`` is computed once per filterbank on the host in float64 and applied by one launch of
``specinv_mel_inverse``.

These names are not exported at the package's top level: ``griffinlim`` next to ``griffin_lim`` would invite mistakes.
"""
from __future__ import annotations

import math
import warnings
from typing import Callable, Optional, Tuple

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


# ---- InverseMelScale ---------------------------------------------------------------------------------------------
# torchaudio.functional.melscale_fbanks restated op for op (same float32 linspace, same slopes, same min / max), so
# that `fb` is bitwise torchaudio's and a state_dict moves between the two modules.
def _hz_to_mel(freq: float, mel_scale: str = "htk") -> float:
    if mel_scale not in ["slaney", "htk"]:
        raise ValueError('mel_scale should be one of "htk" or "slaney".')
    if mel_scale == "htk":
        return 2595.0 * math.log10(1.0 + (freq / 700.0))
    f_min = 0.0
    f_sp = 200.0 / 3
    mels = (freq - f_min) / f_sp
    min_log_hz = 1000.0
    min_log_mel = (min_log_hz - f_min) / f_sp
    logstep = math.log(6.4) / 27.0
    if freq >= min_log_hz:
        mels = min_log_mel + math.log(freq / min_log_hz) / logstep
    return mels


def _mel_to_hz(mels: Tensor, mel_scale: str = "htk") -> Tensor:
    if mel_scale not in ["slaney", "htk"]:
        raise ValueError('mel_scale should be one of "htk" or "slaney".')
    if mel_scale == "htk":
        return 700.0 * (10.0 ** (mels / 2595.0) - 1.0)
    f_min = 0.0
    f_sp = 200.0 / 3
    freqs = f_min + f_sp * mels
    min_log_hz = 1000.0
    min_log_mel = (min_log_hz - f_min) / f_sp
    logstep = math.log(6.4) / 27.0
    log_t = mels >= min_log_mel
    freqs[log_t] = min_log_hz * torch.exp(logstep * (mels[log_t] - min_log_mel))
    return freqs


def _create_triangular_filterbank(all_freqs: Tensor, f_pts: Tensor) -> Tensor:
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    zero = torch.zeros(1)
    down_slopes = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up_slopes = slopes[:, 2:] / f_diff[1:]
    return torch.max(zero, torch.min(down_slopes, up_slopes))


def _melscale_fbanks(n_freqs: int, f_min: float, f_max: float, n_mels: int, sample_rate: int,
                     norm: Optional[str] = None, mel_scale: str = "htk") -> Tensor:
    """(n_freqs, n_mels) triangular filterbank: ``torchaudio.functional.melscale_fbanks``, bit for bit."""
    if norm is not None and norm != "slaney":
        raise ValueError('norm must be one of None or "slaney"')
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_min = _hz_to_mel(f_min, mel_scale=mel_scale)
    m_max = _hz_to_mel(f_max, mel_scale=mel_scale)
    m_pts = torch.linspace(m_min, m_max, n_mels + 2)
    f_pts = _mel_to_hz(m_pts, mel_scale=mel_scale)
    fb = _create_triangular_filterbank(all_freqs, f_pts)
    if norm is not None and norm == "slaney":
        enorm = 2.0 / (f_pts[2:n_mels + 2] - f_pts[:n_mels])
        fb *= enorm.unsqueeze(0)
    if (fb.max(dim=0).values == 0.0).any():
        warnings.warn(
            "At least one mel filterbank has all zero values. "
            f"The value for `n_mels` ({n_mels}) may be set too high. "
            f"Or, the value for `n_freqs` ({n_freqs}) may be set too low."
        )
    return fb


_DRIVERS = ["gels", "gelsy", "gelsd", "gelss"]


def _mel_operator(fb: Tensor, driver: str) -> Tuple[Tensor, int, int]:
    """``(P, f_lo, f_hi)``: ``P = pinv(fb.T)`` of shape (n_stft, n_mels), computed in float64 from the SVD and
    returned in fb's dtype on fb's device, and the rows ``[f_lo, f_hi)`` outside which ``fb`` (hence ``P``) is zero.

    Singular values ``<= sigma_max * max(n_stft, n_mels) * eps64`` are dropped: the default cutoff of
    ``torch.linalg.pinv``, ``matrix_rank`` and ``lstsq(driver="gelsd")``.  With ``driver="gels"`` a rank below
    n_mels raises ``torch.linalg.LinAlgError``, as LAPACK's gels does on the host; the other drivers return the
    minimum-norm solution.  The product is ``torch.linalg.pinv``'s; the rows of ``P`` that no filter covers are zero
    in exact arithmetic and are set to exactly zero (the SVD leaves ~1e-16 there)."""
    A = fb.detach().to("cpu", torch.float64).T                      # fb.T: (n_mels, n_stft)
    n_mels, n_stft = A.shape
    covered = torch.nonzero(A.ne(0).any(dim=0)).flatten()
    f_lo, f_hi = (int(covered[0]), int(covered[-1]) + 1) if covered.numel() else (0, 0)
    U, S, Vh = torch.linalg.svd(A, full_matrices=False)
    keep = S > S.max() * max(n_stft, n_mels) * torch.finfo(torch.float64).eps
    rank = int(keep.sum())
    P = (Vh.mT * torch.where(keep, 1 / S, torch.zeros_like(S)).unsqueeze(-2)) @ U.mT
    P[:f_lo] = 0
    P[f_hi:] = 0
    if driver == "gels" and rank < n_mels:
        raise torch.linalg.LinAlgError(
            "torch.linalg.lstsq: The least squares solution could not be computed because the input matrix does not "
            f"have full rank (rank {rank} of {n_mels}: the mel filterbank has dependent or all-zero filters; "
            "driver='gelsd' returns the minimum-norm solution)")
    return P.to(device=fb.device, dtype=fb.dtype).contiguous(), f_lo, f_hi


class InverseMelScale(torch.nn.Module):
    r"""``torchaudio.transforms.InverseMelScale`` on one sm_100a kernel: same constructor, defaults, ``fb`` buffer and
    checks.  Estimates the linear magnitude spectrogram as ``relu(pinv(fb.T) @ mel)``, the minimum-norm least-squares
    solution torchaudio's ``relu(lstsq(fb.T, mel).solution)`` returns.

    Args:
        n_stft (int): number of STFT bins (``n_fft // 2 + 1``).  n_mels (int): default 128.  sample_rate (int):
        default 16000.  f_min (float): default 0.  f_max (float or None): default ``sample_rate // 2`` (so does 0).
        norm (str or None): None or ``"slaney"``.  mel_scale (str): ``"htk"`` (default) or ``"slaney"``.
        driver (str): ``"gels"`` (default), ``"gelsy"``, ``"gelsd"`` or ``"gelss"``.

    ``pinv(fb.T)`` is computed once per filterbank on the host in float64 and cached on the module, keyed on fb's
    device, dtype and version, so ``.to()``, ``.double()`` and ``load_state_dict`` take effect; ``state_dict()``
    holds only ``fb``.  Input and ``fb`` must share dtype and device; ``.double()`` the module for float64.  A host
    module takes host input, computes on the current CUDA device and returns a host tensor.

    Possible deviations from torchaudio for CUDA inputs: torchaudio documents only ``"gels"`` there and assumes a
    full-rank ``fb``.  Here the rule is the same on every device: ``"gels"`` raises ``torch.linalg.LinAlgError``
    when the rank (with ``torch.linalg.pinv``'s cutoff) is below n_mels, as torchaudio's host path does, and the
    other drivers return the minimum-norm solution.  The result depends only on the values, not on the device.

    There is no gradient: an input that requires grad raises ``NotImplementedError``.  torchaudio's Tacotron2
    Griffin-Lim vocoder calls ``requires_grad_(True)`` on the mel and detaches the result on the next line, a
    leftover of the older gradient-descent InverseMelScale; drop that line when switching to this module.
    """
    __constants__ = ["n_stft", "n_mels", "sample_rate", "f_min", "f_max"]

    def __init__(self, n_stft: int, n_mels: int = 128, sample_rate: int = 16000, f_min: float = 0.0,
                 f_max: Optional[float] = None, norm: Optional[str] = None, mel_scale: str = "htk",
                 driver: str = "gels") -> None:
        super().__init__()
        self.n_stft = n_stft
        self.n_mels = n_mels
        self.sample_rate = sample_rate
        self.f_max = f_max or float(sample_rate // 2)
        self.f_min = f_min
        self.norm = norm
        self.mel_scale = mel_scale
        self.driver = driver
        if f_min > self.f_max:
            raise ValueError("Require f_min: {} <= f_max: {}".format(f_min, self.f_max))
        if driver not in _DRIVERS:
            raise ValueError(f'driver must be one of ["gels", "gelsy", "gelsd", "gelss"]. Found {driver}.')
        fb = _melscale_fbanks(self.n_stft, self.f_min, self.f_max, self.n_mels, self.sample_rate, self.norm,
                              self.mel_scale)
        self.register_buffer("fb", fb)
        self._op_cache = None       # (key, P, f_lo, f_hi); deliberately not a buffer

    def operator(self) -> Tuple[Tensor, int, int]:
        """``(P, f_lo, f_hi)`` of the current ``fb`` (see ``_mel_operator``), recomputed when fb changes."""
        fb = self.fb
        key = (fb.device, fb.dtype, fb._version, fb.data_ptr())
        if self._op_cache is None or self._op_cache[0] != key:
            self._op_cache = (key, *_mel_operator(fb, self.driver))
        return self._op_cache[1:]

    def forward(self, melspec: Tensor) -> Tensor:
        r"""
        Args:
            melspec (Tensor): mel spectrogram ``(..., n_mels, time)``, in fb's dtype, on fb's device.

        Returns:
            Tensor: linear magnitude spectrogram ``(..., n_stft, time)`` on melspec's device.
        """
        if melspec.dim() < 2:
            raise RuntimeError(f"InverseMelScale: expected a (..., n_mels, time) tensor, got shape {list(melspec.shape)}")
        shape = melspec.size()
        n_mels, time = shape[-2], shape[-1]
        freq = self.fb.size(0)
        if self.n_mels != n_mels:
            raise ValueError("Expected an input with {} mel bins. Found: {}".format(self.n_mels, n_mels))
        if melspec.requires_grad:
            raise NotImplementedError("torchaudio_compat.InverseMelScale has no gradient path: the input must not "
                                      "require grad")
        if melspec.dtype != self.fb.dtype:
            raise RuntimeError("torch.linalg.lstsq: Expected input and other to have the same dtype, but got "
                               f"input's dtype {self.fb.dtype} and other's dtype {melspec.dtype}")
        if melspec.device != self.fb.device:
            raise RuntimeError(f"InverseMelScale: fb is on {self.fb.device} and the input on {melspec.device}: move "
                               "the module with .to()")
        if self.fb.dtype not in (torch.float32, torch.float64):
            raise RuntimeError(f"InverseMelScale: dtype {self.fb.dtype} is not supported (float32 / float64 only)")
        P, f_lo, f_hi = self.operator()
        mel = melspec.reshape(math.prod(shape[:-2]), n_mels, time)
        if mel.numel() == 0 or time == 0:
            return torch.zeros(shape[:-2] + (freq, time), dtype=melspec.dtype, device=melspec.device)
        dev = compute_device(mel)
        mel = mel.to(dev, non_blocking=True).contiguous()
        out = torch.empty(mel.shape[0], freq, time, dtype=mel.dtype, device=dev)
        _ops.mel_inverse_direct(P.to(dev), mel, out, f_lo, f_hi)
        out = out.view(shape[:-2] + (freq, time))
        if dev == melspec.device:
            return out
        y = torch.empty(out.shape, dtype=out.dtype, pin_memory=melspec.is_pinned())
        y.copy_(out, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return y
