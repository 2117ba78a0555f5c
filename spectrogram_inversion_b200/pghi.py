"""PGHI: phase-gradient heap integration, a non-iterative phase for a magnitude spectrogram.

Průša, Balazs and Søndergaard, IEEE/ACM TASLP 25(5), 2017, in the frame-causal form of Průša and Holighaus,
EUSIPCO 2017: the phase is integrated from the magnitude alone, through the analytic relation between the
log-magnitude gradient and the phase gradient of a (near-)Gaussian window, along the widest paths of significant
bins.  ``tests/golden/pghi_ref.py``'s ``pghi_heap`` is the definition; the sm_100a kernels of ``csrc/specinv_pghi.cu`` compute its scan
formulation (DESIGN.md section 3.7).
"""
from __future__ import annotations

import math

import torch

from . import _ops
from .engine import compute_device

__all__ = ["pghi"]


def _analysis(n_bins: int, stft_kwargs: dict):
    """(n_fft, hop, win_length) of a onesided spectrum: the defaults and the onesided rule of ``args_helper``
    (torch_specinv/methods.py:21-91), plus an explicit ``n_fft`` for odd sizes, which 2 (F - 1) cannot express."""
    window = stft_kwargs.get("window", None)
    onesided = stft_kwargs.get("onesided", None)
    if onesided is None:
        onesided = not (window is not None and window.is_complex())
    if not onesided:
        raise NotImplementedError("pghi: two-sided spectra are not supported (pass the onesided magnitude)")
    if window is not None and window.is_complex():
        raise NotImplementedError("pghi: complex windows are not supported")
    n_fft = stft_kwargs.get("n_fft", None)
    if n_fft is None:
        n_fft = (n_bins - 1) * 2
    n_fft = int(n_fft)
    if n_fft < 2 or n_fft // 2 + 1 != n_bins:
        raise ValueError(f"pghi: n_fft={n_fft} does not give {n_bins} onesided bins")
    win_length = stft_kwargs.get("win_length", None) or (window.numel() if window is not None else n_fft)
    hop = stft_kwargs.get("hop_length", None) or n_fft // 4
    if not 1 <= int(win_length) <= n_fft:
        raise ValueError(f"pghi: win_length={win_length} must lie in [1, n_fft={n_fft}]")
    if int(hop) < 1:
        raise ValueError(f"pghi: hop_length={hop} must be positive")
    return n_fft, int(hop), int(win_length)


def pghi(spec, gamma=None, tol=1e-5, **stft_kwargs):
    r"""Phase-gradient heap integration (PGHI): a phase for a magnitude spectrogram without iterations.

    The result is a good start for ``griffin_lim`` and ``ADMM``, which take a complex input as their start::

        x = griffin_lim(pghi(mag, **kw), **kw)

    Args:
        spec (Tensor): real onesided magnitude ``(..., F, T)``, float32 or float64, on the host or a CUDA device.
        gamma (float, optional): time-frequency ratio of the window, ``0.25645 * win_length**2`` by default (a Hann
            window's value; pass it for any other window).
        tol (float): bins at or below ``tol * max`` of their signal are not integrated and get phase 0.
        **stft_kwargs: the ``torch.stft`` arguments the magnitude came from (``hop_length``, ``win_length``,
            ``window``, ``onesided``; ``n_fft`` for an odd size).

    Returns:
        ``spec * exp(i phi)``, complex, in ``spec``'s shape and device.  Computed in float64 throughout; only the
        output is rounded to ``spec``'s precision.
    """
    if not isinstance(spec, torch.Tensor):
        raise TypeError("pghi: spec must be a torch.Tensor")
    if spec.is_complex():
        raise ValueError("pghi: spec must be a real magnitude, not a complex spectrum")
    if spec.requires_grad and torch.is_grad_enabled():
        raise NotImplementedError("pghi has no gradient path: detach the magnitude or call it under torch.no_grad()")
    if spec.dtype not in _ops.CDT:
        raise NotImplementedError(f"pghi: dtype {spec.dtype} is not supported (float32 / float64 only)")
    if spec.dim() < 2:
        raise ValueError(f"pghi: spec must be (..., F, T), got shape {list(spec.shape)}")
    if not (isinstance(tol, (int, float)) and 0 < tol < 1):
        raise ValueError(f"pghi: tol={tol} must lie in (0, 1)")
    shape = spec.shape
    F, T = shape[-2], shape[-1]
    n_fft, hop, win_length = _analysis(F, stft_kwargs)
    gamma = 0.25645 * win_length ** 2 if gamma is None else float(gamma)
    if not (gamma > 0 and math.isfinite(gamma)):
        raise ValueError(f"pghi: gamma={gamma} must be positive and finite")
    dev = compute_device(spec)
    m = spec.detach().to(dev).reshape(-1, F, T)
    B = m.shape[0]
    out = torch.empty(B, T, F, dtype=_ops.CDT[spec.dtype], device=dev)
    if B and T:
        _ops.pghi_direct(m, out, n_fft, hop, win_length, gamma, float(tol))
    return out.transpose(1, 2).reshape(shape).to(spec.device)
