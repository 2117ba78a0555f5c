"""torchaudio.functional.griffinlim restated with torch.stft / torch.istft only, so that the tests of
spectrogram_inversion_b200.torchaudio_compat need torch and not torchaudio.  ``griffinlim`` is op for op torchaudio's
code (tests/test_torchaudio_compat_host.py shows it is bit for bit equal whenever torchaudio imports); the pieces are
exposed for the single-iteration parity tests."""
from __future__ import annotations

from typing import Optional

import torch

_CPLX = {torch.float32: torch.complex64, torch.float64: torch.complex128}


def stft(x, window, n_fft, hop_length, win_length):
    return torch.stft(input=x, n_fft=n_fft, hop_length=hop_length, win_length=win_length, window=window, center=True,
                      pad_mode="reflect", normalized=False, onesided=True, return_complex=True)


def istft(spec, window, n_fft, hop_length, win_length, length):
    return torch.istft(spec, n_fft=n_fft, hop_length=hop_length, win_length=win_length, window=window, length=length)


def start_angles(specgram: torch.Tensor, rand_init: bool) -> torch.Tensor:
    """torchaudio's start phases for a (B, F, T) spectrogram (drawn from the global generator when rand_init)."""
    cdt = _CPLX[specgram.dtype]
    if rand_init:
        return torch.rand(specgram.size(), dtype=cdt, device=specgram.device)
    return torch.full(specgram.size(), 1, dtype=cdt, device=specgram.device)


def iteration(x, s_prev, mag, m, window, n_fft, hop_length, win_length, length):
    """One pass of the loop from the signal x and the previous rebuilt spectrum s_prev (None: plain GL):
    returns (x_out, rebuilt)."""
    rebuilt = stft(x, window, n_fft, hop_length, win_length)
    angles = rebuilt
    if s_prev is not None:
        angles = angles - s_prev * m
    angles = angles.div(angles.abs().add(1e-16))
    return istft(mag * angles, window, n_fft, hop_length, win_length, length), rebuilt


def loop(specgram, angles, window, n_fft, hop_length, win_length, n_iter, momentum, length):
    """torchaudio's loop on an already powered (B, F, T) spectrogram and given start angles."""
    momentum = momentum / (1 + momentum)
    tprev = torch.tensor(0.0, dtype=specgram.dtype, device=specgram.device)
    for _ in range(n_iter):
        inverse = istft(specgram * angles, window, n_fft, hop_length, win_length, length)
        rebuilt = stft(inverse, window, n_fft, hop_length, win_length)
        angles = rebuilt
        if momentum:
            angles = angles - tprev.mul_(momentum)
        angles = angles.div(angles.abs().add(1e-16))
        tprev = rebuilt
    return istft(specgram * angles, window, n_fft, hop_length, win_length, length)


def griffinlim(specgram, window, n_fft, hop_length, win_length, power, n_iter, momentum, length: Optional[int],
               rand_init):
    """torchaudio.functional.griffinlim, same arguments, same random draws."""
    if not 0 <= momentum < 1:
        raise ValueError("momentum must be in range [0, 1). Found: {}".format(momentum))
    shape = specgram.size()
    specgram = specgram.reshape([-1] + list(shape[-2:]))
    specgram = specgram.pow(1 / power)
    angles = start_angles(specgram, rand_init)
    waveform = loop(specgram, angles, window, n_fft, hop_length, win_length, n_iter, momentum, length)
    return waveform.reshape(shape[:-2] + waveform.shape[-1:])


def spectral_convergence(x, mag, window, n_fft, hop_length, win_length):
    """|| |STFT(x)| - mag ||_F / || mag ||_F  over the whole batch (mag: (B, F, T), already powered)."""
    s = stft(x.reshape(-1, x.shape[-1]).to(torch.float64), window.to(torch.float64), n_fft, hop_length, win_length)
    mag = mag.reshape(s.shape).to(torch.float64)
    return float(torch.linalg.vector_norm(s.abs() - mag) / torch.linalg.vector_norm(mag))
