"""PGHI on the GPU (csrc/specinv_pghi.cu) against the scan formulation of tests/golden/pghi_ref.py (pghi_phase,
which equals the heap definition bit for bit on tie-free magnitudes: tests/test_pghi_host.py).

The reference is C_ref = mag * exp(i phi) in float64.  Per bin:
  * float32: |C - C_ref| <= 4e-7 mag: the output's rounding to float32 (the kernel computes in float64 too);
  * float64: |C - C_ref| <= 1e-9 mag: re-associated float64 sums of phases kept in [-pi, pi].
The choices (which neighbour reaches a bin) depend on magnitudes only and are exact, so a wrong choice shows as an
error of the size of a phase step.  Small batches split time into chunks of >= 32 frames (T // 32 chunks when
T < 1568 and B <= 3), so T = 64, 65, 95, 96 and 400 put chunk seams at every offset the apply pass can meet."""
import math

import numpy as np
import pytest
import torch

import pghi_ref as P
from oracle import specinv_oracle as O
from spectrogram_inversion_b200 import ADMM, griffin_lim, pghi

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 4e-7, torch.float64: 1e-9}


def signals(B, n, sr=16000, seed=0):
    """Harmonic tones with vibrato and an envelope, a chirp, and a little noise: (B, n) float64."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n, dtype=torch.float64) / sr
    out = []
    for b in range(B):
        f0 = 110 + 60 * torch.rand((), generator=g, dtype=torch.float64)
        f = f0 * (1 + 0.05 * torch.sin(2 * math.pi * (0.5 + b % 3) * t))
        ph = 2 * math.pi * torch.cumsum(f, 0) / sr
        x = sum((0.6 / k) * torch.sin(k * ph) for k in range(1, 12))
        x = x * (0.6 + 0.4 * torch.sin(2 * math.pi * 1.5 * t) ** 2)
        x = x + 0.3 * torch.sin(2 * math.pi * (300 * t + 900 * t ** 2))
        out.append(x + 0.003 * torch.randn(n, generator=g, dtype=torch.float64))
    return torch.stack(out)


def magnitude(B, n_fft, hop, T, dtype, win_length=None, center=True, seed=0):
    wl = win_length or n_fft
    n = (T - 1) * hop + (0 if center else n_fft)
    x = signals(B, max(n, 1), seed=seed)
    X = torch.stft(x, n_fft, hop, win_length=wl, window=torch.hann_window(wl, dtype=torch.float64), center=center,
                   return_complex=True)
    return X.abs()[..., :T].to(dtype).contiguous()


def reference(mag, n_fft, hop, win_length=None, gamma=None, tol=1e-5):
    m = mag.detach().cpu().numpy()
    ph = P.pghi_phase(m.reshape(-1, *m.shape[-2:]), n_fft, hop, win_length, gamma, tol).reshape(m.shape)
    return m.astype(np.float64) * np.exp(1j * ph)


def check(C, mag, ref, dtype):
    assert C.dtype == (torch.complex64 if dtype == torch.float32 else torch.complex128)
    assert C.shape == mag.shape
    c = C.detach().cpu().numpy().astype(np.complex128)
    m = mag.detach().cpu().numpy().astype(np.float64)
    err = np.abs(c - ref)
    bad = err > TOL[dtype] * m
    assert not bad.any(), f"{bad.sum()} bins off, worst {np.max(err / np.maximum(m, 1e-300)):.3e} x mag"


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n_fft,hop,B,T", [(512, 128, 3, 40), (1024, 256, 1, 96), (2048, 512, 1, 65), (400, 100, 3, 64),
                                           (1000, 250, 1, 95), (401, 100, 1, 70)])
def test_against_reference(n_fft, hop, B, T, dtype):
    mag = magnitude(B, n_fft, hop, T, dtype).cuda()
    kw = dict(hop_length=hop, n_fft=n_fft) if n_fft % 2 else dict(hop_length=hop)
    check(pghi(mag, **kw), mag, reference(mag, n_fft, hop), dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_batches_short_window_uncentred(dtype):
    for B in (1, 3, 64):
        T = 400 if B == 1 else 24
        mag = magnitude(B, 1024, 256, T, dtype, win_length=800, center=False, seed=B).cuda()
        check(pghi(mag, hop_length=256, win_length=800), mag, reference(mag, 1024, 256, win_length=800), dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_gamma_and_tol(dtype):
    mag = magnitude(2, 512, 128, 50, dtype, seed=3).cuda()
    check(pghi(mag, gamma=0.2 * 512 ** 2, tol=1e-3, hop_length=128), mag,
          reference(mag, 512, 128, gamma=0.2 * 512 ** 2, tol=1e-3), dtype)


def test_leading_dims_host_input_and_one_frame():
    mag = magnitude(6, 512, 128, 30, torch.float32, seed=4)
    lead = mag.reshape(2, 3, *mag.shape[-2:])
    C = pghi(lead, hop_length=128)
    assert C.device.type == "cpu" and C.shape == lead.shape
    check(C.reshape(mag.shape), mag, reference(mag, 512, 128), torch.float32)
    assert torch.equal(pghi(lead.cuda(), hop_length=128).cpu(), C)
    one = mag[:2, :, :1].cuda()
    check(pghi(one, hop_length=128), one, reference(one, 512, 128), torch.float32)
    check(pghi(mag[0], hop_length=128), mag[0], reference(mag[0], 512, 128), torch.float32)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_silence_and_ties(dtype):
    mag = magnitude(3, 512, 128, 70, dtype, seed=5)
    mag[1] = 0
    mag[2, :, 10:20] = 0                                             # silent frames inside a signal
    q = torch.round(mag / mag.amax() * 64) / 64                      # quantised: many equal magnitudes
    for m in (mag.cuda(), q.cuda()):
        C = pghi(m, hop_length=128)
        check(C, m, reference(m, 512, 128), dtype)
    assert torch.equal(pghi(mag[1:2].cuda(), hop_length=128).real, mag[1:2].cuda())


def test_large_frames_run_from_the_workspace():
    # n_fft 16384 in float64: the per-CTA working set exceeds shared memory and lives in the workspace
    mag = magnitude(1, 16384, 4096, 12, torch.float64).cuda()
    check(pghi(mag, hop_length=4096), mag, reference(mag, 16384, 4096), torch.float64)


def test_one_hour_signal():
    sr, n_fft, hop = 22050, 4096, 1024
    n = 3600 * sr
    g = torch.Generator(device="cuda").manual_seed(0)
    t = torch.arange(n, device="cuda", dtype=torch.float64) / sr
    x = torch.sin(2 * math.pi * (220 * t + 3 * torch.sin(2 * math.pi * 0.3 * t)))
    x = (x + 0.01 * torch.randn(n, generator=g, device="cuda", dtype=torch.float64)).float()
    mag = torch.stft(x, n_fft, hop, window=torch.hann_window(n_fft, device="cuda"), return_complex=True).abs()
    del x, t
    mag[0, 0] = mag.max()          # the threshold is tol * the whole signal's max: put it where the reference sees it
    C = pghi(mag, hop_length=hop)
    assert torch.isfinite(C).all()
    assert torch.allclose(C.abs(), mag, rtol=1e-6, atol=0)
    head = mag[:, :151]
    check(C[:, :150], head[:, :150], reference(head, n_fft, hop)[:, :150], torch.float32)
    assert torch.equal(pghi(mag, hop_length=hop), C)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_runs_are_bit_identical(dtype):
    mag = magnitude(3, 1024, 256, 300, dtype, seed=6).cuda()
    assert torch.equal(pghi(mag, hop_length=256), pghi(mag, hop_length=256))


def _sc_db(x, mag, n_fft, hop):
    Y = torch.stft(x, n_fft, hop, window=torch.hann_window(n_fft, device=x.device, dtype=x.dtype),
                   return_complex=True).abs()
    return float(20 * torch.log10(torch.linalg.norm(Y - mag) / torch.linalg.norm(mag)))


@pytest.mark.parametrize("n_fft,hop", [(1024, 256), (400, 100)])
def test_griffin_lim_from_pghi_ends_lower(n_fft, hop):
    mag = magnitude(4, n_fft, hop, 300, torch.float32, seed=7).cuda()
    w = torch.hann_window(n_fft, device="cuda")
    kw = dict(window=w, hop_length=hop)
    for method in ("griffin_lim", "ADMM"):
        fn = griffin_lim if method == "griffin_lim" else ADMM
        plain = _sc_db(fn(mag, max_iter=64, tol=0, verbose=False, **kw), mag, n_fft, hop)
        start = _sc_db(fn(pghi(mag, **kw), max_iter=64, tol=0, verbose=False, **kw), mag, n_fft, hop)
        assert start < plain, (method, start, plain)
