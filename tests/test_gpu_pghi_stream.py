"""PGHIStream on the GPU (pghi_stream_kernel of csrc/specinv_pghi.cu) against the stream reference
(tests/golden/pghi_stream_ref.py, the scan formulation with the causal threshold), within pghi's bounds per bin:
4e-7 * mag in float32, 1e-9 * mag in float64 (tests/test_gpu_pghi.py).  The waveform output is checked against
torch.istft of the concatenated spectrum output."""
import math

import numpy as np
import pytest
import torch

import pghi_stream_ref as S
from spectrogram_inversion_b200 import PGHIStream, pghi
from spectrogram_inversion_b200.streaming import pghi_emitted_samples
from tests.test_gpu_pghi import TOL, magnitude

pytestmark = pytest.mark.gpu


def stream_ref(mag, n_fft, hop, win_length=None, tol=1e-5):
    m = mag.detach().cpu().numpy()
    ph = S.pghi_stream_phase(m.reshape(-1, *m.shape[-2:]), n_fft, hop, win_length, None, tol).reshape(m.shape)
    return m.astype(np.float64) * np.exp(1j * ph)


def check(C, mag, ref, dtype):
    assert C.shape == mag.shape and C.dtype == (torch.complex64 if dtype == torch.float32 else torch.complex128)
    c = C.detach().cpu().numpy().astype(np.complex128)
    m = mag.detach().cpu().numpy().astype(np.float64)
    err = np.abs(c - ref)
    bad = err > TOL[dtype] * m
    assert not bad.any(), f"{bad.sum()} bins off, worst {np.max(err / np.maximum(m, 1e-300)):.3e} x mag"


def chunkings(T, seed):
    rs = np.random.RandomState(seed)
    rand, left = [], T
    while left > 0:
        k = int(min(left, rs.choice([0, 0, 1, 2, 3, 5, 8, 13])))
        rand.append(k)
        left -= k
    return {"whole": [T], "one": [1] * T, "random": rand}


def run(mag, sizes, output="spectrum", **kw):
    """Push mag (…, F, T) in chunks of `sizes` frames; return the pieces (pushes, then flush)."""
    st = PGHIStream(output=output, **kw)
    pieces, t = [], 0
    for k in sizes:
        pieces.append(st.push(mag[..., t:t + k]))
        t += k
    pieces.append(st.flush())
    return pieces


def fade_in(mag):
    """A level that rises over the first third of the frames: the running max moves for many frames."""
    T = mag.shape[-1]
    ramp = torch.clamp(torch.arange(T, dtype=torch.float64) / max(1, T // 3), max=1.0) ** 2 + 1e-3
    return (mag.double() * ramp.to(mag.device)).to(mag.dtype).contiguous()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n_fft,hop,B,T", [(400, 100, 3, 40), (401, 100, 1, 30), (512, 128, 64, 12),
                                           (1024, 256, 1, 50), (2048, 512, 3, 20), (16384, 4096, 1, 8)])
def test_spectrum_against_reference_in_every_chunking(n_fft, hop, B, T, dtype):
    mag = fade_in(magnitude(B, n_fft, hop, T, dtype, seed=n_fft)).cuda()
    T = mag.shape[-1]                         # an odd n_fft gives one frame less
    kw = dict(hop_length=hop, n_fft=n_fft)
    ref = stream_ref(mag, n_fft, hop)
    outs = []
    for name, sizes in chunkings(T, seed=T).items():
        pieces = run(mag, sizes, **kw)
        assert [p.shape[-1] for p in pieces[:-1]] == [max(0, sum(sizes[:i + 1]) - 1) - max(0, sum(sizes[:i]) - 1)
                                                      for i in range(len(sizes))], name
        assert pieces[-1].shape[-1] == 1
        C = torch.cat(pieces, -1)
        check(C, mag, ref, dtype)
        outs.append(C)
    outs.append(torch.cat(run(mag, chunkings(T, seed=T)["random"], **kw), -1))      # a repeat
    for C in outs[1:]:
        assert torch.equal(C, outs[0])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_equals_offline_pghi_when_the_maximum_is_in_frame_0(dtype):
    mag = magnitude(3, 1024, 256, 60, dtype, seed=2)
    mag[:, 40, 0] = 2 * mag.max()
    mag = mag.cuda()
    C = torch.cat(run(mag, [7, 1, 0, 20, 32], hop_length=256), -1)
    off = pghi(mag, hop_length=256)
    err = (C.to(torch.complex128) - off.to(torch.complex128)).abs()
    assert bool((err <= 2 * TOL[dtype] * mag.double()).all())


def _istft_ref(C, n_fft, hop, window, center, normalized, length):
    return torch.istft(C, n_fft, hop, window=window, center=center, normalized=normalized, length=length)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("case", ["centred", "uncentred", "normalized", "short_window", "hop_one_third"])
def test_waveform_against_istft_of_the_spectrum(case, dtype):
    n_fft, hop, wl, center, normalized = 512, 128, 512, True, False
    if case == "uncentred":
        center = False
    elif case == "normalized":
        normalized = True
    elif case == "short_window":
        wl = 400
    elif case == "hop_one_third":
        n_fft, hop, wl = 480, 160, 480
    B, T = 2, 37
    w = torch.hamming_window(wl, dtype=dtype)     # no zero at the ends: the un-centred envelope never vanishes
    mag = fade_in(magnitude(B, n_fft, hop, T, dtype, win_length=wl, center=center, seed=5)).cuda()
    kw = dict(hop_length=hop, win_length=wl, window=w.cuda(), center=center, normalized=normalized)
    spec = torch.cat(run(mag, chunkings(T, 3)["random"], **kw), -1)
    ref = _istft_ref(spec, n_fft, hop, torch.nn.functional.pad(w, [(n_fft - wl) // 2, (n_fft - wl + 1) // 2]).cuda(),
                     center, normalized, None)
    for name, sizes in chunkings(T, seed=4).items():
        st = PGHIStream(**kw)
        pieces, t = [], 0
        for k in sizes:
            pieces.append(st.push(mag[..., t:t + k]))
            t += k
            assert sum(p.shape[-1] for p in pieces) == pghi_emitted_samples(t, n_fft, hop, center), (name, t)
        pieces.append(st.flush())
        x = torch.cat(pieces, -1)
        assert x.shape == ref.shape, (name, x.shape, ref.shape)
        tol = (1e-5 if dtype == torch.float32 else 1e-12) * float(ref.abs().max())
        assert float((x - ref).abs().max()) <= tol, (name, float((x - ref).abs().max()), tol)


def test_waveform_at_n_fft_32768():
    n_fft, hop, T = 32768, 8192, 9
    mag = magnitude(1, n_fft, hop, T, torch.float32, seed=8).cuda()
    w = torch.hann_window(n_fft, device="cuda")
    spec = torch.cat(run(mag, [2, 3, 4], hop_length=hop, window=w), -1)
    ref = torch.istft(spec, n_fft, hop, window=w)
    x = torch.cat(run(mag, [2, 3, 4], output="waveform", hop_length=hop, window=w), -1)
    assert x.shape == ref.shape
    assert float((x - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


@pytest.mark.parametrize("center", [True, False])
def test_short_streams_silence_and_host_input(center):
    n_fft, hop = 512, 128
    w = torch.hamming_window(n_fft)
    kw = dict(hop_length=hop, window=w, center=center)
    for T in (1, 2):
        mag = magnitude(2, n_fft, hop, T, torch.float32, center=False, seed=T)
        C = torch.cat(run(mag, [T], **kw), -1)
        assert C.device.type == "cpu"
        check(C, mag, stream_ref(mag, n_fft, hop), torch.float32)
        x = torch.cat(run(mag, [T], output="waveform", **kw), -1)
        assert x.device.type == "cpu" and x.shape == (2, (T - 1) * hop + n_fft - (n_fft if center else 0))
        if x.numel():
            assert torch.allclose(x, torch.istft(C, n_fft, hop, window=w, center=center), atol=1e-5 * float(x.abs().max()))
    zero = torch.zeros(257, 10)
    x = torch.cat(run(zero, [3, 3, 4], output="waveform", **kw), -1)
    assert x.shape == ((9 * hop + n_fft - (n_fft if center else 0)),) and not torch.isnan(x).any() and not x.any()
    C = torch.cat(run(zero.cuda(), [10], **kw), -1)
    assert not C.isnan().any() and not C.any()


def test_error_cases():
    st = PGHIStream(hop_length=128)
    with pytest.raises(RuntimeError):
        st.flush()
    st.push(torch.zeros(2, 257, 3, device="cuda"))
    with pytest.raises(AssertionError):
        st.push(torch.zeros(3, 257, 3, device="cuda"))
    with pytest.raises(AssertionError):
        st.push(torch.zeros(2, 257, 3, device="cuda", dtype=torch.float64))
    with pytest.raises(AssertionError):
        st.push(torch.zeros(2, 257, 3))
    with pytest.raises(NotImplementedError):
        st.push(torch.zeros(2, 257, 3, device="cuda", requires_grad=True))
    st.flush()
    with pytest.raises(RuntimeError):
        st.push(torch.zeros(2, 257, 3, device="cuda"))
    with pytest.raises(RuntimeError):
        st.flush()
    with pytest.raises(NotImplementedError):
        PGHIStream(n_fft=401, hop_length=100).push(torch.zeros(201, 3, device="cuda"))


def test_one_hour_stream_keeps_memory_bounded():
    sr, n_fft, hop = 22050, 4096, 1024
    n_frames = 3600 * sr // hop
    t = torch.arange(sr * 20, device="cuda", dtype=torch.float64) / sr
    x = torch.sin(2 * math.pi * (220 * t + 3 * torch.sin(2 * math.pi * 0.3 * t))).float()
    w = torch.hann_window(n_fft, device="cuda")
    block = torch.stft(x, n_fft, hop, window=w, return_complex=True, center=False).abs()     # 20 s of frames
    st = PGHIStream(hop_length=hop, window=w)
    chunk = 256
    pushed, emitted, peak = 0, 0, 0
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    while pushed < n_frames:
        k = min(chunk, n_frames - pushed)
        j = pushed % (block.shape[-1] - chunk)
        y = st.push(block[:, j:j + k])
        pushed += k
        emitted += y.shape[-1]
        assert emitted == pghi_emitted_samples(pushed, n_fft, hop, True)
        if pushed % (50 * chunk) == 0:
            assert bool(torch.isfinite(y).all())
        peak = max(peak, torch.cuda.memory_allocated() - base)
    emitted += st.flush().shape[-1]
    assert emitted == (n_frames - 1) * hop
    assert peak < 64 << 20, peak
