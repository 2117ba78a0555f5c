"""torchaudio_compat.InverseMelScale on the GPU (specinv_mel_inverse).

1. Against the float64 least-squares reference relu(lstsq(fb.T, mel, driver="gelsd").solution) on the host: within
   1e-5 * max|ref| in fp32 and 1e-12 * max|ref| in fp64 wherever the kept condition number is <= 20, over frame counts
   around the kernel's 64-frame tile, batches, leading dimensions, n_mels up to 256 and n_stft up to 4097, for mels
   in the filterbank's range and arbitrary non-negative ones; bins no filter covers are exactly zero.
2. Against torchaudio's own host InverseMelScale on the full-rank configurations (fp32, 1e-5 * max|ref|).
3. Module behaviour: host tensors, .double(), a loaded state_dict, T = 0, requires_grad.
4. The Tacotron2 Griffin-Lim vocoder chain, ours against torchaudio's with the same seed."""
import math
import warnings

import pytest
import torch

import torchaudio_gl_ref as R
from spectrogram_inversion_b200 import torchaudio_compat as TC

pytestmark = pytest.mark.gpu

try:
    import torchaudio.transforms as TAT
except Exception:  # pragma: no cover - torchaudio is optional
    TAT = None

needs_torchaudio = pytest.mark.skipif(TAT is None, reason="torchaudio not importable")
DEV = "cuda"
EPS64 = torch.finfo(torch.float64).eps

TACOTRON2 = dict(n_stft=513, n_mels=80, sample_rate=22050, f_max=8000.0, norm="slaney", mel_scale="slaney")
# every configuration here has a kept condition number <= 20 (checked in _module)
CONFIGS = {
    "tacotron2": TACOTRON2,
    "defaults-201-128": dict(n_stft=201, n_mels=128, sample_rate=16000, driver="gelsd"),     # rank 107
    "1025-256-htk": dict(n_stft=1025, n_mels=256, sample_rate=48000, driver="gelsd"),       # rank 235
    "4097-256-slaney": dict(n_stft=4097, n_mels=256, sample_rate=48000, norm="slaney", mel_scale="slaney"),
    "65-1": dict(n_stft=65, n_mels=1, sample_rate=8000),
}
FULL_RANK = [TACOTRON2,
             dict(n_stft=1025, n_mels=128, sample_rate=44100, norm="slaney", mel_scale="slaney"),
             dict(n_stft=513, n_mels=80, sample_rate=24000, f_max=12000.0, norm="slaney", mel_scale="slaney"),
             dict(n_stft=513, n_mels=80, sample_rate=22050, f_max=8000.0),
             dict(n_stft=1025, n_mels=100, sample_rate=24000, f_max=12000.0, norm="slaney", mel_scale="slaney")]


def _module(kwargs, max_cond=20.0):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = TC.InverseMelScale(**kwargs)
    S = torch.linalg.svdvals(m.fb.T.double())
    kept = S[S > S.max() * max(m.fb.shape) * EPS64]
    cond = float(kept.max() / kept.min())
    assert cond <= max_cond, cond
    return m, cond


def _mel(fb, lead, T, kind, seed):
    """(*lead, n_mels, T) float64 on the host: fb.T @ a non-negative spectrogram ("range"), or arbitrary >= 0."""
    g = torch.Generator().manual_seed(seed)
    if kind == "range":
        spec = torch.rand(*lead, fb.shape[0], T, dtype=torch.float64, generator=g) ** 2
        return fb.T.double() @ spec
    return torch.rand(*lead, fb.shape[1], T, dtype=torch.float64, generator=g) * 3


def _reference(fb, mel64):
    flat = mel64.reshape(-1, *mel64.shape[-2:])
    x = torch.linalg.lstsq(fb.T.double()[None], flat, driver="gelsd").solution
    return torch.relu(x).reshape(*mel64.shape[:-2], fb.shape[0], mel64.shape[-1])


def _check(m, mel64, dtype, tol):
    ref = _reference(m.fb.cpu(), mel64)
    m = m.to(device=DEV, dtype=dtype)
    out = m(mel64.to(device=DEV, dtype=dtype))
    assert out.shape == ref.shape and out.dtype == dtype and out.is_cuda
    err = float((out.cpu().double() - ref).abs().max())
    assert err <= tol * float(ref.abs().max()), (err, float(ref.abs().max()))
    _, f_lo, f_hi = m.operator()
    assert not out[..., :f_lo, :].any() and not out[..., f_hi:, :].any()      # exactly zero where no filter reaches
    return out


@pytest.mark.parametrize("kind", ["range", "arbitrary"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_matches_float64_lstsq_over_shapes(name, dtype, kind):
    m, _ = _module(CONFIGS[name])
    tol = 1e-5 if dtype == torch.float32 else 1e-12
    big = m.fb.shape[0] > 1100
    shapes = [((1,), 1), ((3,), 7), ((1,), 63), ((3,), 64), ((1,), 65), ((2, 3), 7)] + \
             ([] if big else [((3,), 862)])
    for i, (lead, T) in enumerate(shapes):
        _check(m, _mel(m.fb.cpu(), lead, T, kind, 100 + i), dtype, tol)


def test_tacotron2_shape_at_full_batch():
    m, _ = _module(TACOTRON2)
    _check(m, _mel(m.fb, (64,), 862, "range", 7), torch.float32, 1e-5)


def test_ill_conditioned_fp64_with_gelsd():
    kwargs = dict(n_stft=257, n_mels=80, sample_rate=16000, driver="gelsd")
    m, cond = _module(kwargs, max_cond=1e7)
    for kind in ("range", "arbitrary"):
        _check(m, _mel(m.fb.cpu(), (3,), 65, kind, 3), torch.float64, 64 * EPS64 * cond)


@needs_torchaudio
@pytest.mark.parametrize("kwargs", FULL_RANK)
def test_matches_torchaudio_host_module(kwargs):
    ours = TC.InverseMelScale(**kwargs).to(DEV)
    ref_mod = TAT.InverseMelScale(**kwargs)
    for kind in ("range", "arbitrary"):
        mel = _mel(ref_mod.fb, (3,), 65, kind, 5).float()
        ref = ref_mod(mel)
        out = ours(mel.to(DEV)).cpu()
        assert out.shape == ref.shape
        assert float((out - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def test_host_input_returns_host_tensor_and_pinned_stays_pinned():
    m, _ = _module(TACOTRON2)
    mel = _mel(m.fb, (2,), 33, "range", 9).float()
    out = m(mel)
    assert out.device.type == "cpu" and not out.is_pinned()
    ref = m.to(DEV)(mel.to(DEV)).cpu()
    assert torch.equal(out, ref)
    m.cpu()
    out_p = m(mel.pin_memory())
    assert out_p.is_pinned() and torch.equal(out_p, ref)


def test_double_module_gives_fp64_accuracy():
    m, _ = _module(TACOTRON2)
    mel = _mel(m.fb, (2,), 40, "arbitrary", 4)
    ref = _reference(m.fb, mel)
    out = m.double().to(DEV)(mel.to(DEV))
    assert out.dtype == torch.float64
    assert float((out.cpu() - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


def test_loaded_state_dict_invalidates_the_cached_operator():
    m, _ = _module(TACOTRON2)
    m = m.to(DEV)
    mel = _mel(m.fb.cpu(), (2,), 20, "range", 8).float().to(DEV)
    before = m(mel)
    m.load_state_dict({"fb": m.fb * 2})
    after = m(mel)
    assert float((after * 2 - before).abs().max()) <= 1e-5 * float(before.abs().max())


def test_no_frames_and_requires_grad():
    m = TC.InverseMelScale(**TACOTRON2).to(DEV)
    out = m(torch.rand(2, 3, 80, 0, device=DEV))
    assert out.shape == (2, 3, 513, 0) and out.is_cuda
    with pytest.raises(NotImplementedError):
        m(torch.rand(2, 80, 5, device=DEV, requires_grad=True))


# ---- the Tacotron2 Griffin-Lim vocoder chain --------------------------------------------------------------------
def _log_mel(B, T, seed):
    """Log-mel of low-passed noise and tones, as Tacotron2 emits it, and the linear magnitude it came from."""
    g = torch.Generator().manual_seed(seed)
    n = torch.arange((T - 1) * 256, dtype=torch.float64) / 22050
    x = torch.randn(B, n.numel(), dtype=torch.float64, generator=g) * 0.05
    x = torch.nn.functional.avg_pool1d(x[:, None], 5, 1, 2)[:, 0]
    for f in (220.0, 440.0, 1250.0):
        x = x + 0.3 * torch.sin(2 * math.pi * f * n + torch.rand(B, 1, dtype=torch.float64, generator=g))
    w = torch.hann_window(1024, dtype=torch.float64)
    mag = R.stft(x, w, 1024, 256, 1024).abs()
    fb = TC._melscale_fbanks(513, 0.0, 8000.0, 80, 22050, "slaney", "slaney").double()
    mel = (fb.T @ mag).clamp_min(1e-5).log()
    return mel.float(), mag.float()


def _vocode(inv_mel, griffin_lim, log_mel, seed):
    """torchaudio's _GriffinLimVocoder.forward without its requires_grad_ / detach lines."""
    spec = inv_mel(torch.exp(log_mel))
    torch.manual_seed(seed)
    return griffin_lim(spec.to(DEV))


@needs_torchaudio
@pytest.mark.parametrize("n_iter", [1, 2, 32])
def test_tacotron2_vocoder_chain_matches_torchaudio(n_iter):
    log_mel, mag = _log_mel(3, 200, 21)
    gl = dict(n_fft=1024, power=1, hop_length=256, win_length=1024, n_iter=n_iter)
    ref = _vocode(TAT.InverseMelScale(**TACOTRON2), TAT.GriffinLim(**gl).to(DEV), log_mel, 5)   # host lstsq
    ours = _vocode(TC.InverseMelScale(**TACOTRON2).to(DEV), TC.GriffinLim(**gl).to(DEV), log_mel.to(DEV), 5)
    assert ours.shape == ref.shape and ours.dtype == ref.dtype
    if n_iter <= 2:
        peak = float(ref.abs().max())
        assert float((ours - ref).abs().max()) <= 1e-4 * peak
    w = torch.hann_window(1024, device=DEV)
    sc_o = R.spectral_convergence(ours, mag.to(DEV), w, 1024, 256, 1024)
    sc_r = R.spectral_convergence(ref, mag.to(DEV), w, 1024, 256, 1024)
    assert abs(sc_o / sc_r - 1) <= 0.01, (sc_o, sc_r)
