"""spectrogram_inversion_b200.torchaudio_compat on the GPU.

1. One fused iteration (specinv_gl_rebuilt_iter) from identical (x, S_prev) against the float64 restatement of
   torchaudio's loop (tests/golden/torchaudio_gl_ref.py): x_out and s_out within 1e-5 in fp32 and 1e-11 in fp64, on
   the specialised kernels and both generic families, centred and in the padded-buffer (`length`) mode.
2. Whole calls against torchaudio.functional.griffinlim on CUDA with the same seed (the restatement, which is bit for
   bit torchaudio's code, when torchaudio does not import): final spectral convergence within 1 %, equal shapes and
   dtypes, and for n_iter <= 2 the waveforms within 1e-4 of the signal's peak.
3. Leading dimensions, the module, host tensors, no state at momentum 0, requires_grad, the envelope error."""
import pytest
import torch

import torchaudio_gl_ref as R
from spectrogram_inversion_b200 import torchaudio_compat as TC
from spectrogram_inversion_b200.stft_args import StftArgs

pytestmark = pytest.mark.gpu

try:
    import torchaudio.functional as TAF
    import torchaudio.transforms as TAT
    ta_griffinlim = TAF.griffinlim
except Exception:  # pragma: no cover - the restatement is bit for bit torchaudio's code
    TAT = None
    ta_griffinlim = R.griffinlim

_CPLX = {torch.float32: torch.complex64, torch.float64: torch.complex128}
DEV = "cuda"

# (n_fft, hop): the specialised sizes at hop n/4, n/2, n/8, torchaudio's default 400 / 200, a size whose half is not a
# power of two (600) and one that no FFT kernel takes (half = 197, prime: the direct-DFT kernel)
SHAPES = [(512, 128), (1024, 256), (2048, 512), (4096, 1024), (1024, 512), (1024, 128), (400, 200), (400, 100),
          (600, 150), (394, 98)]
FAMILIES = {"default": {}, "generic-mr": {"SPECINV_FORCE_GENERIC": "1"},
            "generic-legacy": {"SPECINV_FORCE_GENERIC": "1", "SPECINV_GENERIC_MR": "0"}}


def _mag(n_fft, hop, B, T, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    F = n_fft // 2 + 1
    m = torch.randn(B, F, T, dtype=torch.float64, device=DEV, generator=g).abs()
    return (m * (0.5 + torch.rand(B, 1, T, dtype=torch.float64, device=DEV, generator=g))).to(dtype)


def _signal_from(mag, window, n_fft, hop, length, seed):
    """A signal of the spectrogram's scale: ISTFT of mag with random phases."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    ph = torch.rand(mag.shape, dtype=torch.float64, device=DEV, generator=g) * (2 * torch.pi)
    return R.istft(mag.to(torch.float64) * torch.exp(1j * ph), window, n_fft, hop, n_fft, length)


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("mode", ["centred", "length"])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("n_fft,hop", SHAPES, ids=[f"{n}-{h}" for n, h in SHAPES])
def test_one_fused_iteration_matches_float64_restatement(n_fft, hop, B, mode, dtype, family, monkeypatch):
    for k, v in FAMILIES[family].items():
        monkeypatch.setenv(k, v)
    T = 9 + (n_fft // hop)
    L0 = (T - 1) * hop
    length = None if mode == "centred" else L0 + hop // 2 + 1
    w64 = torch.hann_window(n_fft, dtype=torch.float64, device=DEV)
    mag = _mag(n_fft, hop, B, T, dtype, 1)
    x = _signal_from(mag, w64, n_fft, hop, length, 2).to(dtype)
    s_prev = R.stft(_signal_from(mag, w64, n_fft, hop, length, 3), w64, n_fft, hop, n_fft).to(_CPLX[dtype])
    m = 0.99 / 1.99
    x_ref, s_ref = R.iteration(x.to(torch.float64), s_prev.to(torch.complex128), mag.to(torch.float64), m, w64, n_fft,
                               hop, n_fft, length)

    args = StftArgs(n_fft=n_fft, hop_length=hop, win_length=n_fft, window=w64.to(dtype), center=True,
                    pad_mode="reflect", normalized=False, onesided=True)
    run = TC._Runner(args, B, T, dtype, torch.device(DEV), length)
    p = run.plan
    if length is None:
        x_in = x.contiguous()
    else:                               # the padded buffer: signal at P, padding re-created by the kernel
        x_in = torch.zeros(B, p.length, dtype=dtype, device=DEV)
        x_in[:, run.P:run.P + run.n_valid] = x[:, :run.n_valid]
        run.restore_padding(x_in)
    x_out = torch.full_like(x_in, float("nan"))
    s_out = p.empty_spec()
    run.iterate(x_in, x_out, p.pack(s_prev), s_out, p.pack(mag), m)
    y = run.output(x_out)
    s = p.unpack(s_out)
    tol = 1e-5 if dtype == torch.float32 else 1e-11
    assert y.shape == x_ref.shape
    ex = float((y.to(torch.float64) - x_ref).abs().max())
    es = float((s.to(torch.complex128) - s_ref).abs().max())
    assert ex <= tol and es <= tol, (ex, es)


def _powered_spec(n_fft, hop, B, T, power, seed, lead=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(B, (T - 1) * hop, device=DEV, generator=g)
    # a smooth-ish, consistent spectrogram: low-passed noise
    x = torch.nn.functional.avg_pool1d(x[:, None], 5, 1, 2)[:, 0]
    w = torch.hann_window(n_fft, device=DEV)
    spec = R.stft(x, w, n_fft, hop, n_fft).abs().pow(power).contiguous()
    return spec if lead is None else spec.reshape(*lead, *spec.shape[-2:])


def _both(spec, window, n_fft, hop, win_length, power, n_iter, momentum, length, rand_init, seed=11):
    torch.manual_seed(seed)
    ours = TC.griffinlim(spec, window, n_fft, hop, win_length, power, n_iter, momentum, length, rand_init)
    torch.manual_seed(seed)
    ref = ta_griffinlim(spec, window, n_fft, hop, win_length, power, n_iter, momentum, length, rand_init)
    return ours, ref


WHOLE = [(1024, 256, 4, 200), (400, 200, 4, 160)]


@pytest.mark.parametrize("length_kind", ["none", "L0", "L0+1", "L0+hop-1"])
@pytest.mark.parametrize("rand_init", [True, False])
@pytest.mark.parametrize("power", [1.0, 2.0])
@pytest.mark.parametrize("momentum", [0.0, 0.99])
@pytest.mark.parametrize("n_fft,hop,B,T", WHOLE, ids=["1024-256", "400-200"])
def test_whole_call_matches_torchaudio(n_fft, hop, B, T, momentum, power, rand_init, length_kind):
    L0 = (T - 1) * hop
    length = {"none": None, "L0": L0, "L0+1": L0 + 1, "L0+hop-1": L0 + hop - 1}[length_kind]
    spec = _powered_spec(n_fft, hop, B, T, power, 5)
    w = torch.hann_window(n_fft, device=DEV)
    ours, ref = _both(spec, w, n_fft, hop, n_fft, power, 32, momentum, length, rand_init)
    assert ours.shape == ref.shape and ours.dtype == ref.dtype and ours.device == ref.device
    mag = spec.pow(1 / power)
    sc_o = R.spectral_convergence(ours, mag, w, n_fft, hop, n_fft)
    sc_r = R.spectral_convergence(ref, mag, w, n_fft, hop, n_fft)
    assert abs(sc_o / sc_r - 1) <= 0.01, (sc_o, sc_r)


@pytest.mark.parametrize("n_iter", [0, 1, 2])
@pytest.mark.parametrize("momentum", [0.0, 0.99])
@pytest.mark.parametrize("n_fft,hop,win_length,length_kind", [
    (1024, 256, 1024, "none"), (1024, 256, 800, "L0+1"), (400, 200, 400, "none"), (400, 100, 300, "L0+hop-1"),
    (256, 160, 256, "L0+hop-1"),            # hop > n_fft / 2: samples past L0 + n_fft / 2 are zeros
])
def test_short_runs_agree_sample_for_sample(n_fft, hop, win_length, length_kind, momentum, n_iter):
    B, T = 3, 40
    L0 = (T - 1) * hop
    length = None if length_kind == "none" else (L0 + 1 if length_kind == "L0+1" else L0 + hop - 1)
    spec = _powered_spec(n_fft, hop, B, T, 2.0, 6)
    w = torch.hann_window(win_length, device=DEV)
    ours, ref = _both(spec, w, n_fft, hop, win_length, 2.0, n_iter, momentum, length, True)
    assert ours.shape == ref.shape and ours.dtype == ref.dtype
    peak = float(ref.abs().max())
    err = float((ours - ref).abs().max())
    assert err <= 1e-4 * peak, (err, peak)           # max-abs within 1e-4 of the signal's peak
    if length is not None and length > L0 + n_fft // 2:
        assert torch.equal(ours[..., L0 + n_fft // 2:], torch.zeros_like(ours[..., L0 + n_fft // 2:]))


def test_fp64_whole_call_matches_restatement():
    n_fft, hop, B, T = 400, 100, 2, 60
    spec = _powered_spec(n_fft, hop, B, T, 2.0, 8).double()
    w = torch.hann_window(n_fft, dtype=torch.float64, device=DEV)
    for length in (None, (T - 1) * hop + 7):
        torch.manual_seed(2)
        ours = TC.griffinlim(spec, w, n_fft, hop, n_fft, 2.0, 8, 0.99, length, True)
        torch.manual_seed(2)
        ref = R.griffinlim(spec, w, n_fft, hop, n_fft, 2.0, 8, 0.99, length, True)
        assert ours.dtype == torch.float64 and ours.shape == ref.shape
        assert float((ours - ref).abs().max()) <= 1e-9 * float(ref.abs().max())


@pytest.mark.parametrize("lead", [(), (2, 3)])
def test_leading_dims_are_flattened_and_restored(lead):
    n_fft, hop, T = 512, 128, 30
    spec = _powered_spec(n_fft, hop, max(1, int(torch.tensor(lead).prod()) if lead else 1), T, 2.0, 9)
    spec = spec.reshape(*lead, n_fft // 2 + 1, T) if lead else spec[0]
    w = torch.hann_window(n_fft, device=DEV)
    ours, ref = _both(spec, w, n_fft, hop, n_fft, 2.0, 2, 0.99, None, True)
    assert ours.shape == ref.shape == (*lead, (T - 1) * hop)
    assert float((ours - ref).abs().max()) <= 1e-4 * float(ref.abs().max())


def test_module_matches_functional_and_moves_like_torchaudio():
    n_fft, T = 400, 50
    spec = _powered_spec(n_fft, 200, 2, T, 2.0, 10)
    mod = TC.GriffinLim(n_fft=n_fft, n_iter=4)
    assert mod.window.device.type == "cpu"
    mod = mod.to(DEV)
    assert mod.window.is_cuda
    torch.manual_seed(4)
    a = mod(spec)
    torch.manual_seed(4)
    b = TC.griffinlim(spec, mod.window, n_fft, 200, n_fft, 2.0, 4, 0.99, None, True)
    assert torch.equal(a, b)
    if TAT is not None:
        ta = TAT.GriffinLim(n_fft=n_fft, n_iter=4).to(DEV)
        torch.manual_seed(4)
        r = ta(spec)
        assert r.shape == a.shape and float((a - r).abs().max()) <= 1e-4 * float(r.abs().max())


def test_host_input_returns_host_tensor():
    n_fft, hop, T = 1024, 256, 40
    spec = _powered_spec(n_fft, hop, 2, T, 2.0, 12)
    w = torch.hann_window(n_fft)
    y_host = TC.griffinlim(spec.cpu(), w, n_fft, hop, n_fft, 2.0, 3, 0.99, None, False)
    y_dev = TC.griffinlim(spec, w.to(DEV), n_fft, hop, n_fft, 2.0, 3, 0.99, None, False)
    assert not y_host.is_cuda and y_dev.is_cuda and y_host.shape == y_dev.shape
    assert float((y_host - y_dev.cpu()).abs().max()) <= 1e-4 * float(y_dev.abs().max())
    # the same seed gives torchaudio's host draw
    torch.manual_seed(5)
    ours = TC.griffinlim(spec.cpu(), w, n_fft, hop, n_fft, 2.0, 0, 0.99, None, True)
    torch.manual_seed(5)
    ref = ta_griffinlim(spec.cpu(), w, n_fft, hop, n_fft, 2.0, 0, 0.99, None, True)
    assert not ours.is_cuda and float((ours - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def test_momentum_zero_keeps_no_state(monkeypatch):
    seen = []
    orig = TC._Runner.iterate

    def spy(self, x_in, x_out, s_in, s_out, mag, m, sums=None):
        seen.append((s_in, s_out, m))
        return orig(self, x_in, x_out, s_in, s_out, mag, m, sums)

    monkeypatch.setattr(TC._Runner, "iterate", spy)
    spec = _powered_spec(1024, 256, 2, 30, 2.0, 13)
    w = torch.hann_window(1024, device=DEV)
    TC.griffinlim(spec, w, 1024, 256, 1024, 2.0, 3, 0.0, None, True)
    assert len(seen) == 3 and all(s_in is None and s_out is None and m == 0 for s_in, s_out, m in seen)
    seen.clear()
    TC.griffinlim(spec, w, 1024, 256, 1024, 2.0, 3, 0.5, None, True)
    assert len(seen) == 3 and all(s_in is not None for s_in, _, _ in seen)


def test_requires_grad_and_envelope_errors(monkeypatch):
    spec = _powered_spec(400, 200, 1, 20, 2.0, 14)[0]
    with pytest.raises(NotImplementedError):
        TC.griffinlim(spec.clone().requires_grad_(), torch.hann_window(400, device=DEV), 400, 200, 400, 2.0, 2, 0.5,
                      None, True)
    calls = []
    monkeypatch.setattr(TC._Runner, "iterate", lambda *a, **k: calls.append(1))
    for length in (None, 19 * 200 + 3):
        with pytest.raises(RuntimeError, match="window overlap add min"):
            TC.griffinlim(spec, torch.hann_window(200, device=DEV), 400, 200, 200, 2.0, 2, 0.5, length, True)
    assert not calls
