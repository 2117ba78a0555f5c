"""CPU checks of spectrogram_inversion_b200.torchaudio_compat: the float64-capable restatement of torchaudio's loop
(tests/golden/torchaudio_gl_ref.py) is bit for bit torchaudio.functional.griffinlim, the arguments are checked before
anything is launched, and GriffinLim has torchaudio's signature, defaults and window buffer."""
import inspect

import pytest
import torch

import torchaudio_gl_ref as R
import spectrogram_inversion_b200
from spectrogram_inversion_b200 import torchaudio_compat as TC

try:
    import torchaudio.functional as TAF
    import torchaudio.transforms as TAT
except Exception:  # pragma: no cover - torchaudio is optional
    TAF = TAT = None

needs_torchaudio = pytest.mark.skipif(TAF is None, reason="torchaudio not importable")


def _spec(n_fft, hop, T, lead=(2,), dtype=torch.float32, power=2.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*lead, (T - 1) * hop, dtype=dtype, generator=g)
    w = torch.hann_window(n_fft, dtype=dtype)
    return R.stft(x.reshape(-1, x.shape[-1]), w, n_fft, hop, n_fft).abs().pow(power).reshape(*lead, n_fft // 2 + 1, T)


@needs_torchaudio
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n_fft,hop,win_length,T,lead,length", [
    (400, 200, 400, 21, (2,), None),
    (400, 100, 300, 17, (), None),
    (512, 128, 512, 12, (2, 3), 11 * 128 + 1),
    (256, 160, 256, 9, (1,), 8 * 160 + 159),        # hop > n_fft / 2: zero tail
])
@pytest.mark.parametrize("momentum,power,rand_init", [(0.99, 2.0, True), (0.0, 1.0, False), (0.5, 2.0, False)])
def test_restatement_is_torchaudio_bit_for_bit(dtype, n_fft, hop, win_length, T, lead, length, momentum, power,
                                               rand_init):
    spec = _spec(n_fft, hop, T, lead, dtype, power)
    w = torch.hann_window(win_length, dtype=dtype)
    args = (spec, w, n_fft, hop, win_length, power, 3, momentum, length, rand_init)
    torch.manual_seed(7)
    ours = R.griffinlim(*args)
    torch.manual_seed(7)
    ref = TAF.griffinlim(*args)
    assert ours.shape == ref.shape and ours.dtype == ref.dtype
    assert torch.equal(ours, ref)


def test_restated_iteration_is_one_pass_of_the_loop():
    """iteration() from (x_{k-1}, S_{k-1}) is exactly the loop's k-th pass (the GPU parity tests drive it)."""
    n_fft, hop, T = 400, 100, 13
    spec = _spec(n_fft, hop, T, (2,), torch.float64).sqrt()
    w = torch.hann_window(n_fft, dtype=torch.float64)
    torch.manual_seed(3)
    angles = R.start_angles(spec, True)
    m = 0.99 / 1.99
    x = R.istft(spec * angles, w, n_fft, hop, n_fft, None)
    s = None
    for _ in range(3):
        x, s = R.iteration(x, s if s is not None else torch.zeros((), dtype=torch.float64), spec, m, w, n_fft, hop,
                           n_fft, None)
    assert torch.equal(x, R.loop(spec, angles, w, n_fft, hop, n_fft, 3, 0.99, None))


def test_momentum_range_is_a_value_error_with_torchaudios_message():
    spec = torch.rand(201, 5)
    w = torch.hann_window(400)
    for bad in (1.0, -0.1, 1.5):
        with pytest.raises(ValueError, match=r"momentum must be in range \[0, 1\)\. Found: "):
            TC.griffinlim(spec, w, 400, 200, 400, 2.0, 4, bad, None, True)
        with pytest.raises(ValueError, match=r"momentum must be in the range \[0, 1\)\. Found: "):
            TC.GriffinLim(momentum=bad)
        if TAF is not None:
            with pytest.raises(ValueError) as ta:
                TAF.griffinlim(spec, w, 400, 200, 400, 2.0, 4, bad, None, True)
            with pytest.raises(ValueError) as ours:
                TC.griffinlim(spec, w, 400, 200, 400, 2.0, 4, bad, None, True)
            assert str(ours.value) == str(ta.value)
            with pytest.raises(ValueError) as ta:
                TAT.GriffinLim(momentum=bad)
            with pytest.raises(ValueError) as ours:
                TC.GriffinLim(momentum=bad)
            assert str(ours.value) == str(ta.value)


def test_frequency_bins_must_match_n_fft():
    w = torch.hann_window(400)
    with pytest.raises(RuntimeError, match="n_fft / 2 \\+ 1 = 201, but got 200"):
        TC.griffinlim(torch.rand(200, 9), w, 400, 200, 400, 2.0, 2, 0.5, None, True)
    if TAF is not None:     # torchaudio fails there too (inside torch.istft)
        with pytest.raises(RuntimeError):
            TAF.griffinlim(torch.rand(200, 9), w, 400, 200, 400, 2.0, 2, 0.5, None, True)


def test_window_hop_and_win_length_checks():
    spec = torch.rand(201, 9)
    with pytest.raises(RuntimeError, match="0 < hop_length <= win_length"):
        TC.griffinlim(spec, torch.hann_window(100), 400, 200, 100, 2.0, 2, 0.5, None, True)
    with pytest.raises(RuntimeError, match="0 < win_length <= n_fft"):
        TC.griffinlim(spec, torch.hann_window(500), 400, 200, 500, 2.0, 2, 0.5, None, True)
    with pytest.raises(RuntimeError, match="size equal to win_length=400"):
        TC.griffinlim(spec, torch.hann_window(300), 400, 200, 400, 2.0, 2, 0.5, None, True)


def _length_ok_in_torchaudio(spec, n_fft, hop, length, n_iter=2):
    if TAF is None:
        return None
    try:
        TAF.griffinlim(spec, torch.hann_window(n_fft), n_fft, hop, n_fft, 2.0, n_iter, 0.5, length, True)
        return True
    except RuntimeError:
        return False


@pytest.mark.parametrize("n_fft,hop,T", [(400, 200, 9), (256, 160, 6), (512, 128, 11)])
def test_valid_length_range(n_fft, hop, T):
    """With n_iter > 0 exactly the lengths with 1 + length // hop == T run in torchaudio; the others raise here before
    any launch (the accepted ones get as far as the device, which this CPU check does not need)."""
    spec = torch.rand(n_fft // 2 + 1, T)
    L0 = (T - 1) * hop
    for length in (L0 - 1, L0 + hop, L0 + 2 * hop, 1):
        with pytest.raises(RuntimeError, match=f"length={length} gives"):
            TC._check(spec.shape, None, n_fft, hop, n_fft, 2, length)
        assert _length_ok_in_torchaudio(spec, n_fft, hop, length) in (False, None)
    for length in (L0, L0 + 1, L0 + hop - 1):
        TC._check(spec.shape, None, n_fft, hop, n_fft, 2, length)
        assert _length_ok_in_torchaudio(spec, n_fft, hop, length) in (True, None)
    # without iterations torchaudio only runs torch.istft, which takes any length
    TC._check(spec.shape, None, n_fft, hop, n_fft, 0, L0 + 5 * hop)
    assert _length_ok_in_torchaudio(spec, n_fft, hop, L0 + 5 * hop, n_iter=0) in (True, None)


def test_window_envelope_case_is_an_istft_error():
    """The configuration the GPU test expects the envelope error for: a periodic Hann window of hop samples leaves the
    frame boundaries uncovered, and torch.istft (hence torchaudio) refuses it."""
    spec = torch.rand(201, 20)
    w = torch.hann_window(200)
    with pytest.raises(RuntimeError, match="window overlap add min"):
        R.griffinlim(spec, w, 400, 200, 200, 2.0, 2, 0.5, None, True)
    if TAF is not None:
        with pytest.raises(RuntimeError, match="window overlap add min"):
            TAF.griffinlim(spec, w, 400, 200, 200, 2.0, 2, 0.5, None, True)


def test_requires_grad_is_not_implemented():
    spec = torch.rand(201, 9, requires_grad=True)
    with pytest.raises(NotImplementedError):
        TC.griffinlim(spec, torch.hann_window(400), 400, 200, 400, 2.0, 2, 0.5, None, True)


def test_griffinlim_signature_matches_torchaudio():
    names = ["specgram", "window", "n_fft", "hop_length", "win_length", "power", "n_iter", "momentum", "length",
             "rand_init"]
    assert list(inspect.signature(TC.griffinlim).parameters) == names
    if TAF is not None:
        assert list(inspect.signature(TAF.griffinlim).parameters) == names


def test_module_defaults_and_buffer_match_torchaudio():
    ours = inspect.signature(TC.GriffinLim.__init__).parameters
    assert {k: p.default for k, p in ours.items() if k != "self"} == {
        "n_fft": 400, "n_iter": 32, "win_length": None, "hop_length": None, "window_fn": torch.hann_window,
        "power": 2.0, "wkwargs": None, "momentum": 0.99, "length": None, "rand_init": True}
    m = TC.GriffinLim()
    assert (m.n_fft, m.n_iter, m.win_length, m.hop_length, m.power, m.momentum, m.length, m.rand_init) == \
        (400, 32, 400, 200, 2.0, 0.99, None, True)
    assert list(m.state_dict()) == ["window"] and torch.equal(m.window, torch.hann_window(400))
    m2 = TC.GriffinLim(n_fft=512, win_length=300, window_fn=torch.hamming_window, wkwargs={"periodic": False}).double()
    assert m2.hop_length == 150 and m2.window.dtype == torch.float64
    assert torch.equal(m2.window, torch.hamming_window(300, periodic=False).double())
    if TAT is not None:
        theirs = inspect.signature(TAT.GriffinLim.__init__).parameters
        assert {k: p.default for k, p in ours.items()} == {k: p.default for k, p in theirs.items()}
        t = TAT.GriffinLim()
        for a in ("n_fft", "n_iter", "win_length", "hop_length", "power", "momentum", "length", "rand_init"):
            assert getattr(m, a) == getattr(t, a), a
        assert list(m.state_dict()) == list(t.state_dict()) and torch.equal(m.window, t.window)
        m.load_state_dict(t.state_dict())


def test_not_exported_at_top_level():
    assert not hasattr(spectrogram_inversion_b200, "griffinlim")
    assert not hasattr(spectrogram_inversion_b200, "GriffinLim")
    assert spectrogram_inversion_b200.torchaudio_compat is TC
    assert TC.__all__ == ["griffinlim", "GriffinLim"]
