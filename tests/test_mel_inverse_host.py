"""CPU checks of torchaudio_compat.InverseMelScale: the filterbank is bit for bit torchaudio's, the module has
torchaudio's signature, defaults, checks and state_dict, the float64 operator is pinv(fb.T), the "gels" rank rule agrees
with torchaudio's host lstsq, and the custom op and the C entry reject bad arguments before any launch."""
import ctypes as C
import inspect
import itertools
import warnings

import pytest
import torch

from spectrogram_inversion_b200 import _ops
from spectrogram_inversion_b200 import torchaudio_compat as TC

try:
    import torchaudio.functional as TAF
    import torchaudio.transforms as TAT
except Exception:  # pragma: no cover - torchaudio is optional
    TAF = TAT = None

needs_torchaudio = pytest.mark.skipif(TAF is None, reason="torchaudio not importable")

TACOTRON2 = dict(n_stft=513, n_mels=80, sample_rate=22050, f_max=8000.0, norm="slaney", mel_scale="slaney")
# (kwargs, torchaudio's host "gels" raises): rank-deficient filterbanks first
GELS_CASES = [
    (dict(n_stft=201, n_mels=128, sample_rate=16000), True),
    (dict(n_stft=513, n_mels=128, sample_rate=22050), True),
    (dict(n_stft=257, n_mels=80, sample_rate=16000), True),
    (TACOTRON2, False),
    (dict(n_stft=1025, n_mels=128, sample_rate=44100, norm="slaney", mel_scale="slaney"), False),
    (dict(n_stft=513, n_mels=80, sample_rate=24000, f_max=12000.0, norm="slaney", mel_scale="slaney"), False),
    (dict(n_stft=513, n_mels=80, sample_rate=22050, f_max=8000.0), False),
    (dict(n_stft=1025, n_mels=100, sample_rate=24000, f_max=12000.0, norm="slaney", mel_scale="slaney"), False),
]


def _fbanks(fn, *args):
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        fb = fn(*args)
    return fb, [str(x.message) for x in w]


@needs_torchaudio
@pytest.mark.parametrize("n_freqs", [65, 201, 257, 513, 1025])
@pytest.mark.parametrize("n_mels", [1, 20, 80, 128, 256])
def test_filterbank_is_torchaudio_bit_for_bit(n_freqs, n_mels):
    grid = itertools.product(["htk", "slaney"], [None, "slaney"], [0.0, 50.0], [None, 8000.0],
                             [8000, 16000, 22050, 44100, 48000])
    for mel_scale, norm, f_min, f_max, sr in grid:
        f_max = f_max or float(sr // 2)
        args = (n_freqs, f_min, f_max, n_mels, sr, norm, mel_scale)
        ours, w_ours = _fbanks(TC._melscale_fbanks, *args)
        ref, w_ref = _fbanks(TAF.melscale_fbanks, *args)
        assert ours.dtype == ref.dtype and torch.equal(ours, ref), args
        assert w_ours == w_ref, args


@needs_torchaudio
def test_signature_and_defaults_match_torchaudio():
    params = lambda cls: [(p.name, p.kind, p.default) for p in inspect.signature(cls.__init__).parameters.values()]
    assert params(TC.InverseMelScale) == params(TAT.InverseMelScale)
    ours, ref = TC.InverseMelScale(201), TAT.InverseMelScale(201)
    for name in ("n_stft", "n_mels", "sample_rate", "f_min", "f_max", "norm", "mel_scale", "driver"):
        assert getattr(ours, name) == getattr(ref, name), name
    assert TC.InverseMelScale(201, f_max=0).f_max == 8000.0       # f_max or sample_rate // 2


@needs_torchaudio
@pytest.mark.parametrize("kwargs", [dict(f_min=9000.0), dict(f_min=100.0, f_max=50.0), dict(driver="gesv"),
                                    dict(norm="area"), dict(mel_scale="mel")])
def test_constructor_errors_match_torchaudio(kwargs):
    with pytest.raises(ValueError) as ref:
        TAT.InverseMelScale(201, **kwargs)
    with pytest.raises(ValueError) as ours:
        TC.InverseMelScale(201, **kwargs)
    assert str(ours.value) == str(ref.value)


@needs_torchaudio
def test_state_dict_round_trips_with_torchaudio():
    ours, ref = TC.InverseMelScale(**TACOTRON2), TAT.InverseMelScale(**TACOTRON2)
    assert list(ours.state_dict()) == ["fb"] and torch.equal(ours.fb, ref.fb)
    ours.operator()                                               # the cached operator is not part of the state
    assert list(ours.state_dict()) == ["fb"]
    scaled = {"fb": ref.fb * 2}
    ours.load_state_dict(scaled)
    assert torch.equal(ours.fb, scaled["fb"])
    ref.load_state_dict(TC.InverseMelScale(**TACOTRON2).state_dict())
    assert torch.equal(ref.fb, ours.fb / 2)


def test_wrong_mel_count_dtype_grad_and_device_raise_before_any_launch():
    m = TC.InverseMelScale(**TACOTRON2)
    with pytest.raises(ValueError, match="Expected an input with 80 mel bins. Found: 81"):
        m(torch.rand(2, 81, 5))
    with pytest.raises(RuntimeError, match="same dtype"):
        m(torch.rand(2, 80, 5, dtype=torch.float64))
    with pytest.raises(NotImplementedError):
        m(torch.rand(2, 80, 5, requires_grad=True))
    with pytest.raises(RuntimeError):
        m(torch.rand(80))


@pytest.mark.parametrize("kwargs", [TACOTRON2, dict(n_stft=201, n_mels=128, sample_rate=16000),
                                    dict(n_stft=257, n_mels=80, sample_rate=16000),
                                    dict(n_stft=4097, n_mels=256, sample_rate=48000, f_max=20000.0)])
def test_operator_is_pinv_of_fb_transposed(kwargs):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = TC.InverseMelScale(**kwargs, driver="gelsd")
    P, f_lo, f_hi = m.operator()
    ref = torch.linalg.pinv(m.fb.T.double())
    assert P.dtype == torch.float32 and P.shape == ref.shape
    assert float((P.double() - ref).abs().max()) <= 1e-6 * float(ref.abs().max())     # rounded to fb's dtype
    m.double()
    P64, lo64, hi64 = m.operator()
    assert P64.dtype == torch.float64 and (lo64, hi64) == (f_lo, f_hi)
    assert float((P64 - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    covered = m.fb.ne(0).any(dim=1)
    assert covered[f_lo:f_hi].all() and not covered[:f_lo].any() and not covered[f_hi:].any()
    assert not P64[:f_lo].any() and not P64[f_hi:].any()


def test_operator_cache_follows_fb():
    m = TC.InverseMelScale(**TACOTRON2)
    P1 = m.operator()[0]
    assert m.operator()[0] is P1                                  # cached
    with torch.no_grad():
        m.fb.mul_(2)                                              # in place: the version changes
    P2 = m.operator()[0]
    assert P2 is not P1 and torch.allclose(P2 * 2, P1)
    assert m.double().operator()[0].dtype == torch.float64


@needs_torchaudio
@pytest.mark.parametrize("kwargs,raises", GELS_CASES)
def test_gels_rank_rule_agrees_with_torchaudio_host(kwargs, raises):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref, ours = TAT.InverseMelScale(**kwargs), TC.InverseMelScale(**kwargs)
    mel = torch.rand(1, kwargs["n_mels"], 4)
    try:
        ref(mel)
        ref_raised = False
    except torch.linalg.LinAlgError:
        ref_raised = True
    assert ref_raised == raises
    if raises:
        with pytest.raises(torch.linalg.LinAlgError, match="^torch.linalg.lstsq: The least squares solution could not "
                                                           "be computed because the input matrix does not have full rank"):
            ours.operator()
        for driver in ("gelsy", "gelsd", "gelss"):                # the minimum-norm solution, no error
            ours.driver = driver
            ours.operator()
    else:
        ours.operator()


def test_mel_op_fake_kernel_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    assert _ops.mel_inverse not in _ops.ALL_OPS and _ops.mel_inverse in _ops.MEL_OPS
    with FakeTensorMode():
        f = lambda *shape, dt=torch.float32: torch.empty(*shape, dtype=dt, device="cuda")
        assert _ops.mel_inverse(f(513, 80), f(3, 80, 7), f(3, 513, 7), 1, 373) is None
        bad = [(f(513, 80), f(3, 81, 7), f(3, 513, 7), 1, 373),          # n_mels disagree
               (f(513, 80), f(3, 80, 7), f(3, 512, 7), 1, 373),          # n_stft disagree
               (f(513, 80), f(3, 80, 7), f(2, 513, 7), 1, 373),          # batch disagree
               (f(513, 80), f(3, 80, 7), f(3, 513, 8), 1, 373),          # frames disagree
               (f(513, 80), f(3, 80, 7, dt=torch.float64), f(3, 513, 7), 1, 373),
               (f(513, 80), f(3, 80, 7), f(3, 513, 7), 5, 4),            # f_lo > f_hi
               (f(513, 80), f(3, 80, 7), f(3, 513, 7), 0, 514)]          # f_hi > n_stft
        for args in bad:
            with pytest.raises(RuntimeError):
                _ops.mel_inverse(*args)


@pytest.fixture(scope="module")
def lib():
    from spectrogram_inversion_b200.build import build_library
    build_library()
    from spectrogram_inversion_b200 import _lib
    return _lib


def _call(lib, **over):
    p = dict(dtype=lib.F32, n_stft=513, n_mels=80, f_lo=1, f_hi=373, B=3, T=7)
    p.update(over)
    ptr = lambda name: None if over.get(name, 1) is None else C.c_void_p(0x1000)
    return lib.lib().specinv_mel_inverse(p["dtype"], ptr("P"), p["n_stft"], p["n_mels"], p["f_lo"], p["f_hi"],
                                         ptr("mel"), ptr("out"), p["B"], p["T"], None)


@pytest.mark.parametrize("over", [dict(dtype=2), dict(dtype=-1), dict(n_stft=0), dict(n_mels=0), dict(B=0),
                                  dict(T=-1), dict(f_lo=-1), dict(f_lo=10, f_hi=9), dict(f_hi=514), dict(P=None),
                                  dict(mel=None), dict(out=None)])
def test_c_entry_rejects_bad_arguments_before_any_launch(lib, over):
    assert _call(lib, **over) == -1


def test_c_entry_launches_nothing_for_no_frames_or_reads_nothing_without_covered_rows(lib):
    assert _call(lib, T=0, P=None, mel=None, out=None) == 0
    # no covered row: P and mel may be NULL, but the zeros still need `out` (not launched here: out=None is invalid)
    assert _call(lib, f_lo=0, f_hi=0, P=None, mel=None, out=None) == -1
