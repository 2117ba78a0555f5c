"""PGHI without a GPU: the reference's scan formulation (tests/golden/pghi_ref.py) against the heap definition, the phase-gradient constants
against the true phase of a Gaussian-window STFT, the quality of the start, and the argument checks of `pghi` and of
the C entry (made before any launch)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import pghi_ref as P
from oracle import specinv_oracle as O


def tie_free(B, F, T, seed):
    rs = np.random.RandomState(seed)
    m = rs.rand(B, F, T) ** 4 + 1e-3              # continuous: every magnitude distinct
    m[rs.rand(B, F, T) < 0.15] = 0.0              # gaps: short islands, one-bin islands among them
    return m


@pytest.mark.parametrize("B,F,T,tol", [(2, 33, 20, 1e-2), (1, 129, 12, 1e-5), (3, 9, 1, 1e-1), (1, 65, 7, 0.3)])
def test_scan_formulation_equals_heap(B, F, T, tol):
    m = tie_free(B, F, T, seed=F + T)
    if T > 4:
        m[:, :, 3] = 0.0                          # a silent frame
    m[0, ::2, 0] = 0.0                            # one-bin islands in frame 0
    n_fft, hop = (F - 1) * 2, max(1, (F - 1) // 2)
    heap = P.pghi_heap_phase(m, n_fft, hop, tol=tol)
    scan = P.pghi_phase(m, n_fft, hop, tol=tol)
    assert np.array_equal(heap, scan)
    assert np.array_equal(P.pghi(m, hop_length=hop, tol=tol), P.pghi_heap(m, hop_length=hop, tol=tol))


def test_scan_formulation_is_deterministic_under_ties():
    m = np.round(tie_free(2, 40, 15, seed=1) * 8) / 8
    a = P.pghi_phase(m, 78, 20, tol=1e-2)
    assert np.array_equal(a, P.pghi_phase(m.copy(), 78, 20, tol=1e-2))
    ch = P.pghi_choices(m[:, :, 3], m[:, :, 4], m[:, :, 3] > 0, m[:, :, 4] > 0)
    assert ((ch == P.PGHI_NONE) == (m[:, :, 4] == 0)).all()


def test_seeded_island_runs_outward_from_its_lowest_maximum():
    mcur = np.array([[0.0, 1.0, 3.0, 2.0, 3.0, 1.0, 0.0]])
    ch = P.pghi_choices(np.zeros_like(mcur), mcur, np.zeros_like(mcur, dtype=bool), mcur > 0)
    assert ch.tolist() == [[P.PGHI_NONE, P.PGHI_RIGHT, P.PGHI_ROOT, P.PGHI_LEFT, P.PGHI_LEFT, P.PGHI_LEFT,
                            P.PGHI_NONE]]


def test_gradient_constants_match_a_gaussian_stft():
    M, a = 1024, 256
    lam = 0.25645 * M ** 2
    g = torch.exp(-math.pi * (torch.arange(M, dtype=torch.float64) - M // 2) ** 2 / lam)
    sr, n = 16000, 32000
    t = torch.arange(n, dtype=torch.float64)
    x = torch.sin(2 * math.pi * (300 * t / sr + 800 * (t / sr) ** 2)) + 0.5 * torch.sin(2 * math.pi * 2000 * t / sr)
    X = torch.stft(x, M, a, window=g, return_complex=True).numpy()[None]
    mg, _, tstep, fstep = P.pghi_steps(np.abs(X), M, a, M, lam, 1e-12)
    sig = mg > 1e-1 * mg.max()                   # the bins that carry the signal (-20 dB)
    ph = np.angle(X)
    st = sig[:, :, 1:] & sig[:, :, :-1]
    st[:, :, [0, -1]] = False
    et = np.angle(np.exp(1j * (ph[:, :, 1:] - ph[:, :, :-1] - tstep[:, :, 1:])))
    sf = sig[:, 1:] & sig[:, :-1]
    sf[:, :, [0, -1]] = False
    ef = np.angle(np.exp(1j * (ph[:, 1:] - ph[:, :-1] - fstep[:, :-1])))
    assert np.median(np.abs(et[st])) < 0.1
    assert np.median(np.abs(ef[sf])) < 0.1


def _signal(kind, n, sr, seed):
    rs = np.random.RandomState(seed)
    t = np.arange(n) / sr
    if kind == "harmonic":
        f0 = 140 * (1 + 0.3 * np.sin(2 * np.pi * 0.7 * t))
        ph = 2 * np.pi * np.cumsum(f0) / sr
        x = sum((0.6 / k) * np.sin(k * ph) for k in range(1, 20)) * (0.5 + 0.5 * np.sin(2 * np.pi * 2 * t) ** 2)
    else:
        x = np.sin(2 * np.pi * (200 * t + 1500 * t ** 2)) + 0.5 * np.sin(2 * np.pi * (3000 * t - 700 * t ** 2))
    return x + 0.003 * rs.randn(n)


@pytest.mark.parametrize("n_fft,hop", [(1024, 256), (400, 100)])
@pytest.mark.parametrize("kind", ["harmonic", "chirp"])
def test_pghi_start_beats_phase_init_by_10_db(n_fft, hop, kind):
    sr = 16000
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(n_fft) / n_fft)
    a = O.args_helper(n_fft // 2 + 1, np.float64, window=w, hop_length=hop)
    x = _signal(kind, sr, sr, seed=n_fft)[None]
    mag = np.abs(O.stft(x, a))

    def sc_of_start(Cs):
        y, _ = O.istft(Cs, a)
        return O.sc(np.abs(O.stft(y, a)), mag)

    start_pghi = sc_of_start(P.pghi(mag, hop_length=hop))
    start_pi = sc_of_start(O.phase_init(mag, window=w, hop_length=hop))
    assert start_pghi < start_pi - 10, (start_pghi, start_pi)


# ---- argument handling of the public function (checked before any device work) ----------------------------------
def _pghi():
    from spectrogram_inversion_b200 import pghi
    return pghi


def test_exported_at_top_level():
    import spectrogram_inversion_b200 as S
    assert "pghi" in S.__all__ and S.pghi is _pghi()


@pytest.mark.parametrize("bad,exc", [
    (dict(spec=torch.zeros(5, 4, dtype=torch.complex64)), ValueError),
    (dict(spec=torch.zeros(5, 4, requires_grad=True)), NotImplementedError),
    (dict(spec=torch.zeros(5, 4, dtype=torch.float16)), NotImplementedError),
    (dict(spec=torch.zeros(5)), ValueError),
    (dict(spec=torch.zeros(5, 4), gamma=0.0), ValueError),
    (dict(spec=torch.zeros(5, 4), gamma=-3.0), ValueError),
    (dict(spec=torch.zeros(5, 4), tol=0.0), ValueError),
    (dict(spec=torch.zeros(5, 4), tol=1.0), ValueError),
    (dict(spec=torch.zeros(5, 4), onesided=False), NotImplementedError),
    (dict(spec=torch.zeros(5, 4), window=torch.ones(8, dtype=torch.complex64)), NotImplementedError),
    (dict(spec=torch.zeros(5, 4), n_fft=10), ValueError),
    (dict(spec=torch.zeros(5, 4), win_length=9), ValueError),
])
def test_refusals(bad, exc):
    with pytest.raises(exc):
        _pghi()(**bad)


def test_argument_parsing():
    from spectrogram_inversion_b200.pghi import _analysis
    assert _analysis(513, {}) == (1024, 256, 1024)
    assert _analysis(201, {"n_fft": 401, "hop_length": 100}) == (401, 100, 401)
    assert _analysis(201, {"n_fft": 400}) == (400, 100, 400)
    assert _analysis(513, {"win_length": 800, "hop_length": 200}) == (1024, 200, 800)
    assert _analysis(513, {"window": torch.ones(700)}) == (1024, 256, 700)
    assert P.pghi_constants(1024, 256, 1024, 0.25645 * 1024 ** 2)[0] == math.pi
    assert P.pghi_constants(1024, 256, 801, 1.0)[0] == 2 * math.pi * 511.5 / 1024


def test_c_entry_checks_arguments_before_any_launch():
    from spectrogram_inversion_b200 import _lib
    try:
        lib = _lib.lib()
    except RuntimeError:
        pytest.skip("libspecinv_b200.so is not built")
    n = C.c_size_t(0)
    inv = -1
    assert lib.specinv_pghi_workspace_bytes(0, 1, 513, 10, None) == inv
    assert lib.specinv_pghi_workspace_bytes(2, 1, 513, 10, C.byref(n)) == inv
    assert lib.specinv_pghi_workspace_bytes(0, 0, 513, 10, C.byref(n)) == inv
    assert lib.specinv_pghi_workspace_bytes(0, 1, 1, 10, C.byref(n)) == inv
    assert lib.specinv_pghi_workspace_bytes(0, 1, 513, 0, C.byref(n)) == inv
    assert lib.specinv_pghi_workspace_bytes(0, 65536, 513, 10, C.byref(n)) == inv
    p = C.c_void_p(16)
    ok = dict(dtype=0, mag=p, sb=513 * 10, sf=10, st=1, out=p, batch=1, n_bins=513, n_frames=10, n_fft=1024, hop=256,
              win_length=1024, gamma=1e5, tol=1e-5, workspace=p, workspace_bytes=1 << 20, stream=None)
    for key, val in [("mag", None), ("out", None), ("workspace", None), ("n_fft", 1000), ("hop", 0),
                     ("win_length", 1025), ("gamma", 0.0), ("gamma", float("inf")), ("tol", 0.0), ("tol", 1.0),
                     ("dtype", 5), ("n_frames", 0)]:
        args = dict(ok, **{key: val})
        assert lib.specinv_pghi(*args.values()) == inv, key
