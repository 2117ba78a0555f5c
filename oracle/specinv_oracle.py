"""CPU oracle for the iterative STFT/ISTFT phase-retrieval hot path (numpy).

TEST INFRASTRUCTURE ONLY.  This module is a from-the-math restatement of what
``torch_specinv`` 0.2.1 computes on the path named in BASELINE.json
(griffin_lim / ADMM / RTISI_LA / sc, snr, ser).  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import it; the product package
(``spectrogram_inversion_b200``) never does and has no CPU fallback.

Parity pin: the reference's own test-suite holds no numeric vectors
("parity unpinned" there, SURVEY.md section 8c), so this oracle is pinned
against outputs of the unmodified reference itself, imported from
/root/reference in the build container by ``tests/golden/make_golden.py`` and
committed as ``tests/golden/*.npz``; ``tests/test_oracle_golden.py`` checks
every function below against them (fp64: <=1e-10, fp32: <=2e-5).

Unlike the reference (which hides the iteration state in closures) every
algorithm here is an explicit ``state -> state`` step so the CUDA kernels can be
compared one iteration at a time from identical state.

Reference citations are ``torch_specinv/<file>:<lines>`` of the upstream tree.
The FFT / padding arithmetic lives upstream in PyTorch (``torch.stft``,
``torch.fft``; pin ``torch>=1.6.0``, upstream setup.py:18); its published
definition is restated here with ``numpy.fft`` (pocketfft).
"""
from __future__ import annotations

import math
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field
from typing import Callable, Dict, Optional, Tuple

import numpy as np

EPS = 1e-16  # magnitude-projection epsilon, methods.py:246, :394, :472

_PAD_NP = {"reflect": "reflect", "constant": "constant",
           "replicate": "edge", "circular": "wrap"}


# --------------------------------------------------------------------------- #
# kwargs normalisation  (methods.py:21-91)
# --------------------------------------------------------------------------- #
@dataclass
class StftArgs:
    """Normalised STFT arguments; ``window`` is already zero-padded to n_fft."""
    n_fft: int
    hop_length: int
    win_length: int
    window: np.ndarray
    center: bool = True
    pad_mode: str = "reflect"
    normalized: bool = False
    onesided: bool = True

    @property
    def n_bins(self) -> int:
        return self.n_fft // 2 + 1 if self.onesided else self.n_fft

    @property
    def pad(self) -> int:
        return self.n_fft // 2 if self.center else 0

    def signal_length(self, n_frames: int) -> int:
        # conv_transpose1d output-size rule, methods.py:127-128,148
        return (n_frames - 1) * self.hop_length + self.n_fft - 2 * self.pad


def real_dtype(dtype) -> np.dtype:
    dtype = np.dtype(dtype)
    if dtype == np.complex64:
        return np.dtype(np.float32)
    if dtype == np.complex128:
        return np.dtype(np.float64)
    return dtype


def args_helper(n_bins: int, dtype, **stft_kwargs) -> StftArgs:
    """methods.py:21-91: defaults :34-41, onesided rule :59-63, n_fft inference
    :65-68, win/hop defaults :70-77, centred zero-padding of the window :79-83.
    Unknown keys are ignored (:42-46)."""
    win_length = stft_kwargs.get("win_length", None)
    window = stft_kwargs.get("window", None)
    hop_length = stft_kwargs.get("hop_length", None)
    center = stft_kwargs.get("center", True)
    pad_mode = stft_kwargs.get("pad_mode", "reflect")
    normalized = stft_kwargs.get("normalized", False)
    onesided = stft_kwargs.get("onesided", None)
    rdt = real_dtype(dtype)

    if window is not None:
        window = np.asarray(window)
    if onesided is None:
        onesided = not (window is not None and np.iscomplexobj(window))
    n_fft = (n_bins - 1) * 2 if onesided else n_bins
    if not win_length:
        win_length = n_fft
    if not hop_length:
        hop_length = n_fft // 4
    if window is None:
        window = np.ones(win_length, dtype=rdt)
    assert n_fft >= win_length
    if n_fft > win_length:
        left = (n_fft - win_length) // 2
        right = (n_fft - win_length + 1) // 2
        window = np.pad(window, (left, right))
        win_length = n_fft
    return StftArgs(n_fft=n_fft, hop_length=int(hop_length), win_length=int(win_length),
                    window=window, center=bool(center), pad_mode=pad_mode,
                    normalized=bool(normalized), onesided=bool(onesided))


# --------------------------------------------------------------------------- #
# STFT / ISTFT / OLA primitives
# --------------------------------------------------------------------------- #
def n_frames_of(length: int, a: StftArgs) -> int:
    return 1 + (length + 2 * a.pad - a.n_fft) // a.hop_length


def frame_signal(x: np.ndarray, a: StftArgs) -> np.ndarray:
    """(B, L) -> (B, T, n_fft) un-windowed frames of the (optionally padded) signal."""
    if a.center:
        x = np.pad(x, ((0, 0), (a.pad, a.pad)), mode=_PAD_NP[a.pad_mode])
    T = 1 + (x.shape[1] - a.n_fft) // a.hop_length
    idx = (np.arange(T) * a.hop_length)[:, None] + np.arange(a.n_fft)[None, :]
    return x[:, idx]


def stft(x: np.ndarray, a: StftArgs) -> np.ndarray:
    """torch.stft as called at methods.py:241, :464, :385 -> (B, F, T) complex.

    pad n_fft//2 both sides with pad_mode when center; frame t = padded samples
    [t*hop, t*hop+n_fft) * window; DFT X[k] = sum_n fr[n] exp(-2 pi i k n / N);
    * N^-1/2 when normalized; keep k <= N/2 when onesided."""
    fr = frame_signal(x, a) * a.window.astype(x.dtype, copy=False)
    spec = np.fft.rfft(fr, axis=-1) if a.onesided else np.fft.fft(fr, axis=-1)
    if a.normalized:
        spec = spec * x.dtype.type(a.n_fft ** -0.5)
    return np.swapaxes(spec, 1, 2)


def ola(frames: np.ndarray, hop: int, weight: np.ndarray, padding: int) -> np.ndarray:
    """methods.py:127-128 without the normalisation: y[b, m] = sum_t
    weight[m+P-t*hop] * frames[b, t, m+P-t*hop];  frames is (B, T, n)."""
    B, T, n = frames.shape
    fw = frames * weight.astype(frames.dtype, copy=False)
    nblk = (n + hop - 1) // hop
    buf = np.zeros((B, T + nblk, hop), dtype=frames.dtype)
    for r in range(nblk):
        seg = fw[:, :, r * hop:(r + 1) * hop]
        buf[:, r:r + T, :seg.shape[2]] += seg
    y = buf.reshape(B, -1)[:, :(T - 1) * hop + n]
    return y[:, padding:y.shape[1] - padding] if padding else y


def ola_envelope(T: int, a: StftArgs, padding: Optional[int] = None, dtype=np.float64) -> np.ndarray:
    """methods.py:129-131: env[m] = sum_t window^2[m+P-t*hop]  (no epsilon)."""
    padding = a.pad if padding is None else padding
    ones = np.ones((1, T, a.n_fft), dtype=dtype)
    w = a.window.astype(dtype, copy=False)
    return ola(ones, a.hop_length, w * w, padding)[0]


def inverse_frames(spec: np.ndarray, a: StftArgs) -> np.ndarray:
    """methods.py:141-146: (B, F, T) complex -> (B, T, n_fft) real time frames.
    irfft ignores Im(DC) and Im(Nyquist); two-sided takes ifft(...).real."""
    s = np.swapaxes(spec, 1, 2)
    norm = "ortho" if a.normalized else "backward"
    if a.onesided:
        return np.fft.irfft(s, n=a.n_fft, axis=-1, norm=norm)
    return np.fft.ifft(s, n=a.n_fft, axis=-1, norm=norm).real


def istft(spec: np.ndarray, a: StftArgs, env: Optional[np.ndarray] = None
          ) -> Tuple[np.ndarray, np.ndarray]:
    """methods.py:135-150: inverse FFT per frame, windowed OLA, divide by env."""
    fr = inverse_frames(spec, a)
    if env is None:
        env = ola_envelope(fr.shape[1], a, dtype=fr.dtype)
    with np.errstate(divide="ignore", invalid="ignore"):
        x = ola(fr, a.hop_length, a.window, a.pad) / env
    return x, env


def project(q: np.ndarray, mag: np.ndarray) -> np.ndarray:
    """methods.py:246-247 / :394-396 / :472-473: q * mag / (|q| + 1e-16)."""
    rdt = real_dtype(q.dtype)
    return q * mag / (np.abs(q) + rdt.type(EPS))


# --------------------------------------------------------------------------- #
# metrics (metrics.py:4-43) and the two sums the fused epilogue produces
# --------------------------------------------------------------------------- #
def metric_sums(est_mag: np.ndarray, mag: np.ndarray) -> Tuple[float, float, float]:
    """d = sum (|s|-m)^2, e = sum |s|^2, g = sum m^2, accumulated in fp64."""
    est = est_mag.astype(np.float64)
    m = mag.astype(np.float64)
    return float(((est - m) ** 2).sum()), float((est ** 2).sum()), float((m ** 2).sum())


def sc(inp, target) -> float:
    """metrics.py:14: 20*(log10||in-tg|| - log10||tg||) in dB."""
    d, _, g = metric_sums(inp, target)
    return 20.0 * (math.log10(math.sqrt(d)) - math.log10(math.sqrt(g)))


def snr(inp, target) -> float:
    """metrics.py:28-29: -10*log10(sum((in-tg)/||tg||)^2)."""
    d, _, g = metric_sums(inp, target)
    return -10.0 * math.log10(d / g)


def ser(inp, target) -> float:
    """metrics.py:43: 10*(log10 sum in^2 - log10 sum (in-tg)^2)."""
    d, e, _ = metric_sums(inp, target)
    return 10.0 * (math.log10(e) - math.log10(d))


def mse(inp, target) -> float:
    d, _, _ = metric_sums(inp, target)
    return d / inp.size


METRICS: Dict[str, Callable] = {"SC": sc, "SNR": snr, "SER": ser}  # methods.py:14-18


def metric_from_sums(name: str, d: float, e: float, g: float) -> float:
    name = name.upper()
    if name == "SC":
        return 10.0 * math.log10(d / g) if d > 0 else -math.inf
    if name == "SNR":
        return -10.0 * math.log10(d / g) if d > 0 else math.inf
    if name == "SER":
        return 10.0 * (math.log10(e) - math.log10(d)) if d > 0 else math.inf
    raise AssertionError(name)


# --------------------------------------------------------------------------- #
# one-shot phase initialiser (methods.py:572-615)
# --------------------------------------------------------------------------- #
def phase_init_phase(mag: np.ndarray, bins: Optional[Tuple[int, int]] = None, **stft_kwargs
                     ) -> Tuple[np.ndarray, np.ndarray]:
    """The running phase of ``phase_init`` for a (B, F, T) or (F, T) magnitude: ``(phase, phase_f64)``,
    the reference's phase rounded to the magnitude's real dtype and the float64 running sum it was
    rounded from.

    ``bins=(k0, k1)`` computes bins [k0, k1) only, shape (B, k1-k0, T): a bin's frequency comes from
    peaks at k-1 .. k+1, which look at magnitudes k-2 .. k+2, so only bins [k0-2, k1+2) are read and
    k stays absolute in omega.  The result equals the same bins of the whole-spectrum call."""
    m = mag[None] if mag.ndim == 2 else mag
    a = args_helper(m.shape[-2], m.dtype, **stft_kwargs)
    rdt = m.dtype
    F = m.shape[1]
    k0, k1 = (0, F) if bins is None else (int(bins[0]), int(bins[1]))
    assert 0 <= k0 < k1 <= F, (k0, k1, F)
    lo, hi = max(k0 - 2, 0), min(k1 + 2, F)
    m = m[:, lo:hi]
    phase = np.zeros(m.shape, dtype=rdt)
    # strict local maxima of the window's interior: absolute bins lo+1 .. hi-2, inside 1 .. F-2 (:597-598)
    mask = np.zeros(m.shape, dtype=bool)
    mask[:, 1:-1] = (m[:, 1:-1] > m[:, 2:]) & (m[:, 1:-1] > m[:, :-2])
    i1, i2, i3 = np.nonzero(mask)
    b = m[i1, i2, i3]
    av = m[i1, i2 - 1, i3]
    r = m[i1, i2 + 1, i3]
    p = rdt.type(0.5) * (av - r) / (av - rdt.type(2) * b + r)
    # methods.py:605: idx2.float() + p promotes to the dtype of p (= spec dtype)
    k = (i2 + lo).astype(rdt)
    omega = rdt.type(2 * math.pi) * (k + p) / rdt.type(a.n_fft) * rdt.type(a.hop_length)
    phase[i1, i2, i3] = omega
    phase[i1, i2 - 1, i3] = omega
    phase[i1, i2 + 1, i3] = omega
    # torch's CPU cumsum accumulates float32 inputs in float64 (acc_type) and rounds every output
    phase_f64 = np.cumsum(phase[:, k0 - lo:k1 - lo].astype(np.float64), axis=2)
    return phase_f64.astype(rdt), phase_f64


def phase_init(mag: np.ndarray, **stft_kwargs) -> np.ndarray:
    """Simplified SPSI: strict local maxima along freq for 1<=k<=F-2 (:597-598),
    parabolic offset p (:604), omega = 2 pi (k+p)/n_fft*hop (:605), written to bins
    k, k-1, k+1 in that order so later writes win (:607-609), cumulative sum over
    time (:611), C = mag * exp(i phi) (:612-614)."""
    shape = mag.shape
    m = mag[None] if mag.ndim == 2 else mag
    phase, _ = phase_init_phase(m, **stft_kwargs)
    cdt = np.result_type(m.dtype, np.complex64)
    out = m * np.exp(phase.astype(cdt) * cdt.type(1j))
    return out.reshape(shape)


# --------------------------------------------------------------------------- #
# Griffin-Lim / fast Griffin-Lim  (methods.py:193-270)
# --------------------------------------------------------------------------- #
@dataclass
class GLState:
    x: np.ndarray          # (B, L) current signal estimate
    q: np.ndarray          # (B, F, T) previous momentum-modified spectrum ("pre_spec")
    env: np.ndarray        # (L,) window^2 overlap-add envelope
    out_mag: Optional[np.ndarray] = None  # |STFT(x)| seen by the last step (metric input)


def gl_init(C: np.ndarray, a: StftArgs) -> GLState:
    """methods.py:232-233: q_0 = C, x_0 = ISTFT(C)."""
    x, env = istft(C, a)
    return GLState(x=x, q=C.copy(), env=env)


def gl_step(st: GLState, mag: np.ndarray, lr: float, a: StftArgs) -> GLState:
    """One closure call, methods.py:237-250:  s = STFT(x); out = |s|;
    q = s - lr*q_prev; x = ISTFT(q * mag / (|q| + 1e-16))."""
    rdt = st.x.dtype
    s = stft(st.x, a)
    q = s - st.q * rdt.type(lr)
    x, _ = istft(project(q, mag), a, st.env)
    return GLState(x=x, q=q, env=st.env, out_mag=np.abs(s))


# --------------------------------------------------------------------------- #
# ADMM  (methods.py:415-506)
# --------------------------------------------------------------------------- #
@dataclass
class ADMMState:
    x: np.ndarray
    X: np.ndarray
    U: np.ndarray
    env: np.ndarray
    out_mag: Optional[np.ndarray] = None


def admm_init(C: np.ndarray, a: StftArgs) -> ADMMState:
    """methods.py:452-456: X_0 = C, U_0 = 0, x_0 = ISTFT(C)  (Y = X + U is implied)."""
    x, env = istft(C, a)
    return ADMMState(x=x, X=C.copy(), U=np.zeros_like(C), env=env)


def admm_step(st: ADMMState, mag: np.ndarray, rho: float, a: StftArgs) -> ADMMState:
    """methods.py:458-483 with Y eliminated (Y == X + U at every call)."""
    rdt = st.x.dtype
    R = stft(st.x, a)
    Z = (rdt.type(rho) * (st.X + st.U) + R) / rdt.type(1 + rho)
    U = st.U + st.X - Z
    X = project(Z - U, mag)
    x, _ = istft(X + U, a, st.env)
    return ADMMState(x=x, X=X, U=U, env=st.env, out_mag=np.abs(R))


# --------------------------------------------------------------------------- #
# host iteration driver  (methods.py:153-190)
# --------------------------------------------------------------------------- #
@dataclass
class LoopLog:
    iterations: int = 0
    evaluations: list = field(default_factory=list)  # (iter, metric, mse)


def training_loop(step: Callable[[], np.ndarray], target: np.ndarray, max_iter: int,
                  tol: float, eva_iter: int, metric: str) -> LoopLog:
    """methods.py:153-190: evaluate when i % eva_iter == eva_iter-1; the first
    evaluated MSE is init_loss; stop when (prev-cur)/init < tol and prev > cur."""
    assert eva_iter > 0
    assert max_iter > 0
    assert tol >= 0
    metric = metric.upper()
    assert metric in METRICS
    log = LoopLog()
    init_loss = None
    previous = None
    for i in range(max_iter):
        out = step()
        log.iterations = i + 1
        if i % eva_iter == eva_iter - 1:
            m = METRICS[metric](out, target)
            l2 = mse(out, target)
            log.evaluations.append((i, m, l2))
            if not init_loss:
                init_loss = l2
            elif (previous - l2) / init_loss < tol and previous > l2:
                break
            previous = l2
    return log


def _format_spec(spec: np.ndarray, **kw) -> Tuple[np.ndarray, np.ndarray]:
    """methods.py:99-111."""
    assert 4 > spec.ndim > 1
    if spec.ndim == 2:
        spec = spec[None]
    if not np.iscomplexobj(spec):
        return phase_init(spec, **kw), spec
    return spec, np.abs(spec)


def _squeeze_like(x: np.ndarray, spec: np.ndarray) -> np.ndarray:
    """methods.py:267-270: keep the batch dim only for 3-D input."""
    return x if spec.ndim == 3 else x[0]


def griffin_lim(spec, max_iter=200, tol=1e-6, alpha=0.99, verbose=True, eva_iter=10,
                metric="sc", return_log=False, **stft_kwargs):
    assert alpha >= 0
    C, mag = _format_spec(np.asarray(spec), **stft_kwargs)
    a = args_helper(mag.shape[-2], mag.dtype, **stft_kwargs)
    st = [gl_init(C, a)]
    lr = alpha / (1 + alpha)

    def step():
        st[0] = gl_step(st[0], mag, lr, a)
        return st[0].out_mag

    log = training_loop(step, mag, max_iter, tol, eva_iter, metric)
    x = _squeeze_like(st[0].x, np.asarray(spec))
    return (x, log) if return_log else x


def ADMM(spec, max_iter=1000, tol=1e-6, rho=0.1, verbose=1, eva_iter=10, metric="sc",
         return_log=False, **stft_kwargs):
    assert eva_iter > 0 and max_iter > 0 and tol >= 0
    assert metric.upper() in METRICS
    C, mag = _format_spec(np.asarray(spec), **stft_kwargs)
    a = args_helper(mag.shape[-2], mag.dtype, **stft_kwargs)
    st = [admm_init(C, a)]

    def step():
        st[0] = admm_step(st[0], mag, rho, a)
        return st[0].out_mag

    log = training_loop(step, mag, max_iter, tol, eva_iter, metric)
    x = _squeeze_like(st[0].x, np.asarray(spec))
    return (x, log) if return_log else x


# --------------------------------------------------------------------------- #
# RTISI-LA  (methods.py:273-412)
# --------------------------------------------------------------------------- #
@dataclass
class RTISISetup:
    a: StftArgs
    look_ahead: int
    num_keep: int
    synth_coeff: float
    asym1: np.ndarray
    asym2: np.ndarray
    mag_pad: np.ndarray     # (B, F, T + 2*LA)
    steps: int
    lr: float
    asymmetric: bool
    max_iter: int


@dataclass
class RTISIState:
    buf: np.ndarray         # (B, K+LA+1, n_fft) un-windowed time frames: kept then active
    pre: Optional[np.ndarray]  # (B, F, LA+1) previous momentum-modified spectrum
    step: int = 0
    commits: list = field(default_factory=list)


def rtisi_setup(mag: np.ndarray, look_ahead=-1, asymmetric_window=False, max_iter=25,
                alpha=0.99, **stft_kwargs) -> RTISISetup:
    """methods.py:295-339."""
    assert max_iter > 0
    assert alpha >= 0
    assert not np.iscomplexobj(mag)
    assert 4 > mag.ndim > 1
    m = mag[None] if mag.ndim == 2 else mag
    a = args_helper(m.shape[-2], m.dtype, **stft_kwargs)
    rdt = m.dtype
    w = a.window.astype(rdt, copy=False)
    synth = rdt.type(a.hop_length) / (w @ w)                      # :318
    K = (a.win_length - 1) // a.hop_length                        # :322
    LA = K if look_ahead < 0 else look_ahead                      # :323-324
    wf = w[::-1]
    asym1 = np.zeros(a.win_length, dtype=rdt)                     # :326-330
    for i in range(K):
        s = (i + 1) * a.hop_length
        asym1[s:] += wf[:a.win_length - s]
    asym1 = asym1 * synth
    asym2 = np.zeros(a.win_length, dtype=rdt)                     # :332-336
    for i in range(K + 1):
        s = i * a.hop_length
        asym2[s:] += wf[:a.win_length - s]
    asym2 = asym2 * synth
    mag_pad = np.pad(m, ((0, 0), (0, 0), (LA, LA)))               # :339
    return RTISISetup(a=a, look_ahead=LA, num_keep=K, synth_coeff=float(synth), asym1=asym1,
                      asym2=asym2, mag_pad=mag_pad, steps=m.shape[2],
                      lr=alpha / (1 + alpha), asymmetric=bool(asymmetric_window),
                      max_iter=max_iter)


def _irfft_frames(S: np.ndarray, a: StftArgs) -> np.ndarray:
    norm = "ortho" if a.normalized else "backward"
    if a.onesided:
        return np.fft.irfft(S, n=a.n_fft, axis=-1, norm=norm)
    return np.fft.ifft(S, n=a.n_fft, axis=-1, norm=norm).real


def _rfft_frames(fr: np.ndarray, a: StftArgs) -> np.ndarray:
    norm = "ortho" if a.normalized else "backward"
    if a.onesided:
        return np.fft.rfft(fr, axis=-1, norm=norm)
    return np.fft.fft(fr, axis=-1, norm=norm)


def rtisi_init(su: RTISISetup) -> RTISIState:
    """methods.py:353-358: kept frames zero, active frames zero except the newest
    which is the zero-phase inverse transform of the first real magnitude frame."""
    a, LA, K = su.a, su.look_ahead, su.num_keep
    B = su.mag_pad.shape[0]
    rdt = su.mag_pad.dtype
    buf = np.zeros((B, K + LA + 1, a.n_fft), dtype=rdt)
    first = su.mag_pad[:, :, LA].astype(np.result_type(rdt, np.complex64))
    buf[:, -1] = _irfft_frames(first, a)
    return RTISIState(buf=buf, pre=None, step=0, commits=[])


def rtisi_inner(su: RTISISetup, st: RTISIState, j: int) -> RTISIState:
    """One inner iteration j of outer step st.step, methods.py:365-398.
    Spectra are handled frame-major here: (B, LA+1, F)."""
    a, LA, K = su.a, su.look_ahead, su.num_keep
    rdt = st.buf.dtype
    hop, n = a.hop_length, a.n_fft
    w = a.window.astype(rdt, copy=False)
    i = st.step
    # :365-370 overlap-add of all K+LA+1 frames with window*synth_coeff, padding 0,
    # no envelope; drop the first K*hop samples
    y = ola(st.buf, hop, w * rdt.type(su.synth_coeff), 0)[:, K * hop:]
    idx = (np.arange(LA + 1) * hop)[:, None] + np.arange(n)[None, :]
    fr = y[:, idx]                                                  # (B, LA+1, n)
    if su.asymmetric:                                               # :371-383
        win = np.broadcast_to(w, (LA + 1, n)).copy()
        win[-1] = su.asym2 if j else su.asym1
        S = _rfft_frames(fr * win, a)
    else:                                                           # :385 (torch.stft, center=False)
        S = np.fft.rfft(fr * w, axis=-1) if a.onesided else np.fft.fft(fr * w, axis=-1)
        if a.normalized:
            S = S * rdt.type(n ** -0.5)
    lr = rdt.type(su.lr)
    if j:                                                           # :387-388
        S = S - lr * st.pre
    elif i:                                                         # :389-391
        S = np.concatenate((S[:, :-1] - lr * st.pre[:, 1:], S[:, -1:]), axis=1)
    pre = S                                                         # :392
    tgt = np.swapaxes(su.mag_pad[:, :, i:i + LA + 1], 1, 2)         # :396
    S = S * tgt / (np.abs(S) + rdt.type(EPS))                       # :394-396
    buf = st.buf.copy()
    buf[:, K:] = _irfft_frames(S, a)                                # :398
    return RTISIState(buf=buf, pre=pre, step=i, commits=st.commits)


def rtisi_commit(su: RTISISetup, st: RTISIState) -> RTISIState:
    """methods.py:401-404: commit the oldest active frame, slide by one, newest = 0."""
    K = su.num_keep
    commits = st.commits + [st.buf[:, K].copy()]
    buf = np.zeros_like(st.buf)
    buf[:, :-1] = st.buf[:, 1:]
    return RTISIState(buf=buf, pre=st.pre, step=st.step + 1, commits=commits)


def rtisi_finish(su: RTISISetup, st: RTISIState) -> np.ndarray:
    """methods.py:406-408: drop the first LA commits; x = OLA(commits*w)/env, trimmed."""
    a = su.a
    frames = np.stack(st.commits[su.look_ahead:], axis=1)            # (B, T, n)
    padding = a.win_length // 2 if a.center else 0
    env = ola_envelope(frames.shape[1], a, padding=padding, dtype=frames.dtype)
    with np.errstate(divide="ignore", invalid="ignore"):
        return ola(frames, a.hop_length, a.window, padding) / env


def RTISI_LA(spec, look_ahead=-1, asymmetric_window=False, max_iter=25, alpha=0.99,
             verbose=1, **stft_kwargs):
    spec = np.asarray(spec)
    su = rtisi_setup(spec, look_ahead, asymmetric_window, max_iter, alpha, **stft_kwargs)
    st = rtisi_init(su)
    for _ in range(su.steps + su.look_ahead):                        # :363
        for j in range(max_iter):                                    # :364
            st = rtisi_inner(su, st, j)
        st = rtisi_commit(su, st)
    return _squeeze_like(rtisi_finish(su, st), spec)


# --------------------------------------------------------------------------- #
# multi-threaded batch driver used only for the CPU baseline timing in bench.py
# --------------------------------------------------------------------------- #
def run_batched(fn: Callable, spec: np.ndarray, n_threads: int, **kw) -> np.ndarray:
    """Split the batch dimension over ``n_threads`` host threads (pocketfft and the
    big numpy element-wise loops release the GIL).  Signals are independent on this
    path (SURVEY.md section 8e) so this is the same arithmetic as one call."""
    B = spec.shape[0]
    n_threads = max(1, min(n_threads, B))
    chunks = np.array_split(np.arange(B), n_threads)
    with ThreadPoolExecutor(n_threads) as ex:
        outs = list(ex.map(lambda c: fn(spec[c[0]:c[-1] + 1], **kw), chunks))
    return np.concatenate(outs, axis=0)
