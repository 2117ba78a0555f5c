"""The reference for PGHI (phase-gradient heap integration), numpy only; the tests compare
spectrogram_inversion_b200.pghi against it.

Průša, Balazs and Søndergaard, IEEE/ACM TASLP 25(5), 2017; the frame-causal heap of Průša and Holighaus, EUSIPCO
2017.  ``pghi_heap`` is the definition; ``pghi`` is the scan formulation the CUDA kernel computes, with the same
arithmetic in the same order, so the two agree bit for bit wherever the magnitudes of every pair of adjacent frames
are distinct (tests/test_pghi_host.py).  Everything is float64; only the output is cast."""
from __future__ import annotations

import heapq
import math
from typing import Optional, Tuple

import numpy as np

TWO_PI = 2 * math.pi


def pghi_wrap(x):
    """The running phase is reduced to [-pi, pi] after every addition, which changes exp(i phi) by rounding
    only and keeps its absolute error at the 1e-15 rad level over any number of frames."""
    return x - TWO_PI * np.rint(x / TWO_PI)


def pghi_constants(n_fft: int, hop: int, win_length: int, gamma: float) -> Tuple[float, float, float]:
    """(K0, K1, K2): the bin step's 2 pi c / M with c the window centre inside the frame, and the gradient
    factors a M / gamma and gamma / (M a)."""
    M, a, wl = int(n_fft), int(hop), int(win_length)
    c = (M - wl) // 2 + wl / 2
    return 2 * math.pi * c / M, a * M / gamma, gamma / (M * a)


def pghi_steps(mag: np.ndarray, n_fft: int, hop: int, win_length: int, gamma: float, tol: float):
    """Per signal of a (B, F, T) magnitude: (mag64, sig, tstep, fstep).  tstep[b, m, n] is the time step from
    frame n-1 to n (n >= 1; column 0 unused), fstep[b, m, n] the bin step from m to m+1 in frame n (m <= F-2)."""
    m64 = mag.astype(np.float64)
    B, F, T = m64.shape
    K0, K1, K2 = pghi_constants(n_fft, hop, win_length, gamma)
    thr = tol * np.maximum(m64.reshape(B, -1).max(axis=1), 0.0)[:, None, None]
    sig = m64 > thr
    with np.errstate(divide="ignore"):
        s = np.log(np.maximum(m64, thr))
    Dm = np.zeros_like(s)
    Dn = np.zeros_like(s)
    with np.errstate(invalid="ignore"):     # -inf - -inf only in silent signals, where nothing is significant
        Dm[:, 1:-1] = 0.5 * (s[:, 2:] - s[:, :-2])
        Dn[:, :, 1:-1] = 0.5 * (s[:, :, 2:] - s[:, :, :-2])
        base = TWO_PI * ((np.arange(F) * int(hop)) % int(n_fft)) / int(n_fft)
        tstep = np.zeros_like(s)
        tstep[:, :, 1:] = base[None, :, None] + K1 * (0.5 * (Dm[:, :, :-1] + Dm[:, :, 1:]))
        fstep = np.zeros_like(s)
        fstep[:, :-1] = K0 - K2 * (0.5 * (Dn[:, :-1] + Dn[:, 1:]))
    return m64, sig, tstep, fstep


def _pghi_out(mag: np.ndarray, phase: np.ndarray) -> np.ndarray:
    cdt = np.result_type(mag.dtype, np.complex64)
    return (mag.astype(np.float64) * np.exp(1j * phase)).astype(cdt)


def _pghi_gamma(win_length: int, gamma: Optional[float]) -> float:
    return 0.25645 * win_length ** 2 if gamma is None else float(gamma)


def pghi_heap_phase(mag: np.ndarray, n_fft: int, hop: int, win_length: Optional[int] = None,
                    gamma: Optional[float] = None, tol: float = 1e-5) -> np.ndarray:
    """The definition: the frame-causal heap integration, one signal after another.  (B, F, T) -> phase."""
    wl = int(win_length or n_fft)
    mg, sig, tstep, fstep = pghi_steps(mag, n_fft, hop, wl, _pghi_gamma(wl, gamma), tol)
    B, F, T = mg.shape
    ph = np.zeros((B, F, T))
    for b in range(B):
        for n in range(T):
            done = ~sig[b, :, n]
            h = [(-mg[b, m, n - 1], m, 0) for m in np.nonzero(sig[b, :, n - 1])[0]] if n else []
            heapq.heapify(h)
            while not done.all():
                if not h:
                    m = int(np.argmax(np.where(done, -1.0, mg[b, :, n])))
                    done[m] = True
                    ph[b, m, n] = pghi_wrap(ph[b, m, n - 1] + tstep[b, m, n]) if n else 0.0
                    heapq.heappush(h, (-mg[b, m, n], m, 1))
                    continue
                _, m, cur = heapq.heappop(h)
                if not cur:
                    if not done[m]:
                        done[m] = True
                        ph[b, m, n] = pghi_wrap(ph[b, m, n - 1] + tstep[b, m, n])
                        heapq.heappush(h, (-mg[b, m, n], m, 1))
                    continue
                if m + 1 < F and not done[m + 1]:
                    done[m + 1] = True
                    ph[b, m + 1, n] = pghi_wrap(ph[b, m, n] + fstep[b, m, n])
                    heapq.heappush(h, (-mg[b, m + 1, n], m + 1, 1))
                if m >= 1 and not done[m - 1]:
                    done[m - 1] = True
                    ph[b, m - 1, n] = pghi_wrap(ph[b, m, n] - fstep[b, m - 1, n])
                    heapq.heappush(h, (-mg[b, m - 1, n], m - 1, 1))
    return ph


def pghi_heap(mag: np.ndarray, n_fft: Optional[int] = None, hop_length: Optional[int] = None,
              win_length: Optional[int] = None, gamma: Optional[float] = None, tol: float = 1e-5) -> np.ndarray:
    """PGHI by its definition (the heap); (F, T) or (B, F, T) real -> complex of the same shape."""
    m = mag[None] if mag.ndim == 2 else mag
    n_fft = int(n_fft or (m.shape[1] - 1) * 2)
    ph = pghi_heap_phase(m, n_fft, int(hop_length or n_fft // 4), win_length, gamma, tol)
    return _pghi_out(m, ph).reshape(mag.shape)


# choice codes of the scan formulation
PGHI_NONE, PGHI_ROOT, PGHI_LEFT, PGHI_RIGHT = 0, 1, 2, 3


def pghi_choices(mprev: np.ndarray, mcur: np.ndarray, sig_prev: np.ndarray, sig_cur: np.ndarray) -> np.ndarray:
    """Which neighbour reaches each bin of a frame, from the magnitudes of frames n-1 and n alone; (B, F) each.

    The widest path: S is the time source (mag[m, n-1] where both bins are significant), A the left reach
    A[m] = min(mag[m-1, n], max(S[m-1], A[m-1])) inside a run of significant bins, B the right reach, mirrored.
    The largest of the three wins, ties going to time, then left, then right.  An island (run of significant
    bins) with no time source is seeded at its maximum, the lowest bin on ties: bins left of the seed are
    reached from the right and bins right of it from the left.  -1 stands for "no path"."""
    Bn, F = mcur.shape
    S = np.where(sig_prev & sig_cur, mprev, -1.0)
    A = np.full((Bn, F), -1.0)
    PL = np.full((Bn, F), -1.0)       # max of the island's bins left of m
    for m in range(1, F):
        on = sig_cur[:, m - 1]
        A[:, m] = np.where(on, np.minimum(mcur[:, m - 1], np.maximum(S[:, m - 1], A[:, m - 1])), -1.0)
        PL[:, m] = np.where(on, np.maximum(mcur[:, m - 1], PL[:, m - 1]), -1.0)
    Bv = np.full((Bn, F), -1.0)
    PR = np.full((Bn, F), -1.0)
    for m in range(F - 2, -1, -1):
        on = sig_cur[:, m + 1]
        Bv[:, m] = np.where(on, np.minimum(mcur[:, m + 1], np.maximum(S[:, m + 1], Bv[:, m + 1])), -1.0)
        PR[:, m] = np.where(on, np.maximum(mcur[:, m + 1], PR[:, m + 1]), -1.0)
    W = np.maximum(S, np.maximum(A, Bv))
    sourced = np.where(S == W, PGHI_ROOT, np.where(A == W, PGHI_LEFT, PGHI_RIGHT))
    seeded = np.where((mcur > PL) & (mcur >= PR), PGHI_ROOT,
                      np.where((PL >= mcur) & (PL >= PR), PGHI_LEFT, PGHI_RIGHT))
    return np.where(sig_cur, np.where(W >= 0, sourced, seeded), PGHI_NONE)


def pghi_phase(mag: np.ndarray, n_fft: int, hop: int, win_length: Optional[int] = None,
               gamma: Optional[float] = None, tol: float = 1e-5) -> np.ndarray:
    """The scan formulation, vectorised over the batch: per frame the choices (``pghi_choices``), then the
    phases along each run from its root: a root integrates in time from the same bin, phi[m, n-1] + tstep (0 in
    frame 0), and phi[m] = phi[m-1] + fstep[m-1] to the right of it, phi[m] = phi[m+1] - fstep[m] to the left,
    wrapped after every addition exactly as in ``pghi_heap_phase``."""
    wl = int(win_length or n_fft)
    mg, sig, tstep, fstep = pghi_steps(mag, n_fft, hop, wl, _pghi_gamma(wl, gamma), tol)
    Bn, F, T = mg.shape
    ph = np.zeros((Bn, F, T))
    zero = np.zeros((Bn, F), dtype=bool)
    for n in range(T):
        prev = (mg[:, :, n - 1], sig[:, :, n - 1]) if n else (np.zeros((Bn, F)), zero)
        ch = pghi_choices(prev[0], mg[:, :, n], prev[1], sig[:, :, n])
        p = np.zeros((Bn, F))
        root = pghi_wrap(ph[:, :, n - 1] + tstep[:, :, n]) if n else np.zeros((Bn, F))
        for m in range(F):
            p[:, m] = np.where(ch[:, m] == PGHI_ROOT, root[:, m], p[:, m])
            if m:
                p[:, m] = np.where(ch[:, m] == PGHI_LEFT, pghi_wrap(p[:, m - 1] + fstep[:, m - 1, n]), p[:, m])
        for m in range(F - 2, -1, -1):
            p[:, m] = np.where(ch[:, m] == PGHI_RIGHT, pghi_wrap(p[:, m + 1] - fstep[:, m, n]), p[:, m])
        ph[:, :, n] = p
    return ph


def pghi(mag: np.ndarray, n_fft: Optional[int] = None, hop_length: Optional[int] = None,
         win_length: Optional[int] = None, gamma: Optional[float] = None, tol: float = 1e-5) -> np.ndarray:
    """PGHI by the scan formulation; (F, T) or (B, F, T) real -> complex of the same shape.  ``n_fft`` defaults
    to 2 (F - 1), ``hop_length`` to n_fft // 4, ``win_length`` to n_fft, ``gamma`` to 0.25645 win_length^2
    (a Hann window's)."""
    m = mag[None] if mag.ndim == 2 else mag
    n_fft = int(n_fft or (m.shape[1] - 1) * 2)
    ph = pghi_phase(m, n_fft, int(hop_length or n_fft // 4), win_length, gamma, tol)
    return _pghi_out(m, ph).reshape(mag.shape)
