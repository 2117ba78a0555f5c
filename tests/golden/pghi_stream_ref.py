"""The reference for PGHI on a stream (spectrogram_inversion_b200.PGHIStream), numpy only.

The one new definition is the threshold.  Offline PGHI (pghi_ref) uses thr = tol * max over the whole signal, which a
stream cannot know.  The step that computes frame n uses instead

    thr_n = tol * max(mag[b, :, 0 .. min(n + 1, N - 1)])          (``pghi_stream_threshold``)

which is everything that step reads anyway (frame n+1 only for the time derivative), and uses it for everything: the
significance of frames n-1 and n, and s = log(max(mag, thr_n)) for frames n-1, n and n+1.  thr_n does not decrease,
so a bin significant in frame n-1 under thr_n was significant under thr_{n-1} and has an integrated phase to continue
from.  Everything else is pghi_ref's arithmetic in pghi_ref's order: ``pghi_stream_heap`` is the heap with a per-step
threshold, ``pghi_stream`` the scan formulation with it, and with a constant threshold both reduce to pghi_ref's
``pghi_heap_phase`` and ``pghi_phase`` bit for bit."""
from __future__ import annotations

import heapq
from typing import Optional

import numpy as np

from pghi_ref import (PGHI_LEFT, PGHI_RIGHT, PGHI_ROOT, TWO_PI, _pghi_gamma, pghi_choices, pghi_constants,
                      pghi_wrap)


def pghi_stream_threshold(mag: np.ndarray, tol: float) -> np.ndarray:
    """(B, F, T) -> (B, T): thr_n = tol * max(mag[b, :, 0 .. min(n + 1, T - 1)])."""
    m64 = mag.astype(np.float64)
    fmax = np.maximum(m64.max(axis=1), 0.0)                     # (B, T)
    run = np.maximum.accumulate(fmax, axis=1)
    ahead = np.concatenate([run[:, 1:], run[:, -1:]], axis=1)   # max over frames 0 .. min(n + 1, T - 1)
    return tol * ahead


def pghi_stream_steps(mag: np.ndarray, n_fft: int, hop: int, win_length: int, gamma: float, thr: np.ndarray):
    """pghi_ref.pghi_steps with thr (B, T) per step: (mag64, sig_prev, sig_cur, tstep, fstep), each (B, F, T).
    sig_prev[:, :, n] is frame n-1's significance under thr_n (False for n = 0), sig_cur[:, :, n] frame n's."""
    m64 = mag.astype(np.float64)
    B, F, T = m64.shape
    K0, K1, K2 = pghi_constants(n_fft, hop, win_length, gamma)
    base = TWO_PI * ((np.arange(F) * int(hop)) % int(n_fft)) / int(n_fft)
    sig_prev = np.zeros((B, F, T), dtype=bool)
    sig_cur = np.zeros((B, F, T), dtype=bool)
    tstep = np.zeros((B, F, T))
    fstep = np.zeros((B, F, T))
    for n in range(T):
        t = thr[:, n][:, None]
        lo, hi = max(0, n - 1), min(T, n + 2)
        with np.errstate(divide="ignore"):
            s = np.log(np.maximum(m64[:, :, lo:hi], t[:, :, None]))     # frames n-1 (if any), n, n+1 (if any)
        c = n - lo
        sig_cur[:, :, n] = m64[:, :, n] > t
        with np.errstate(invalid="ignore"):     # -inf - -inf only in silent signals, where nothing is significant
            Dm = np.zeros((B, F, hi - lo))
            Dm[:, 1:-1] = 0.5 * (s[:, 2:] - s[:, :-2])
            if n:
                sig_prev[:, :, n] = m64[:, :, n - 1] > t
                tstep[:, :, n] = base[None, :] + K1 * (0.5 * (Dm[:, :, c - 1] + Dm[:, :, c]))
            Dn = np.zeros((B, F))
            if 1 <= n < T - 1:
                Dn = 0.5 * (s[:, :, c + 1] - s[:, :, c - 1])
            fstep[:, :-1, n] = K0 - K2 * (0.5 * (Dn[:, :-1] + Dn[:, 1:]))
    return m64, sig_prev, sig_cur, tstep, fstep


def _thr(mag: np.ndarray, tol: float, thr: Optional[np.ndarray]) -> np.ndarray:
    return pghi_stream_threshold(mag, tol) if thr is None else thr


def pghi_stream_heap(mag: np.ndarray, n_fft: int, hop: int, win_length: Optional[int] = None,
                     gamma: Optional[float] = None, tol: float = 1e-5, thr: Optional[np.ndarray] = None) -> np.ndarray:
    """The definition: pghi_ref.pghi_heap_phase with the per-step threshold.  (B, F, T) -> phase.  ``thr`` (B, T)
    overrides the running-max rule (a constant one gives pghi_heap_phase)."""
    wl = int(win_length or n_fft)
    mg, sigp, sigc, tstep, fstep = pghi_stream_steps(mag, n_fft, hop, wl, _pghi_gamma(wl, gamma),
                                                      _thr(mag, tol, thr))
    B, F, T = mg.shape
    ph = np.zeros((B, F, T))
    for b in range(B):
        for n in range(T):
            done = ~sigc[b, :, n]
            h = [(-mg[b, m, n - 1], m, 0) for m in np.nonzero(sigp[b, :, n])[0]] if n else []
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


def pghi_stream_phase(mag: np.ndarray, n_fft: int, hop: int, win_length: Optional[int] = None,
                      gamma: Optional[float] = None, tol: float = 1e-5, thr: Optional[np.ndarray] = None) -> np.ndarray:
    """The scan formulation (pghi_ref.pghi_phase) with the per-step threshold; the kernels compute it."""
    wl = int(win_length or n_fft)
    mg, sigp, sigc, tstep, fstep = pghi_stream_steps(mag, n_fft, hop, wl, _pghi_gamma(wl, gamma),
                                                      _thr(mag, tol, thr))
    Bn, F, T = mg.shape
    ph = np.zeros((Bn, F, T))
    for n in range(T):
        mprev = mg[:, :, n - 1] if n else np.zeros((Bn, F))
        ch = pghi_choices(mprev, mg[:, :, n], sigp[:, :, n], sigc[:, :, n])
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


def pghi_stream(mag: np.ndarray, n_fft: Optional[int] = None, hop_length: Optional[int] = None,
                win_length: Optional[int] = None, gamma: Optional[float] = None, tol: float = 1e-5) -> np.ndarray:
    """What a PGHIStream returns in total (``output="spectrum"``), by the scan formulation; (F, T) or (B, F, T) real
    -> complex of the same shape.  Defaults as pghi_ref.pghi."""
    m = mag[None] if mag.ndim == 2 else mag
    n_fft = int(n_fft or (m.shape[1] - 1) * 2)
    ph = pghi_stream_phase(m, n_fft, int(hop_length or n_fft // 4), win_length, gamma, tol)
    cdt = np.result_type(mag.dtype, np.complex64)
    return (m.astype(np.float64) * np.exp(1j * ph)).astype(cdt).reshape(mag.shape)
