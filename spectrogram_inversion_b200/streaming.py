"""Streaming RTISI-LA and PGHI: magnitude frames in as they are produced, final samples (or frames) out as soon as
they are final."""
from __future__ import annotations

import dataclasses
import math

import torch

from . import _ops
from .engine import StftPlan, compute_device, host_copy
from .methods import _rtisi_checks
from .pghi import _analysis
from .stft_args import args_helper

__all__ = ["RTISIStream", "emitted_samples", "PGHIStream", "pghi_emitted_samples"]


def emitted_samples(n_frames: int, n_fft: int, hop: int, look_ahead: int, center: bool) -> int:
    """E(n) = clamp((n - LA) * hop - P, 0, L(n)): the samples per signal an RTISIStream has returned once n frames
    have been pushed (LA = (n_fft - 1) // hop for look_ahead < 0, P = n_fft // 2 when centred)."""
    LA = (n_fft - 1) // hop if look_ahead < 0 else look_ahead
    P = n_fft // 2 if center else 0
    return max(0, min((n_frames - LA) * hop - P, (n_frames - 1) * hop + n_fft - 2 * P))


def pghi_emitted_samples(n_frames: int, n_fft: int, hop: int, center: bool) -> int:
    """E(n) = clamp((n - 1) * hop - P, 0, L(n)): the samples per signal a PGHIStream with ``output="waveform"`` has
    returned once n frames have been pushed (P = n_fft // 2 when centred, L(n) = (n - 1) * hop + n_fft - 2P).  That is
    ``emitted_samples`` with a look-ahead of one frame."""
    return emitted_samples(n_frames, n_fft, hop, 1, center)


class _FrameStream:
    """The push / flush protocol of the frame streams.  The first chunk fixes the number of dimensions, F, B, the dtype
    and the device of every later one; the frames a step still needs are kept on the compute device between pushes;
    results go back as the chunks came (host or CUDA, with or without the batch dimension).

    A subclass defines ``_start(chunk)``, its set-up at the first push, which calls ``_capture`` (and
    ``_start_envelope`` when it needs 1/envelope windows), and ``_last()``, the final step of ``flush()``, which
    returns what was not returned yet and drops the subclass's own buffers."""

    def __init__(self, stft_kwargs: dict):
        self._stft_kwargs = stft_kwargs
        self._n = 0                # frames pushed
        self._started = False
        self._closed = False

    def _check_open(self) -> None:
        if self._closed:
            raise RuntimeError(f"{type(self).__name__}: the stream was flushed and is closed")

    # ---- set-up at the first push ---------------------------------------------------------------------------
    def _capture(self, chunk: torch.Tensor) -> None:
        self._ndim, self._F, self._dtype, self._in_device = chunk.dim(), chunk.shape[-2], chunk.dtype, chunk.device
        self._B = chunk.shape[0] if chunk.dim() == 3 else 1
        self._host = not chunk.is_cuda
        self._pinned = self._host and chunk.is_pinned()
        self._dev = compute_device(chunk)
        self._hist = torch.empty(self._B, self._F, 0, dtype=self._dtype, device=self._dev)   # frames kept

    def _start_envelope(self, stft_kwargs: dict) -> None:
        """The STFT arguments and the plan that ``_inv_env_window`` gathers from."""
        shape_only = torch.empty(self._B, self._F, 0, dtype=self._dtype, device=self._dev)
        # no stream pads a signal: a constant pad mode keeps short plans (a flush of a few frames) valid for make_dims
        self._args = a = dataclasses.replace(args_helper(shape_only, **stft_kwargs), pad_mode="constant")
        self._P = a.pad
        # shortest plan whose envelope has head, interior and tail apart: (T0 - 1) * hop >= n_fft
        self._T0 = (a.n_fft - 1) // a.hop_length + 2
        self._plan = StftPlan(a, self._T0, self._B, self._dtype, self._dev)

    def _inv_env_window(self, x0: int, length: int, total_frames: int = -1) -> torch.Tensor:
        """1/envelope of samples [x0, x0 + length) of the signal (total_frames -1: not known yet), gathered from the
        short plan, or from a plan of the whole signal when it has fewer than T0 frames."""
        a = self._args
        out = torch.empty(length, dtype=self._dtype, device=self._dev)
        if 0 <= total_frames < self._T0:
            plan = StftPlan(a, total_frames, self._B, self._dtype, self._dev)
        else:
            plan = self._plan
        _ops.plan_inv_env_window(plan.buf, out, x0, total_frames, a.n_fft, a.hop_length, plan.T, a.center,
                                 a.normalized, a.onesided)
        return out

    # ---- every push ------------------------------------------------------------------------------------------
    def _append(self, chunk: torch.Tensor):
        """Set the stream up at the first chunk, check a later one against it, and append its frames to the kept
        ones: returns (window, frame0), window (B, F, rows) on the compute device with row r holding frame
        frame0 + r."""
        if not self._started:
            self._start(chunk)
            self._started = True
        assert chunk.dim() == self._ndim and chunk.shape[-2] == self._F, (tuple(chunk.shape), self._ndim, self._F)
        assert (chunk.shape[0] if chunk.dim() == 3 else 1) == self._B, (tuple(chunk.shape), self._B)
        assert chunk.dtype == self._dtype and chunk.device == self._in_device, (chunk.dtype, chunk.device)
        work = (chunk if chunk.dim() == 3 else chunk.unsqueeze(0)).detach().to(self._dev, non_blocking=True)
        frame0 = self._n - self._hist.shape[-1]
        window = torch.cat([self._hist, work], -1) if work.shape[-1] else self._hist
        self._n += work.shape[-1]
        return window, frame0

    def _keep(self, window: torch.Tensor, k: int) -> None:
        """Keep the last k frames of the window (all of them when it has fewer) for the next push."""
        self._hist = window[..., window.shape[-1] - min(k, window.shape[-1]):].clone()

    def _result(self, out: torch.Tensor) -> torch.Tensor:
        """``out`` (B, ...) on the compute device as the caller gets it: without the batch dimension for 2-D chunks,
        as a host copy for host chunks."""
        if self._ndim == 2:
            out = out[0]
        return host_copy(out, self._pinned) if self._host else out

    # ---- public ------------------------------------------------------------------------------------------------
    def flush(self) -> torch.Tensor:
        """What was not returned yet; closes the stream."""
        self._check_open()
        if self._n == 0:
            raise RuntimeError(f"{type(self).__name__}.flush: no frame has been pushed")
        out = self._last()
        self._closed = True
        self._plan = self._hist = None
        return out


class RTISIStream(_FrameStream):
    r"""RTISI-LA on a spectrogram that arrives a few frames at a time (a TTS or vocoder front end).

    ``RTISIStream(look_ahead, asymmetric_window, max_iter, alpha, **stft_kwargs)`` takes ``RTISI_LA``'s arguments
    with the same defaults and checks (an unknown keyword is a ``TypeError`` unless ``asymmetric_window``).

    * ``push(chunk)``: ``chunk`` holds ``k >= 0`` real magnitude frames, ``(F, k)`` or ``(B, F, k)``; returns the
      samples that became final, ``(n,)`` or ``(B, n)``.  The first push fixes F, B, the number of dimensions, the
      dtype and the device; a later chunk that differs is an ``AssertionError``.  The B signals advance in lockstep.
    * ``flush()``: the remaining samples; the stream is closed afterwards.

    Semantics:

    * ``torch.cat([push_1, ..., push_k, flush()], -1)`` is bit for bit ``RTISI_LA(torch.cat(chunks, -1), same
      arguments, verbose=0)``, for every chunking.  Returned samples never change.
    * After ``n`` frames in total exactly ``E(n) = clamp((n - LA) * hop - P, 0, L(n))`` samples per signal have been
      returned: ``LA`` is the resolved look-ahead (``(n_fft - 1) // hop`` for -1), ``P = n_fft // 2`` when centred,
      else 0, and ``L(n) = (n - 1) * hop + n_fft - 2P``.  That is the earliest a sample is final: step ``i`` needs
      frame ``i`` and its commit finishes the block ``[(i - LA) * hop - P, (i - LA + 1) * hop - P)``.  A block can
      cross ``L(n)`` (``look_ahead = 0``, centred, ``hop > n_fft / 2``); its samples past ``L(n)`` are held back
      and ``flush()`` releases those below the final length.
    * A CUDA chunk is processed on the current stream and the result is a device tensor, without synchronising; a
      host chunk gives a host tensor (like ``RTISI_LA``).
    * Device memory does not grow with the number of frames: the sliding state, the last ``LA`` magnitude frames,
      a plan of ``(n_fft - 1) // hop + 2`` frames and the buffers of one push.
    * No gradients: a chunk that requires grad raises ``NotImplementedError`` (``RTISI_LA`` is differentiable).
      ``flush()`` before any frame, and ``push`` / ``flush`` after ``flush()``, raise ``RuntimeError``.
    """

    def __init__(self, look_ahead=-1, asymmetric_window=False, max_iter=25, alpha=0.99, **stft_kwargs):
        _rtisi_checks(None, max_iter, alpha, asymmetric_window, stft_kwargs)
        super().__init__(stft_kwargs)
        self.look_ahead, self.asymmetric_window = int(look_ahead), bool(asymmetric_window)
        self.max_iter, self.alpha = int(max_iter), float(alpha)
        self._steps = 0            # outer steps run
        self._emitted = 0          # samples per signal returned

    def _start(self, chunk: torch.Tensor) -> None:
        self._capture(chunk)
        self._start_envelope(self._stft_kwargs)
        a, dev = self._args, self._dev
        n, hop = a.n_fft, a.hop_length
        self._LA = (n - 1) // hop if self.look_ahead < 0 else self.look_ahead
        self._window = a.window.detach().to(device=dev, dtype=chunk.dtype).contiguous()
        self._synth_coeff = float(hop / (self._window @ self._window))            # as RTISI_LA (methods.py:318)
        self._scratch = torch.empty(2 * n, dtype=chunk.dtype, device=dev)
        nbytes = _ops.rtisi_state_bytes(self._scratch, n, hop, 1, self._B, a.normalized, a.onesided, self._LA)
        self._state = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self._pending = torch.empty(self._B, 0, dtype=chunk.dtype, device=dev)         # computed, not yet returned

    # ---- helpers -----------------------------------------------------------------------------------------------
    def _block_end(self, step: int) -> int:
        """End of the samples finished by the steps before `step`."""
        return max(0, (step - self._LA) * self._args.hop_length - self._P)

    def _run(self, mag_ext: torch.Tensor, frame0: int, step_end: int, final: bool):
        """Steps [self._steps, step_end) on magnitude frames [frame0, frame0 + mag_ext.shape[-1]); returns the
        samples they finish."""
        a = self._args
        x0 = self._block_end(self._steps)
        x1 = self._block_end(step_end)
        if final:
            L = max(0, a.signal_length(self._n))
            x0, x1 = min(x0, L), L
        x = torch.empty(self._B, x1 - x0, dtype=self._dtype, device=self._dev)
        if final and x1 == x0:
            return x                              # nothing of the signal left to compute
        mag = StftPlan(a, mag_ext.shape[-1], self._B, self._dtype, self._dev, tables=False)
        pm = mag.pack(mag_ext) if mag_ext.shape[-1] else mag.empty_spec(real=True)
        _ops.rtisi_la_stream(self._plan.buf, self._window, pm.main, pm.nyq, x,
                             self._inv_env_window(x0, x1 - x0, self._n if final else -1), self._scratch, self._state,
                             self._n, frame0, x0, self._LA, self.asymmetric_window, self.max_iter, self.alpha,
                             self._synth_coeff, self._steps, step_end, final, a.n_fft, a.hop_length, a.center,
                             a.normalized, a.onesided)
        self._steps = step_end
        return x

    def _emit(self, x: torch.Tensor, upto: int) -> torch.Tensor:
        """Return samples [emitted, upto) of pending ++ x and keep the rest pending."""
        avail = torch.cat([self._pending, x], 1) if self._pending.shape[1] else x
        take = upto - self._emitted
        out = avail[:, :take]
        self._pending = avail[:, take:].clone() if take < avail.shape[1] else avail[:, :0]
        self._emitted = upto
        return self._result(out.contiguous())

    # ---- public ------------------------------------------------------------------------------------------------
    def push(self, chunk: torch.Tensor) -> torch.Tensor:
        """Append k >= 0 magnitude frames, (F, k) or (B, F, k); return the samples that became final."""
        self._check_open()
        if chunk.requires_grad:
            raise NotImplementedError("RTISIStream has no gradient path: use RTISI_LA for a differentiable inversion")
        _rtisi_checks(chunk, self.max_iter, self.alpha, self.asymmetric_window, self._stft_kwargs)
        mag_ext, frame0 = self._append(chunk)
        x = self._run(mag_ext, frame0, self._n, False) if chunk.shape[-1] else self._pending[:, :0]
        self._keep(mag_ext, self._LA)
        a = self._args
        return self._emit(x, emitted_samples(self._n, a.n_fft, a.hop_length, self._LA, a.center))

    def _last(self) -> torch.Tensor:
        x = self._run(self._hist, self._n - self._hist.shape[-1], self._n + self._LA, True)
        out = self._emit(x, max(0, self._args.signal_length(self._n)))
        self._state = self._pending = self._scratch = None
        return out


class PGHIStream(_FrameStream):
    r"""PGHI on a spectrogram that arrives a few frames at a time: one frame of look-ahead, no iterations.

    ``PGHIStream(gamma=None, tol=1e-5, output="waveform", **stft_kwargs)``: ``gamma``, ``tol`` and ``stft_kwargs``
    take ``pghi``'s meaning, defaults and checks.

    * ``push(chunk)``: ``chunk`` holds ``k >= 0`` real magnitude frames, ``(F, k)`` or ``(B, F, k)``, float32 or
      float64; returns what became final.  The first push fixes F, B, the number of dimensions, the dtype and the
      device; a later chunk that differs is an ``AssertionError``.
    * ``flush()``: the rest; the stream is closed afterwards.
    * ``output="spectrum"``: the complex frames that became final, ``(F, k')`` or ``(B, F, k')``.
      ``output="waveform"``: their samples, ``(n,)`` or ``(B, n)``, the ISTFT of the frames with the same
      ``stft_kwargs``.

    Semantics:

    * Frame j is final once frame j+1 has been pushed, or at ``flush()``, where the last frame has a zero time
      derivative like ``pghi``'s.  After n frames ``output="spectrum"`` has returned ``max(0, n - 1)`` frames, and
      ``output="waveform"`` exactly ``pghi_emitted_samples(n, ...)`` samples per signal: a sample is final when every
      frame covering it is.  Returned values never change.
    * The threshold is causal: the step that computes frame n uses ``tol * max`` over frames ``0 .. n + 1`` (``pghi``
      uses the whole signal's max).  So the frames do not depend on how the stream is cut into chunks, and they
      equal ``pghi``'s when a signal's loudest bin lies in frame 0 or 1 (DESIGN.md section 3.7.1).
    * A CUDA chunk is processed on the current stream and the result is a device tensor, without synchronising; a
      host chunk gives a host tensor.
    * Device memory does not grow with the number of frames: the per-signal state, the last two frames, the
      overlap-add carry of ``n_fft - hop`` samples, a plan of ``(n_fft - 1) // hop + 2`` frames and one push's
      buffers.
    * The waveform needs an even n_fft (the ISTFT's sizes: up to 32768 in float32, 16384 in float64) and
      ``hop_length <= win_length``; otherwise ``NotImplementedError``.
    * No gradients: a chunk that requires grad raises ``NotImplementedError``.  ``flush()`` before any frame, and
      ``push`` / ``flush`` after ``flush()``, raise ``RuntimeError``.
    """

    def __init__(self, gamma=None, tol=1e-5, output="waveform", **stft_kwargs):
        if not (isinstance(tol, (int, float)) and 0 < tol < 1):
            raise ValueError(f"PGHIStream: tol={tol} must lie in (0, 1)")
        if gamma is not None and not (float(gamma) > 0 and math.isfinite(float(gamma))):
            raise ValueError(f"PGHIStream: gamma={gamma} must be positive and finite")
        if output not in ("waveform", "spectrum"):
            raise ValueError(f"PGHIStream: output={output!r} must be 'waveform' or 'spectrum'")
        if stft_kwargs.get("n_fft") is not None:
            _analysis(int(stft_kwargs["n_fft"]) // 2 + 1, stft_kwargs)        # refuse bad options before any frame
        super().__init__(stft_kwargs)
        self.gamma, self.tol, self.output = gamma, float(tol), output
        self._final = 0            # frames final

    def _start(self, chunk: torch.Tensor) -> None:
        n_fft, hop, wl = _analysis(chunk.shape[-2], self._stft_kwargs)
        gamma = 0.25645 * wl ** 2 if self.gamma is None else float(self.gamma)
        if self.output == "waveform":
            if n_fft % 2:
                raise NotImplementedError(f"PGHIStream: output='waveform' needs an even n_fft (got {n_fft}); "
                                          "output='spectrum' takes any")
            if hop > wl:
                raise NotImplementedError(f"PGHIStream: output='waveform' needs hop_length <= win_length "
                                          f"({hop} > {wl}): the envelope would vanish between frames")
        self._capture(chunk)
        self._an = (n_fft, hop, wl, gamma)
        self._state = torch.empty(_ops.pghi_stream_state_bytes(chunk.dtype, self._B, self._F), dtype=torch.uint8,
                                  device=self._dev)
        if self.output == "waveform":
            self._start_envelope({k: v for k, v in self._stft_kwargs.items() if k != "n_fft"})
            self._ola = None       # (frames, un-centred unit-envelope plan): plain windowed overlap-add
            self._carry = torch.zeros(self._B, n_fft - hop, dtype=chunk.dtype, device=self._dev)

    # ---- the steps ---------------------------------------------------------------------------------------------
    def _frames(self, window: torch.Tensor, frame0: int, n_final: int, final: bool) -> torch.Tensor:
        """Finalise frames [self._final, self._final + n_final) from magnitude rows frame0 + r: (B, n_final, F)."""
        n_fft, hop, wl, gamma = self._an
        out = torch.empty(self._B, n_final, self._F, dtype=_ops.CDT[self._dtype], device=self._dev)
        if n_final:                # nothing final yet (the window may even be empty)
            _ops.pghi_stream_direct(window, frame0, n_final, final, self._state, out, n_fft, hop, wl, gamma,
                                    self.tol)
        return out

    def _samples(self, frames: torch.Tensor, first: int, final: bool) -> torch.Tensor:
        """The output samples that frames [first, first + k) finish: overlap-add, carry, 1/envelope, trim."""
        a = self._args
        n_fft, hop = a.n_fft, a.hop_length
        k = frames.shape[1]
        T = max(k, self._T0)
        if self._ola is None or self._ola[0] != T:
            plan = StftPlan(dataclasses.replace(a, center=False), T, self._B, self._dtype, self._dev)
            plan.set_unit_envelope()
            self._ola = (T, plan)
        plan = self._ola[1]
        if k < T:
            frames = torch.cat([frames, frames.new_zeros(self._B, T - k, self._F)], 1)
        y = plan.istft(plan.pack(frames.transpose(1, 2)))       # padded samples first * hop + j
        z = y[:, :(k - 1) * hop + n_fft]
        z[:, :n_fft - hop] += self._carry
        if not final:
            self._carry = z[:, k * hop:].clone()
            z = z[:, :k * hop]
        o0 = first * hop - self._P                               # output sample of z[:, 0]
        o1 = o0 + z.shape[1]
        if final:
            o1 = min(o1, a.signal_length(self._n))
        x0 = max(0, o0)
        if o1 <= x0:
            return z[:, :0]
        return z[:, x0 - o0:o1 - o0] * self._inv_env_window(x0, o1 - x0, self._n if final else -1)

    def _run(self, window: torch.Tensor, frame0: int, n_final: int, final: bool) -> torch.Tensor:
        first = self._final
        frames = self._frames(window, frame0, n_final, final)
        self._final += n_final
        if self.output == "spectrum":
            out = frames.transpose(1, 2)
        elif n_final:
            out = self._samples(frames, first, final)
        else:
            out = torch.empty(self._B, 0, dtype=self._dtype, device=self._dev)
        return self._result(out)

    # ---- public ------------------------------------------------------------------------------------------------
    def push(self, chunk: torch.Tensor) -> torch.Tensor:
        """Append k >= 0 magnitude frames, (F, k) or (B, F, k); return the frames or samples that became final."""
        self._check_open()
        if chunk.requires_grad:
            raise NotImplementedError("PGHIStream has no gradient path: detach the magnitude")
        if chunk.is_complex():
            raise ValueError("PGHIStream: a chunk must be a real magnitude, not a complex spectrum")
        if chunk.dtype not in _ops.CDT:
            raise NotImplementedError(f"PGHIStream: dtype {chunk.dtype} is not supported (float32 / float64 only)")
        if chunk.dim() not in (2, 3):
            raise ValueError(f"PGHIStream: a chunk must be (F, k) or (B, F, k), got shape {list(chunk.shape)}")
        window, frame0 = self._append(chunk)
        out = self._run(window, frame0, max(0, self._n - 1 - self._final), False)
        self._keep(window, self._n - max(0, self._final - 1))      # frames [final - 1, n)
        return out

    def _last(self) -> torch.Tensor:
        out = self._run(self._hist, self._n - self._hist.shape[-1], self._n - self._final, True)
        self._state = self._ola = self._carry = None
        return out
