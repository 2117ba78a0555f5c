"""Streaming RTISI-LA: magnitude frames in as they are produced, final samples out as soon as they are final."""
from __future__ import annotations

import dataclasses

import torch

from . import _ops
from .engine import StftPlan, compute_device
from .methods import _rtisi_checks
from .stft_args import args_helper

__all__ = ["RTISIStream", "emitted_samples"]


def emitted_samples(n_frames: int, n_fft: int, hop: int, look_ahead: int, center: bool) -> int:
    """E(n) = clamp((n - LA) * hop - P, 0, L(n)): the samples per signal an RTISIStream has returned once n frames
    have been pushed (LA = (n_fft - 1) // hop for look_ahead < 0, P = n_fft // 2 when centred)."""
    LA = (n_fft - 1) // hop if look_ahead < 0 else look_ahead
    P = n_fft // 2 if center else 0
    return max(0, min((n_frames - LA) * hop - P, (n_frames - 1) * hop + n_fft - 2 * P))


class RTISIStream:
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
        self.look_ahead, self.asymmetric_window = int(look_ahead), bool(asymmetric_window)
        self.max_iter, self.alpha = int(max_iter), float(alpha)
        self._stft_kwargs = stft_kwargs
        self._n = 0                # frames pushed
        self._steps = 0            # outer steps run
        self._emitted = 0          # samples per signal returned
        self._started = False
        self._closed = False

    # ---- set-up at the first push ---------------------------------------------------------------------------
    def _start(self, chunk: torch.Tensor) -> None:
        self._ndim, self._F, self._dtype, self._in_device = chunk.dim(), chunk.shape[-2], chunk.dtype, chunk.device
        self._host = not chunk.is_cuda
        self._pinned = self._host and chunk.is_pinned()
        work = chunk if chunk.dim() == 3 else chunk.unsqueeze(0)
        self._B = work.shape[0]
        self._dev = dev = compute_device(chunk)
        # RTISI-LA never pads: a constant pad mode keeps short plans (flush of a few frames) valid for make_dims
        shape_only = torch.empty(work.shape[:-1] + (0,), dtype=work.dtype, device=dev)
        args = dataclasses.replace(args_helper(shape_only, **self._stft_kwargs), pad_mode="constant")
        self._args = args
        n, hop = args.n_fft, args.hop_length
        K = (n - 1) // hop
        self._LA = K if self.look_ahead < 0 else self.look_ahead
        self._P = n // 2 if args.center else 0
        # shortest plan whose envelope has head, interior and tail apart: (T0 - 1) * hop >= n_fft
        self._T0 = K + 2
        self._plan = StftPlan(args, self._T0, self._B, chunk.dtype, dev)
        self._window = args.window.detach().to(device=dev, dtype=chunk.dtype).contiguous()
        self._synth_coeff = float(hop / (self._window @ self._window))            # as RTISI_LA (methods.py:318)
        self._scratch = torch.empty(2 * n, dtype=chunk.dtype, device=dev)
        nbytes = _ops.rtisi_state_bytes(self._scratch, n, hop, 1, self._B, args.normalized, args.onesided, self._LA)
        self._state = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self._hist = torch.empty(self._B, self._F, 0, dtype=chunk.dtype, device=dev)   # last LA frames pushed
        self._pending = torch.empty(self._B, 0, dtype=chunk.dtype, device=dev)         # computed, not yet returned
        self._started = True

    def _check_open(self) -> None:
        if self._closed:
            raise RuntimeError("RTISIStream: the stream was flushed and is closed")

    # ---- helpers -----------------------------------------------------------------------------------------------
    def _length(self, n_frames: int) -> int:
        """L(n): the reference's output length for n frames."""
        a = self._args
        return (n_frames - 1) * a.hop_length + a.n_fft - 2 * self._P

    def _block_end(self, step: int) -> int:
        """End of the samples finished by the steps before `step`."""
        return max(0, (step - self._LA) * self._args.hop_length - self._P)

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

    def _run(self, mag_ext: torch.Tensor, frame0: int, step_end: int, final: bool):
        """Steps [self._steps, step_end) on magnitude frames [frame0, frame0 + mag_ext.shape[-1]); returns the
        samples they finish."""
        a = self._args
        x0 = self._block_end(self._steps)
        x1 = self._block_end(step_end)
        if final:
            L = max(0, self._length(self._n))
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
        if self._ndim == 2:
            out = out[0]
        if not out.is_contiguous():
            out = out.contiguous()
        if not self._host:
            return out
        host = torch.empty(out.shape, dtype=out.dtype, pin_memory=self._pinned)
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(self._dev).synchronize()
        return host

    # ---- public ------------------------------------------------------------------------------------------------
    def push(self, chunk: torch.Tensor) -> torch.Tensor:
        """Append k >= 0 magnitude frames, (F, k) or (B, F, k); return the samples that became final."""
        self._check_open()
        if chunk.requires_grad:
            raise NotImplementedError("RTISIStream has no gradient path: use RTISI_LA for a differentiable inversion")
        _rtisi_checks(chunk, self.max_iter, self.alpha, self.asymmetric_window, self._stft_kwargs)
        if not self._started:
            self._start(chunk)
        assert chunk.dim() == self._ndim and chunk.shape[-2] == self._F, (tuple(chunk.shape), self._ndim, self._F)
        assert (chunk.shape[0] if chunk.dim() == 3 else 1) == self._B, (tuple(chunk.shape), self._B)
        assert chunk.dtype == self._dtype and chunk.device == self._in_device, (chunk.dtype, chunk.device)
        k = chunk.shape[-1]
        work = (chunk if chunk.dim() == 3 else chunk.unsqueeze(0)).detach().to(self._dev, non_blocking=True)
        frame0 = self._n - self._hist.shape[-1]
        mag_ext = torch.cat([self._hist, work], -1) if k else self._hist
        self._n += k
        x = self._run(mag_ext, frame0, self._n, False) if k else self._pending[:, :0]
        self._hist = mag_ext[..., mag_ext.shape[-1] - min(self._LA, mag_ext.shape[-1]):].clone()
        a = self._args
        return self._emit(x, emitted_samples(self._n, a.n_fft, a.hop_length, self._LA, a.center))

    def flush(self) -> torch.Tensor:
        """The samples not returned yet; closes the stream."""
        self._check_open()
        if self._n == 0:
            raise RuntimeError("RTISIStream.flush: no frame has been pushed")
        x = self._run(self._hist, self._n - self._hist.shape[-1], self._n + self._LA, True)
        out = self._emit(x, max(0, self._length(self._n)))
        self._closed = True
        self._plan = self._state = self._hist = self._pending = self._scratch = None
        return out
