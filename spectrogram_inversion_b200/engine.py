"""Device-side state and drivers for the fused iterations.

Everything numerical is done by the CUDA kernels behind ``_ops``; this module only owns
buffers (PyTorch is the allocator / stream provider) and the host loop that the reference
keeps in ``_training_loop`` (torch_specinv/methods.py:153-190)."""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple

import torch
from tqdm import tqdm

from . import _lib, _ops
from .stft_args import StftArgs

_CDT = {torch.float32: torch.complex64, torch.float64: torch.complex128}


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError("spectrogram_inversion_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _lib.lib()


def compute_device(t: torch.Tensor) -> torch.device:
    """CUDA tensors run in place; host tensors are staged through the current CUDA device."""
    require_cuda()
    return t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device())


@dataclass
class SplitSpec:
    """Split frame-major spectrum: main (B, T, row), nyq (B, T) or empty when two-sided."""
    main: torch.Tensor
    nyq: torch.Tensor

    def like(self) -> "SplitSpec":
        return SplitSpec(torch.empty_like(self.main), torch.empty_like(self.nyq))

    def zeros_like(self) -> "SplitSpec":
        return SplitSpec(torch.zeros_like(self.main), torch.zeros_like(self.nyq))


class StftPlan:
    """Twiddles, scaled windows and 1/envelope for one (stft args, T, B, dtype, device)."""

    def __init__(self, args: StftArgs, n_frames: int, batch: int, dtype: torch.dtype, device: torch.device,
                 tables: bool = True):
        require_cuda()
        if dtype not in _CDT:
            raise NotImplementedError(f"dtype {dtype} is not supported (float32 / float64 only)")
        if args.pad_mode not in _lib.PAD_MODES:
            raise NotImplementedError(f"pad_mode {args.pad_mode!r} is not supported")
        n = args.n_fft
        if n < 16 or n > 8192:
            raise NotImplementedError(f"n_fft={n}: the sm_100a kernels need an n_fft in [16, 8192] (sizes whose half "
                                      "factors into 2 .. 13 run the FFT kernels, other sizes the direct-DFT tile kernel)")
        self.args, self.T, self.B, self.dtype, self.device = args, int(n_frames), int(batch), dtype, device
        self.cdtype = _CDT[dtype]
        self.pad_mode = _lib.PAD_MODES[args.pad_mode]
        self.length = args.signal_length(self.T)
        self.row = n // 2 if args.onesided else n
        self.n_bins = args.n_bins
        self._k = (n, args.hop_length, args.center, self.pad_mode, args.normalized, args.onesided)
        self.buf = None
        d = _lib.make_desc(n, args.hop_length, self.T, self.B, args.center, self.pad_mode, args.normalized,
                           args.onesided, _ops._DT[dtype])
        self.desc, self.desc_ref = d, _lib.C.byref(d)      # struct specinv_desc of this plan (kept alive here)
        if not tables:          # layout conversion / phase_init only
            return
        nbytes = _lib.C.c_size_t(0)
        _lib.check(_lib.lib().specinv_plan_bytes(_lib.C.byref(d), _lib.C.byref(nbytes)), "plan_bytes")
        self.buf = torch.empty(nbytes.value, dtype=torch.uint8, device=device)
        window = args.window.detach().to(device=device, dtype=dtype).contiguous()
        _ops.plan_init(self.buf, window, n, args.hop_length, self.T, self.B, args.center, self.pad_mode,
                       args.normalized, args.onesided)

    # ---- buffers ---------------------------------------------------------------------------
    def empty_spec(self, real: bool = False) -> SplitSpec:
        dt = self.dtype if real else self.cdtype
        main = torch.empty(self.B, self.T, self.row, dtype=dt, device=self.device)
        nyq = torch.empty((self.B, self.T) if self.args.onesided else (0,), dtype=dt, device=self.device)
        return SplitSpec(main, nyq)

    def empty_signal(self) -> torch.Tensor:
        return torch.empty(self.B, self.length, dtype=self.dtype, device=self.device)

    # ---- layout ----------------------------------------------------------------------------
    def pack(self, spec: torch.Tensor) -> SplitSpec:
        """(B, F, T) tensor with any strides -> split layout (real or complex)."""
        assert spec.shape == (self.B, self.n_bins, self.T), (spec.shape, (self.B, self.n_bins, self.T))
        want = self.cdtype if spec.is_complex() else self.dtype
        spec = spec.detach().to(device=self.device, dtype=want)
        out = self.empty_spec(real=not spec.is_complex())
        _ops.pack(spec, out.main, out.nyq, self.args.n_fft, self.args.onesided)
        return out

    def unpack(self, s: SplitSpec) -> torch.Tensor:
        """split layout -> (B, F, T) complex with the physical layout torch.stft produces
        (frame-major: strides (F*T, 1, F))."""
        out = torch.empty(self.B, self.T, self.n_bins, dtype=self.cdtype, device=self.device).transpose(1, 2)
        _ops.unpack(s.main, s.nyq, out, self.args.n_fft, self.args.onesided)
        return out

    # ---- one-shot setup --------------------------------------------------------------------
    def phase_init(self, mag: SplitSpec) -> SplitSpec:
        """split magnitude -> split complex start, the reference's phase_init (methods.py:572-615)."""
        out = self.empty_spec()
        _ops.phase_init(mag.main, mag.nyq, out.main, out.nyq, self.args.n_fft, self.args.hop_length,
                        self.args.onesided)
        return out

    def spec_abs(self, c: SplitSpec) -> SplitSpec:
        """|C| of a complex split spectrum (target magnitude of a complex start, methods.py:110)."""
        out = self.empty_spec(real=True)
        _ops.spec_abs(c.main, c.nyq, out.main, out.nyq, self.args.n_fft, self.args.onesided)
        return out

    # ---- primitives ------------------------------------------------------------------------
    def stft(self, x: torch.Tensor, out: Optional[SplitSpec] = None) -> SplitSpec:
        out = out or self.empty_spec()
        _ops.stft(self.buf, x, out.main, out.nyq, *self._k)
        return out

    def istft(self, s: SplitSpec, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = out if out is not None else self.empty_signal()
        _ops.istft(self.buf, s.main, s.nyq, out, *self._k)
        return out


def spec_sums(a: SplitSpec, b: SplitSpec) -> torch.Tensor:
    """3 doubles: sum (a-b)^2, sum a^2, sum b^2 over a real split spectrum pair."""
    out = torch.zeros(3, dtype=torch.float64, device=a.main.device)
    _ops.metric_sums(a.main, b.main, out)
    if a.nyq.numel():
        _ops.metric_sums(a.nyq, b.nyq, out)
    return out


def evaluates(i: int, eva_iter: int) -> bool:
    """Whether iteration ``i`` (from 0) of the reference loop evaluates the metric (methods.py:153-190)."""
    return i % eva_iter == eva_iter - 1


class _Solver:
    """Common ping-pong state for the fused iterations."""

    def __init__(self, plan: StftPlan, mag: SplitSpec):
        self.plan, self.mag = plan, mag
        self.x = [plan.empty_signal(), plan.empty_signal()]
        self.cur = 0
        self.sums = torch.zeros(2, dtype=torch.float64, device=plan.device)
        self._nosums = torch.empty(0, dtype=torch.float64, device=plan.device)
        self.n_bins_total = plan.B * plan.n_bins * plan.T
        self.g = float(spec_sums(mag, mag)[2].item())   # sum mag^2 (constant per call)
        self.iterations = 0
        # Iterations are launched straight through ctypes (`_ops.iter_direct`, ~6 us of host time each), which keeps
        # even the smallest config GPU-bound (cfg1: 24 us of kernel per iteration).
        self._ptrs = [None, None]      # per ping-pong parity: (tensors, their device pointers)

    def _launch_direct(self, what: str, tensors: tuple, coef: float, sums: torch.Tensor) -> None:
        c = self._ptrs[self.cur]
        if c is None or len(c[0]) != len(tensors) or any(a is not b for a, b in zip(c[0], tensors)):
            c = self._ptrs[self.cur] = (tensors, _ops.pointers(tensors))      # (re)built when a buffer was replaced
        _ops.iter_direct(self._fn, what, self.plan.device, self.plan.desc_ref, c[1], coef,
                         sums.data_ptr() if sums.numel() else None)

    @property
    def signal(self) -> torch.Tensor:
        return self.x[self.cur]

    def _launch(self, sums: torch.Tensor) -> None:
        raise NotImplementedError

    def step(self, evaluate: bool = False, read: bool = True) -> Optional[Tuple[float, float]]:
        """One fused iteration.  With ``evaluate`` returns (d, e) = (sum (|s|-mag)^2, sum |s|^2) of
        the spectrogram the iteration started from -- exactly the ``output`` the reference's closure
        returns (methods.py:242, :465) -- which costs one device->host sync like the reference's
        ``.item()`` calls (methods.py:181-182).  ``read=False`` leaves the two sums on the device
        (``self.sums``): the evaluation is computed but the host does not wait for it."""
        if evaluate:
            self.sums.zero_()
            self._launch(self.sums)
        else:
            self._launch(self._nosums)
        self.cur ^= 1
        self.iterations += 1
        if evaluate and read:
            d, e = self.sums.tolist()
            return d, e
        return None

    def run_many(self, n: int, iter0: int, eva_iter: int, evaluate: bool = True) -> None:
        """Iterations iter0 .. iter0 + n - 1 of the reference loop (methods.py:178-190) without host synchronisation:
        those that ``evaluates`` run the fused metric epilogue when ``evaluate`` (the last pair of sums stays in
        ``self.sums``)."""
        for i in range(iter0, iter0 + n):
            self.step(evaluate=evaluate and evaluates(i, eva_iter), read=False)


class GriffinLimSolver(_Solver):
    """State machine of griffin_lim (methods.py:225-255): q_0 = C, x_0 = ISTFT(C), then
    q_n = STFT(x_{n-1}) - lr q_{n-1};  x_n = ISTFT(proj(q_n))."""

    def __init__(self, plan: StftPlan, C: SplitSpec, mag: SplitSpec, alpha: float):
        super().__init__(plan, mag)
        self.lr = alpha / (1 + alpha)                     # methods.py:235
        # alpha = 0 is plain Griffin-Lim: q_n = STFT(x_{n-1}) needs no momentum state, so none is kept or moved
        self.plain = self.lr == 0
        self.q = None if self.plain else [C, C.like()]
        self._fn = _lib.lib().specinv_gl_iter
        plan.istft(C, self.x[0])                          # methods.py:233
        # Small problems (B * T frames fit the SMs' shared memory): runs of iterations go through ONE persistent kernel
        # with the state resident on chip (csrc/specinv_resident.cu) instead of one launch per iteration.
        self._resident_ws = None
        if not self.plain and plan.dtype == torch.float32 and os.environ.get("SPECINV_RESIDENT", "1") != "0":
            nbytes = _lib.C.c_size_t(0)
            if _lib.lib().specinv_gl_run_workspace_bytes(plan.desc_ref, _lib.C.byref(nbytes)) == 0:
                self._resident_ws = torch.empty(nbytes.value, dtype=torch.uint8, device=plan.device)

    def run_many(self, n: int, iter0: int, eva_iter: int, evaluate: bool = True) -> None:
        if self._resident_ws is None or n < 2:
            return super().run_many(n, iter0, eva_iter, evaluate)
        p, i, o = self.plan, self.cur, self.cur ^ 1
        n_eval = sum(1 for k in range(iter0, iter0 + n) if evaluates(k, eva_iter)) if evaluate else 0
        sums = torch.zeros(2 * n_eval, dtype=torch.float64, device=p.device) if n_eval else None
        stream = torch.cuda.current_stream(p.device).cuda_stream
        with torch.cuda.device(p.device):
            code = _lib.lib().specinv_gl_run(
                p.desc_ref, p.buf.data_ptr(), self.x[i].data_ptr(), self.x[o].data_ptr(), self.q[i].main.data_ptr(),
                self.q[i].nyq.data_ptr(), self.q[o].main.data_ptr(), self.q[o].nyq.data_ptr(), self.mag.main.data_ptr(),
                self.mag.nyq.data_ptr(), self.lr, int(n), int(iter0), int(eva_iter),
                sums.data_ptr() if sums is not None else None, self._resident_ws.data_ptr(), stream)
        _ops._ok(code, "gl_run")
        if sums is not None:
            self.sums.copy_(sums[-2:])
        self.cur ^= 1
        self.iterations += n

    def check_resident(self) -> None:
        """Raise if a CTA of the last persistent run timed out waiting for a neighbour (synchronises)."""
        if self._resident_ws is None:
            return
        status = _lib.C.c_uint32(0)
        with torch.cuda.device(self.plan.device):
            _ops._ok(_lib.lib().specinv_gl_run_status(self.plan.desc_ref, self._resident_ws.data_ptr(), _lib.C.byref(status),
                                                      torch.cuda.current_stream(self.plan.device).cuda_stream), "gl_run_status", 0)
        if status.value:
            raise RuntimeError(f"persistent Griffin-Lim kernel: neighbour wait timed out at iteration {status.value}")

    def _launch(self, sums: torch.Tensor) -> None:
        p, i, o = self.plan, self.cur, self.cur ^ 1
        qi = (None, None, None, None) if self.plain else (self.q[i].main, self.q[i].nyq, self.q[o].main, self.q[o].nyq)
        self._launch_direct("gl_iter", (p.buf, self.x[i], self.x[o], *qi, self.mag.main, self.mag.nyq), self.lr, sums)

    @property
    def q_state(self) -> SplitSpec:
        if self.plain:
            raise RuntimeError("plain Griffin-Lim (alpha = 0) keeps no momentum state")
        return self.q[self.cur]


class ADMMSolver(_Solver):
    """State machine of ADMM (methods.py:452-490) with the redundant Y = X + U eliminated."""

    def __init__(self, plan: StftPlan, C: SplitSpec, mag: SplitSpec, rho: float):
        super().__init__(plan, mag)
        self.rho = float(rho)
        self.X = [C, C.like()]
        self.U = [C.zeros_like(), C.like()]
        self._fn = _lib.lib().specinv_admm_iter
        plan.istft(C, self.x[0])                          # methods.py:453

    def _launch(self, sums: torch.Tensor) -> None:
        p, i, o = self.plan, self.cur, self.cur ^ 1
        self._launch_direct("admm_iter",
                            (p.buf, self.x[i], self.x[o], self.X[i].main, self.X[i].nyq, self.U[i].main, self.U[i].nyq,
                             self.X[o].main, self.X[o].nyq, self.U[o].main, self.U[o].nyq, self.mag.main, self.mag.nyq),
                            self.rho, sums)


def metric_value(name: str, d: float, e: float, g: float) -> float:
    """sc / snr / ser from the three sums (metrics.py:14, :28-29, :43)."""
    def l10(v: float) -> float:
        return math.log10(v) if v > 0 else -math.inf
    if name == "SC":
        return 10.0 * (l10(d) - l10(g))
    if name == "SNR":
        return -10.0 * (l10(d) - l10(g))
    if name == "SER":
        return 10.0 * (l10(e) - l10(d))
    raise AssertionError(name)


METRIC_NAMES = ("SC", "SNR", "SER")   # methods.py:14-18


def training_loop(solver, max_iter: int, tol: float, verbose, eva_iter: int, metric: str,
                  history: Optional[List] = None, reduce_sums: Optional[Callable] = None) -> int:
    """Host loop with the reference's evaluation cadence and early-stop rule (methods.py:153-190).

    ``solver`` needs ``step(evaluate) -> (d, e) | None``, ``g`` and ``n_bins_total``; with ``run_many`` (every
    ``_Solver``) the iterations between evaluations run without a host synchronisation.  ``reduce_sums``
    (multi-GPU): maps the local ``(d, e)`` of an evaluation to the global ones (an all-reduce), so that the
    metric, the loss and therefore the stopping decision are those of the whole batch on every rank --
    the reference evaluates over the entire batch (methods.py:181-182); ``solver.g`` / ``n_bins_total`` must
    then be global too."""
    assert eva_iter > 0
    assert max_iter > 0
    assert tol >= 0
    metric = metric.upper()
    assert metric in METRIC_NAMES
    bar = {metric: 0}
    init_loss = None
    previous_loss = None
    done = 0
    run_many = getattr(solver, "run_many", None)
    if tol == 0 and not verbose and history is None and reduce_sums is None and run_many is not None:
        # With tol == 0 the stopping rule `(previous - loss) / init < 0 and previous > loss` (methods.py:187) can
        # never fire and nothing displays the metric: the evaluations are still computed at the reference's cadence
        # (the fused epilogue runs on the same iterations) but the host does not wait for the two sums.
        run_many(max_iter, 0, eva_iter)
        return max_iter
    with tqdm(total=max_iter, disable=not verbose) as pbar:
        i = 0
        while i < max_iter:
            if not evaluates(i, eva_iter):
                if run_many is None:
                    solver.step()
                    i += 1
                else:
                    # the iterations up to the next evaluation (or the end) in one go
                    n = min(eva_iter - 1 - i % eva_iter, max_iter - i)
                    run_many(n, i, eva_iter, evaluate=False)
                    i += n
                done = i
                continue
            d, e = solver.step(evaluate=True)
            if reduce_sums is not None:
                d, e = reduce_sums(d, e)
            done = i + 1
            bar[metric] = metric_value(metric, d, e, solver.g)
            l2_loss = d / solver.n_bins_total
            if history is not None:
                history.append((i, bar[metric], l2_loss))
            pbar.set_postfix(**bar, loss=l2_loss)
            pbar.update(eva_iter)
            if not init_loss:
                init_loss = l2_loss
            elif (previous_loss - l2_loss) / init_loss < tol and previous_loss > l2_loss:
                break
            previous_loss = l2_loss
            i += 1
    return done
