"""Public algorithm API with the reference's signatures (torch_specinv/methods.py:193, :273, :415,
:572), running on the sm_100a kernels of libspecinv_b200.so.  No CPU / PyTorch fallback."""
from __future__ import annotations

import math

import torch
from tqdm import tqdm

from . import _ops, autograd
from .engine import ADMMSolver, GriffinLimSolver, METRIC_NAMES, StftPlan, compute_device, host_copy, training_loop
from .stft_args import args_helper, real_dtype_of

__all__ = ["griffin_lim", "RTISI_LA", "ADMM", "L_BFGS", "phase_init"]

pi2 = 2 * math.pi
_TORCH_STFT_KEYS = frozenset(("hop_length", "win_length", "window", "center", "pad_mode", "normalized", "onesided",
                              "return_complex", "align_to_window"))


def _pop_aliases(kw: dict, max_iter, eva_iter):
    """BASELINE.json / the reference README spell these ``maxiter`` / ``evaiter``; the reference code
    itself only knows max_iter / eva_iter (methods.py:193-200).  Accept both."""
    if "maxiter" in kw:
        max_iter = kw.pop("maxiter")
    if "evaiter" in kw:
        eva_iter = kw.pop("evaiter")
    return max_iter, eva_iter


def _setup(spec: torch.Tensor, stft_kwargs: dict):
    """Input formatting of the reference (methods.py:99-111 and :225-227) on the device, in the split
    layout: 2-D -> 3-D; a real input is the target magnitude and gets its start from phase_init, a
    complex input is the start and its modulus the target."""
    shape = spec.shape
    assert 4 > len(shape) > 1
    dev = compute_device(spec)
    work = spec.detach()
    if len(shape) == 2:
        work = work.unsqueeze(0)
    work = work.to(dev, non_blocking=True)
    args = args_helper(work, **stft_kwargs)
    B, _, T = work.shape
    plan = StftPlan(args, T, B, real_dtype_of(work.dtype), dev)
    if work.is_complex():
        C = plan.pack(work)
        return plan, C, plan.spec_abs(C)
    mag = plan.pack(work)
    return plan, plan.phase_init(mag), mag


def _diff_setup(spec: torch.Tensor, stft_kwargs: dict):
    """Input handling of the differentiable path: everything stays attached to ``spec``'s graph."""
    assert 4 > len(spec.shape) > 1
    dev = compute_device(spec)
    work = spec.unsqueeze(0) if len(spec.shape) == 2 else spec
    work = work.to(dev)
    args = args_helper(work, **stft_kwargs)
    args.window = args.window.detach().to(device=dev, dtype=real_dtype_of(work.dtype))
    return work, args


def _diff_finish(x: torch.Tensor, spec: torch.Tensor) -> torch.Tensor:
    if not (spec.shape[0] == 1 and len(spec.shape) == 3):
        x = x.squeeze(0)
    return x.to(spec.device)


def _finish(x: torch.Tensor, spec: torch.Tensor) -> torch.Tensor:
    """methods.py:267-270: drop the batch dim unless the input was (1, F, T)."""
    if not (spec.shape[0] == 1 and len(spec.shape) == 3):
        x = x.squeeze(0)
    return x.clone() if spec.is_cuda else host_copy(x, spec.is_pinned())


def _pipeline_chunks(spec: torch.Tensor, tol: float, verbose, state_arrays: int = 1) -> int:
    """Host (non-CUDA) batches are processed in batch chunks so that the host->device copy of the next chunk and
    the device->host copy of the previous result overlap the iterations of the current one.  The signals of a
    batch only interact through the batch-global early-stop test (methods.py:186-190), which can never fire with
    ``tol == 0`` ((prev - cur) / init < 0 and prev > cur contradict each other), and through the progress bar; so
    with ``tol == 0`` and no progress bar the chunked run returns exactly what the whole-batch run returns."""
    if spec.is_cuda or len(spec.shape) != 3 or tol != 0 or verbose:
        return 1
    B, F, T = spec.shape
    # at most 4 chunks: 4 / 6 / 8 / 16 measured within noise of each other at cfg2 (DESIGN.md section 7)
    n = int(max(1, min(4, B, (B * T) // 60000)))
    # ... and small enough for the device: a chunk holds its input, the magnitudes, the ping-pong state (two complex
    # arrays for Griffin-Lim, four for ADMM) and two signals; keep that within 80 % of the free memory
    per_signal = F * T * spec.element_size() * (2 if not spec.is_complex() else 1) * (1 + 0.5 + 2 * state_arrays + 1)
    if not torch.cuda.is_available():
        return n
    dev = compute_device(spec)
    # cudaMemGetInfo takes a context-wide lock and was measured to stall this call for 15 - 85 ms now and then
    # (the whole e2e tail of bench.py).  Ask the driver only when the batch could come anywhere
    # near the device's memory; otherwise the static total minus torch's own live allocations is estimate enough.
    total = _total_memory(dev)
    if B * per_signal / n > 0.25 * (total - torch.cuda.memory_allocated(dev)):
        free = torch.cuda.mem_get_info(dev)[0]
        if free > 0:
            n = max(n, min(B, -(-int(B * per_signal) // int(0.8 * free))))
    return n


_TOTAL_MEMORY = {}


def _total_memory(dev: torch.device) -> int:
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _TOTAL_MEMORY:
        _TOTAL_MEMORY[key] = torch.cuda.get_device_properties(key).total_memory
    return _TOTAL_MEMORY[key]


_SIDE_STREAMS = {}


def _side_streams(dev: torch.device):
    """The copy-in / copy-out streams of the host pipeline, created ONCE per device.  torch hands out side streams
    round-robin from a pool of 32 and its caching allocator keeps freed blocks per stream: with fresh streams per call
    the staged input chunks (3 x 236 MiB at cfg2) could not be reused until the pool wrapped around 16 calls later --
    every call paid three cudaMallocs, some of them 100-250 ms (measured, tools/e2e_tail.py)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
    return st


def _run_host_pipelined(spec, n_chunks, make_solver, max_iter, eva_iter, metric, stft_kwargs):
    dev = compute_device(spec)
    cur = torch.cuda.current_stream(dev)
    s_in, s_out = _side_streams(dev)
    s_in.wait_stream(cur)
    B = spec.shape[0]
    bounds = [(B * k) // n_chunks for k in range(n_chunks + 1)]

    def stage(k):
        with torch.cuda.stream(s_in):
            t = spec[bounds[k]:bounds[k + 1]].detach().to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(s_in)
        return t, ev

    out, keep = None, []
    nxt = stage(0)
    for k in range(n_chunks):
        work, ev = nxt
        if k + 1 < n_chunks:
            nxt = stage(k + 1)
        cur.wait_event(ev)
        work.record_stream(cur)
        plan, C, mag = _setup(work, stft_kwargs)
        solver = make_solver(plan, C, mag)
        training_loop(solver, max_iter, 0.0, False, eva_iter, metric)
        x = solver.signal
        if out is None:
            out = torch.empty((B, x.shape[1]), dtype=x.dtype, pin_memory=spec.is_pinned())
        done = torch.cuda.Event()
        done.record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(done)
            out[bounds[k]:bounds[k + 1]].copy_(x, non_blocking=True)
        keep.append(x)                       # alive until the copy stream has drained
        del plan, C, mag, solver, work
    s_out.synchronize()
    return out


def griffin_lim(spec, max_iter=200, tol=1e-6, alpha=0.99, verbose=True, eva_iter=10, metric="sc",
                **stft_kwargs):
    r"""Griffin-Lim / fast Griffin-Lim phase reconstruction (drop-in for
    ``torch_specinv.griffin_lim``, methods.py:193-270).

    Args:
        spec (Tensor): magnitude (real) or initial complex estimate, ``(F, T)`` or ``(B, F, T)``.
        max_iter (int): number of iterations.
        tol (float): early-stop tolerance on the relative MSE decrease. Default ``1e-6``.
        alpha (float): momentum of fast Griffin-Lim, 0 disables it. Default ``0.99``.
        verbose (bool): progress bar.
        eva_iter (int): evaluate the metric every ``eva_iter`` iterations. Default ``10``.
        metric (str): ``'sc'``, ``'snr'`` or ``'ser'``.
        **stft_kwargs: the ``torch.stft`` arguments the spectrogram was computed with.

    Returns:
        the time-domain signal, ``(L,)`` or ``(B, L)``.
    """
    assert alpha >= 0
    max_iter, eva_iter = _pop_aliases(stft_kwargs, max_iter, eva_iter)
    assert eva_iter > 0
    assert max_iter > 0
    assert tol >= 0
    assert metric.upper() in METRIC_NAMES
    if autograd.wants_grad(spec):     # the reference's output is differentiable w.r.t. spec (test_griffin.py:54,65-66)
        work, args = _diff_setup(spec, stft_kwargs)
        return _diff_finish(autograd.griffin_lim_diff(work, args, max_iter, tol, alpha, verbose, eva_iter, metric), spec)
    n_chunks = _pipeline_chunks(spec, tol, verbose)
    if n_chunks > 1:
        return _run_host_pipelined(spec, n_chunks, lambda p, c, m: GriffinLimSolver(p, c, m, alpha), max_iter, eva_iter,
                                   metric, stft_kwargs)
    plan, C, mag = _setup(spec, stft_kwargs)
    solver = GriffinLimSolver(plan, C, mag, alpha)
    training_loop(solver, max_iter, tol, verbose, eva_iter, metric)
    return _finish(solver.signal, spec)


def ADMM(spec, max_iter=1000, tol=1e-6, rho=0.1, verbose=1, eva_iter=10, metric="sc", **stft_kwargs):
    r"""ADMM phase recovery (drop-in for ``torch_specinv.ADMM``, methods.py:415-506)."""
    max_iter, eva_iter = _pop_aliases(stft_kwargs, max_iter, eva_iter)
    assert eva_iter > 0
    assert max_iter > 0
    assert tol >= 0
    assert metric.upper() in METRIC_NAMES
    if autograd.wants_grad(spec):
        work, args = _diff_setup(spec, stft_kwargs)
        return _diff_finish(autograd.admm_diff(work, args, max_iter, tol, rho, verbose, eva_iter, metric), spec)
    n_chunks = _pipeline_chunks(spec, tol, verbose, state_arrays=2)
    if n_chunks > 1:
        return _run_host_pipelined(spec, n_chunks, lambda p, c, m: ADMMSolver(p, c, m, rho), max_iter, eva_iter, metric,
                                   stft_kwargs)
    plan, C, mag = _setup(spec, stft_kwargs)
    solver = ADMMSolver(plan, C, mag, rho)
    training_loop(solver, max_iter, tol, verbose, eva_iter, metric)
    return _finish(solver.signal, spec)


def _rtisi_checks(spec, max_iter, alpha, asymmetric_window, stft_kwargs) -> None:
    """The argument checks of RTISI_LA, shared with RTISIStream (``spec`` None: the options only)."""
    assert max_iter > 0
    assert alpha >= 0
    if spec is not None:
        assert not spec.is_complex()
        assert 4 > len(spec.shape) > 1
    if not asymmetric_window:
        # the reference hands the caller's kwargs to torch.stft on this path (methods.py:308-310, :385), so an unknown
        # key is a TypeError there (griffin_lim / ADMM and the asymmetric path silently ignore it, :42-46)
        for key in stft_kwargs:
            if key not in _TORCH_STFT_KEYS:
                raise TypeError(f"stft() got an unexpected keyword argument '{key}'")


def RTISI_LA(spec, look_ahead=-1, asymmetric_window=False, max_iter=25, alpha=0.99, verbose=1, **stft_kwargs):
    r"""Real-Time Iterative Spectrogram Inversion with Look-Ahead (drop-in for
    ``torch_specinv.RTISI_LA``, methods.py:273-412).  ``RTISIStream`` runs the same algorithm on frames that
    arrive a few at a time."""
    _rtisi_checks(spec, max_iter, alpha, asymmetric_window, stft_kwargs)
    if autograd.wants_grad(spec):
        work, args = _diff_setup(spec, stft_kwargs)
        return _diff_finish(autograd.rtisi_diff(work, args, look_ahead, asymmetric_window, max_iter, alpha, verbose), spec)
    dev = compute_device(spec)
    work = spec.detach()
    if len(spec.shape) == 2:
        work = work.unsqueeze(0)
    work = work.to(dev, non_blocking=True)
    args = args_helper(work, **stft_kwargs)
    B, _, T = work.shape
    plan = StftPlan(args, T, B, work.dtype, dev)
    mag = plan.pack(work)
    window = args.window.detach().to(device=dev, dtype=work.dtype).contiguous()
    synth_coeff = float(args.hop_length / (window @ window))                 # methods.py:318
    x = plan.empty_signal()
    scratch = torch.empty(2 * args.n_fft, dtype=work.dtype, device=dev)
    if not verbose:
        _ops.rtisi_la(plan.buf, window, mag.main, mag.nyq, x, scratch, int(look_ahead), bool(asymmetric_window),
                      int(max_iter), float(alpha), synth_coeff, *plan._k)
        return _finish(x, spec)
    # the reference's progress bar counts outer steps (methods.py:362, :400): the persistent kernel is cut at step
    # boundaries, its sliding state parked in HBM in between (bit-identical to the uncut run)
    LA = (args.n_fft - 1) // args.hop_length if look_ahead < 0 else int(look_ahead)
    steps = T + LA
    state = torch.empty(_ops.rtisi_state_bytes(x, args.n_fft, args.hop_length, T, B, args.normalized, args.onesided, LA),
                        dtype=torch.uint8, device=dev)
    chunk = max(1, -(-steps // 40))
    with tqdm(total=steps, disable=not verbose) as pbar:
        for s0 in range(0, steps, chunk):
            s1 = min(steps, s0 + chunk)
            _ops.rtisi_la_steps(plan.buf, window, mag.main, mag.nyq, x, scratch, state, LA, bool(asymmetric_window),
                                int(max_iter), float(alpha), synth_coeff, s0, s1, *plan._k)
            torch.cuda.current_stream(dev).synchronize()          # the bar shows work that is done
            pbar.update(s1 - s0)
    return _finish(x, spec)


def phase_init(spec, **stft_kwargs):
    r"""One-shot phase initialiser (simplified SPSI), drop-in for ``torch_specinv.phase_init``
    (methods.py:572-615): instantaneous frequency of each strict spectral peak (parabolic
    interpolation) assigned to the peak bin and its two neighbours, integrated over time."""
    assert not spec.is_complex()
    shape = spec.shape
    if len(spec.shape) == 2:
        spec = spec.unsqueeze(0)
    assert len(spec.shape) == 3
    dev = compute_device(spec)
    m = spec.detach().to(dev)
    args = args_helper(m, **stft_kwargs)
    B, _, T = m.shape
    plan = StftPlan(args, T, B, m.dtype, dev, tables=False)
    out = plan.unpack(plan.phase_init(plan.pack(m)))
    return out.reshape(shape).to(spec.device)


def L_BFGS(spec, transform_fn, samples=None, init_x0=None, outer_max_iter=1000, tol=1e-6, verbose=1, eva_iter=10,
           metric="sc", **kwargs):
    r"""Inversion of an arbitrary differentiable representation with ``torch.optim.LBFGS`` (same signature and
    loop as ``torch_specinv.L_BFGS``, methods.py:509-569).

    This function is generic autograd on a USER transform -- nothing of it is STFT specific and none of the
    sm_100a kernels apply (SURVEY.md section 2: out of scope); it is provided so that the package exports the same
    five names as the reference.  It runs wherever ``spec`` lives, on plain PyTorch.
    """
    if init_x0 is None:
        init_x0 = spec.new_empty(*samples).normal_(std=1e-6)
    x = torch.nn.Parameter(init_x0)
    optimizer = torch.optim.LBFGS([x], **kwargs)

    def inner():
        optimizer.zero_grad()
        loss = torch.nn.functional.mse_loss(transform_fn(x), spec)
        loss.backward()
        return loss

    def outer():
        optimizer.step(inner)
        with torch.no_grad():
            return transform_fn(x)

    autograd._loop(outer, spec.detach(), outer_max_iter, tol, verbose, eva_iter, metric)
    return x.detach()
