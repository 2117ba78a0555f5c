"""Differentiable path (SURVEY.md section 8f, row 2).

The reference's outputs are differentiable with respect to ``spec`` -- its tests call ``.backward()``
(test/test_griffin.py:54,65-66).  The fused iteration kernels are forward only, so when the caller asks for
gradients (``spec.requires_grad`` under ``torch.enable_grad``) the algorithms run UNFUSED here: the transforms
are this library's own STFT / ISTFT kernels wrapped in ``torch.autograd.Function``s whose backward passes are
again those kernels (the adjoint of an STFT is an un-normalised ISTFT and vice versa); the point-wise updates
between them are ordinary differentiable tensor expressions on the device.  This path follows the reference
op by op (methods.py:237-250, :458-483, :363-404, :572-615); it is not the benchmarked path.

Adjoints (real signal, G = dL/dRe + i dL/dIm, N = n_fft, c_k = 1 for k in {0, N/2}, 2 otherwise):
  S = STFT(xp):    dL/dxp = OLA_t( wa * N * irfft(G / c) )           -> ISTFT kernel on a unit-envelope plan
  x = ISTFT(S):    dL/dS  = c * STFT_ws( zero-pad(dL/dx / env) )     -> STFT kernel
with wa / ws the analysis / synthesis windows (their scale ratio is N, or 1 when ``normalized``); two-sided
spectra use c = 1 (methods.py:145-146)."""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
import torch
import torch.nn.functional as F
from tqdm import tqdm

from . import _lib, _ops
from .engine import METRIC_NAMES, StftPlan, metric_value
from .stft_args import StftArgs

pi2 = 2 * math.pi


def wants_grad(spec: torch.Tensor) -> bool:
    return torch.is_grad_enabled() and spec.requires_grad


def _desc_of(plan: StftPlan):
    a = plan.args
    return _lib.make_desc(a.n_fft, a.hop_length, plan.T, plan.B, a.center, plan.pad_mode, a.normalized, a.onesided,
                          _ops._DT[plan.dtype])


class Transforms:
    """Differentiable ``stft`` / ``istft`` of one (stft args, n_frames, batch) on the CUDA kernels."""

    def __init__(self, args: StftArgs, n_frames: int, batch: int, dtype: torch.dtype, device: torch.device):
        self.args = args
        self.pad = args.pad
        nc = dataclasses.replace(args, center=False)
        self.plan = StftPlan(args, n_frames, batch, dtype, device)          # as the caller sees it
        self.plan_nc = StftPlan(nc, n_frames, batch, dtype, device)         # un-centred, over the padded length
        self.plan_raw = StftPlan(nc, n_frames, batch, dtype, device)        # un-centred, unit envelope: plain OLA
        d = _desc_of(self.plan_raw)
        stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().specinv_plan_unit_envelope(C.byref(d), C.c_void_p(self.plan_raw.buf.data_ptr()),
                                                             stream), "plan_unit_envelope")
            self.env = torch.empty(self.plan.length, dtype=dtype, device=device)
            d2 = _desc_of(self.plan)
            _lib.check(_lib.lib().specinv_plan_envelope(C.byref(d2), C.c_void_p(self.plan.buf.data_ptr()),
                                                        C.c_void_p(self.env.data_ptr()), stream), "plan_envelope")
        n = args.n_fft
        self.ratio = 1.0 if args.normalized else float(n)                   # analysis scale / synthesis scale
        F_ = args.n_bins
        c = torch.ones(F_, dtype=dtype, device=device)
        if args.onesided:
            c[1:n // 2] = 2.0
        self.c = c[None, :, None]

    # -- raw kernels on (B, F, T) tensors -------------------------------------------------------------
    def _stft_nc(self, xp: torch.Tensor) -> torch.Tensor:
        return self.plan_nc.unpack(self.plan_nc.stft(xp.contiguous()))

    def _istft_raw(self, spec: torch.Tensor) -> torch.Tensor:
        return self.plan_raw.istft(self.plan_raw.pack(spec))

    def _istft(self, spec: torch.Tensor) -> torch.Tensor:
        return self.plan.istft(self.plan.pack(spec))

    # -- differentiable transforms ---------------------------------------------------------------------
    def stft(self, x: torch.Tensor) -> torch.Tensor:
        """torch.stft(x, **args) (methods.py:241): the centre padding is torch's own (differentiable) pad, the
        transform of the padded signal is the kernel."""
        if self.pad:
            x = F.pad(x[:, None, :], (self.pad, self.pad), mode=self.args.pad_mode)[:, 0, :]
        return _StftFn.apply(x, self)

    def istft(self, spec: torch.Tensor) -> torch.Tensor:
        """_istft (methods.py:135-150)."""
        return _IstftFn.apply(spec, self)


class _StftFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xp, tr: Transforms):
        ctx.tr = tr
        return tr._stft_nc(xp.detach())

    @staticmethod
    def backward(ctx, g):
        tr = ctx.tr
        return tr._istft_raw(g / tr.c) * tr.ratio, None


class _IstftFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec, tr: Transforms):
        ctx.tr = tr
        return tr._istft(spec.detach())

    @staticmethod
    def backward(ctx, gx):
        tr = ctx.tr
        gp = gx / tr.env
        if tr.pad:
            gp = F.pad(gp, (tr.pad, tr.pad))
        return tr._stft_nc(gp) * (tr.c / tr.ratio), None


# ---------------------------------------------------------------------------------------------------------
def phase_init_diff(spec: torch.Tensor, n_fft: int, hop: int) -> torch.Tensor:
    """phase_init (methods.py:572-615) as dense differentiable tensor expressions: a bin takes the frequency of
    the peak below it, else of the peak above it, else its own (the reference's write order :607-609).

    The arithmetic is the reference's CPU arithmetic: a true division by n_fft (a CUDA tensor divided by a
    Python number is a multiplication by its reciprocal, which differs in the last bit when n_fft is not a
    power of two), and the running phase summed in float64 and rounded to the input dtype (torch's CPU cumsum
    accumulates float32 in float64; a float32 sum drifts by radians over a few thousand frames)."""
    lo, mid, hi = spec[:, :-2], spec[:, 1:-1], spec[:, 2:]
    peak = (mid > hi) & (mid > lo)
    den = torch.where(peak, lo - 2 * mid + hi, torch.ones_like(mid))
    p = 0.5 * (lo - hi) / den
    k = torch.arange(1, spec.shape[1] - 1, device=spec.device, dtype=spec.dtype)[None, :, None]
    n = torch.tensor(n_fft, device=spec.device, dtype=spec.dtype)
    own = torch.where(peak, pi2 * (k + p) / n * hop, torch.zeros_like(mid))
    own = F.pad(own, [0, 0, 1, 1])
    pk = F.pad(peak, [0, 0, 1, 1])
    up, pk_up = F.pad(own[:, 1:], [0, 0, 0, 1]), F.pad(pk[:, 1:], [0, 0, 0, 1])        # the bin above
    dn, pk_dn = F.pad(own[:, :-1], [0, 0, 1, 0]), F.pad(pk[:, :-1], [0, 0, 1, 0])      # the bin below
    omega = torch.where(pk_dn, dn, torch.where(pk_up, up, own))
    phase = torch.cumsum(omega.double(), 2).to(spec.dtype)
    return spec * torch.exp(phase * 1j)


def _format(spec: torch.Tensor, args: StftArgs):
    """_spec_formatter (methods.py:99-111) on the device."""
    if spec.is_complex():
        return spec, spec.abs()
    return phase_init_diff(spec, args.n_fft, args.hop_length), spec


def _loop(closure, target: torch.Tensor, max_iter: int, tol: float, verbose, eva_iter: int, metric: str) -> None:
    """_training_loop (methods.py:153-190); the evaluation reads three sums like the fused path."""
    metric = metric.upper()
    assert metric in METRIC_NAMES
    init_loss = previous = None
    g = float((target.detach().double() ** 2).sum())
    n = target.numel()
    with tqdm(total=max_iter, disable=not verbose) as pbar:
        for i in range(max_iter):
            out = closure()
            if i % eva_iter == eva_iter - 1:
                with torch.no_grad():
                    d = float(((out.double() - target.double()) ** 2).sum())
                    e = float((out.double() ** 2).sum())
                loss = d / n
                pbar.set_postfix(**{metric: metric_value(metric, d, e, g)}, loss=loss)
                pbar.update(eva_iter)
                if not init_loss:
                    init_loss = loss
                elif (previous - loss) / init_loss < tol and previous > loss:
                    break
                previous = loss


def griffin_lim_diff(work: torch.Tensor, args: StftArgs, max_iter, tol, alpha, verbose, eva_iter, metric):
    """griffin_lim (methods.py:225-265) with differentiable transforms; ``work`` is (B, F, T) on the device."""
    B, _, T = work.shape
    tr = Transforms(args, T, B, args.window.dtype, work.device)
    cmplx, target = _format(work, args)
    st = {"x": tr.istft(cmplx), "pre": cmplx.clone()}
    lr = alpha / (1 + alpha)

    def closure():
        new_spec = tr.stft(st["x"])
        output = new_spec.abs()
        new_spec = new_spec - st["pre"] * lr
        st["pre"] = new_spec
        new_spec = new_spec * target / (new_spec.abs() + 1e-16)
        st["x"] = tr.istft(new_spec)
        return output

    _loop(closure, target, max_iter, tol, verbose, eva_iter, metric)
    return st["x"]


def admm_diff(work: torch.Tensor, args: StftArgs, max_iter, tol, rho, verbose, eva_iter, metric):
    """ADMM (methods.py:445-501) with differentiable transforms."""
    B, _, T = work.shape
    tr = Transforms(args, T, B, args.window.dtype, work.device)
    X, target = _format(work, args)
    st = {"X": X, "Y": X.clone(), "U": torch.zeros_like(X), "x": tr.istft(X)}

    def closure():
        rec = tr.stft(st["x"])
        output = rec.abs()
        Z = (rho * st["Y"] + rec) / (1 + rho)
        U = st["U"] + st["X"] - Z
        Xn = Z - U
        Xn = Xn * target / (Xn.abs() + 1e-16)
        Y = Xn + U
        st.update(X=Xn, Y=Y, U=U, x=tr.istft(Y))
        return output

    _loop(closure, target, max_iter, tol, verbose, eva_iter, metric)
    return st["x"]


def rtisi_diff(work: torch.Tensor, args: StftArgs, look_ahead, asymmetric_window, max_iter, alpha, verbose):
    """RTISI_LA (methods.py:305-408) with differentiable transforms.  Frame-wise rfft / irfft are the STFT /
    ISTFT kernels on a rectangular window with hop = n_fft (frames laid end to end); the overlap-adds of the
    handful of buffered frames are ``F.fold`` (they are (K + LA + 1)-frame tensors, not the signal)."""
    B, _, T = work.shape
    n, hop, dev, dt = args.n_fft, args.hop_length, work.device, args.window.dtype
    window = args.window
    synth = hop / (window @ window)
    K = (args.win_length - 1) // hop
    LA = K if look_ahead < 0 else int(look_ahead)
    NA = LA + 1
    ones = torch.ones(n, dtype=dt, device=dev)
    rect = dataclasses.replace(args, hop_length=n, window=ones, center=False, win_length=n)
    fr = Transforms(rect, NA, B, dt, dev)                 # rfft / irfft of NA frames laid end to end
    fr1 = Transforms(rect, 1, B, dt, dev)
    nc = dataclasses.replace(args, center=False)
    st_nc = Transforms(nc, NA, B, dt, dev)                # torch.stft(x, center=False) of the (LA hop + n) buffer

    def irfft(spec, t):                                   # (B, F, nf) -> (B, n, nf)
        return t.istft(spec).reshape(B, spec.shape[2], n).transpose(1, 2)

    def rfft(frames, t):                                  # (B, n, nf) -> (B, F, nf)
        return t.stft(frames.transpose(1, 2).reshape(B, -1))

    def ola(frames, weight):                              # _ola with padding=0, norm_envelope=1 (methods.py:114-132)
        nf = frames.shape[2]
        return F.fold(frames * weight[None, :, None], (1, (nf - 1) * hop + n), (1, n), stride=(1, hop))[:, 0, 0]

    flip = window.flip(0)
    asym1, asym2 = torch.zeros_like(window), torch.zeros_like(window)
    for i in range(K):
        asym1[(i + 1) * hop:] += flip[:n - (i + 1) * hop]
    for i in range(K + 1):
        asym2[i * hop:] += flip[:n - i * hop]
    asym1, asym2 = asym1 * synth, asym2 * synth

    target = F.pad(work, [LA, LA])
    kept = work.new_zeros(B, n, K)
    update = torch.cat((work.new_zeros(B, n, LA), irfft(target[..., LA, None] + 0j, fr1)), 2)
    lr = alpha / (1 + alpha)
    commits = []
    pre = None
    with tqdm(total=T + LA, disable=not verbose) as pbar:
        for i in range(T + LA):
            for j in range(max_iter):
                x = ola(torch.cat((kept, update), 2), window * synth)[:, K * hop:]
                if asymmetric_window:
                    view = x.unfold(1, n, hop).transpose(1, 2)
                    last = view[:, :, -1:] * (asym2 if j else asym1)[:, None]
                    new_spec = rfft(torch.cat((view[:, :, :-1] * window[:, None], last), 2), fr)
                else:
                    new_spec = st_nc.stft(x)
                if j:
                    new_spec = new_spec - lr * pre
                elif i:
                    new_spec = torch.cat((new_spec[:, :, :-1] - lr * pre[:, :, 1:], new_spec[:, :, -1:]), 2)
                pre = new_spec
                new_spec = new_spec * target[..., i:i + NA] / (new_spec.abs() + 1e-16)
                update = irfft(new_spec, fr)
            pbar.update()
            commits.append(update[:, :, 0])
            kept = torch.cat((kept[:, :, 1:], update[:, :, :1]), 2)
            update = F.pad(update[:, :, 1:], [0, 1])
    frames = torch.stack(commits[LA:], 2)
    nf = frames.shape[2]
    y = F.fold(frames * window[None, :, None], (1, (nf - 1) * hop + n), (1, n), stride=(1, hop))[:, 0, 0]
    env = F.fold((window * window)[None, :, None].expand(1, n, nf), (1, (nf - 1) * hop + n), (1, n), stride=(1, hop))[:, 0, 0]
    P = args.pad
    if P:
        y, env = y[:, P:-P], env[:, P:-P]
    return y / env
