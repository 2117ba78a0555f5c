"""The streamed-frame generic kernel (csrc/specinv_generic_stream.cu) on the GPU: the shapes whose tile (K halo frames
plus one owned frame) does not fit in shared memory, and n_fft up to 32768 (fp32) / 16384 (fp64).

1. One iteration of every op from the oracle's state: x, the state and the metric sums.
2. Routing from torch.profiler kernel names: the streamed kernel runs at these shapes and not at the tile kernels'.
3. Whole runs against the oracle / torchaudio, the differentiable path, determinism, and the refusals."""
import numpy as np
import pytest
import torch

import torchaudio_gl_ref as R
from oracle import specinv_oracle as O

pytestmark = pytest.mark.gpu

STREAM = "stream_tile_kernel"

# (n_fft, hop, dtype): the shapes no tile kernel holds (tests/test_large_frames_host.py pins that), and n_fft > 8192
SHAPES = [(8192, 2048, np.float64), (4096, 512, np.float64), (2048, 128, np.float64), (6000, 750, np.float64),
          (8192, 1024, np.float32), (4096, 256, np.float32), (6000, 375, np.float32),
          (16384, 4096, np.float32), (12000, 3000, np.float32), (32768, 8192, np.float32), (16384, 4096, np.float64)]


def _id(n, h, dt, extra=""):
    return f"{n}-{h}-{'fp64' if dt == np.float64 else 'fp32'}{extra}"


def frames_for(n_fft, hop, B):
    """T that spans at least three CTA ranges (launch_stream: ranges of max(ceil(T / floor(148 / B)), 4 K) frames)."""
    K = (n_fft - 1) // hop
    T = 12 * K + 2
    want = max(1, 148 // B)
    rng = max(-(-T // want), 4 * K)
    assert -(-T // rng) >= 3
    return T


CASES = [pytest.param(n, h, dt, B, frames_for(n, h, B), {}, id=_id(n, h, dt, f"-B{B}"))
         for n, h, dt in SHAPES for B in (1, 3)]
# the options, one shape each; T = 3 < K + 1 = 4 (no range has an owned frame without halo)
CASES += [
    pytest.param(16384, 4096, np.float32, 2, 14, {"onesided": False}, id="two-sided"),
    pytest.param(16384, 4096, np.float32, 1, 14, {"center": False}, id="uncentred"),
    pytest.param(12000, 3000, np.float32, 3, 14, {"pad_mode": "constant"}, id="pad-constant"),
    pytest.param(8192, 2048, np.float64, 1, 14, {"pad_mode": "replicate"}, id="pad-replicate"),
    pytest.param(32768, 8192, np.float32, 1, 14, {"pad_mode": "circular"}, id="pad-circular"),
    pytest.param(8192, 2048, np.float64, 3, 14, {"normalized": True}, id="normalized"),
    pytest.param(16384, 4096, np.float32, 2, 14, {"win_length": 12000}, id="short-window"),
    pytest.param(16384, 4096, np.float32, 1, 3, {"pad_mode": "constant"}, id="T-below-K+1"),
]


def close(a, b, tol, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()))
    err = float(np.abs(a - b).max())
    assert err <= tol * scale, (what, err, tol * scale)


def make_case(n_fft, hop, dtype, B, T, opts, seed=0):
    """(kwargs for the package, oracle args, C, mag, x): a consistent spectrogram with random phases."""
    rs = np.random.RandomState(seed)
    opts = dict(opts)
    wl = opts.pop("win_length", n_fft)
    w = (0.54 - 0.46 * np.cos(2 * np.pi * np.arange(wl) / wl)).astype(dtype)    # Hamming: no zero envelope
    kw = dict(window=w, hop_length=hop, win_length=wl, **opts)
    F = n_fft if opts.get("onesided", True) is False else n_fft // 2 + 1
    oa = O.args_helper(F, dtype, **kw)
    assert oa.n_fft == n_fft
    L = oa.signal_length(T)
    mag = np.abs(O.stft(rs.randn(B, L).astype(dtype), oa)).astype(dtype)
    assert mag.shape == (B, F, T)
    C = (mag * np.exp(2j * np.pi * rs.rand(*mag.shape))).astype(np.complex128 if dtype == np.float64 else np.complex64)
    return kw, oa, C, mag


def tkw(kw):
    return {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}


def plan_for(kw, mag):
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    magt = torch.from_numpy(mag).cuda()
    return StftPlan(args_helper(magt, **tkw(kw)), mag.shape[2], mag.shape[0], magt.dtype, torch.device("cuda")), magt


@pytest.mark.parametrize("n_fft,hop,dtype,B,T,opts", CASES)
def test_one_iteration_from_the_oracles_state(n_fft, hop, dtype, B, T, opts):
    from spectrogram_inversion_b200 import _lib, _ops
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver
    kw, oa, C, mag = make_case(n_fft, hop, dtype, B, T, opts)
    plan, magt = plan_for(kw, mag)
    tol = 1e-10 if dtype == np.float64 else 1e-5
    rel = 1e-10 if dtype == np.float64 else 1e-4
    Cs = plan.pack(torch.from_numpy(C))
    close(plan.unpack(Cs), C, 0.0, "pack / unpack")
    xo, env = O.istft(C, oa)
    assert np.isfinite(xo).all()
    close(plan.istft(Cs), xo, tol, "istft")
    close(plan.unpack(plan.stft(torch.from_numpy(xo).cuda())), O.stft(xo, oa), tol, "stft")

    def check_sums(d, e, s_mag, what):
        do, eo, _ = O.metric_sums(s_mag, mag)
        assert abs(d - do) <= rel * do and abs(e - eo) <= rel * eo, (what, d, do, e, eo)

    # GL, momentum 0.99 and plain (alpha 0)
    for alpha in (0.99, 0.0):
        solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), alpha)
        st = O.gl_init(C, oa)
        solver.x[solver.cur].copy_(torch.from_numpy(st.x))
        d, e = solver.step(evaluate=True)
        st = O.gl_step(st, mag, alpha / (1 + alpha), oa)
        close(solver.signal, st.x, tol, f"GL alpha {alpha} x")
        if alpha:
            close(plan.unpack(solver.q_state), st.q, tol, "GL q")
        check_sums(d, e, st.out_mag, f"GL alpha {alpha}")

    # GLR (torchaudio's recurrence): state out = s = STFT(x), x_out = ISTFT(proj(s - m s_prev))
    m = 0.99 / 1.99
    rs = np.random.RandomState(1)
    s_prev = (C * np.exp(2j * np.pi * rs.rand(*C.shape))).astype(C.dtype)
    x_in = torch.from_numpy(xo).cuda()
    x_out = torch.full_like(x_in, float("nan"))
    s_in, s_out = plan.pack(torch.from_numpy(s_prev)), plan.empty_spec()
    mg = plan.pack(magt)
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    _ops.iter_direct(_lib.lib().specinv_gl_rebuilt_iter, "gl_rebuilt_iter", plan.device, plan.desc_ref,
                     _ops.pointers((plan.buf, x_in, x_out, s_in.main, s_in.nyq, s_out.main, s_out.nyq, mg.main, mg.nyq)),
                     m, sums.data_ptr())
    s = O.stft(xo, oa)
    x_ref, _ = O.istft(O.project(s - s_prev * oa.window.dtype.type(m), mag), oa, env)
    close(x_out, x_ref, tol, "GLR x")
    close(plan.unpack(s_out), s, tol, "GLR state")
    d, e = sums.tolist()
    check_sums(d, e, np.abs(s), "GLR")

    # ADMM
    solver = ADMMSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.1)
    st = O.admm_init(C, oa)
    rs = np.random.RandomState(2)
    st.U = (0.1 * C * np.exp(2j * np.pi * rs.rand(*C.shape))).astype(C.dtype)
    i = solver.cur
    solver.x[i].copy_(torch.from_numpy(st.x))
    solver.U[i] = plan.pack(torch.from_numpy(st.U))
    d, e = solver.step(evaluate=True)
    X0, U0 = st.X, st.U
    st = O.admm_step(st, mag, 0.1, oa)
    close(solver.signal, st.x, tol, "ADMM x")
    close(plan.unpack(solver.U[solver.cur]), st.U, tol, "ADMM U")
    # X = proj(q), q = Z - U: an error dq of q turns the phase by dq / |q|, so X is compared within
    # tol * scale * (1 + mag / |q|) (the projection's condition number)
    q = (X0 + U0 - st.U) - st.U
    Xg = plan.unpack(solver.X[solver.cur]).cpu().numpy()
    scale = max(1.0, float(np.abs(st.X).max()))
    bound = tol * scale * (1 + mag / np.maximum(np.abs(q), 1e-30))
    assert (np.abs(Xg - st.X) <= bound).all(), ("ADMM X", float((np.abs(Xg - st.X) / bound).max()))
    check_sums(d, e, st.out_mag, "ADMM")


ROUTED = [(n, h, dt, True) for n, h, dt in SHAPES] + [
    (8192, 2048, np.float32, False), (4096, 1024, np.float64, False), (400, 100, np.float32, False),
    (1024, 256, np.float32, False)]

_ROUTING_CHILD = """
import json, sys
import numpy as np, torch
from torch.profiler import ProfilerActivity, profile
from tests.test_gpu_large_frames import ROUTED, frames_for, make_case, plan_for
from spectrogram_inversion_b200.engine import GriffinLimSolver
out = []
for n_fft, hop, dtype, _ in ROUTED:
    kw, _, C, mag = make_case(n_fft, hop, dtype, 2, frames_for(n_fft, hop, 2), {})
    plan, magt = plan_for(kw, mag)
    solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.99)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        solver.step(evaluate=True)
        torch.cuda.synchronize()
    out.append(sorted({e.name for e in prof.events() if e.device_type.name == "CUDA"}))
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def routed_kernels():
    """Kernel names of one GL iteration per ROUTED shape, profiled in a child process (a profiler session leaves
    state behind that would hide kernels from later sessions of this process)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.path.join(root, "tests", "golden")]))
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", _ROUTING_CHILD], cwd=root, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("i", range(len(ROUTED)), ids=[_id(n, h, dt) for n, h, dt, _ in ROUTED])
def test_routing(i, routed_kernels):
    names = routed_kernels[i]
    assert any(STREAM in n for n in names) == ROUTED[i][3], names


def _sc(x, mag, oa):
    d, _, g = O.metric_sums(np.abs(O.stft(x, oa)), mag)
    return float(np.sqrt(d / g))


def test_griffin_lim_whole_run_fp32_16384():
    import spectrogram_inversion_b200 as S
    kw, oa, C, mag = make_case(16384, 4096, np.float32, 2, 30, {}, seed=3)
    y = S.griffin_lim(torch.from_numpy(C).cuda(), max_iter=50, tol=0, alpha=0.99, verbose=False, **tkw(kw))
    yo = O.griffin_lim(C, max_iter=50, tol=0, alpha=0.99, verbose=False, **kw)
    sc, sco = _sc(y.cpu().numpy(), mag, oa), _sc(yo, mag, oa)
    assert abs(sc / sco - 1) <= 0.01, (sc, sco)


def test_admm_whole_run_fp64_8192():
    import spectrogram_inversion_b200 as S
    kw, oa, C, mag = make_case(8192, 2048, np.float64, 2, 40, {}, seed=4)
    y = S.ADMM(torch.from_numpy(C).cuda(), max_iter=30, tol=0, rho=0.1, verbose=False, **tkw(kw))
    yo = O.ADMM(C, max_iter=30, tol=0, rho=0.1, verbose=False, **kw)
    sc, sco = _sc(y.cpu().numpy(), mag, oa), _sc(yo, mag, oa)
    assert abs(sc / sco - 1) <= 0.01, (sc, sco)


def _powered_spec(n_fft, hop, B, T, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, (T - 1) * hop, device="cuda", generator=g)
    x = torch.nn.functional.avg_pool1d(x[:, None], 5, 1, 2)[:, 0]
    return R.stft(x, torch.hann_window(n_fft, device="cuda"), n_fft, hop, n_fft).abs().pow(2).contiguous()


@pytest.mark.parametrize("n_iter", [1, 2, 32])
def test_torchaudio_compat_griffinlim_16384(n_iter):
    """Final spectral convergence within 1 % of torchaudio's on CUDA (same seed).  Sample for sample, short runs are
    held to the float64 restatement from the same start phases: torchaudio's own float32 waveform is 4e-3 of the peak
    away from it at this shape (the projection a / |a| amplifies the float32 rounding of small bins)."""
    from spectrogram_inversion_b200 import torchaudio_compat as TC
    try:
        import torchaudio.functional as TAF
        ta_griffinlim = TAF.griffinlim
    except Exception:  # pragma: no cover - the restatement is bit for bit torchaudio's code
        ta_griffinlim = R.griffinlim
    n_fft, hop = 16384, 4096
    spec = _powered_spec(n_fft, hop, 2, 40, 5)
    w = torch.hann_window(n_fft, device="cuda")
    torch.manual_seed(11)
    ours = TC.griffinlim(spec, w, n_fft, hop, n_fft, 2.0, n_iter, 0.99, None, True)
    torch.manual_seed(11)
    ref = ta_griffinlim(spec, w, n_fft, hop, n_fft, 2.0, n_iter, 0.99, None, True)
    assert ours.shape == ref.shape
    mag = spec.sqrt()
    if n_iter <= 2:
        torch.manual_seed(11)
        angles = R.start_angles(mag, True).to(torch.complex128)
        r64 = R.loop(mag.double(), angles, w.double(), n_fft, hop, n_fft, n_iter, 0.99, None)
        assert float((ours.double() - r64).abs().max()) <= 1e-4 * float(r64.abs().max())
    sc_o = R.spectral_convergence(ours, mag, w, n_fft, hop, n_fft)
    sc_r = R.spectral_convergence(ref, mag, w, n_fft, hop, n_fft)
    assert abs(sc_o / sc_r - 1) <= 0.01, (sc_o, sc_r)


def test_griffin_lim_gradient_fp64_8192():
    """griffin_lim with requires_grad (autograd.py: the differentiable transforms run the streamed kernel) against
    the same two iterations restated with float64 torch.stft / torch.istft."""
    import spectrogram_inversion_b200 as S
    n_fft, hop, B, T = 8192, 2048, 2, 20
    kw, oa, C, mag = make_case(n_fft, hop, np.float64, B, T, {}, seed=6)
    w = torch.from_numpy(kw["window"]).cuda()
    spec = torch.from_numpy(C).cuda().requires_grad_()
    y = S.griffin_lim(spec, max_iter=2, tol=0, alpha=0.99, verbose=False, window=w, hop_length=hop)
    g = torch.Generator(device="cuda").manual_seed(7)
    gy = torch.randn(y.shape, dtype=torch.float64, device="cuda", generator=g)
    (gs,) = torch.autograd.grad(y, spec, gy)

    spec2 = torch.from_numpy(C).cuda().requires_grad_()
    magt = spec2.abs()
    L = (T - 1) * hop

    def istft(S_):
        return torch.istft(S_, n_fft, hop, n_fft, w, center=True, length=L)

    def stft(x):
        return torch.stft(x, n_fft, hop, n_fft, w, center=True, pad_mode="reflect", return_complex=True)

    lr = 0.99 / 1.99
    q = spec2
    x = istft(spec2)
    for _ in range(2):
        s = stft(x)
        q = s - lr * q
        x = istft(magt * q / (q.abs() + 1e-16))
    (gr,) = torch.autograd.grad(x, spec2, gy)
    assert float((y.detach() - x.detach()).abs().max()) <= 1e-10 * float(x.abs().max())
    assert float((gs - gr).abs().max()) <= 1e-8 * float(gr.abs().max())


def test_runs_are_bit_identical():
    from spectrogram_inversion_b200.engine import GriffinLimSolver
    kw, _, C, mag = make_case(32768, 8192, np.float32, 3, 40, {}, seed=8)
    plan, magt = plan_for(kw, mag)
    outs = []
    for _ in range(2):
        solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.99)
        for _ in range(3):
            solver.step()
        outs.append((solver.signal.clone(), solver.q_state.main.clone(), solver.q_state.nyq.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_phase_init_and_pack_at_16384():
    from tests.test_gpu_phase_init import check_against_oracle, fused
    g = torch.Generator(device="cuda").manual_seed(9)
    for dtype in (torch.float32, torch.float64):
        magt = torch.rand(2, 8193, 50, generator=g, device="cuda", dtype=dtype)
        check_against_oracle(fused(magt, 4096), magt, 4096, True, f"phase_init 16384 {dtype}")


def test_refusals():
    import spectrogram_inversion_b200 as S
    mag = torch.rand(1, 8193, 12, device="cuda")
    with pytest.raises(NotImplementedError):
        S.RTISI_LA(mag, max_iter=2, verbose=0)
    with pytest.raises(NotImplementedError):          # one fp64 frame of 32768 does not fit in shared memory
        S.griffin_lim(torch.rand(1, 16385, 12, device="cuda", dtype=torch.float64), max_iter=2, verbose=False)
    with pytest.raises(NotImplementedError):          # over the limit
        S.griffin_lim(torch.rand(1, 16386, 12, device="cuda"), max_iter=2, verbose=False)
    with pytest.raises(NotImplementedError):          # half = 8193 = 3 * 2731
        S.griffin_lim(torch.rand(1, 8194, 12, device="cuda"), max_iter=2, verbose=False)
