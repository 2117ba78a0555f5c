"""GPU parity: the CUDA kernels (through the C ABI / torch.library ops) against the numpy oracle
and against the golden vectors produced by the unmodified reference.

Tolerances: BASELINE.json north_star -- single-iteration max-abs <= 1e-5 in fp32 from identical
state (scaled by max(1, |x|max)); fp64 is held to 1e-10."""
import os

import numpy as np
import pytest
import torch

import cases
from oracle import specinv_oracle as O

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(__file__), "golden")
GL = np.load(os.path.join(G, "gl.npz"))
ADMM = np.load(os.path.join(G, "admm.npz"))
PRIM = np.load(os.path.join(G, "primitives.npz"))
LOOP = np.load(os.path.join(G, "loop.npz"))
MISC = np.load(os.path.join(G, "misc.npz"))
RTISI = np.load(os.path.join(G, "rtisi.npz"))


def tol_of(dtype):
    return 1e-10 if np.dtype(dtype) == np.float64 else 1e-5


def close(a, b, tol, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    fin = np.isfinite(b)
    assert (np.isfinite(a) == fin).all(), what
    scale = max(1.0, float(np.abs(b[fin]).max())) if fin.any() else 1.0
    err = float(np.abs(a[fin] - b[fin]).max()) if fin.any() else 0.0
    assert err <= tol * scale, (what, err, tol * scale)


def build(case):
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    inp = cases.make_case_inputs(case)
    C = inp["C"] if inp["C"].ndim == 3 else inp["C"][None]
    mag = inp["mag"] if inp["mag"].ndim == 3 else inp["mag"][None]
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    dev = torch.device("cuda")
    magt = torch.from_numpy(mag).to(dev)
    args = args_helper(magt, **kw)
    plan = StftPlan(args, mag.shape[2], mag.shape[0], magt.dtype, dev)
    oa = O.args_helper(mag.shape[1], mag.dtype, **inp["kwargs"])
    return inp, C, mag, plan, oa


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_stft_istft_primitives(case, generic_kernel):
    inp, C, mag, plan, oa = build(case)
    name = case["name"]
    tol = tol_of(case["dtype"])
    Cs = plan.pack(torch.from_numpy(C))
    close(plan.unpack(Cs), C, 0.0, "pack/unpack round trip")
    x = plan.istft(Cs)
    close(x, PRIM[f"{name}/istft_x"], tol, "istft vs reference")
    xo, env = O.istft(C, oa)
    close(x, xo, tol, "istft vs oracle")
    if np.isfinite(xo).all():
        S = plan.unpack(plan.stft(torch.from_numpy(xo).cuda()))
        close(S, O.stft(xo, oa), tol * 10, "stft vs oracle")
        if f"{name}/stft_of_x" in PRIM:
            close(S, PRIM[f"{name}/stft_of_x"], tol * 20, "stft vs reference")


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_griffin_lim_iterations_from_identical_state(case, generic_kernel):
    from spectrogram_inversion_b200.engine import GriffinLimSolver
    inp, C, mag, plan, oa = build(case)
    tol = tol_of(case["dtype"])
    for alpha in cases.GL_ALPHAS:
        solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(torch.from_numpy(mag)), alpha)
        st = O.gl_init(C, oa)
        close(solver.signal, st.x, tol, "x0")
        for k in (1, 2, 3):
            # restart the CUDA step from the ORACLE's state so every step is a single-iteration test
            solver.x[solver.cur].copy_(torch.from_numpy(st.x))
            if not solver.plain:      # alpha = 0: no momentum state at all (NULL q pointers through the ABI)
                solver.q[solver.cur] = plan.pack(torch.from_numpy(st.q))
                solver.q[solver.cur ^ 1] = solver.q[solver.cur].like()
            d, e = solver.step(evaluate=True)
            st = O.gl_step(st, mag, alpha / (1 + alpha), oa)
            close(solver.signal, st.x, tol, f"x after step {k} alpha {alpha}")
            if not solver.plain:
                close(plan.unpack(solver.q_state), st.q, tol * 10, f"q after step {k}")
            do, eo, go = O.metric_sums(st.out_mag, mag)
            rel = 1e-4 if case["dtype"] == "float32" else 1e-10
            assert abs(d - do) <= rel * max(do, 1e-30) + 1e-12 and abs(e - eo) <= rel * eo
            assert abs(solver.g - go) <= rel * go


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_griffin_lim_matches_reference_golden(case, generic_kernel):
    import spectrogram_inversion_b200 as S
    inp = cases.make_case_inputs(case)
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    tol = tol_of(case["dtype"])
    C = torch.from_numpy(inp["C"]).cuda()
    for alpha in cases.GL_ALPHAS:
        for k in cases.ITER_COUNTS:
            y = S.griffin_lim(C, max_iter=k, tol=0, alpha=alpha, verbose=False, eva_iter=1, **kw)
            assert y.is_cuda
            close(y, GL[f"{case['name']}/a{alpha}/k{k}"], tol * (4 ** (k - 1)), f"a{alpha} k{k}")


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_admm_iterations_and_golden(case, generic_kernel):
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200.engine import ADMMSolver
    inp, C, mag, plan, oa = build(case)
    tol = tol_of(case["dtype"])
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    for rho in cases.ADMM_RHOS:
        solver = ADMMSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(torch.from_numpy(mag)), rho)
        st = O.admm_init(C, oa)
        for k in (1, 2, 3):
            i = solver.cur
            solver.x[i].copy_(torch.from_numpy(st.x))
            solver.X[i] = plan.pack(torch.from_numpy(st.X))
            solver.U[i] = plan.pack(torch.from_numpy(st.U))
            solver.X[i ^ 1] = solver.X[i].like()
            solver.U[i ^ 1] = solver.U[i].like()
            solver.step(evaluate=(k == 2))
            st = O.admm_step(st, mag, rho, oa)
            close(solver.signal, st.x, tol * 2, f"x step {k} rho {rho}")
            # X = proj(2Z - U - X_prev) is a discontinuous map where |2Z - U - X_prev| is small against
            # its terms (cancellation), so fp32 state parity is held looser than the signal parity
            stol = 1e-9 if case["dtype"] == "float64" else 1e-3
            close(plan.unpack(solver.X[solver.cur]), st.X, stol, "X")
            close(plan.unpack(solver.U[solver.cur]), st.U, stol, "U")
        for k in cases.ITER_COUNTS:
            y = S.ADMM(torch.from_numpy(inp["C"]).cuda(), max_iter=k, tol=0, rho=rho, verbose=False, eva_iter=1, **kw)
            close(y, ADMM[f"{case['name']}/r{rho}/k{k}"], tol * 2 * (4 ** (k - 1)), f"r{rho} k{k}")


@pytest.mark.parametrize("case", cases.LOOP_CASES, ids=lambda c: c["name"])
def test_early_stop_like_reference(case):
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, training_loop
    inp, C, mag, plan, oa = build(case)
    for algo in ("gl", "admm"):
        Cs, ms = plan.pack(torch.from_numpy(C)), plan.pack(torch.from_numpy(mag))
        solver = GriffinLimSolver(plan, Cs, ms, 0.99) if algo == "gl" else ADMMSolver(plan, Cs, ms, 0.1)
        hist = []
        n = training_loop(solver, case["max_iter"], case["tol"], False, case["eva_iter"], case["metric"], hist)
        assert n == int(LOOP[f"{case['name']}/{algo}/iters"]), (algo, n)
        close(solver.signal, LOOP[f"{case['name']}/{algo}/x"], 1e-7 if algo == "gl" else 5e-2, algo)


@pytest.mark.parametrize("i", [0, 1])
def test_metrics_like_reference(i):
    import spectrogram_inversion_b200 as S
    a, b = MISC[f"metric{i}/a"], MISC[f"metric{i}/b"]
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    rel = 1e-5 if i == 0 else 1e-12
    for fn in ("sc", "snr", "ser"):
        got = getattr(S, fn)(ta, tb)
        assert got.ndim == 0 and got.is_cuda and got.dtype == ta.dtype
        want = float(MISC[f"metric{i}/{fn}"])
        assert abs(float(got) - want) <= rel * max(1.0, abs(want)), (fn, float(got), want)
    assert S.spectral_convergence is S.sc
    # host tensors are staged through the GPU and come back on the host
    assert not S.sc(torch.from_numpy(a), torch.from_numpy(b)).is_cuda


def test_public_api_shapes_and_asserts():
    import spectrogram_inversion_b200 as S
    for shape in [(4410,), (2, 4410), (1, 4410)]:
        for dtype in (torch.float32, torch.float64):
            x = torch.randn(*shape, dtype=dtype, device="cuda")
            spec = torch.stft(x, 256, return_complex=True, window=torch.ones(256, dtype=dtype, device="cuda"))
            for fn in (S.griffin_lim, S.ADMM):
                y = fn(spec, max_iter=4, verbose=False)
                assert y.ndim == x.ndim and y.dtype == dtype and y.is_cuda
                if y.ndim > 1:
                    assert y.shape[0] == x.shape[0] and y.shape[1] <= x.shape[1]
    spec = torch.stft(torch.randn(2048, device="cuda"), 128, return_complex=True,
                      window=torch.hann_window(128, device="cuda"))
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, alpha=-1)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, max_iter=0)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, eva_iter=0)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, tol=-1)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, metric="nope")
    with pytest.raises(AssertionError):
        S.ADMM(spec, metric="nope")
    with pytest.raises(AssertionError):
        S.RTISI_LA(spec)                     # complex input is rejected (methods.py:297)
    with pytest.raises(AssertionError):
        S.RTISI_LA(spec.abs(), max_iter=0)
    # host input -> host output (staged through the GPU, never computed on the CPU)
    y = S.griffin_lim(spec.cpu(), max_iter=2, verbose=False, window=torch.hann_window(128), maxiter=3)
    assert not y.is_cuda


def test_full_run_spectral_convergence_within_1pct():
    """north_star: final spectral convergence after the full iteration count within 1 % of the
    reference's (here: of the oracle's, which is pinned to the reference)."""
    import spectrogram_inversion_b200 as S
    rs = np.random.RandomState(3)
    x = rs.randn(4, 48000).astype(np.float32)
    w = cases.window_of("hann", 256, np.float32)
    a = O.args_helper(129, np.float32, window=w, hop_length=64)
    mag = np.abs(O.stft(x, a))
    C = (mag * np.exp(2j * np.pi * rs.rand(*mag.shape))).astype(np.complex64)
    for algo, kw in (("griffin_lim", dict(alpha=0.99)), ("ADMM", dict(rho=0.1))):
        yo = getattr(O, algo)(C, max_iter=64, tol=0, window=w, hop_length=64, **kw)
        yg = getattr(S, algo)(torch.from_numpy(C).cuda(), max_iter=64, tol=0, verbose=False,
                              window=torch.from_numpy(w).cuda(), hop_length=64, **kw)
        sco = O.sc(np.abs(O.stft(yo, a)), mag)
        scg = O.sc(np.abs(O.stft(yg.cpu().numpy(), a)), mag)
        # 1 % on the linear spectral-convergence ratio == 0.0864 dB
        assert abs(scg - sco) <= 20 * np.log10(1.01) + 0.05 * abs(sco) * 0, (algo, scg, sco)


# ---------------------------------------------------------------------------------------------
# fast path (n_fft = 1024, hop = 256): many frames, several chunks per signal, every edge mode
# ---------------------------------------------------------------------------------------------
FAST_CASES = [
    dict(B=3, T=101, center=True, pad_mode="reflect", normalized=False, window="hann"),
    dict(B=2, T=57, center=True, pad_mode="constant", normalized=True, window="hann"),
    dict(B=2, T=40, center=True, pad_mode="replicate", normalized=False, window="hamming"),
    dict(B=1, T=333, center=True, pad_mode="circular", normalized=False, window="hann"),
    dict(B=5, T=64, center=False, pad_mode="reflect", normalized=False, window="hamming"),
    dict(B=2, T=30, center=True, pad_mode="reflect", normalized=False, window=None, win_length=700),
]


@pytest.mark.parametrize("fc", FAST_CASES, ids=lambda c: f"B{c['B']}_T{c['T']}_{c['pad_mode']}_c{int(c['center'])}")
def test_fast_path_1024_against_oracle(fc):
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    rs = np.random.RandomState(fc["T"])
    n_fft, hop = 1024, 256
    B, T = fc["B"], fc["T"]
    kw = dict(hop_length=hop, center=fc["center"], pad_mode=fc["pad_mode"], normalized=fc["normalized"])
    wl = fc.get("win_length", n_fft)
    if fc["window"] is not None:
        kw["window"] = cases.window_of(fc["window"], wl, np.float32)
    if wl != n_fft:
        kw["win_length"] = wl
    oa = O.args_helper(n_fft // 2 + 1, np.float32, **kw)
    mag = (np.abs(rs.randn(B, 513, T) + 1j * rs.randn(B, 513, T)) * 8).astype(np.float32)
    C = (mag * np.exp(2j * np.pi * rs.rand(B, 513, T))).astype(np.complex64)
    tkw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    magt = torch.from_numpy(mag).cuda()
    plan = StftPlan(args_helper(magt, **tkw), T, B, torch.float32, torch.device("cuda"))

    # Griffin-Lim, three single steps each restarted from the oracle's state
    solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.99)
    st = O.gl_init(C, oa)
    close(solver.signal, st.x, 1e-5, "fast ISTFT (x_0)")
    for k in range(3):
        solver.x[solver.cur].copy_(torch.from_numpy(st.x))
        solver.q[solver.cur] = plan.pack(torch.from_numpy(st.q))
        solver.q[solver.cur ^ 1] = solver.q[solver.cur].like()
        out = solver.step(evaluate=(k != 1))
        st = O.gl_step(st, mag, 0.99 / 1.99, oa)
        close(solver.signal, st.x, 1e-5, f"fast GL x step {k}")
        close(plan.unpack(solver.q_state), st.q, 1e-4, f"fast GL q step {k}")
        if out is not None:
            do, eo, _ = O.metric_sums(st.out_mag, mag)
            assert abs(out[0] - do) <= 1e-4 * do and abs(out[1] - eo) <= 1e-4 * eo

    # ADMM
    solver = ADMMSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.1)
    st = O.admm_init(C, oa)
    for k in range(2):
        i = solver.cur
        solver.x[i].copy_(torch.from_numpy(st.x))
        solver.X[i] = plan.pack(torch.from_numpy(st.X)); solver.U[i] = plan.pack(torch.from_numpy(st.U))
        solver.X[i ^ 1] = solver.X[i].like(); solver.U[i ^ 1] = solver.U[i].like()
        solver.step(evaluate=(k == 1))
        st = O.admm_step(st, mag, 0.1, oa)
        close(solver.signal, st.x, 2e-5, f"fast ADMM x step {k}")
        close(plan.unpack(solver.U[solver.cur]), st.U, 1e-3, "fast ADMM U")


def test_fast_and_generic_kernels_agree(monkeypatch):
    """The specialised 1024/256 kernel and the generic tile kernel are two implementations of the
    same iteration: run 5 free-running iterations with each and compare."""
    from spectrogram_inversion_b200.engine import GriffinLimSolver, StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    rs = np.random.RandomState(5)
    B, T = 4, 200
    mag = (np.abs(rs.randn(B, 513, T) + 1j * rs.randn(B, 513, T)) * 8).astype(np.float32)
    C = (mag * np.exp(2j * np.pi * rs.rand(B, 513, T))).astype(np.complex64)
    w = torch.hann_window(1024, device="cuda")
    magt = torch.from_numpy(mag).cuda()
    plan = StftPlan(args_helper(magt, window=w, hop_length=256), T, B, torch.float32, torch.device("cuda"))
    outs = []
    for force in ("0", "1"):
        monkeypatch.setenv("SPECINV_FORCE_GENERIC", force)
        s = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.99)
        sums = [s.step(evaluate=True) for _ in range(5)]
        outs.append((s.signal.clone(), sums))
    close(outs[0][0], outs[1][0].cpu().numpy(), 2e-4, "fast vs generic after 5 iterations")
    for (d0, e0), (d1, e1) in zip(outs[0][1], outs[1][1]):
        assert abs(d0 - d1) <= 1e-4 * d1 and abs(e0 - e1) <= 1e-4 * e1


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_phase_init_and_magnitude_entry_match_reference(case):
    """Real-magnitude entry: the fused phase_init kernel against the reference's phase_init, and
    griffin_lim(mag) (phase_init inside) against the reference after 2 iterations."""
    import spectrogram_inversion_b200 as S
    inp = cases.make_case_inputs(case)
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    mag = torch.from_numpy(inp["mag"]).cuda()
    f32 = case["dtype"] == "float32"
    pi = S.phase_init(mag, **kw)
    assert pi.shape == mag.shape and pi.is_complex() and pi.is_cuda
    # fp32: the phase reaches O(1e3) rad, so one ulp of phase is ~1e-4 rad of angle error
    close(pi, PRIM[f"{case['name']}/phase_init"], 5e-4 if f32 else 1e-9, "phase_init")
    close(pi, O.phase_init(inp["mag"], **inp["kwargs"]), 5e-4 if f32 else 1e-9, "phase_init vs oracle")
    y = S.griffin_lim(mag, max_iter=2, tol=0, alpha=0.99, verbose=False, **kw)
    close(y, GL[f"{case['name']}/mag_in/k2"], 2e-3 if f32 else 1e-8, "griffin_lim(mag)")


@pytest.mark.parametrize("case", cases.RTISI_CASES, ids=lambda c: c["name"])
def test_rtisi_la_matches_reference(case):
    """Whole RTISI-LA runs (small T, few inner iterations so round-off is not yet amplified) against the
    reference's output and the oracle's."""
    import spectrogram_inversion_b200 as S
    inp = cases.make_case_inputs(case)
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    mag = torch.from_numpy(inp["mag"]).cuda()
    y = S.RTISI_LA(mag, look_ahead=case["look_ahead"], asymmetric_window=case["asym"], max_iter=case["max_iter"],
                   alpha=case["alpha"], verbose=0, **kw)
    f32 = case["dtype"] == "float32"
    close(y, RTISI[case["name"]], 5e-3 if f32 else 1e-7, "vs reference")
    yo = O.RTISI_LA(inp["mag"], look_ahead=case["look_ahead"], asymmetric_window=case["asym"],
                    max_iter=case["max_iter"], alpha=case["alpha"], **inp["kwargs"])
    close(y, yo, 5e-3 if f32 else 1e-7, "vs oracle")


def test_rtisi_la_shapes_and_quality():
    import spectrogram_inversion_b200 as S
    for shape in [(4410,), (2, 4410), (1, 4410)]:
        for dtype in (torch.float32, torch.float64):
            x = torch.randn(*shape, dtype=dtype, device="cuda")
            spec = torch.stft(x, 256, return_complex=True, window=torch.ones(256, dtype=dtype, device="cuda")).abs()
            y = S.RTISI_LA(spec, max_iter=4, verbose=0)
            assert y.ndim == x.ndim and y.dtype == dtype and y.is_cuda
            if y.ndim > 1:
                assert y.shape[0] == x.shape[0] and y.shape[1] <= x.shape[1]
    # a longer run at the cfg3 frame shape: spectral convergence comparable with the oracle's
    rs = np.random.RandomState(1)
    w = cases.window_of("hann", 1024, np.float32)
    a = O.args_helper(513, np.float32, window=w, hop_length=256)
    mag = np.abs(O.stft(rs.randn(2, 12000).astype(np.float32), a))
    yo = O.RTISI_LA(mag, look_ahead=3, max_iter=8, alpha=0.99, window=w, hop_length=256)
    yg = S.RTISI_LA(torch.from_numpy(mag).cuda(), look_ahead=3, max_iter=8, alpha=0.99, verbose=0,
                    window=torch.from_numpy(w).cuda(), hop_length=256)
    sco = O.sc(np.abs(O.stft(yo, a)), mag)
    scg = O.sc(np.abs(O.stft(yg.cpu().numpy(), a)), mag)
    assert abs(scg - sco) <= 0.02 * abs(sco) + 0.2, (scg, sco)


RTISI_FAST_CASES = [
    dict(B=3, T=6, look_ahead=3, asym=False, max_iter=1, alpha=0.99, center=True, normalized=False, window="hann"),
    dict(B=3, T=8, look_ahead=3, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann"),
    dict(B=2, T=7, look_ahead=-1, asym=True, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann"),
    dict(B=1, T=7, look_ahead=1, asym=True, max_iter=2, alpha=0.5, center=False, normalized=True, window="hamming"),
    dict(B=5, T=8, look_ahead=0, asym=False, max_iter=2, alpha=0.0, center=True, normalized=False, window="hann"),
    dict(B=2, T=8, look_ahead=2, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window=None, win_length=700),
    dict(B=3, T=14, look_ahead=3, asym=False, max_iter=3, alpha=0.99, center=True, normalized=False, window="hann"),
    # n_fft = 512 / hop = 128: 8 values per lane, four signals per CTA
    dict(B=5, T=9, look_ahead=3, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=512),
    dict(B=4, T=7, look_ahead=-1, asym=True, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=512),
    dict(B=1, T=8, look_ahead=1, asym=True, max_iter=3, alpha=0.5, center=False, normalized=True, window="hamming", n_fft=512),
    dict(B=9, T=8, look_ahead=0, asym=False, max_iter=2, alpha=0.0, center=True, normalized=False, window="hann", n_fft=512),
    dict(B=2, T=12, look_ahead=2, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window=None, win_length=300, n_fft=512),
    # n_fft = 2048 / hop = 512: two warps per frame
    dict(B=3, T=7, look_ahead=3, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=2048),
    dict(B=2, T=6, look_ahead=-1, asym=True, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=2048),
    dict(B=1, T=6, look_ahead=1, asym=True, max_iter=3, alpha=0.5, center=False, normalized=True, window="hamming", n_fft=2048),
    dict(B=4, T=6, look_ahead=0, asym=False, max_iter=2, alpha=0.0, center=True, normalized=False, window="hann", n_fft=2048),
    dict(B=2, T=9, look_ahead=2, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window=None, win_length=1500, n_fft=2048),
    # batches beyond one signal per SM (148): two / four signals share a CTA
    dict(B=151, T=6, look_ahead=3, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann"),
    dict(B=151, T=6, look_ahead=3, asym=True, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=512),
    dict(B=299, T=6, look_ahead=2, asym=False, max_iter=2, alpha=0.99, center=True, normalized=False, window="hann", n_fft=512),
]


@pytest.mark.parametrize("rc", RTISI_FAST_CASES, ids=lambda c: f"n{c.get('n_fft', 1024)}_B{c['B']}_T{c['T']}_la{c['look_ahead']}_asym{int(c['asym'])}_it{c['max_iter']}")
def test_rtisi_fast_kernel_1024_against_oracle(rc, monkeypatch):
    """The register-FFT RTISI-LA kernel (n_fft = 1024 / hop = 256, 512 / 128, 2048 / 512) against the oracle in float64.  fp32 trajectories of
    RTISI-LA drift apart quickly (the projection divides by |S|; SURVEY.md section 7: fp32 vs fp64 of the REFERENCE
    decorrelate over a full run), so the yardstick is the drift of two other fp32 implementations from the same fp64
    run -- the oracle in float32 and the generic shared-memory kernel on either of its two FFTs: an indexing mistake
    gives O(1) errors."""
    import spectrogram_inversion_b200 as S
    rs = np.random.RandomState(rc["T"])
    n_fft = rc.get("n_fft", 1024)
    hop = n_fft // 4
    kw = dict(hop_length=hop, center=rc["center"], normalized=rc["normalized"])
    wl = rc.get("win_length", n_fft)
    if rc["window"] is not None:
        kw["window"] = cases.window_of(rc["window"], wl, np.float32)
    if wl != n_fft:
        kw["win_length"] = wl
    oa = O.args_helper(n_fft // 2 + 1, np.float32, **kw)
    n_samples = (rc["T"] - 1) * hop + (0 if rc["center"] else n_fft)
    mag = np.abs(O.stft(rs.randn(rc["B"], n_samples).astype(np.float32), oa)).astype(np.float32)
    assert mag.shape == (rc["B"], n_fft // 2 + 1, rc["T"])
    run = dict(look_ahead=rc["look_ahead"], asymmetric_window=rc["asym"], max_iter=rc["max_iter"], alpha=rc["alpha"])
    y32 = O.RTISI_LA(mag, **run, **kw)
    kw64 = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    y64 = O.RTISI_LA(mag.astype(np.float64), **run, **kw64)
    tkw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    outs = {}
    # "1": the generic kernel on the mixed-radix passes, "1b": on the radix-2^2 passes (SPECINV_GENERIC_MR=0)
    for force in ("0", "1", "1b"):
        monkeypatch.setenv("SPECINV_FORCE_GENERIC", force[0])
        monkeypatch.setenv("SPECINV_GENERIC_MR", "0" if force.endswith("b") else "1")
        outs[force] = S.RTISI_LA(torch.from_numpy(mag).cuda(), verbose=0, **run, **tkw).cpu().numpy()

    def rel_l2(a, b):
        return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
    assert outs["0"].shape == y64.shape and np.isfinite(outs["0"]).all()
    drift = max(rel_l2(y32, y64), rel_l2(outs["1"], y64), rel_l2(outs["1b"], y64))
    assert drift < 0.1, drift                              # the horizon is short enough for the comparison to mean something
    assert rel_l2(outs["0"], y64) <= 4 * drift + 1e-5, (rel_l2(outs["0"], y64), drift)
    assert rel_l2(outs["0"], outs["1"]) <= 4 * drift + 1e-5


# ---------------------------------------------------------------------------------------------
# fast paths for n_fft = 2048, hop = 512 (two warps per frame), n_fft = 4096, hop = 1024 (four warps per frame)
# and n_fft = 512, hop = 128 (one warp per frame, 8 values per lane)
# ---------------------------------------------------------------------------------------------
FAST2048_CASES = [
    dict(B=40, T=130, center=True, pad_mode="reflect", normalized=False),
    dict(B=37, T=77, center=True, pad_mode="constant", normalized=True),
    dict(B=64, T=64, center=False, pad_mode="reflect", normalized=False),
    dict(B=1, T=9, center=True, pad_mode="reflect", normalized=False),
    dict(B=3, T=41, center=True, pad_mode="circular", normalized=False),
    dict(B=7, T=120, center=True, pad_mode="reflect", normalized=False, n_fft=512),
    dict(B=3, T=61, center=True, pad_mode="circular", normalized=True, n_fft=512),
    dict(B=4, T=33, center=False, pad_mode="reflect", normalized=False, n_fft=512),
    dict(B=1, T=7, center=True, pad_mode="constant", normalized=False, n_fft=512),
    dict(B=9, T=50, center=True, pad_mode="replicate", normalized=False, n_fft=4096),
    dict(B=2, T=33, center=False, pad_mode="reflect", normalized=True, n_fft=4096),
    dict(B=1, T=301, center=True, pad_mode="reflect", normalized=False, n_fft=4096),
    # hop = n_fft / 2 and n_fft / 8 (ov = frames overlapping on a sample)
    dict(B=5, T=90, center=True, pad_mode="reflect", normalized=False, n_fft=1024, ov=2),
    dict(B=5, T=90, center=True, pad_mode="reflect", normalized=False, n_fft=1024, ov=8),
    dict(B=3, T=40, center=False, pad_mode="reflect", normalized=True, n_fft=1024, ov=8),
    dict(B=6, T=70, center=True, pad_mode="constant", normalized=False, n_fft=512, ov=2),
    dict(B=6, T=70, center=True, pad_mode="circular", normalized=False, n_fft=512, ov=8),
    dict(B=2, T=17, center=False, pad_mode="reflect", normalized=False, n_fft=512, ov=2),
    dict(B=4, T=50, center=True, pad_mode="replicate", normalized=False, n_fft=2048, ov=2),
    dict(B=4, T=50, center=True, pad_mode="reflect", normalized=True, n_fft=2048, ov=8),
    dict(B=2, T=40, center=True, pad_mode="reflect", normalized=False, n_fft=4096, ov=2),
    dict(B=2, T=40, center=False, pad_mode="reflect", normalized=False, n_fft=4096, ov=8),
    dict(B=1, T=300, center=True, pad_mode="reflect", normalized=False, n_fft=1024, ov=2),
]


@pytest.mark.parametrize("fc", FAST2048_CASES,
                         ids=lambda c: f"n{c.get('n_fft', 2048)}_ov{c.get('ov', 4)}_B{c['B']}_T{c['T']}_{c['pad_mode']}_c{int(c['center'])}")
def test_fast_path_2048_against_oracle(fc):
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    rs = np.random.RandomState(fc["T"])
    n_fft = fc.get("n_fft", 2048)
    hop, F = n_fft // fc.get("ov", 4), n_fft // 2 + 1
    B, T = fc["B"], fc["T"]
    w = cases.window_of("hann" if fc["center"] else "hamming", n_fft, np.float32)
    kw = dict(hop_length=hop, center=fc["center"], pad_mode=fc["pad_mode"], normalized=fc["normalized"], window=w)
    oa = O.args_helper(F, np.float32, **kw)
    mag = (np.abs(rs.randn(B, F, T) + 1j * rs.randn(B, F, T)) * 8).astype(np.float32)
    C = (mag * np.exp(2j * np.pi * rs.rand(B, F, T))).astype(np.complex64)
    tkw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    magt = torch.from_numpy(mag).cuda()
    plan = StftPlan(args_helper(magt, **tkw), T, B, torch.float32, torch.device("cuda"))
    solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.99)
    st = O.gl_init(C, oa)
    close(solver.signal, st.x, 1e-5, "fast ISTFT (x_0)")
    for k in range(2):
        solver.x[solver.cur].copy_(torch.from_numpy(st.x))
        solver.q[solver.cur] = plan.pack(torch.from_numpy(st.q))
        solver.q[solver.cur ^ 1] = solver.q[solver.cur].like()
        out = solver.step(evaluate=(k == 1))
        st = O.gl_step(st, mag, 0.99 / 1.99, oa)
        close(solver.signal, st.x, 1e-5, f"fast2048 GL x step {k}")
        close(plan.unpack(solver.q_state), st.q, 1e-4, f"fast2048 GL q step {k}")
        if out is not None:
            do, eo, _ = O.metric_sums(st.out_mag, mag)
            assert abs(out[0] - do) <= 1e-4 * do and abs(out[1] - eo) <= 1e-4 * eo
    # plain Griffin-Lim (alpha = 0): the no-momentum variant of the kernel (NULL q pointers), 2 steps + sums
    solver = GriffinLimSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.0)
    assert solver.plain and solver.q is None
    st = O.gl_init(C, oa)
    for k in range(2):
        solver.x[solver.cur].copy_(torch.from_numpy(st.x))
        out = solver.step(evaluate=(k == 1))
        st = O.gl_step(st, mag, 0.0, oa)
        close(solver.signal, st.x, 1e-5, f"plain GL x step {k}")
        if out is not None:
            do, eo, _ = O.metric_sums(st.out_mag, mag)
            assert abs(out[0] - do) <= 1e-4 * do and abs(out[1] - eo) <= 1e-4 * eo
    solver = ADMMSolver(plan, plan.pack(torch.from_numpy(C)), plan.pack(magt), 0.1)
    st = O.admm_init(C, oa)
    solver.step(evaluate=True)
    st = O.admm_step(st, mag, 0.1, oa)
    close(solver.signal, st.x, 2e-5, "fast2048 ADMM x")
    close(plan.unpack(solver.U[solver.cur]), st.U, 1e-3, "fast2048 ADMM U")


def test_host_batches_are_pipelined_in_chunks_with_identical_results():
    """tol == 0, no progress bar, host input: the batch is processed in chunks (copies overlap compute); the signals
    of a batch are independent then, so the result must equal the whole-batch (CUDA input) run bit for bit."""
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200 import methods
    rs = np.random.RandomState(3)
    B, T = 6, 22000                      # enough frames for the chunked path (>= 2 chunks of 60000 frames)
    mag = torch.from_numpy((np.abs(rs.randn(B, 129, T)) * 3).astype(np.float32))
    assert methods._pipeline_chunks(mag, 0.0, False) == 2
    assert methods._pipeline_chunks(mag, 1e-6, False) == 1 and methods._pipeline_chunks(mag.cuda(), 0.0, False) == 1
    # a host batch too large for the device is cut into as many chunks as it takes to fit 80 % of the free memory
    free = torch.cuda.mem_get_info()[0]
    big = torch.empty(1, dtype=torch.float32).expand(40000, 513, 938)           # 77 GB of magnitudes, stride 0
    need = 40000 * 513 * 938 * 4 * 9
    assert methods._pipeline_chunks(big, 0.0, False) == max(4, -(-need // int(0.8 * free)))
    assert methods._pipeline_chunks(big, 0.0, False, state_arrays=2) > methods._pipeline_chunks(big, 0.0, False)
    w = torch.hann_window(256)
    for fn, kw in ((S.griffin_lim, dict(alpha=0.99)), (S.ADMM, dict(rho=0.1))):
        y_host = fn(mag.pin_memory(), max_iter=3, tol=0, verbose=False, eva_iter=2, window=w, hop_length=64, **kw)
        y_dev = fn(mag.cuda(), max_iter=3, tol=0, verbose=False, eva_iter=2, window=w.cuda(), hop_length=64, **kw)
        assert not y_host.is_cuda and y_host.shape == y_dev.shape
        assert torch.equal(y_host, y_dev.cpu())


def test_evaluating_and_non_reading_loops_give_identical_signals(monkeypatch):
    """training_loop with a history reads the sums at every evaluation and runs the iterations between evaluations
    through run_many; with tol == 0 and nothing watching the metric it runs the whole job through run_many and the
    host never waits for the sums.  Same kernels on the same buffers at the same cadence: the signals must agree bit
    for bit, and the last sums left on the device must be those of the last evaluation.  (The persistent
    small-problem kernel is switched off: it is another kernel, compared in test_gpu_resident.py.)"""
    monkeypatch.setenv("SPECINV_RESIDENT", "0")
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, StftPlan, training_loop
    from spectrogram_inversion_b200.stft_args import args_helper
    rs = np.random.RandomState(9)
    mag = torch.from_numpy((np.abs(rs.randn(2, 513, 40)) * 3).astype(np.float32)).cuda()
    w = torch.hann_window(1024, device="cuda")
    plan = StftPlan(args_helper(mag, window=w, hop_length=256), 40, 2, torch.float32, mag.device)
    pm = plan.pack(mag)
    for make in (lambda: GriffinLimSolver(plan, plan.phase_init(pm), pm, 0.99), lambda: ADMMSolver(plan, plan.phase_init(pm), pm, 0.1)):
        a, c = make(), make()
        ha = []
        na = training_loop(a, 23, 0.0, False, 4, "sc", history=ha)       # runs of 3 plain iterations, tail of 3
        nc = training_loop(c, 23, 0.0, False, 4, "sc")
        assert na == nc == 23 and a.iterations == c.iterations == 23
        assert torch.equal(c.signal, a.signal)
        d_last = float(c.sums[0].item())
        assert abs(d_last / c.n_bins_total - ha[-1][2]) <= 1e-12 * abs(ha[-1][2])


@pytest.mark.parametrize("ov", [4, 2, 8])
@pytest.mark.parametrize("n_fft", [512, 1024, 2048, 4096])
def test_specialised_kernels_on_tiny_frame_counts(n_fft, ov, monkeypatch):
    """T = 1 .. 6 frames (fewer frames than the 3-frame halo, no interior hop, ranges of one frame), several signals:
    the specialised kernel must agree with the generic one (and not hang on its TMA / mbarrier pipeline)."""
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, StftPlan
    from spectrogram_inversion_b200.stft_args import StftArgs
    dev = torch.device("cuda")
    hop, F = n_fft // ov, n_fft // 2 + 1
    g = torch.Generator(device=dev).manual_seed(n_fft)
    for center, pad_mode in ((False, "reflect"), (True, "constant"), (True, "replicate")):
        for T in (range(1, 7) if ov == 4 else sorted({1, 2, 3, ov - 1, ov, ov + 1, 2 * ov + 1})):
            if center and T < 2:
                continue
            B = 5
            args = StftArgs(n_fft, hop, n_fft, torch.hamming_window(n_fft, device=dev), center, pad_mode, False, True)
            plan = StftPlan(args, T, B, torch.float32, dev)
            mag = torch.rand(B, F, T, device=dev, generator=g) * 4
            C = mag * torch.exp(2j * torch.pi * torch.rand(B, F, T, device=dev, generator=g))
            outs = []
            for force in ("0", "1"):
                monkeypatch.setenv("SPECINV_FORCE_GENERIC", force)
                for Cls, coef in ((GriffinLimSolver, 0.99), (ADMMSolver, 0.1), (GriffinLimSolver, 0.0)):
                    s_ = Cls(plan, plan.pack(C), plan.pack(mag), coef)
                    sums = [s_.step(evaluate=True) for _ in range(2)]
                    outs.append((s_.signal.clone(), sums))
            for (xa, sa), (xb, sb) in zip(outs[:3], outs[3:]):
                fin = torch.isfinite(xb)
                assert (torch.isfinite(xa) == fin).all(), (center, T)
                scale = max(1.0, float(xb[fin].abs().max())) if fin.any() else 1.0
                assert float((xa[fin] - xb[fin]).abs().max()) <= 5e-5 * scale, (n_fft, center, pad_mode, T)
                for (d0, e0), (d1, e1) in zip(sa, sb):
                    if np.isfinite(d1) and np.isfinite(e1):
                        assert abs(d0 - d1) <= 1e-4 * abs(d1) + 1e-6 and abs(e0 - e1) <= 1e-4 * abs(e1) + 1e-6


FASTREF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fast.npz"))


@pytest.mark.parametrize("case", cases.FASTREF_CASES, ids=lambda c: c["name"])
def test_specialised_kernels_match_the_reference_itself(case):
    """The specialised kernels' shapes against outputs of the UNMODIFIED reference (tests/golden/fast.npz, written by
    tests/golden/make_golden_fast.py): one and two iterations from the same complex start, the magnitude entry
    (phase_init inside) and RTISI-LA."""
    import spectrogram_inversion_b200 as S
    inp = cases.make_case_inputs(case)
    kw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    C, mag, name = torch.from_numpy(inp["C"]).cuda(), torch.from_numpy(inp["mag"]).cuda(), case["name"]
    y = S.griffin_lim(C, max_iter=1, tol=0, alpha=0.99, verbose=False, eva_iter=1, **kw)
    close(y, FASTREF[f"{name}/gl_k1"], 1e-5, "GL 1 iteration vs reference")       # north_star: <= 1e-5 in fp32
    y = S.griffin_lim(C, max_iter=2, tol=0, alpha=0.99, verbose=False, eva_iter=1, **kw)
    close(y, FASTREF[f"{name}/gl_k2"], 5e-5, "GL 2 iterations vs reference")
    y = S.ADMM(C, max_iter=1, tol=0, rho=0.1, verbose=False, eva_iter=1, **kw)
    close(y, FASTREF[f"{name}/admm_k1"], 1e-5, "ADMM 1 iteration vs reference")
    y = S.griffin_lim(mag, max_iter=2, tol=0, alpha=0.99, verbose=False, **kw)
    close(y, FASTREF[f"{name}/gl_mag_k2"], 2e-3, "griffin_lim(mag) vs reference")
    y = S.griffin_lim(C, max_iter=2, tol=0, alpha=0.0, verbose=False, eva_iter=1, **kw)
    close(y, FASTREF[f"{name}/gl_plain_k2"], 5e-5, "plain GL (alpha = 0) 2 iterations vs reference")
    if f"{name}/rtisi_la3_k1" in FASTREF:
        y = S.RTISI_LA(mag, look_ahead=3, max_iter=1, alpha=0.99, verbose=0, **kw)
        close(y, FASTREF[f"{name}/rtisi_la3_k1"], 5e-3, "RTISI-LA vs reference")


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("onesided", [True, False])
def test_layout_conversion_is_exact_for_every_stride_pattern(dtype, onesided):
    """pack / unpack between the reference's (B, F, T) tensors and the split frame-major layout: contiguous input (32 x 32
    tile transposes), frame-major input = what torch.stft returns (the row-copy kernel), a strided view of a larger
    tensor, real and complex; all bit-exact."""
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import StftArgs
    dev = torch.device("cuda")
    n_fft, B, T = 128, 3, 45
    F = n_fft // 2 + 1 if onesided else n_fft
    plan = StftPlan(StftArgs(n_fft, 32, n_fft, torch.hann_window(n_fft, device=dev, dtype=dtype), True, "reflect", False,
                             onesided), T, B, dtype, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    for cplx in (False, True):
        base = torch.randn(B, F, T, device=dev, dtype=dtype, generator=g)
        if cplx:
            base = torch.complex(base, torch.randn(B, F, T, device=dev, dtype=dtype, generator=g))
        frame_major = base.transpose(1, 2).contiguous().transpose(1, 2)            # strides (F*T, 1, F)
        wide = torch.zeros(B, F + 3, 2 * T, device=dev, dtype=base.dtype)
        wide[:, 1:F + 1, ::2] = base
        views = {"contiguous": base, "frame-major": frame_major, "strided view": wide[:, 1:F + 1, ::2]}
        assert frame_major.stride() == (F * T, 1, F)
        ref = None
        for name, v in views.items():
            s = plan.pack(v)
            got = torch.cat([s.main, s.nyq.unsqueeze(-1)], dim=-1) if onesided else s.main      # (B, T, F)
            assert torch.equal(got, base.transpose(1, 2)), name
            if cplx:
                assert torch.equal(plan.unpack(s), base), name


def test_random_configurations_specialised_vs_fp64_generic():
    """tools/fuzz_fast_vs_generic.py: random (n_fft, hop, B, T, padding, window length, algorithm) draws; the specialised
    fp32 kernels must stay within 4x the generic fp32 kernel's distance (+1e-5) from the generic fp64 result."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "fuzz_fast_vs_generic.py"), "100", "3"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 101 and lines[-1].startswith("worst"), r.stdout[-1000:]
    bad = [ln for ln in lines if "MISMATCH" in ln]
    assert not bad, "\n".join(bad)
