"""RTISI-LA cut at outer-step boundaries (specinv_rtisi_la_steps): the persistent kernels save / restore their
sliding state, which gives
  * the reference's per-step progress bar (methods.py:362, :400) without changing a bit of the result, and
  * PER-STEP PARITY FROM IDENTICAL STATE (SURVEY.md section 8c): the oracle's state before outer step i is loaded into
    the kernel, one outer step (max_iter inner iterations + commit, methods.py:364-404) runs on the GPU, and the state
    that comes back is compared with the oracle's -- no chaotic amplification over hundreds of steps in between.
Both kernels: the register kernel (n_fft 512 / 1024 / 2048, hop = n_fft / 4, look_ahead <= 3) and the generic
shared-memory kernel (everything else, fp32 / fp64)."""
import numpy as np
import pytest
import torch

import cases
from oracle import specinv_oracle as O

pytestmark = pytest.mark.gpu


def _setup(n_fft, hop, B, T, dtype, seed, **kw):
    rs = np.random.RandomState(seed)
    w = cases.window_of(kw.pop("win", "hann"), n_fft, dtype)
    okw = dict(kw, window=w, hop_length=hop)
    oa = O.args_helper(n_fft // 2 + 1, dtype, **okw)
    n_samples = (T - 1) * hop + (0 if okw.get("center", True) else n_fft)
    mag = np.abs(O.stft(rs.randn(B, n_samples).astype(dtype), oa)).astype(dtype)
    assert mag.shape[2] == T
    return w, okw, oa, mag


def _gpu_objects(mag, okw, look_ahead):
    from spectrogram_inversion_b200 import _ops
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    dev = torch.device("cuda")
    magt = torch.from_numpy(mag).to(dev)
    tkw = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in okw.items()}
    args = args_helper(magt, **tkw)
    B, _, T = mag.shape
    plan = StftPlan(args, T, B, magt.dtype, dev)
    pm = plan.pack(magt)
    window = args.window.to(dev).contiguous()
    coeff = float(args.hop_length / (window @ window))
    LA = (args.n_fft - 1) // args.hop_length if look_ahead < 0 else look_ahead
    nbytes = _ops.rtisi_state_bytes(magt, args.n_fft, args.hop_length, T, B, args.normalized, args.onesided, LA)
    return plan, pm, window, coeff, LA, nbytes, args


def _run_steps(plan, pm, window, coeff, LA, args, x, state, cuts, asym, max_iter, alpha):
    from spectrogram_inversion_b200 import _ops
    scratch = torch.empty(2 * args.n_fft, dtype=x.dtype, device=x.device)
    for s0, s1 in zip(cuts[:-1], cuts[1:]):
        _ops.rtisi_la_steps(plan.buf, window, pm.main, pm.nyq, x, scratch, state, LA, asym, max_iter, alpha, coeff, s0, s1,
                            *plan._k)


CUT_CASES = [
    dict(n_fft=1024, B=3, T=14, la=3, asym=False, it=3, dtype="float32"),
    dict(n_fft=1024, B=151, T=9, la=2, asym=True, it=2, dtype="float32"),        # two signals per CTA
    dict(n_fft=512, B=5, T=12, la=3, asym=False, it=2, dtype="float32"),
    dict(n_fft=2048, B=2, T=9, la=-1, asym=True, it=2, dtype="float32"),
    dict(n_fft=1024, B=2, T=10, la=3, asym=False, it=2, dtype="float32", generic=True),
    dict(n_fft=256, B=3, T=15, la=-1, asym=False, it=3, dtype="float64"),
    dict(n_fft=256, B=2, T=11, la=1, asym=True, it=2, dtype="float32", center=False, win="hamming"),
    dict(n_fft=400, B=2, T=11, la=-1, asym=False, it=2, dtype="float32"),           # mixed-radix passes (200 = 8 * 5 * 5)
    dict(n_fft=256, B=2, T=11, la=2, asym=False, it=2, dtype="float32", legacy=True),   # radix-2^2 passes
]


@pytest.mark.parametrize("c", CUT_CASES, ids=lambda c: f"n{c['n_fft']}_B{c['B']}_la{c['la']}_{c['dtype']}{'_generic' if c.get('generic') else ''}{'_legacy' if c.get('legacy') else ''}")
def test_cut_runs_are_bit_identical_to_one_run(c, monkeypatch):
    monkeypatch.setenv("SPECINV_GENERIC_MR", "0" if c.get("legacy") else "1")
    import spectrogram_inversion_b200 as S
    monkeypatch.setenv("SPECINV_FORCE_GENERIC", "1" if c.get("generic") else "0")
    hop = c["n_fft"] // 4
    kw = {k: c[k] for k in ("center", "win") if k in c}
    w, okw, oa, mag = _setup(c["n_fft"], hop, c["B"], c["T"], np.dtype(c["dtype"]), seed=c["T"], **kw)
    plan, pm, window, coeff, LA, nbytes, args = _gpu_objects(mag, okw, c["la"])
    steps = c["T"] + LA
    tkw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in okw.items()}
    want = S.RTISI_LA(torch.from_numpy(mag).cuda(), look_ahead=c["la"], asymmetric_window=c["asym"], max_iter=c["it"],
                      alpha=0.99, verbose=0, **tkw)
    for cuts in ([0, 1, 2, steps], [0, steps // 2, steps - 1, steps], list(range(steps + 1))):
        x = torch.full_like(want, float("nan"))
        state = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        _run_steps(plan, pm, window, coeff, LA, args, x, state, cuts, c["asym"], c["it"], 0.99)
        assert torch.equal(x, want), cuts
    # the progress-bar path of the public API cuts the run the same way
    got = S.RTISI_LA(torch.from_numpy(mag).cuda(), look_ahead=c["la"], asymmetric_window=c["asym"], max_iter=c["it"],
                     alpha=0.99, verbose=1, **tkw)
    assert torch.equal(got, want)


def _canonical(su, st, dtype):
    """The oracle's state before outer step st.step in the layout of specinv_rtisi_la_steps (include/specinv_b200.h)."""
    a, K, LA = su.a, su.num_keep, su.look_ahead
    N, F = a.n_fft, a.n_fft // 2 + 1
    B = st.buf.shape[0]
    inv_scale = N ** -0.5 if a.normalized else 1.0 / N
    w = a.window.astype(np.float64)
    frames = st.buf[:, K:].astype(np.float64) / inv_scale                       # un-normalised inverse FFT samples
    pre = np.zeros((B, LA + 1, F), dtype=np.complex128)
    if st.pre is not None:
        pre[:, :LA] = st.pre[:, 1:]                                            # frame a of the next step had index a + 1
    kept = st.buf[:, :K].astype(np.float64) * (w * su.synth_coeff)
    carry = np.zeros((B, N))
    out = st.commits[LA:]                                                       # committed output frames so far
    for back, fr in enumerate(reversed(out[-K:] if (len(out) and K) else [])):  # back = 0: the last one
        sh = (back + 1) * a.hop_length
        if sh < N:
            carry[:, :N - sh] += (fr.astype(np.float64) * w)[:, sh:]
    pre_ri = np.stack([pre.real, pre.imag], axis=-1)
    flat = np.concatenate([frames.reshape(B, -1), pre_ri.reshape(B, -1), kept.reshape(B, -1), carry], axis=1)
    return flat.astype(dtype), dict(frames=frames * inv_scale, pre=pre, kept=kept, carry=carry)


STEP_CASES = [
    dict(n_fft=1024, B=3, T=12, la=3, asym=False, dtype="float32"),
    dict(n_fft=1024, B=3, T=12, la=3, asym=True, dtype="float32"),
    dict(n_fft=1024, B=150, T=10, la=2, asym=False, dtype="float32"),                   # two signals per CTA
    dict(n_fft=1024, B=2, T=12, la=3, asym=True, dtype="float32"),
    dict(n_fft=512, B=4, T=12, la=2, asym=False, dtype="float32"),
    dict(n_fft=2048, B=2, T=10, la=3, asym=False, dtype="float32"),
    dict(n_fft=1024, B=2, T=12, la=3, asym=False, dtype="float32", generic=True),
    dict(n_fft=256, B=3, T=14, la=-1, asym=True, dtype="float64"),
    dict(n_fft=256, B=3, T=14, la=-1, asym=True, dtype="float64", legacy=True),     # radix-2^2 passes (SPECINV_GENERIC_MR=0)
    dict(n_fft=400, B=2, T=12, la=3, asym=False, dtype="float32"),                  # mixed radix: 200 = 8 * 5 * 5
    dict(n_fft=600, B=2, T=10, la=-1, asym=True, dtype="float64"),                  # 300 = 4 * 5 * 5 * 3
    dict(n_fft=250, B=2, T=10, la=1, asym=False, dtype="float64"),                  # odd half 125 = 5^3, hop 62
    dict(n_fft=1144, B=1, T=8, la=2, asym=False, dtype="float32"),                  # 572 = 4 * 13 * 11
]


@pytest.mark.parametrize("c", STEP_CASES, ids=lambda c: f"n{c['n_fft']}_B{c['B']}_la{c['la']}_asym{int(c['asym'])}_{c['dtype']}{'_generic' if c.get('generic') else ''}{'_legacy' if c.get('legacy') else ''}")
def test_one_outer_step_from_the_oracles_state(c, monkeypatch):
    """Outer step i (its max_iter inner iterations j = 0 .. max_iter-1 and the commit) from the ORACLE's state, for
    several i (start-up, steady state, tail where the look-ahead runs past the spectrogram) and max_iter = 1, 2:
    frames to 1e-5 absolute (unit-scale signals) x 4 per extra inner iteration, spectra relative to their scale."""
    monkeypatch.setenv("SPECINV_FORCE_GENERIC", "1" if c.get("generic") else "0")
    monkeypatch.setenv("SPECINV_GENERIC_MR", "0" if c.get("legacy") else "1")
    dtype = np.dtype(c["dtype"])
    f32 = dtype == np.float32
    hop = c["n_fft"] // 4
    w, okw, oa, mag = _setup(c["n_fft"], hop, c["B"], c["T"], dtype, seed=3 * c["T"])
    plan, pm, window, coeff, LA, nbytes, args = _gpu_objects(mag, okw, c["la"])
    steps = c["T"] + LA
    for max_iter in (1, 2):
        su = O.rtisi_setup(mag, look_ahead=c["la"], asymmetric_window=c["asym"], max_iter=max_iter, alpha=0.99, **okw)
        st = O.rtisi_init(su)
        states = []                                           # oracle state before every outer step
        for i in range(steps):
            states.append(st)
            for j in range(max_iter):
                st = O.rtisi_inner(su, st, j)
            st = O.rtisi_commit(su, st)
        states.append(st)
        for i in sorted({1, 2, LA + 2, c["T"] // 2, min(c["T"], steps - 2), steps - 2}):   # (the last step saves no state)
            flat, _ = _canonical(su, states[i], dtype)
            state = torch.from_numpy(np.ascontiguousarray(flat)).cuda().view(torch.uint8).reshape(-1)
            assert state.numel() == nbytes
            x = torch.zeros(c["B"], plan.length, dtype=pm.main.dtype, device="cuda")
            _run_steps(plan, pm, window, coeff, LA, args, x, state, [i, i + 1], c["asym"], max_iter, 0.99)
            got = state.view(torch.from_numpy(flat).dtype).reshape(c["B"], -1).cpu().numpy().astype(np.float64)
            want_flat, parts = _canonical(su, states[i + 1], np.float64)
            N, F, NA, K = args.n_fft, args.n_fft // 2 + 1, LA + 1, su.num_keep
            inv_scale = N ** -0.5 if args.normalized else 1.0 / N
            o = 0
            fr_g = got[:, o:o + NA * N].reshape(c["B"], NA, N) * inv_scale; o += NA * N
            pre_g = got[:, o:o + 2 * NA * F].reshape(c["B"], NA, F, 2); o += 2 * NA * F
            kept_g = got[:, o:o + K * N].reshape(c["B"], K, N); o += K * N
            carry_g = got[:, o:o + N]
            tol = (1e-5 if f32 else 1e-10) * 4 ** (max_iter - 1)
            assert np.abs(fr_g - parts["frames"]).max() <= tol * max(1.0, np.abs(parts["frames"]).max()), \
                ("frames", i, max_iter, np.abs(fr_g - parts["frames"]).max())
            pre_c = pre_g[..., 0] + 1j * pre_g[..., 1]
            ps = max(1.0, np.abs(parts["pre"]).max())
            # (relative to the largest spectrum value; with 150 signals a bin behind a tiny |S| of the first inner
            # iteration reaches 1.7e-5 in the second one)
            assert np.abs(pre_c[:, :LA] - parts["pre"][:, :LA]).max() <= (1e-5 if f32 else 1e-11) * ps * 4 ** (max_iter - 1), \
                ("pre", i, max_iter, np.abs(pre_c[:, :LA] - parts["pre"][:, :LA]).max(), ps)
            assert np.abs(kept_g - parts["kept"]).max() <= tol * max(1.0, np.abs(parts["kept"]).max()), ("kept", i, max_iter)
            assert np.abs(carry_g - parts["carry"]).max() <= tol * max(1.0, np.abs(parts["carry"]).max()), ("carry", i, max_iter)


@pytest.mark.parametrize("seed", range(14))
def test_random_configurations_one_step_from_oracle_state(seed, monkeypatch):
    """The configurations tools/fuzz_rtisi.py draws (n_fft, look_ahead, asymmetric, alpha, win_length, normalized,
    centre, batch sizes that put 1 / 2 / 4 signals on a CTA), judged per OUTER STEP from the oracle's state instead of
    over whole runs.  Round 1's whole-run fuzz saw the register kernel up to 6.5x further from the fp64 run than the
    generic kernel in two cases (n_fft=2048 la=0 wl=1866; n_fft=512 la=0 alpha=0): whole runs amplify every rounding
    difference step after step (the projection S * mag / |S| divides by |S|, and |S| ~ 0 bins are common when the
    look-ahead is 0), so two correct fp32 implementations can differ by 1e-2 after three inner iterations of a dozen
    steps.  From identical state one step agrees to 1e-5; those two configurations are seeds 0 and 1 here."""
    import random
    rnd = random.Random(seed)
    if seed == 0:
        n_fft, la, asym, alpha, wl, normalized, center, B, T = 2048, 0, False, 0.99, 1866, False, True, 3, 9
    elif seed == 1:
        n_fft, la, asym, alpha, wl, normalized, center, B, T = 512, 0, False, 0.0, 512, False, True, 5, 8
    else:
        n_fft = rnd.choice([512, 1024, 2048, 256])
        la = rnd.choice([-1, 0, 1, 2, 3])
        asym = rnd.random() < 0.4
        alpha = rnd.choice([0.99, 0.99, 0.5, 0.0])
        wl = n_fft if rnd.random() < 0.6 else rnd.randrange(n_fft // 2 + 1, n_fft)
        normalized = rnd.random() < 0.3
        center = rnd.random() < 0.7
        B = rnd.choice([1, 2, 3, 5, 150, 299] if n_fft in (512, 1024) else [1, 2, 3])
        T = rnd.choice([6, 9, 14])
    hop = n_fft // 4
    dtype = np.dtype(np.float32)
    rs = np.random.RandomState(seed)
    w = cases.window_of("hann" if center else "hamming", wl, dtype)
    okw = dict(window=w, hop_length=hop, center=center, normalized=normalized)
    if wl != n_fft:
        okw["win_length"] = wl
    oa = O.args_helper(n_fft // 2 + 1, dtype, **okw)
    mag = np.abs(O.stft(rs.randn(B, (T - 1) * hop + (0 if center else n_fft)).astype(dtype), oa)).astype(dtype)
    plan, pm, window, coeff, LA, nbytes, args = _gpu_objects(mag, okw, la)
    steps = T + LA
    max_iter = rnd.choice([1, 2])
    su = O.rtisi_setup(mag, look_ahead=la, asymmetric_window=asym, max_iter=max_iter, alpha=alpha, **okw)
    st = O.rtisi_init(su)
    i0 = rnd.randrange(1, steps - 1)
    for i in range(i0):
        for j in range(max_iter):
            st = O.rtisi_inner(su, st, j)
        st = O.rtisi_commit(su, st)
    flat, _ = _canonical(su, st, dtype)
    for j in range(max_iter):
        st = O.rtisi_inner(su, st, j)
    st = O.rtisi_commit(su, st)
    _, parts = _canonical(su, st, np.float64)
    state = torch.from_numpy(np.ascontiguousarray(flat)).cuda().view(torch.uint8).reshape(-1)
    assert state.numel() == nbytes
    x = torch.zeros(B, plan.length, dtype=torch.float32, device="cuda")
    _run_steps(plan, pm, window, coeff, LA, args, x, state, [i0, i0 + 1], asym, max_iter, alpha)
    got = state.view(torch.float32).reshape(B, -1).cpu().numpy().astype(np.float64)
    N, NA = n_fft, LA + 1
    inv_scale = N ** -0.5 if normalized else 1.0 / N
    fr_g = got[:, :NA * N].reshape(B, NA, N) * inv_scale
    err = np.abs(fr_g - parts["frames"]).max()
    assert err <= 1e-5 * 4 ** (max_iter - 1) * max(1.0, np.abs(parts["frames"]).max()), (err, n_fft, la, asym, alpha, wl, i0)
