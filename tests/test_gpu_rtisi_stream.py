"""Streaming RTISI-LA (RTISIStream, specinv_rtisi_la_stream): pushes concatenated with the flush are bit for bit
RTISI_LA on the whole spectrogram, on both kernel families and for every chunking; the emitted count follows
E(n); memory does not grow with the stream; the 1/envelope windows gathered from the short plan equal a full plan's.
Bit patterns are compared (.view(int)), so NaN / inf positions count."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

_INT = {torch.float32: torch.int32, torch.float64: torch.int64}


def _bits(t):
    return t.contiguous().view(_INT[t.dtype])


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _mag(n_fft, hop, B, T, dtype, seed, center=True, win="hann", win_length=None, normalized=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    wl = win_length or n_fft
    w = (torch.hann_window if win == "hann" else torch.hamming_window)(wl, dtype=dtype, device="cuda")
    n = (T - 1) * hop + (0 if center else n_fft)
    x = torch.randn(B, n, dtype=dtype, device="cuda", generator=g)
    S = torch.stft(x, n_fft, hop, wl, w, center=center, normalized=normalized, onesided=True, return_complex=True)
    assert S.shape[-1] == T
    kw = dict(window=w, hop_length=hop, center=center, normalized=normalized)
    if win_length:
        kw["win_length"] = win_length
    return S.abs().contiguous(), kw


def _chunkings(T, LA, seed):
    rnd = random.Random(seed)
    sizes = []
    while sum(sizes) < T:
        sizes.append(rnd.choice([0, 0, 1, max(1, LA - 1), 2, 3, 5]))
    sizes[-1] -= sum(sizes) - T
    rest = []
    while sum(rest) < T - 1:
        rest.append(rnd.choice([0, 1, 2, 4, 7]))
    if rest:
        rest[-1] -= sum(rest) - (T - 1)
    return {"whole": [T], "single_frames": [1] * T, "random": sizes, "first_one": [1] + rest}


def _stream(mag, sizes, la, asym, it, kw, check_count=True):
    from spectrogram_inversion_b200 import RTISIStream
    from spectrogram_inversion_b200.streaming import emitted_samples
    s = RTISIStream(look_ahead=la, asymmetric_window=asym, max_iter=it, alpha=0.99, **kw)
    outs, t = [], 0
    n_fft = (mag.shape[-2] - 1) * 2
    for k in sizes:
        outs.append(s.push(mag[..., t:t + k]))
        t += k
        if check_count:
            got = sum(o.shape[-1] for o in outs)
            assert got == emitted_samples(t, n_fft, kw["hop_length"], la, kw.get("center", True)), (t, got)
    outs.append(s.flush())
    return torch.cat(outs, -1)


STREAM_CASES = [
    dict(n_fft=1024, B=3, T=14, la=3, asym=False, it=3, dtype=torch.float32),
    dict(n_fft=1024, B=151, T=9, la=2, asym=True, it=2, dtype=torch.float32),       # two signals per CTA
    dict(n_fft=512, B=5, T=12, la=-1, asym=True, it=2, dtype=torch.float32),
    dict(n_fft=2048, B=2, T=9, la=-1, asym=True, it=2, dtype=torch.float32),
    dict(n_fft=1024, B=2, T=10, la=3, asym=False, it=2, dtype=torch.float32, generic=True),
    dict(n_fft=1024, B=2, T=10, la=0, asym=False, it=2, dtype=torch.float32),       # flush releases the carry
    dict(n_fft=256, B=3, T=15, la=-1, asym=False, it=3, dtype=torch.float64),
    dict(n_fft=256, B=2, T=11, la=0, asym=True, it=2, dtype=torch.float64, center=False),
    dict(n_fft=256, B=2, T=11, la=1, asym=True, it=2, dtype=torch.float32, center=False, win="hamming"),
    dict(n_fft=400, B=2, T=11, la=-1, asym=False, it=2, dtype=torch.float32),      # mixed radix: 200 = 8 * 5 * 5
    dict(n_fft=250, B=2, T=10, la=1, asym=False, it=2, dtype=torch.float64),       # odd half 125, hop 62
    dict(n_fft=1024, B=2, T=10, la=2, asym=True, it=2, dtype=torch.float32, win_length=800),
    dict(n_fft=512, B=2, T=10, la=3, asym=False, it=2, dtype=torch.float32, normalized=True),
]


def _case_id(c):
    extra = "".join(f"_{k}" for k in ("generic", "normalized", "win_length") if c.get(k))
    return f"n{c['n_fft']}_B{c['B']}_la{c['la']}_{str(c['dtype'])[6:]}{extra}{'' if c.get('center', True) else '_nocenter'}"


@pytest.mark.parametrize("c", STREAM_CASES, ids=_case_id)
def test_pushes_and_flush_equal_rtisi_la(c, monkeypatch):
    monkeypatch.setenv("SPECINV_FORCE_GENERIC", "1" if c.get("generic") else "0")
    import spectrogram_inversion_b200 as S
    mag, kw = _mag(c["n_fft"], c["n_fft"] // 4, c["B"], c["T"], c["dtype"], seed=c["T"] + c["n_fft"],
                   center=c.get("center", True), win=c.get("win", "hann"), win_length=c.get("win_length"),
                   normalized=c.get("normalized", False))
    want = S.RTISI_LA(mag, look_ahead=c["la"], asymmetric_window=c["asym"], max_iter=c["it"], alpha=0.99, verbose=0,
                      **kw)
    LA = (c["n_fft"] - 1) // (c["n_fft"] // 4) if c["la"] < 0 else c["la"]
    for name, sizes in _chunkings(c["T"], LA, seed=c["T"]).items():
        got = _stream(mag, sizes, c["la"], c["asym"], c["it"], kw)
        assert _same_bits(got, want), (name, sizes, (got - want).abs().max().item() if got.shape == want.shape else got.shape)


@pytest.mark.parametrize("T", [1, 2, 3, 4, 6])
def test_emitted_count_when_blocks_cross_the_length_and_short_streams(T, monkeypatch):
    """look_ahead = 0, centred, hop > n_fft / 2 (generic kernel): the block of the newest frame reaches past L(n); those
    samples wait for the next push or are dropped by the flush.  And streams of T <= look_ahead frames in total."""
    import spectrogram_inversion_b200 as S
    monkeypatch.setenv("SPECINV_FORCE_GENERIC", "0")
    if T >= 2:          # (reflect padding needs P < L: RTISI_LA itself takes T >= 2 here)
        mag, kw = _mag(256, 160, 2, T, torch.float32, seed=T)
        want = S.RTISI_LA(mag, look_ahead=0, max_iter=3, alpha=0.99, verbose=0, **kw)
        for sizes in ([T], [1] * T, [0, 1, 0] + [1] * (T - 1)):
            assert _same_bits(_stream(mag, sizes, 0, False, 3, kw), want), sizes
    for n_fft, la in ((1024, 3), (256, -1)) if T <= 3 else ():     # T <= LA: nothing is emitted before the flush
        mag, kw = _mag(n_fft, n_fft // 4, 2, T, torch.float32, seed=T, center=False)
        want = S.RTISI_LA(mag, look_ahead=la, asymmetric_window=True, max_iter=2, alpha=0.99, verbose=0, **kw)
        for sizes in ([T], [1] * T):
            assert _same_bits(_stream(mag, sizes, la, True, 2, kw), want), (n_fft, sizes)


def test_long_stream_memory_does_not_grow():
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200 import RTISIStream
    T, step = 7007, 7
    mag, kw = _mag(1024, 256, 4, T, torch.float32, seed=5)
    s = RTISIStream(look_ahead=3, max_iter=2, **kw)
    outs = []
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    peaks = {}
    for i, t in enumerate(range(0, T, step)):
        outs.append(s.push(mag[..., t:t + step]).cpu())
        if i + 1 in (100, 1000):
            peaks[i + 1] = torch.cuda.max_memory_allocated()
    outs.append(s.flush().cpu())
    assert peaks[1000] <= peaks[100], peaks
    want = S.RTISI_LA(mag, look_ahead=3, max_iter=2, alpha=0.99, verbose=0, **kw).cpu()
    assert _same_bits(torch.cat(outs, -1), want)


def _full_inv_env(n_fft, hop, T, center, dtype):
    from spectrogram_inversion_b200 import _ops
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    import dataclasses
    w = torch.hann_window(n_fft, dtype=dtype, device="cuda")
    args = dataclasses.replace(args_helper(torch.empty(1, n_fft // 2 + 1, T, dtype=dtype, device="cuda"), window=w,
                                           hop_length=hop, center=center), pad_mode="constant")
    plan = StftPlan(args, T, 1, dtype, "cuda")
    out = torch.empty(plan.length, dtype=dtype, device="cuda")
    _ops.plan_inv_env_window(plan.buf, out, 0, T, n_fft, hop, T, center, False, True)   # the plan's own values
    env = plan.envelope()
    torch.cuda.synchronize()
    assert _same_bits(out, 1 / env)               # (an independent read of the same plan)
    return w, out


@pytest.mark.parametrize("n_fft,hop,center,dtype", [(1024, 256, True, torch.float32), (250, 62, True, torch.float64),
                                                    (256, 64, False, torch.float32)])
def test_inv_env_windows_equal_a_full_plan(n_fft, hop, center, dtype):
    from spectrogram_inversion_b200 import RTISIStream
    K = (n_fft - 1) // hop
    T0 = K + 2
    s = None
    for T in sorted({1, 2, K, K + 1, T0 - 1, T0, 40000}):
        L = (T - 1) * hop + n_fft - 2 * (n_fft // 2 if center else 0)
        if L < 1:
            continue
        w, want = _full_inv_env(n_fft, hop, T, center, dtype)
        if s is None:
            s = RTISIStream(look_ahead=1, max_iter=1, window=w, hop_length=hop, center=center)
            s.push(torch.zeros(n_fft // 2 + 1, 1, dtype=dtype, device="cuda"))
        assert _same_bits(s._inv_env_window(0, L, T), want), T
        if T == 40000:
            assert not torch.isfinite(want).all() or center        # un-centred hann: inf at the first sample
            rnd = random.Random(T)
            for _ in range(20):        # windows of a stream whose end is not known yet (before the tail)
                x0 = rnd.randrange(0, L - 4 * n_fft)
                n = rnd.randrange(0, 3 * n_fft)
                assert _same_bits(s._inv_env_window(x0, n), want[x0:x0 + n]), (x0, n)


def test_shapes_devices_and_errors():
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200 import RTISIStream
    mag, kw = _mag(512, 128, 1, 12, torch.float32, seed=1)
    want = S.RTISI_LA(mag[0], look_ahead=2, max_iter=2, verbose=0, **kw)
    s = RTISIStream(look_ahead=2, max_iter=2, **kw)                  # 2-D chunks -> 1-D samples
    parts = [s.push(mag[0, :, :5]), s.push(mag[0, :, 5:])]
    assert all(p.dim() == 1 and p.is_cuda for p in parts)
    with pytest.raises(AssertionError):
        s.push(mag[..., :1])                                         # 3-D after 2-D
    with pytest.raises(AssertionError):
        s.push(mag[0, :-1, :1])                                      # other F
    with pytest.raises(AssertionError):
        s.push(mag[0, :, :1].double())                               # other dtype
    with pytest.raises(AssertionError):
        s.push(mag[0, :, :1].cpu())                                  # other device
    with pytest.raises(NotImplementedError):
        s.push(mag[0, :, :1].clone().requires_grad_())
    with pytest.raises(AssertionError):
        s.push(mag[0, :, :1].to(torch.complex64))
    parts.append(s.flush())
    assert _same_bits(torch.cat(parts), want)
    with pytest.raises(RuntimeError):
        s.push(mag[0, :, :1])
    with pytest.raises(RuntimeError):
        s.flush()
    # 3-D with one signal keeps the batch dimension, as RTISI_LA does
    s = RTISIStream(look_ahead=2, max_iter=2, **kw)
    got = torch.cat([s.push(mag[..., :7]), s.push(mag[..., 7:]), s.flush()], -1)
    assert _same_bits(got, S.RTISI_LA(mag, look_ahead=2, max_iter=2, verbose=0, **kw))
    # host chunks give host samples
    hkw = dict(kw, window=kw["window"].cpu())
    s = RTISIStream(look_ahead=2, max_iter=2, **hkw)
    host = mag.cpu()
    parts = [s.push(host[..., :3]), s.push(host[..., 3:3]), s.push(host[..., 3:]), s.flush()]
    assert all(not p.is_cuda for p in parts)
    assert _same_bits(torch.cat(parts, -1), S.RTISI_LA(host, look_ahead=2, max_iter=2, verbose=0, **hkw))
    with pytest.raises(TypeError):
        RTISIStream(bogus=1, **kw)
    with pytest.raises(RuntimeError):
        RTISIStream(**kw).flush()
