"""phase_init on the GPU (csrc/specinv_phase_init.cu, autograd.phase_init_diff) against the reference's phase at
real signal lengths, on both of the kernel's paths: the single pass, and the time split that small batches take
(per-chunk phase sums, a scan over the chunks, the apply pass).

The reference is C_ref = mag * exp(i phi) in float64, phi the oracle's phase (oracle.phase_init_phase, which
reproduces the reference's phase bit for bit: tests/test_oracle_golden.py).  Per bin:
  * float32: |C - C_ref| <= 4e-7 mag: two ulps of sincosf, one of the product, the rounding of the reduced angle;
    the float64 range reduction adds < 1e-10 rad.  One ulp of phase is visible from |phi| >= 8 rad.
  * float64: |C - C_ref| <= mag (1e-14 + T 2^-53 |phi|): re-associated float64 sums.  One omega (>= 0.1 rad here)
    lost or counted twice at a chunk seam is far above it."""
import re

import numpy as np
import pytest
import torch

from oracle import specinv_oracle as O

pytestmark = pytest.mark.gpu

SEG = 30                 # bins per warp of phase_init_kernel (PI_SEG)
WARP_SLOTS = 148 * 64    # resident warps the host's chunk rule fills


def chunking(B, F, T):
    """phase_init_t's time split: (chunks, chunk_len).  Time is split when the (signal, 30-bin segment) pairs leave
    warp slots idle, into chunks of >= 32 frames; chunks == 1 is the single-pass kernel."""
    segs = -(-F // SEG)
    chunks = max(1, min(WARP_SLOTS // (B * segs), T // 32))
    chunk_len = -(-T // chunks)
    return -(-T // chunk_len), chunk_len


def n_bins(n_fft, onesided):
    return n_fft // 2 + 1 if onesided else n_fft


def rand_mag(B, F, T, dtype, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(B, F, T, generator=g, device="cuda", dtype=dtype)


def plan_of(magt, hop, onesided):
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    B, _, T = magt.shape
    return StftPlan(args_helper(magt, hop_length=hop, onesided=onesided), T, B, magt.dtype, magt.device, tables=False)


def fused(magt, hop, onesided=True):
    """the fused kernel through the plan: (B, F, T) CUDA magnitude -> (B, F, T) complex"""
    plan = plan_of(magt, hop, onesided)
    return plan.unpack(plan.phase_init(plan.pack(magt)))


def fused_ex(magt, hop, onesided, phase_in=None):
    """specinv_phase_init_ex over one frame range: (C, phase_out), phase_in / phase_out (B, F) float64"""
    from spectrogram_inversion_b200 import _ops
    B, F, _ = magt.shape
    plan = plan_of(magt, hop, onesided)
    mag = plan.pack(magt)
    out = plan.empty_spec()
    pin = phase_in.contiguous() if phase_in is not None else torch.empty(0, dtype=torch.float64, device=magt.device)
    pout = torch.empty(B, F, dtype=torch.float64, device=magt.device)
    _ops.phase_init_ex(mag.main, mag.nyq, out.main, out.nyq, pin, pout, plan.args.n_fft, hop, onesided)
    return plan.unpack(out), pout


def check(C, mag, phase, phase_f64, what, k0=0):
    """C (B, K, T) from the GPU against mag * exp(i phase) under the bound of the module docstring; bins k0 .. of
    the spectrum."""
    C = C.detach().cpu().numpy() if isinstance(C, torch.Tensor) else np.asarray(C)
    assert C.shape == mag.shape == phase.shape, (what, C.shape, mag.shape, phase.shape)
    T = mag.shape[-1]
    m = mag.astype(np.float64)
    ref = m * np.exp(1j * phase.astype(np.float64))
    err = np.abs(C.astype(np.complex128) - ref)
    if mag.dtype == np.float32:
        bound = 4e-7 * m
    else:
        bound = m * (1e-14 + T * 2.0 ** -53 * np.abs(phase_f64))
    bad = ~(err <= bound)
    if bad.any():
        ratio = np.where(bad, err / np.maximum(bound, np.finfo(np.float64).tiny), 0)
        b, k, t = np.unravel_index(np.argmax(ratio), ratio.shape)
        ph = phase[b, k, t]
        dphi = np.angle(C[b, k, t].astype(np.complex128) * np.conj(ref[b, k, t]))
        ulp = float(np.spacing(np.abs(ph)))
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.size} bins over the bound; worst (b, k, t) = "
                    f"({b}, {k + k0}, {t}): |C - C_ref| = {err[b, k, t]:.3e} > {bound[b, k, t]:.3e} at mag "
                    f"{m[b, k, t]:.4g}, |phi| = {abs(float(ph)):.9g} rad, phase error {dphi / ulp:+.2f} ulp")


def check_against_oracle(C, magt, hop, onesided, what):
    mag = magt.cpu().numpy()
    ph, ph64 = O.phase_init_phase(mag, hop_length=hop, onesided=onesided)
    check(C, mag, ph, ph64, what)
    return mag, ph, ph64


# ---------------------------------------------------------------------------------------------------------------
# shape matrix: (id, B, n_fft, hop, T, onesided, also float64, expected (chunks, chunk_len, frames of the last chunk))
SHAPES = [
    # single pass over long signals: enough (signal, segment) pairs to fill the machine
    ("single-1024-B528-T100", 528, 1024, 256, 100, True, False, (1, 100, 100)),
    ("single-4096-B140-T70", 140, 4096, 1024, 70, True, True, (1, 70, 70)),
    # the chunk rule's boundary at one signal of 1024/256
    ("1024-T63", 1, 1024, 256, 63, True, True, (1, 63, 63)),
    ("1024-T64", 1, 1024, 256, 64, True, False, (2, 32, 32)),
    ("1024-T65", 1, 1024, 256, 65, True, True, (2, 33, 32)),
    # a last chunk shorter than the kernel's unroll of 4 frames
    ("cfg1-2048-T1292", 1, 2048, 512, 1292, True, True, (40, 33, 5)),
    ("4096-T5000", 1, 4096, 1024, 5000, True, False, (136, 37, 5)),
    # n_fft not a power of two, chunked
    ("400-B64-T1001", 64, 400, 100, 1001, True, True, (21, 48, 41)),
    ("120-T2000", 1, 120, 30, 2000, True, False, (61, 33, 20)),         # F = 61: a one-bin last segment
    ("600-B3-T900", 3, 600, 150, 900, True, True, (28, 33, 9)),          # F = 301: a one-bin last segment
    ("1000-B2-T1500", 2, 1000, 250, 1500, True, False, (46, 33, 15)),
    ("250-T1200", 1, 250, 50, 1200, True, False, (37, 33, 12)),          # odd n_fft / 2
    # two-sided: F = n_fft, the Nyquist bin (if any) is a bin of the main array
    ("two-sided-96-B2", 2, 96, 24, 800, False, True, (25, 32, 32)),
    ("two-sided-75", 1, 75, 25, 1000, False, True, (31, 33, 10)),
    ("two-sided-255", 1, 255, 64, 700, False, False, (21, 34, 20)),
]
SHAPE_PARAMS = [pytest.param(s, np.float32, id=f"{s[0]}-f32") for s in SHAPES] + \
               [pytest.param(s, np.float64, id=f"{s[0]}-f64") for s in SHAPES if s[6]]


@pytest.mark.parametrize("shape,dtype", SHAPE_PARAMS)
def test_phase_init_matches_reference_phase(shape, dtype):
    name, B, n_fft, hop, T, onesided, _, expect = shape
    F = n_bins(n_fft, onesided)
    chunks, chunk_len = chunking(B, F, T)
    assert (chunks, chunk_len, T - (chunks - 1) * chunk_len) == expect, "the case no longer covers its path"
    magt = rand_mag(B, F, T, torch.float32 if dtype == np.float32 else torch.float64, seed=n_fft + T)
    assert plan_of(magt, hop, onesided).args.n_fft == n_fft
    if name.startswith("600"):      # through the public entry, with a kwarg phase_init must ignore
        import spectrogram_inversion_b200 as S
        C = S.phase_init(magt, hop_length=hop, normalized=True)
    else:
        C = fused(magt, hop, onesided)
    check_against_oracle(C, magt, hop, onesided, name)


def test_chunk_rule_matches_the_launched_kernels():
    """`chunking` above restates the host's rule; the kernels the profiler sees must be the ones it predicts."""
    from torch.profiler import ProfilerActivity, profile
    for B, n_fft, T in ((1, 1024, 63), (1, 1024, 64), (528, 1024, 100), (64, 400, 1001)):
        F = n_bins(n_fft, True)
        magt = rand_mag(B, F, T, torch.float32, seed=1)
        plan = plan_of(magt, n_fft // 4, True)
        mag = plan.pack(magt)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            plan.phase_init(mag)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events()]
        modes = sorted({int(m) for n in names for m in re.findall(r"phase_init_kernel<float, ?(\d)", n)})
        scans = sum("phase_scan_kernel" in n for n in names)
        split = chunking(B, F, T)[0] > 1
        assert (modes, scans) == (([1, 2], 1) if split else ([0], 0)), (B, n_fft, T, modes, scans)


def test_cfg5_length_signal_in_three_bands():
    """One hour at 4096/1024 (BASELINE cfg5: 168 751 frames, 137 chunks): the phase reaches ~5e8 rad, where a float
    ulp is 32 rad and only the float64 range reduction keeps sin / cos right.  Three 64-bin bands go through the
    oracle: the bottom, the middle (two segment seams) and the top with the Nyquist bin."""
    B, n_fft, hop, T = 1, 4096, 1024, 168751
    F = n_bins(n_fft, True)
    assert chunking(B, F, T) == (137, 1232)
    magt = rand_mag(B, F, T, torch.float32, seed=5)
    C = fused(magt, hop)
    mag = magt.cpu().numpy()
    del magt
    top = 0.0
    for k0 in (0, 1000, F - 64):
        ph, ph64 = O.phase_init_phase(mag, bins=(k0, k0 + 64), hop_length=hop)
        check(C[:, k0:k0 + 64], mag[:, k0:k0 + 64], ph, ph64, f"cfg5 bins {k0}..{k0 + 63}", k0)
        top = max(top, float(np.abs(ph64).max()))
    assert top > 4e8


# ---------------------------------------------------------------------------------------------------------------
# crafted magnitudes: background in [0, 1), planted values above it
def _crafted(pattern, F, T, chunk_len, seed):
    rs = np.random.RandomState(seed)
    m = rs.uniform(0.0, 1.0, (1, F, T)).astype(np.float32)
    ks = np.arange(F)

    def peak(k, t):
        k = k[(k >= 1) & (k <= F - 2)]
        m[0, k, t] = rs.uniform(1.5, 2.5, len(k))

    for t in range(T):
        if pattern == "edge-peaks":           # k = 1 / 2 alternately, F - 2 (= M - 1: the Nyquist bin takes its omega)
            peak(np.array([1 + t % 2, F - 2]), t)
        elif pattern == "seam-peaks":         # every k = 28, 29, 0, 1 (mod 30): the segment seams and the halo lanes
            peak(ks[ks % SEG == (28, 29, 0, 1)[t % 4]], t)
        elif pattern == "peaks-around-a-bin":  # peaks at c - 1 and c + 1: bin c takes the omega of c - 1 (:607-609)
            c = ks[(ks % SEG == (29, 0, 15, 1)[t % 4]) & (ks >= 2) & (ks <= F - 3)]
            peak(c - 1, t)
            peak(c + 1, t)
            m[0, c, t] = rs.uniform(0.0, 0.5, len(c))
        elif pattern == "plateaus":            # mid == hi / mid == lo across a seam: no strict peak there
            k = ks[(ks % SEG == 29) & (ks <= F - 3)]
            v = rs.uniform(1.5, 2.5, len(k)).astype(np.float32)
            m[0, k, t] = v
            m[0, k + 1, t] = v
            if t % 2:
                m[0, k - 1, t] = v
    if pattern == "silent":                   # all-zero frames inside chunks and one whole silent chunk
        m[:, :, [3, 4, chunk_len + 1, T - 1]] = 0
        m[:, :, 2 * chunk_len:3 * chunk_len] = 0
    return m


@pytest.mark.parametrize("n_fft", [1024, 400])
@pytest.mark.parametrize("pattern", ["edge-peaks", "seam-peaks", "peaks-around-a-bin", "plateaus", "silent"])
def test_crafted_magnitudes(pattern, n_fft):
    hop, T = n_fft // 4, 200
    F = n_bins(n_fft, True)
    chunks, chunk_len = chunking(1, F, T)
    assert chunks == 6
    mag = _crafted(pattern, F, T, chunk_len, seed=n_fft)
    magt = torch.from_numpy(mag).cuda()
    _, ph, _ = check_against_oracle(fused(magt, hop), magt, hop, True, pattern)
    if pattern == "peaks-around-a-bin":
        # the planted bins c (k = 29 mod 30 at t = 0) advanced by the omega of their lower peak: check the oracle
        # does what the kernel was compared with
        c = np.arange(29, F - 2, SEG)
        lo, mid, hi = mag[0, c - 2, 0], mag[0, c - 1, 0], mag[0, c, 0]
        p = np.float32(0.5) * (lo - hi) / (lo - np.float32(2) * mid + hi)
        om = np.float32(2 * np.pi) * ((c - 1).astype(np.float32) + p) / np.float32(n_fft) * np.float32(hop)
        assert np.array_equal(ph[0, c, 0], om)
    if pattern == "silent":
        assert (ph[..., 2 * chunk_len:3 * chunk_len] == ph[..., 2 * chunk_len - 1:2 * chunk_len]).all()


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("n_fft", [1024, 400])
def test_frame_range_carry(n_fft, dtype):
    """specinv_phase_init_ex: phase_out is the reference's float64 running phase at the last frame (bit for bit from
    float32 magnitudes: float64 sums of float32 omegas are exact), and frame ranges run with the two-pass scheme of
    griffin_lim_frame_sharded (advance of every range from zero, exclusive sum, run again with that start) put
    together the whole-signal output."""
    B, hop, T = 2, n_fft // 4, 700
    F = n_bins(n_fft, True)
    f32 = dtype == np.float32
    magt = rand_mag(B, F, T, torch.float32 if f32 else torch.float64, seed=n_fft)
    C, pout = fused_ex(magt, hop, True)
    mag, ph, ph64 = check_against_oracle(C, magt, hop, True, "whole signal")
    last = ph64[..., -1]
    got = pout.cpu().numpy()
    if f32:
        assert np.array_equal(got, last), int((got != last).sum())
    else:
        assert (np.abs(got - last) <= T * 2.0 ** -53 * np.abs(last)).all()
    assert np.array_equal(fused(magt, hop).cpu().numpy(), C.cpu().numpy())    # phase_init == phase_init_ex
    for edges in ((0, 640, 700), (0, 250, 290, 700)):
        ranges = list(zip(edges[:-1], edges[1:]))
        paths = [chunking(B, F, b - a)[0] > 1 for a, b in ranges]
        assert paths[1:] == ([False] if len(ranges) == 2 else [False, True])   # a short single pass / a split range
        advs = [fused_ex(magt[..., a:b].contiguous(), hop, True)[1] for a, b in ranges]
        start = torch.zeros_like(advs[0])
        parts, outs = [], []
        for (a, b), adv in zip(ranges, advs):
            Cr, pr = fused_ex(magt[..., a:b].contiguous(), hop, True, start if a else None)
            parts.append(Cr)
            outs.append(pr)
            start = start + adv
        Cs = torch.cat(parts, 2)
        if f32:
            assert torch.equal(Cs, C), edges
            assert torch.equal(outs[-1], pout) and torch.equal(start, pout)
        else:
            check(Cs, mag, ph, ph64, f"ranges {edges}")


# ---------------------------------------------------------------------------------------------------------------
def test_public_phase_init_on_a_host_tensor():
    import spectrogram_inversion_b200 as S
    hop, T = 100, 2003
    mag = np.random.RandomState(3).rand(201, T).astype(np.float32)
    out = S.phase_init(torch.from_numpy(mag), hop_length=hop)
    assert out.device.type == "cpu" and out.dtype == torch.complex64 and out.shape == mag.shape
    assert chunking(1, 201, T)[0] > 1
    ph, ph64 = O.phase_init_phase(mag, hop_length=hop)
    check(out.numpy()[None], mag[None], ph, ph64, "S.phase_init")


@pytest.mark.parametrize("n_fft", [1024, 400])
def test_differentiable_phase_init_matches_reference_phase(n_fft):
    """autograd.phase_init_diff (the path taken when spec.requires_grad) on a CUDA float32 magnitude: against the
    reference's phase, and against the fused kernel."""
    from spectrogram_inversion_b200.autograd import phase_init_diff
    hop, T = n_fft // 4, 2000
    magt = rand_mag(1, n_bins(n_fft, True), T, torch.float32, seed=n_fft + 1)
    spec = magt.clone().requires_grad_(True)
    with torch.enable_grad():
        C = phase_init_diff(spec, n_fft, hop)
    assert C.requires_grad and C.dtype == torch.complex64
    mag, _, _ = check_against_oracle(C, magt, hop, True, "phase_init_diff")
    diff = (C.detach() - fused(magt, hop)).abs().cpu().numpy()
    assert (diff <= 8e-7 * mag).all(), float((diff / np.maximum(mag, 1e-30)).max())
    C.real.sum().backward()
    assert spec.grad is not None and torch.isfinite(spec.grad).all()
