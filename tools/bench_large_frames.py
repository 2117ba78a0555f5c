"""Time the streamed-frame generic kernel (csrc/specinv_generic_stream.cu) at the large-frame shapes, against
torchaudio.functional.griffinlim on CUDA.

    python tools/bench_large_frames.py [--iters 20] [--n-iter 32] [--shapes all|quick]

Per shape: one fused Griffin-Lim iteration (momentum 0.99, no metric) timed with CUDA events, median over --iters
launches after a warm-up, and its algorithmic bandwidth: the signal read and written once, and per bin the state
read and written and the magnitude read (5 reals).  The recompute ratio counts the halo frames the CTA ranges of
launch_stream process per owned frame.  Then whole calls of torchaudio_compat.griffinlim and torchaudio's griffinlim
(n_iter = --n-iter, the same seed).  Every signal is 48 kHz audio; the working sets are larger than the 126 MB L2."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SR = 48000
# (n_fft, hop, dtype, batch, seconds)
SHAPES = [(8192, 2048, torch.float64, 8, 30), (4096, 256, torch.float32, 16, 30),
          (16384, 4096, torch.float32, 16, 60), (32768, 8192, torch.float32, 16, 60)]


def card() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:  # pragma: no cover
        return f"{torch.cuda.get_device_name(0)} (power limit unknown: {ex})"


def recompute_ratio(T: int, B: int, K: int) -> float:
    """Halo frames per owned frame of launch_stream's ranges: max(ceil(T / floor(148 / B)), 4 K) owned frames."""
    want = max(1, 148 // B)
    rng = min(max(-(-T // want), 4 * max(K, 1)), T)
    halo = sum(min(K, t0) for t0 in range(0, T, rng))
    return halo / T


def cuda_ms(fn, iters: int):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in ev)
    return ts[len(ts) // 2]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--n-iter", type=int, default=32)
    ap.add_argument("--shapes", default="all", choices=["all", "quick"])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_large_frames needs a CUDA device")
    from spectrogram_inversion_b200 import torchaudio_compat as TC
    from spectrogram_inversion_b200.engine import GriffinLimSolver, StftPlan
    from spectrogram_inversion_b200.stft_args import StftArgs
    try:
        import torchaudio.functional as TAF
        ta = TAF.griffinlim
    except Exception as ex:
        ta = None
        print(f"torchaudio not importable ({ex}): its column is empty")
    print(f"card: {card()}")
    dev = torch.device("cuda")
    shapes = SHAPES if args.shapes == "all" else [(n, h, dt, 2, 5) for n, h, dt, _, _ in SHAPES]
    for n_fft, hop, dtype, B, secs in shapes:
        T = secs * SR // hop + 1
        K = (n_fft - 1) // hop
        g = torch.Generator(device=dev).manual_seed(0)
        F = n_fft // 2 + 1
        mag = torch.rand(B, F, T, dtype=dtype, device=dev, generator=g)
        C = mag * torch.exp(2j * torch.pi * torch.rand(B, F, T, dtype=dtype, device=dev, generator=g))
        w = torch.hann_window(n_fft, dtype=dtype, device=dev)
        sa = StftArgs(n_fft=n_fft, hop_length=hop, win_length=n_fft, window=w, center=True, pad_mode="reflect",
                      normalized=False, onesided=True)
        plan = StftPlan(sa, T, B, dtype, dev)
        solver = GriffinLimSolver(plan, plan.pack(C), plan.pack(mag), 0.99)
        for _ in range(3):
            solver.step()
        ms = cuda_ms(solver.step, args.iters)
        es = torch.finfo(dtype).bits // 8
        nbytes = 2 * B * plan.length * es + 5 * B * T * F * es
        del solver, plan, C
        spec = mag.pow(2)
        torch.cuda.synchronize()

        def ours():
            torch.manual_seed(1)
            TC.griffinlim(spec, w, n_fft, hop, n_fft, 2.0, args.n_iter, 0.99, None, True)

        def theirs():
            torch.manual_seed(1)
            ta(spec, w, n_fft, hop, n_fft, 2.0, args.n_iter, 0.99, None, True)

        ours()
        call = cuda_ms(ours, 3)
        ta_call = None
        if ta is not None:
            theirs()
            ta_call = cuda_ms(theirs, 3)
        name = "fp64" if dtype == torch.float64 else "fp32"
        print(f"{name} {n_fft}/{hop} B={B} x {secs} s (T={T}, K={K}): {ms:.3f} ms/iteration, "
              f"{nbytes / ms / 1e6:.0f} GB/s algorithmic ({nbytes / 1e6:.0f} MB), recompute "
              f"{recompute_ratio(T, B, K):.3f} halo frames per owned frame | griffinlim n_iter={args.n_iter}: "
              f"{call:.1f} ms" + (f" vs torchaudio {ta_call:.1f} ms ({ta_call / call:.1f}x)" if ta_call else ""),
              flush=True)
        del spec, mag
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
