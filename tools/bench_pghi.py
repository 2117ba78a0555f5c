"""Time `pghi` on a B200 and produce the start-quality table from the GPU path.

    python tools/bench_pghi.py [--out results/bench_pghi.json]

* `pghi` call time at the cfg2 shape (B = 512 ten-second clips at 22.05 kHz, 1024/256, float32) and on one one-hour
  signal at 4096/1024, with CUDA events after warm-up; beside it one fused fast Griffin-Lim iteration at the cfg2 shape.
  The cfg2 magnitude (905 MB) is larger than the 126 MB L2, so every call reads it from HBM.
* The quality table: spectral convergence of the start (STFT of its ISTFT against the magnitude) and after 16 and 64
  fast Griffin-Lim iterations (alpha 0.99), from zero phase, `phase_init` and `pghi`, on a 3 s vibrato harmonic tone
  with an amplitude envelope and noise at 22.05 kHz, 1024/256, Hann window.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spectrogram_inversion_b200 import griffin_lim, pghi, phase_init  # noqa: E402
from spectrogram_inversion_b200.engine import GriffinLimSolver, StftPlan  # noqa: E402
from spectrogram_inversion_b200.stft_args import args_helper  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name(0)


def harmonic(B, n, sr, seed=0, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    t = torch.arange(n, device=device, dtype=torch.float64) / sr
    f0 = 100 + 100 * torch.rand(B, 1, generator=g, device=device, dtype=torch.float64)
    f = f0 * (1 + 0.3 * torch.sin(2 * math.pi * 0.7 * t))
    ph = 2 * math.pi * torch.cumsum(f, -1) / sr
    x = sum((0.6 / k) * torch.sin(k * ph) for k in range(1, 30)) * (0.5 + 0.5 * torch.sin(2 * math.pi * 2 * t) ** 2)
    return x + 0.003 * torch.randn(x.shape, generator=g, device=device, dtype=torch.float64)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"card": card()}
    sr, M, a = 22050, 1024, 256
    w = torch.hann_window(M, device="cuda")

    x = harmonic(512, 10 * sr, sr).float()
    mag = torch.stft(x, M, a, window=w, return_complex=True).abs()
    del x
    res["cfg2_shape"] = list(mag.shape)
    res["pghi_cfg2_ms"] = timed(lambda: pghi(mag, hop_length=a), 10)
    plan = StftPlan(args_helper(mag, window=w, hop_length=a), mag.shape[2], mag.shape[0], torch.float32, mag.device)
    C0 = pghi(mag, hop_length=a)
    solver = GriffinLimSolver(plan, plan.pack(C0), plan.pack(mag), 0.99)
    res["gl_iteration_cfg2_ms"] = timed(lambda: solver.step(), 20)
    del plan, solver, C0, mag
    torch.cuda.empty_cache()

    x = harmonic(1, 3600 * sr, sr)[0].float()
    mag = torch.stft(x, 4096, 1024, window=torch.hann_window(4096, device="cuda"), return_complex=True).abs()
    del x
    res["hour_shape"] = list(mag.shape)
    res["pghi_one_hour_ms"] = timed(lambda: pghi(mag, hop_length=1024), 3)
    del mag
    torch.cuda.empty_cache()

    x = harmonic(1, 3 * sr, sr, seed=1)[0]
    wd = torch.hann_window(M, device="cuda", dtype=torch.float64)
    mag = torch.stft(x, M, a, window=wd, return_complex=True).abs()

    def sc(C):
        y = torch.istft(C, M, a, window=wd)
        Y = torch.stft(y, M, a, window=wd, return_complex=True).abs()
        return float(20 * torch.log10(torch.linalg.norm(Y - mag) / torch.linalg.norm(mag)))

    def sc_x(y):
        Y = torch.stft(y, M, a, window=wd, return_complex=True).abs()
        return float(20 * torch.log10(torch.linalg.norm(Y - mag) / torch.linalg.norm(mag)))

    table = {}
    for name, C in (("zero phase", mag.to(torch.complex128)), ("phase_init", phase_init(mag, window=wd, hop_length=a)),
                    ("pghi", pghi(mag, hop_length=a))):
        row = {"start": sc(C)}
        for k in (16, 64):
            row[f"gl{k}"] = sc_x(griffin_lim(C, max_iter=k, tol=0, alpha=0.99, verbose=False, window=wd, hop_length=a))
        table[name] = row
    res["quality_db"] = table
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
