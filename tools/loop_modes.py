"""Host / device time of engine.training_loop on a small problem (cfg1 shape): synchronising evaluations (history
given) or not.

    python tools/loop_modes.py
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spectrogram_inversion_b200.engine import GriffinLimSolver, StftPlan, training_loop  # noqa: E402
from spectrogram_inversion_b200.stft_args import StftArgs  # noqa: E402

dev = torch.device("cuda")
n_fft, hop, T = 2048, 512, 1292
args = StftArgs(n_fft, hop, n_fft, torch.hann_window(n_fft, device=dev), True, "reflect", False, True)
plan = StftPlan(args, T, 1, torch.float32, dev)
x = torch.randn(1, plan.length, device=dev)
S = plan.stft(x)
mag = plan.spec_abs(S)


def run(label, hist, reps=3):
    for r in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        solver = GriffinLimSolver(plan, S, mag, 0.3)
        t1 = time.perf_counter()
        training_loop(solver, 100, 0.0, False, 10, "sc", history=[] if hist else None)
        t2 = time.perf_counter()
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        training_loop(solver, 100, 0.0, False, 10, "sc", history=[] if hist else None)
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        print(f"{label:28s} rep {r}: solver init {1e3 * (t1 - t0):6.2f} ms, first loop host {1e3 * (t2 - t1):6.2f} ms "
              f"(+{1e3 * (t3 - t2):5.2f} ms to drain), second loop {1e3 * (t4 - t3):6.2f} ms")
        del solver


run("sync evals", True)
run("blind evals", False)
