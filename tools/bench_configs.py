"""Device-resident timing of all five BASELINE.json configs (kernel iteration time, not the headline bench).

    python tools/bench_configs.py [cfg1 cfg2 cfg3 cfg4 cfg5] [--scale 1.0]
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spectrogram_inversion_b200 as S  # noqa: E402
from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, StftPlan  # noqa: E402
from spectrogram_inversion_b200.stft_args import StftArgs  # noqa: E402

CFG = {
    "cfg1": dict(algo="gl", B=1, N=661500, sr=22050, n_fft=2048, hop=512, iters=100, alpha=0.3),
    "cfg2": dict(algo="gl", B=512, N=240000, sr=24000, n_fft=1024, hop=256, iters=64, alpha=0.99),
    "cfg3": dict(algo="rtisi", B=256, N=240000, sr=24000, n_fft=1024, hop=256, iters=25, alpha=0.99, la=3),
    "cfg3s": dict(algo="rtisi", B=256, N=160000, sr=16000, n_fft=512, hop=128, iters=25, alpha=0.99, la=3),
    "cfg3l": dict(algo="rtisi", B=128, N=441000, sr=44100, n_fft=2048, hop=512, iters=25, alpha=0.99, la=3),
    "cfg4": dict(algo="admm", B=128, N=882000, sr=44100, n_fft=2048, hop=512, iters=100, rho=0.1),
    "cfg2p": dict(algo="gl", B=512, N=240000, sr=24000, n_fft=1024, hop=256, iters=64, alpha=0.0),      # plain GL
    "cfg5p": dict(algo="gl", B=1, N=172800000, sr=48000, n_fft=4096, hop=1024, iters=10, alpha=0.0),
    "cfg5": dict(algo="gl", B=1, N=172800000, sr=48000, n_fft=4096, hop=1024, iters=10, alpha=0.99),
}
names = [a for a in sys.argv[1:] if a in CFG] or list(CFG)
dev = torch.device("cuda")
PEAK = 6545.3
for name in names:
    c = CFG[name]
    n_fft, hop, B = c["n_fft"], c["hop"], c["B"]
    T = 1 + c["N"] // hop
    args = StftArgs(n_fft, hop, n_fft, torch.hann_window(n_fft, device=dev), True, "reflect", False, True)
    plan = StftPlan(args, T, B, torch.float32, dev)
    torch.manual_seed(0)
    x = torch.randn(B, plan.length, device=dev)
    Sx = plan.stft(x)
    mag = plan.spec_abs(Sx)
    del x
    F = n_fft // 2 + 1
    audio = B * c["N"] / c["sr"]
    if c["algo"] == "rtisi":
        magt = plan.unpack(Sx).abs()
        del Sx
        for _ in range(2):
            torch.cuda.synchronize(); t = time.perf_counter()
            y = S.RTISI_LA(magt, look_ahead=c["la"], max_iter=c["iters"], alpha=c["alpha"], verbose=0,
                           window=args.window, hop_length=hop)
            torch.cuda.synchronize(); dt = time.perf_counter() - t
        print(f"{name}: RTISI_LA B={B} T={T} {n_fft}/{hop} LA={c['la']} max_iter={c['iters']}: {dt*1e3:.1f} ms total, "
              f"{audio * c['iters'] / dt:.0f} audio-s*it/s, {dt / ((T + c['la']) * c['iters']) * 1e6:.2f} us / inner iteration")
        continue
    ph = torch.exp(2j * torch.pi * torch.rand(Sx.main.shape, device=dev))
    Sx.main.copy_(mag.main * ph)
    del ph
    solver = GriffinLimSolver(plan, Sx, mag, c["alpha"]) if c["algo"] == "gl" else ADMMSolver(plan, Sx, mag, c["rho"])
    for _ in range(3):
        solver.step()
    n = min(c["iters"], 20)
    solver.run_many(n, 0, 1, evaluate=False)      # what training_loop does between evaluations
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    solver.run_many(n, 0, 1, evaluate=False)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    per_bin = (20 if c["alpha"] > 0 else 4) if c["algo"] == "gl" else 36
    gb = (per_bin * B * F * T + 8 * B * plan.length) / 1e9
    print(f"{name}: {c['algo']} B={B} T={T} {n_fft}/{hop}: {ms:.4f} ms/iter, {gb / ms * 1e3:.0f} GB/s algorithmic "
          f"({gb / ms * 1e3 / PEAK * 100:.1f} % of {PEAK:.0f}), {audio / ms * 1e3:.0f} audio-s*it/s")
    del solver, Sx, mag, plan
    torch.cuda.empty_cache()
