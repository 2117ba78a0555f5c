"""torchaudio's InverseMelScale and its InverseMelScale -> GriffinLim chain against
spectrogram_inversion_b200.torchaudio_compat on the same seeded input.

    python tools/bench_torchaudio_mel.py [--reps 5] [--warmup 2] [--out result.json]

Shape: torchaudio's Tacotron2 Griffin-Lim vocoder (n_stft 513, n_mels 80, 22.05 kHz, f_max 8 kHz, slaney scale and
norm; GriffinLim n_fft 1024 / hop 256, power 1, n_iter 32) on B = 64 ten-second clips (T = 862 frames).  The mel is
torchaudio's MelSpectrogram (power 1) of seeded noise plus tones.

Reported: ms per InverseMelScale call (module forward, CUDA input) and per chain call for both implementations
(median of --reps calls timed with CUDA events after --warmup calls); if torchaudio's CUDA lstsq rejects the system or
fails, that is printed and torchaudio's InverseMelScale runs on the host (input copied there and back inside the
timed call).  The kernel alone (specinv_mel_inverse, P precomputed) is timed over 50 back-to-back launches, and its
achieved FLOP/s and bytes/s are derived from shape-based counts: 2 * covered_rows * n_mels * B * T FLOP, and
B * T * (n_mels + n_stft) * 4 bytes (mel read once, output written once; P is 160 KB).  Both bounds are given against
the measured FFMA peak (73.7 TFLOP/s, DESIGN.md) and 7.7 TB/s.  The final spectral convergence of both chains is
against the linear magnitude of the same signal.  The card's name and power limit are read in the same run."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from spectrogram_inversion_b200 import _ops  # noqa: E402
from spectrogram_inversion_b200 import torchaudio_compat as TC  # noqa: E402
import torchaudio_gl_ref as R  # noqa: E402

SR, N_FFT, HOP, N_MELS, B, SECONDS, N_ITER = 22050, 1024, 256, 80, 64, 10, 32
MEL = dict(n_stft=N_FFT // 2 + 1, n_mels=N_MELS, sample_rate=SR, f_min=0.0, f_max=8000.0, mel_scale="slaney",
           norm="slaney")
GL = dict(n_fft=N_FFT, power=1, hop_length=HOP, win_length=N_FFT, n_iter=N_ITER)
FFMA_PEAK, HBM_BW = 73.7e12, 7.7e12


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:
        return f"{torch.cuda.get_device_name(0)} (power limit not read: {ex})"


def make_signal(seed=0):
    """B clips of SECONDS s: low-passed noise plus three tones with random phases."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = torch.arange(SR * SECONDS, device="cuda") / SR
    x = torch.randn(B, n.numel(), device="cuda", generator=g) * 0.05
    x = torch.nn.functional.avg_pool1d(x[:, None], 5, 1, 2)[:, 0]
    for f in (220.0, 440.0, 1250.0):
        x = x + 0.3 * torch.sin(2 * math.pi * f * n + 2 * math.pi * torch.rand(B, 1, device="cuda", generator=g))
    return x


def time_calls(fn, reps, warmup, inner=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b) / inner)
    return statistics.median(ms), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import torchaudio.transforms as TAT

    x = make_signal()
    mel = TAT.MelSpectrogram(SR, n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS, f_max=8000.0, mel_scale="slaney",
                             norm="slaney", power=1).cuda()(x).contiguous()
    w = torch.hann_window(N_FFT, device="cuda")
    mag = R.stft(x, w, N_FFT, HOP, N_FFT).abs()
    T = mel.shape[-1]
    result = {"card": card(), "torch": torch.__version__, "B": B, "T": T, "n_stft": MEL["n_stft"], "n_mels": N_MELS}

    ours_inv = TC.InverseMelScale(**MEL).cuda()
    ta_inv = TAT.InverseMelScale(**MEL).cuda()
    try:
        ta_inv(mel[:2])
        torch.cuda.synchronize()
        ta_device = "cuda"
        ta_fn = ta_inv
    except Exception as ex:
        print(f"torchaudio InverseMelScale on CUDA failed ({type(ex).__name__}: {ex}); timing it on the host",
              flush=True)
        ta_device = "cpu"
        ta_inv = ta_inv.cpu()
        ta_fn = lambda m: ta_inv(m.cpu()).to("cuda")
    result["torchaudio_inverse_mel_device"] = ta_device

    # InverseMelScale alone
    inv = {}
    for impl, fn in (("specinv_b200", ours_inv), ("torchaudio", ta_fn)):
        med, all_ms = time_calls(lambda: fn(mel), a.reps, a.warmup)
        inv[impl] = {"ms_per_call": round(med, 4), "calls_ms": [round(v, 4) for v in all_ms]}
    inv["speedup"] = round(inv["torchaudio"]["ms_per_call"] / inv["specinv_b200"]["ms_per_call"], 1)
    spec_o, spec_r = ours_inv(mel), ta_fn(mel)
    inv["max_abs_diff_over_peak"] = float((spec_o - spec_r).abs().max() / spec_r.abs().max())
    result["inverse_mel"] = inv
    print(json.dumps({"inverse_mel": inv}), flush=True)

    # the kernel alone, from shape-derived counts
    P, f_lo, f_hi = ours_inv.operator()
    out = torch.empty_like(spec_o)
    med, _ = time_calls(lambda: _ops.mel_inverse_direct(P, mel, out, f_lo, f_hi), a.reps, a.warmup, inner=50)
    flop = 2.0 * (f_hi - f_lo) * N_MELS * B * T
    nbytes = 4.0 * B * T * (N_MELS + MEL["n_stft"])
    t = med * 1e-3
    kern = {"us": round(med * 1e3, 2), "covered_rows": f_hi - f_lo, "gflop": round(flop / 1e9, 3),
            "mbytes": round(nbytes / 1e6, 1), "tflops": round(flop / t / 1e12, 2), "tbytes_s": round(nbytes / t / 1e12, 3),
            "ffma_bound_us": round(flop / FFMA_PEAK * 1e6, 1), "hbm_bound_us": round(nbytes / HBM_BW * 1e6, 1)}
    kern["larger_bound"] = "ffma" if kern["ffma_bound_us"] >= kern["hbm_bound_us"] else "hbm"
    kern["share_of_larger_bound"] = round(max(kern["ffma_bound_us"], kern["hbm_bound_us"]) / kern["us"], 3)
    result["kernel"] = kern
    print(json.dumps({"kernel": kern}), flush=True)

    # the chain: InverseMelScale -> GriffinLim(n_iter=32)
    chains = {"specinv_b200": (ours_inv, TC.GriffinLim(**GL).cuda()),
              "torchaudio": (ta_fn, TAT.GriffinLim(**GL).cuda())}
    chain = {}
    for impl, (im, gl) in chains.items():
        fn = lambda: gl(im(mel))
        med, all_ms = time_calls(fn, a.reps, a.warmup)
        torch.manual_seed(1234)
        y = fn()
        sc = R.spectral_convergence(y, mag, w, N_FFT, HOP, N_FFT)
        chain[impl] = {"ms_per_call": round(med, 3), "calls_ms": [round(v, 3) for v in all_ms], "final_sc": sc}
        del y
    chain["speedup"] = round(chain["torchaudio"]["ms_per_call"] / chain["specinv_b200"]["ms_per_call"], 2)
    chain["inverse_mel_share_specinv"] = round(inv["specinv_b200"]["ms_per_call"] / chain["specinv_b200"]["ms_per_call"],
                                               4)
    result["chain"] = chain
    print(json.dumps({"chain": chain}), flush=True)
    print(json.dumps(result))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
