"""Whole calls of torchaudio's CUDA griffinlim against spectrogram_inversion_b200.torchaudio_compat.griffinlim on the
same seeded inputs.

    python tools/bench_torchaudio_gl.py [--reps 5] [--warmup 2] [--out result.json]

Shapes:
  fast     B = 64 ten-second clips at 22.05 kHz, n_fft 1024 / hop 256 (T = 862 frames), n_iter 32, momentum 0.99:
           the specialised fused kernel;
  generic  torchaudio's defaults: n_fft 400 / hop 200 at 16 kHz, B = 64 ten-second clips (T = 801), n_iter 32,
           momentum 0.99: the generic (mixed-radix) fused kernel.
Per shape and implementation: ms per call (median of --reps calls timed with CUDA events after --warmup calls of the
same shape), ms per iteration (the call over n_iter), and the final spectral convergence
|| |STFT(y)| - mag ||_F / || mag ||_F of the output of a call with the same seed.  The card's name and power limit are
read in the same run (nvidia-smi query only).  The input spectrogram (~0.9 GB at the fast shape) is larger than the
L2 cache."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from spectrogram_inversion_b200 import torchaudio_compat as TC  # noqa: E402
import torchaudio_gl_ref as R  # noqa: E402

SHAPES = {
    "fast": dict(sr=22050, n_fft=1024, hop=256, B=64, seconds=10, n_iter=32, momentum=0.99),
    "generic": dict(sr=16000, n_fft=400, hop=200, B=64, seconds=10, n_iter=32, momentum=0.99),
}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:
        return f"{torch.cuda.get_device_name(0)} (power limit not read: {ex})"


def make_spec(c, seed=0):
    """Power spectrogram (power 2) of low-passed noise, B clips of `seconds` s."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = c["sr"] * c["seconds"]
    x = torch.randn(c["B"], n, device="cuda", generator=g)
    x = torch.nn.functional.avg_pool1d(x[:, None], 5, 1, 2)[:, 0]
    w = torch.hann_window(c["n_fft"], device="cuda")
    return R.stft(x, w, c["n_fft"], c["hop"], c["n_fft"]).abs().pow(2).contiguous(), w


def time_calls(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="fast,generic")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import torchaudio.functional as TAF
    impls = {"torchaudio": TAF.griffinlim, "specinv_b200": TC.griffinlim}
    result = {"card": card(), "torch": torch.__version__, "shapes": {}}
    for name in a.shapes.split(","):
        c = SHAPES[name]
        spec, w = make_spec(c)
        call = (spec, w, c["n_fft"], c["hop"], c["n_fft"], 2.0, c["n_iter"], c["momentum"], None, True)
        row = {"B": c["B"], "T": spec.shape[-1], "n_fft": c["n_fft"], "hop": c["hop"], "n_iter": c["n_iter"],
               "sr": c["sr"], "seconds": c["seconds"]}
        for impl, fn in impls.items():
            med, all_ms = time_calls(lambda: fn(*call), a.reps, a.warmup)
            torch.manual_seed(1234)
            y = fn(*call)
            sc = R.spectral_convergence(y, spec.sqrt(), w, c["n_fft"], c["hop"], c["n_fft"])
            row[impl] = {"ms_per_call": round(med, 3), "ms_per_iter": round(med / c["n_iter"], 4),
                         "calls_ms": [round(v, 3) for v in all_ms], "final_sc": sc}
            del y
        row["speedup"] = round(row["torchaudio"]["ms_per_call"] / row["specinv_b200"]["ms_per_call"], 2)
        result["shapes"][name] = row
        print(json.dumps({name: row}), flush=True)
        del spec
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
